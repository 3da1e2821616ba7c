#!/usr/bin/env python
"""Verify-then-release decrypt of ONE message sharded over N GPUs (PeerExchange.decrypt_verified, the two-pass
agcm_stream_decrypt_verified_peer) against the releasing decrypt of the same inputs (PeerExchange.crypt(1, ...), the
fused one-pass kernel), the two alternated in one run.

  python tools/bench_peer_verified.py --gpus N [--reps 10] [--warmup 3] [--out FILE]

Workload: the config 2 shape -- one 2^30 B message, AES-256, 16 B AAD, key / IV / AAD / payload from default_rng(1) --
cut into counter ranges by shard_plan, one rank per GPU (re-executed under torch.distributed.run as bench.py does).
Before anything is timed every rank checks its plaintext and ok flag from both forms against OpenSSL (`cryptography`),
and that a forged tag leaves ok = 0 and the output untouched on every rank.  Each repetition barriers the ranks, then
times one call of each form with CUDA events on the calling stream (both forms make the stream wait for the exchange, so
the time runs until ok is valid); the figure is the mean over repetitions, the maximum over ranks.  At N <= 2 the host
forms (pinned buffers, PeerExchange.crypt_host / decrypt_verified_host) are timed the same way with a host clock around
the synchronous call.  Prints the card's name, power limit and the SM clock sampled during the timed loop, then one JSON
line per form (rank 0)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

TOTAL = 1 << 30
SENT = 0x5A


def inputs():
    """config 2 constants (bench.stream_inputs) and the payload drawn after them"""
    rng = np.random.default_rng(1)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    iv = rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
    aad = rng.integers(0, 256, 16, dtype=np.uint8).tobytes()
    return key, iv, aad, rng.bytes(TOTAL)


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file (rank 0)")
    a = ap.parse_args()
    if a.reps < 10:
        ap.error("--reps must be at least 10")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus > 1 and world == 1:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29543", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    rank, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    import aesgcm_b200
    from aesgcm_b200.parallel import PeerExchange, shard_plan
    from bench import ClockSampler
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
            torch.cuda.synchronize()

    def allreduce(x, op):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return t.item()

    key, iv, aad, pt = inputs()
    from cryptography.hazmat.primitives.ciphers.aead import AESGCM
    sealed = memoryview(AESGCM(key).encrypt(iv, pt, aad))
    tag = bytes(sealed[-16:])
    bad_tag = bytes([tag[0] ^ 1]) + tag[1:]
    sh = shard_plan(TOTAL, world)[rank]
    lo, hi = sh.byte_offset, sh.byte_offset + sh.n_bytes

    eng = aesgcm_b200.GcmEngine(local_rank)
    eng.set_key(key)
    if world > 1:
        px = PeerExchange(eng)
    else:   # a world of one: the context's own exchange buffer, no process group
        px = PeerExchange.__new__(PeerExchange)
        px.buf = torch.zeros(4096, dtype=torch.uint8, device=dev)
        eng.peer_setup(0, 1, [px.buf.data_ptr()])
        px.engine, px.group, px.rank, px.world = eng, None, 0, 1

    U8 = lambda b: torch.from_numpy(np.frombuffer(b, np.uint8).copy()).to(dev)   # noqa: E731
    d_ct, d_want = U8(sealed[lo:hi]), U8(pt[lo:hi])
    d_pt = torch.empty_like(d_ct)
    d_aad, d_tag, d_bad = U8(aad), U8(tag), U8(bad_tag)
    d_ok = torch.zeros(1, dtype=torch.uint8, device=dev)
    release = lambda t: px.crypt(1, iv, d_aad, sh, d_ct, d_pt, TOTAL, t, d_ok)                 # noqa: E731
    verified = lambda t: px.decrypt_verified(iv, d_aad, sh, d_ct, d_pt, TOTAL, t, d_ok)        # noqa: E731

    # correctness first: both forms against OpenSSL's plaintext, and the forged tag refused everywhere
    good = True
    for fn, t, authentic in ((release, d_tag, True), (verified, d_tag, True), (verified, d_bad, False)):
        d_pt.fill_(SENT)
        d_ok.fill_(7)
        barrier()
        fn(t)
        torch.cuda.synchronize()
        good = good and int(d_ok.item()) == int(authentic)
        good = good and (torch.equal(d_pt, d_want) if authentic else bool((d_pt == SENT).all()))
    checked = allreduce(float(good), dist.ReduceOp.MIN if dist else None) == 1.0
    if not checked:
        sys.exit("rank %d: output differs from OpenSSL" % rank)

    cards = [card(local_rank)]
    if dist:
        cards = [None] * world
        dist.all_gather_object(cards, card(local_rank))
    lines = [{"cards": cards, "world": world}]

    def timed(form, rel, ver, host_clock):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        for _ in range(a.warmup):
            rel()
            ver()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.mark_start()
        t_rel = t_ver = 0.0
        for _ in range(a.reps):
            for f, (e0, e1), acc in ((rel, ev[:2], "rel"), (ver, ev[2:], "ver")):
                barrier()
                t0 = time.perf_counter()
                e0.record()
                f()
                e1.record()
                torch.cuda.synchronize()
                ms = (time.perf_counter() - t0) * 1e3 if host_clock else e0.elapsed_time(e1)
                if acc == "rel":
                    t_rel += ms
                else:
                    t_ver += ms
        sampler.mark_stop()
        clocks = sampler.finish()
        t_rel = allreduce(t_rel / a.reps, dist.ReduceOp.MAX if dist else None)
        t_ver = allreduce(t_ver / a.reps, dist.ReduceOp.MAX if dist else None)
        rec = {"world": world, "form": form, "message_bytes": TOTAL, "shard_bytes_max": shard_plan(TOTAL, world)[0].n_bytes,
               "reps": a.reps, "release_ms": round(t_rel, 4), "verified_ms": round(t_ver, 4),
               "release_GBps": round(TOTAL / t_rel / 1e6, 1), "verified_GBps": round(TOTAL / t_ver / 1e6, 1),
               "verified_over_release_time": round(t_ver / t_rel, 3), "checked_vs_openssl": checked,
               "sm_clock_rank0": clocks}
        lines.append(rec)

    timed("device (HBM-resident shard), CUDA events", lambda: release(d_tag), lambda: verified(d_tag), False)

    if world <= 2:
        h_ct = torch.empty(sh.n_bytes, dtype=torch.uint8, pin_memory=True).numpy()
        h_pt = torch.empty(sh.n_bytes, dtype=torch.uint8, pin_memory=True).numpy()
        h_ct[:] = np.frombuffer(sealed[lo:hi], np.uint8)
        want = np.frombuffer(pt, np.uint8, count=sh.n_bytes, offset=lo)
        ok_rel = px.crypt_host(1, iv, aad, sh, h_ct, h_pt, TOTAL, tag)
        good = ok_rel and np.array_equal(h_pt, want)
        h_pt[:] = SENT
        ok_ver = px.decrypt_verified_host(iv, aad, sh, h_ct, h_pt, TOTAL, tag)
        good = good and ok_ver and np.array_equal(h_pt, want)
        h_pt[:] = SENT
        good = good and not px.decrypt_verified_host(iv, aad, sh, h_ct, h_pt, TOTAL, bad_tag) and bool((h_pt == SENT).all())
        if allreduce(float(good), dist.ReduceOp.MIN if dist else None) != 1.0:
            sys.exit("rank %d: host-form output differs from OpenSSL" % rank)
        timed("host (pinned buffers, synchronous call), host clock",
              lambda: px.crypt_host(1, iv, aad, sh, h_ct, h_pt, TOTAL, tag),
              lambda: px.decrypt_verified_host(iv, aad, sh, h_ct, h_pt, TOTAL, tag), True)

    if rank == 0:
        for rec in lines:
            print(json.dumps(rec), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
            with open(a.out, "a") as f:
                for rec in lines:
                    f.write(json.dumps(rec) + "\n")
    barrier()   # no rank frees its context while a peer may still read its exchange buffer
    eng.close()
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
