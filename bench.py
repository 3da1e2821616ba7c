#!/usr/bin/env python
"""bench.py -- AES-GCM enc+tag throughput of the B200 engine (BASELINE.json metric).

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one fused GCTR+GHASH pass (encrypt + tag) over one synthetic stream resident in HBM.
N=1: BASELINE config 2, AES-256, one 2^30-byte stream, 16 B AAD.
N>1 (torchrun, one rank per GPU), three curves in one run:
  * headline `value` (weak scaling): one stream of N x 2^30 bytes split by counter range, 2^30 bytes
    per GPU; every step ends with the 16-byte-per-rank exchange over NVLink peer memory and the tag
    finish on every rank, all inside the timed region;
  * `strong_scaling`: config 2 exactly as SURVEY 8(d) writes it -- ONE 2^30-byte stream cut into
    2^30/N-byte counter ranges;
  * `batched_split`: configs 3 and 4 (2^20 messages) split over the ranks with
    parallel.batch_split, no collective on the data path.
Before anything is timed, every N runs the SAME step on a 64 MiB x N stream and compares the tag and
every ciphertext byte with OpenSSL (`cryptography`) on the host: `parity_checked`.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

METRIC = "aes_gcm_enc_tag_throughput"
UNIT = "GB/s"
SHARD_BYTES = 1 << 30
AAD_BYTES = 16
PARITY_BYTES_PER_RANK = 64 << 20
DUMP_WINDOW = 4096      # bytes per sampled ciphertext window (--dump-outputs)
DUMP_WINDOWS = 2048     # windows over all ranks: 8 MiB of ciphertext, 32 MiB as float32


def stream_inputs():
    """BASELINE config 2 constants: key / IV / AAD from default_rng(1)."""
    rng = np.random.default_rng(1)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    iv = rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
    aad = rng.integers(0, 256, AAD_BYTES, dtype=np.uint8).tobytes()
    return key, iv, aad


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.path = None
        exe = shutil.which("nvidia-smi")
        if not exe:
            return
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        self.f = open(self.path, "w")
        self.proc = subprocess.Popen([exe, "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                      "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        self.t0 = self.t1 = None

    def mark_start(self):
        self.t0 = time.time()

    def mark_stop(self):
        self.t1 = time.time()

    def finish(self):
        if not self.proc:
            return None
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        rows = []
        import datetime
        with open(self.path) as f:
            for line in f:
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(c[1]), float(c[2]), c[4], c[5], c[6], c[7], c[8]))
                except Exception:
                    continue
        os.unlink(self.path)
        if not rows:
            return None
        inside = [r for r in rows if self.t0 and self.t1 and self.t0 - 0.05 <= r[0] <= self.t1 + 0.05]
        scope = "timed region"
        if not inside:
            inside, scope = rows, "whole bench (timed region shorter than the sampling period)"
        sm = sorted(r[1] for r in inside)
        reasons = set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in inside:
            for nm, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": inside[0][2], "reasons": sorted(reasons), "samples": len(inside),
                "scope": scope}


# --------------------------------------------------------------------------- CPU baselines
def openssl_speed(cores, seconds=2):
    """`openssl speed -evp aes-256-gcm` on the host (AES-NI/VAES+PCLMUL), cache-resident 16 KiB
    buffers: an upper bound for the host, not a streaming figure.  GB/s or None."""
    exe = shutil.which("openssl")
    if not exe:
        return None
    try:
        out = subprocess.run([exe, "speed", "-evp", "aes-256-gcm", "-bytes", "16384", "-seconds", str(seconds), "-multi",
                              str(cores)], capture_output=True, text=True, timeout=60).stdout
        for line in out.splitlines():
            if line.lower().startswith("aes-256-gcm") or line.startswith("evp"):
                tok = line.split()[-1]
                if tok.endswith("k"):
                    return float(tok[:-1]) * 1000.0 / 1e9
    except Exception:
        return None
    return None


def _mp_aesgcm_worker(idx, n_bytes, reps, barrier, q):
    try:
        from cryptography.hazmat.primitives.ciphers.aead import AESGCM
        key, iv, aad = stream_inputs()
        pt = np.random.default_rng(100 + idx).integers(0, 256, n_bytes, dtype=np.uint8).tobytes()
        a = AESGCM(key)
        a.encrypt(iv, pt[: 1 << 20], aad)
        barrier.wait(timeout=120)
        t0 = time.perf_counter()
        for _ in range(reps):
            a.encrypt(iv, pt, aad)
        q.put((n_bytes * reps, t0, time.perf_counter()))
    except Exception as ex:  # pragma: no cover
        q.put(("error", str(ex), 0))


def openssl_multiprocess_stream(total_bytes, procs, reps=2):
    """The honest strong CPU baseline for config 2: `total_bytes` of AES-256-GCM encrypt+tag through
    OpenSSL (cryptography.AESGCM: VAES + VPCLMULQDQ) on ALL host cores, one process per core, each
    encrypting its own total/procs-byte slice as one message out of DRAM (the AEAD API cannot start
    a counter range, so the slices are independent messages: the same AES and GHASH work).
    -> dict or None."""
    try:
        import multiprocessing as mp
        from cryptography.hazmat.primitives.ciphers.aead import AESGCM  # noqa: F401
    except Exception:
        return None
    try:
        ctx = mp.get_context("fork")
        per = max(1 << 20, total_bytes // procs)
        barrier, q = ctx.Barrier(procs), ctx.Queue()
        ps = [ctx.Process(target=_mp_aesgcm_worker, args=(i, per, reps, barrier, q)) for i in range(procs)]
        for p in ps:
            p.start()
        res = [q.get(timeout=300) for _ in ps]
        for p in ps:
            p.join(timeout=60)
        if any(r[0] == "error" for r in res):
            return {"error": [r[1] for r in res if r[0] == "error"][0]}
        nbytes = sum(r[0] for r in res)
        dt = max(r[2] for r in res) - min(r[1] for r in res)
        return {"GBps": round(nbytes / dt / 1e9, 3), "processes": procs, "bytes_per_process": per, "passes": reps,
                "what": "cryptography.AESGCM(key).encrypt, one message per process, wall clock from the first start to the last end"}
    except Exception as ex:
        return {"error": "%s: %s" % (type(ex).__name__, ex)}


def python_model_rates():
    """The reference model's calling patterns (tb/gcm_model.py) on one host core with the AES-GCM
    library that IS installed (`cryptography`/OpenSSL): whole message, and the testbench's
    one-<=16-byte-block-per-call streaming.  GB/s each, or None."""
    try:
        from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
        from cryptography.hazmat.primitives.ciphers.aead import AESGCM
    except Exception:
        return None
    key, iv, aad = stream_inputs()
    res = {}
    pt = np.random.default_rng(1).integers(0, 256, 64 << 20, dtype=np.uint8).tobytes()
    t0 = time.perf_counter()
    AESGCM(key).encrypt(iv, pt, aad)
    res["whole_message_64MiB_1core_GBps"] = round(len(pt) / (time.perf_counter() - t0) / 1e9, 3)
    n = 1 << 20
    enc = Cipher(algorithms.AES(key), modes.GCM(iv)).encryptor()
    enc.authenticate_additional_data(aad)
    t0 = time.perf_counter()
    for i in range(0, n, 16):
        enc.update(pt[i:i + 16])
    enc.finalize()
    res["per_16B_call_streaming_1MiB_1core_GBps"] = round(n / (time.perf_counter() - t0) / 1e9, 5)
    return res


def pycryptodome_rates():
    """The reference's ACTUAL backend (tb/gcm_model.py:1,18), probed at run time: whole-message
    encrypt_and_digest and the testbench's per-16-byte pattern (tb/gcm_model.py:22,26,35)."""
    try:
        try:
            from Crypto.Cipher import AES
        except ImportError:
            from Cryptodome.Cipher import AES
    except Exception as ex:
        return {"available": False, "error": "%s: %s" % (type(ex).__name__, ex)}
    key, iv, aad = stream_inputs()
    pt = np.random.default_rng(1).integers(0, 256, 64 << 20, dtype=np.uint8).tobytes()
    res = {"available": True}
    c = AES.new(key, AES.MODE_GCM, nonce=iv)
    c.update(aad)
    t0 = time.perf_counter()
    c.encrypt_and_digest(pt)
    res["whole_message_64MiB_1core_GBps"] = round(len(pt) / (time.perf_counter() - t0) / 1e9, 3)
    n = 1 << 20
    c = AES.new(key, AES.MODE_GCM, nonce=iv)
    c.update(aad)
    t0 = time.perf_counter()
    for i in range(0, n, 16):
        c.encrypt(pt[i:i + 16])
    c.digest()
    res["per_16B_call_streaming_1MiB_1core_GBps"] = round(n / (time.perf_counter() - t0) / 1e9, 5)
    return res


def cpu_reference_rate(sample_bytes, threads, steps, warmup):
    """Times the CPU restatement of the reference datapath (oracle/gcm_oracle.c, all host
    threads) on the first `sample_bytes` of the config-2 stream.  -> (GB/s, seconds per step)."""
    from oracle import cpu_oracle as o
    key, iv, aad = stream_inputs()
    pt = np.random.default_rng(1).integers(0, 256, sample_bytes, dtype=np.uint8)
    for _ in range(warmup):
        o.gcm_crypt(key, iv, aad, pt[: max(1 << 16, sample_bytes // 16)], threads=threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.gcm_crypt(key, iv, aad, pt, threads=threads)
    dt = (time.perf_counter() - t0) / steps
    return sample_bytes / dt / 1e9, dt


def calibrate_sample(threads, target_s):
    from oracle import cpu_oracle as o
    key, iv, aad = stream_inputs()
    n = 1 << 20
    pt = np.random.default_rng(1).integers(0, 256, n, dtype=np.uint8)
    o.gcm_crypt(key, iv, aad, pt[:65536], threads=threads)
    t0 = time.perf_counter()
    o.gcm_crypt(key, iv, aad, pt, threads=threads)
    rate = n / (time.perf_counter() - t0)
    s = int(rate * target_s) >> 20 << 20
    return max(1 << 20, min(s, SHARD_BYTES))


def cpu_baseline_block(cores, sample, val, dt, passes, quick):
    """The `cpu_baseline` object shared by both arms.  `value` is the port of the reference
    datapath (the contract's kind "port"); the strong baselines ride beside it."""
    return {"value": round(val, 6), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "first %d MiB of the config-2 stream, %d pass(es), oracle/gcm_oracle.c with %d threads (%.1f s per pass)"
                      % (sample >> 20, passes, cores, dt),
            "openssl_allcores_full_stream": None if quick else openssl_multiprocess_stream(SHARD_BYTES, cores),
            "openssl_speed_evp_aes256gcm_allcores_GBps": None if quick else openssl_speed(cores),
            "python_cryptography_aesgcm": None if quick else python_model_rates(),
            "pycryptodome": pycryptodome_rates()}


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    budget = float(os.environ.get("AGCM_BENCH_REF_BUDGET_S", "150"))  # seconds for the whole arm
    per_step = max(0.2, min(5.0, budget / max(1, args.steps + 1)))
    sample = calibrate_sample(cores, per_step)
    val, dt = cpu_reference_rate(sample, cores, args.steps, min(args.warmup, 1))
    quick = budget < 30
    line = {
        "impl": "reference", "metric": METRIC, "value": round(val, 6), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": cpu_baseline_block(cores, sample, val, dt, args.steps, quick),
        "e2e": {"value": round(val, 6), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(n_gpus):
    return {"workload": "BASELINE config 2: AES-256-GCM encrypt+tag, one stream of %d x 2^30 B, %d B AAD, counter-range "
                        "split (2^30 B per GPU)" % (n_gpus, AAD_BYTES),
            "bytes_per_gpu": SHARD_BYTES, "aad_bytes": AAD_BYTES, "key_bits": 256,
            "parallelism": ("counter-range x%d + 16 B/rank exchange (%s)" % (n_gpus, os.environ.get("AGCM_BENCH_EXCHANGE", "peer-memory stores posted by the bulk kernel's tail, one-warp finish on a side stream"))) if n_gpus > 1 else "single GPU",
            "l2": "inputs (1 GiB read + 1 GiB written per step and GPU) exceed the 126 MB L2; no flush needed"}


# --------------------------------------------------------------------------- GPU arm
def expected_aesgcm(key, iv, aad, pt):
    """(ct, tag, checker name) from OpenSSL; the oracle port if `cryptography` is missing."""
    try:
        from cryptography.hazmat.primitives.ciphers.aead import AESGCM
        out = AESGCM(key).encrypt(iv, pt, aad if aad else None)
        return out[:-16], out[-16:], "cryptography AESGCM (OpenSSL)"
    except ImportError:
        from oracle import cpu_oracle as o
        ct, tag = o.gcm_crypt(key, iv, aad, np.frombuffer(pt, dtype=np.uint8), threads=os.cpu_count() or 1)
        return ct, tag, "oracle/gcm_oracle.c"


def batched_split(eng, torch, dist, dev, rank, world, iters=5, weak=False):
    """BASELINE configs 3 and 4 with the messages split over the ranks (parallel.batch_split):
    independent messages, NO collective on the data path.  Device-resident, CUDA events, max over
    ranks.  Three messages per rank are checked against OpenSSL before timing.
    weak=False: the 2^20 messages of the config over all ranks (strong scaling: 2^20 / N per GPU);
    weak=True: 2^20 messages PER GPU (the batch grows with the machine)."""
    from aesgcm_b200.parallel import batch_split

    def timeit(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        if dist:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def openssl_msg(key, iv, aad, pt):
        ct, tag, _ = expected_aesgcm(key, iv, aad, pt)
        return ct, tag

    res = []
    n_total, length, stride = (1 << 20) * (world if weak else 1), 1500, 1504
    lo, hi = batch_split(n_total, world, rank)
    n_msgs = hi - lo
    rng = np.random.default_rng(2)
    key3 = rng.integers(0, 256, 24, dtype=np.uint8).tobytes()
    ivs_all = rng.integers(0, 256, 12 * n_total, dtype=np.uint8)      # message i has the same IV at every N
    gen = torch.Generator(device=dev)
    gen.manual_seed(200 + rank)
    d_buf = torch.randint(0, 256, (n_msgs * stride,), dtype=torch.uint8, device=dev, generator=gen)
    d_out = torch.empty_like(d_buf)
    d_iv = torch.from_numpy(ivs_all[12 * lo:12 * hi].copy()).to(dev)
    d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device=dev)
    d_ok = torch.zeros(n_msgs, dtype=torch.uint8, device=dev)
    eng.set_key(key3)
    eng.set_key(eng.round_keys())  # shared PRE-EXPANDED key
    run3 = lambda: eng.batch_crypt_uniform_device(0, d_iv, None, 0, 0, d_buf, d_out, length, stride, d_tags, n_msgs=n_msgs)
    run3()
    torch.cuda.synchronize()
    checked = 0
    for m in sorted({0, n_msgs // 2, n_msgs - 1}):
        pt = d_buf[m * stride:m * stride + length].cpu().numpy().tobytes()
        ct, tag = openssl_msg(key3, ivs_all[12 * (lo + m):12 * (lo + m + 1)].tobytes(), b"", pt)
        assert d_out[m * stride:m * stride + length].cpu().numpy().tobytes() == ct, "config 3: ciphertext differs from OpenSSL"
        assert d_tags[16 * m:16 * m + 16].cpu().numpy().tobytes() == tag, "config 3: tag differs from OpenSSL"
        checked += 1
    ms = timeit(run3)
    shape = "%d x 2^20" % world if weak else "2^20"
    res.append({"workload": "config 3: AES-192 encrypt+tag, %s x 1500 B at a 1504 B stride, per-message IV, shared "
                            "pre-expanded key; messages split over %d rank(s), no collective" % (shape, world),
                "scaling": "weak" if weak else "strong",
                "ms": round(ms, 4), "payload_GBps": round(n_total * length / ms / 1e6, 1),
                "msgs_per_rank": n_msgs, "openssl_checked_msgs_per_rank": checked})
    del d_buf, d_out
    alen = 64
    d_keys = torch.randint(0, 256, (n_msgs * 32,), dtype=torch.uint8, device=dev, generator=gen)
    d_aad = torch.randint(0, 256, (n_msgs * alen,), dtype=torch.uint8, device=dev, generator=gen)
    d_pt = torch.randint(0, 256, (n_msgs * stride,), dtype=torch.uint8, device=dev, generator=gen)
    d_ct = torch.empty_like(d_pt)
    d_back = torch.empty_like(d_pt)
    eng.batch_crypt_perkey_uniform_device(256, 0, d_keys, d_iv, d_aad, alen, alen, d_pt, d_ct, length, stride, d_tags, n_msgs=n_msgs)
    torch.cuda.synchronize()
    for m in sorted({0, n_msgs // 2, n_msgs - 1}):
        k = d_keys[32 * m:32 * m + 32].cpu().numpy().tobytes()
        a = d_aad[alen * m:alen * (m + 1)].cpu().numpy().tobytes()
        pt = d_pt[m * stride:m * stride + length].cpu().numpy().tobytes()
        ct, tag = openssl_msg(k, ivs_all[12 * (lo + m):12 * (lo + m + 1)].tobytes(), a, pt)
        assert d_ct[m * stride:m * stride + length].cpu().numpy().tobytes() == ct, "config 4: ciphertext differs from OpenSSL"
        assert d_tags[16 * m:16 * m + 16].cpu().numpy().tobytes() == tag, "config 4: tag differs from OpenSSL"
    # 0.1 % of the tags corrupted (BASELINE.md 5 row 4): the ok flags must say exactly which
    tags_in = d_tags.clone()
    bad = torch.arange(7, n_msgs, 1000, device=dev)
    tags_in[16 * bad + 5] = tags_in[16 * bad + 5] ^ 0x10
    ms = timeit(lambda: eng.batch_crypt_perkey_uniform_device(256, 1, d_keys, d_iv, d_aad, alen, alen, d_ct, d_back, length,
                                                              stride, tags_in, d_ok, n_msgs=n_msgs))
    torch.cuda.synchronize()
    want_ok = torch.ones(n_msgs, dtype=torch.uint8, device=dev)
    want_ok[bad] = 0
    assert torch.equal(d_ok, want_ok), "config 4: ok flags do not match the corrupted tags"
    assert torch.equal(d_back.view(n_msgs, stride)[:, :length], d_pt.view(n_msgs, stride)[:, :length]), "config 4 round trip failed"
    res.append({"workload": "config 4: AES-256 decrypt+verify, %s x 1500 B at a 1504 B pitch, distinct key per message (schedule "
                            "on device), 64 B AAD, 0.1 %% of the tags corrupted; messages split over %d rank(s), no collective"
                            % (shape, world),
                "scaling": "weak" if weak else "strong",
                "ms": round(ms, 4), "payload_GBps": round(n_total * length / ms / 1e6, 1),
                "Mmsg_per_s": round(n_total / ms / 1e3, 1), "msgs_per_rank": n_msgs, "openssl_checked_msgs_per_rank": 3,
                "bad_tags_per_rank": int(bad.numel())})
    return res


def dump_outputs(out_dir, rank, world, d_ct, d_tag):
    """Writes what the last timed step handed its caller, so that two builds can be compared output
    for output: the 16-byte tag (tag.npy) and a fixed sample of this rank's ciphertext, DUMP_WINDOWS /
    world windows of DUMP_WINDOW bytes at window indices drawn by default_rng(3), one row per window
    in stream order (ciphertext_sample.npy, or ciphertext_sample_rank<r>.npy when N > 1).  Bytes are
    stored as float32."""
    import torch
    n_win = d_ct.numel() // DUMP_WINDOW
    pick = np.sort(np.random.default_rng(3).choice(n_win, min(n_win, DUMP_WINDOWS // world), replace=False))
    windows = d_ct[:n_win * DUMP_WINDOW].view(n_win, DUMP_WINDOW).index_select(0, torch.from_numpy(pick).to(d_ct.device))
    os.makedirs(out_dir, exist_ok=True)
    name = "ciphertext_sample.npy" if world == 1 else "ciphertext_sample_rank%d.npy" % rank
    np.save(os.path.join(out_dir, name), windows.cpu().numpy().astype(np.float32))
    if rank == 0:
        np.save(os.path.join(out_dir, "tag.npy"), d_tag.cpu().numpy().astype(np.float32))


def run_ours(args, rank, world, local_rank):
    import torch
    import aesgcm_b200
    from aesgcm_b200.parallel import shard_plan

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    key, iv, aad = stream_inputs()
    eng = aesgcm_b200.GcmEngine(local_rank)
    eng.set_key(key)
    d_aad = torch.from_numpy(np.frombuffer(aad, dtype=np.uint8).copy()).to(dev)
    d_tag = torch.zeros(16, dtype=torch.uint8, device=dev)
    d_part = torch.zeros(16, dtype=torch.uint8, device=dev)
    d_parts = torch.zeros((world, 16), dtype=torch.uint8, device=dev)

    # N > 1: the 16-byte partials cross NVLink as peer-memory stores from the bulk kernel's own tail;
    # AGCM_BENCH_EXCHANGE=nccl selects part + all_gather + finish
    exchange = os.environ.get("AGCM_BENCH_EXCHANGE", "peer") if world > 1 else "none"
    px = None
    if exchange == "peer":
        try:
            from aesgcm_b200.parallel import PeerExchange
            px = PeerExchange(eng)
        except Exception as ex:  # symmetric memory not available on this node: use the library exchange
            px = None
            exchange = "nccl (peer-memory rendezvous failed: %s)" % type(ex).__name__
            os.environ["AGCM_BENCH_EXCHANGE"] = exchange

    def make_step(total, shard, d_in, d_out):
        def step():
            if world == 1:
                eng.stream_crypt_device(0, iv, d_aad, d_in, d_out, d_tag)
            elif px is not None:
                # deferred: the one-warp finish of this message waits for the world's flags on the
                # engine's side stream while the next message's bulk kernel already runs
                px.crypt(0, iv, d_aad, shard, d_in, d_out, total, d_tag, defer=True)
            else:
                eng.stream_part_device(0, iv, shard.first_block, d_in, d_out, shard.blocks_after, d_part)
                dist.all_gather_into_tensor(d_parts.view(-1), d_part)
                eng.stream_finish_device(0, iv, d_parts, world, d_aad, total, d_tag)
        return step

    def join():
        if px is not None:
            px.join()

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
            torch.cuda.synchronize()

    def allmax(x):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- parity, before anything is timed: the SAME step on a 64 MiB x N stream against OpenSSL
    p_total = PARITY_BYTES_PER_RANK * world
    p_shard = shard_plan(p_total, world)[rank]
    p_pt = np.random.default_rng(7).integers(0, 256, p_total, dtype=np.uint8)   # identical on every rank
    want_ct, want_tag, checker = expected_aesgcm(key, iv, aad, p_pt.tobytes())
    dp_in = torch.from_numpy(p_pt[p_shard.byte_offset:p_shard.byte_offset + p_shard.n_bytes].copy()).to(dev)
    dp_out = torch.zeros_like(dp_in)
    barrier()   # the ranks made their inputs at different speeds: line up before the first exchange (its wait is bounded)
    make_step(p_total, p_shard, dp_in, dp_out)()
    join()
    torch.cuda.synchronize()
    got_ct = dp_out.cpu().numpy().tobytes()
    ok_ct = got_ct == want_ct[p_shard.byte_offset:p_shard.byte_offset + p_shard.n_bytes]
    ok_tag = d_tag.cpu().numpy().tobytes() == want_tag
    bad = allmax(0.0 if (ok_ct and ok_tag) else 1.0)
    assert bad == 0.0, "parity check against %s failed (rank %d: ct %s, tag %s)" % (checker, rank, ok_ct, ok_tag)
    parity = {"checked": True, "against": checker, "stream_bytes": p_total, "ct_bytes_compared_per_rank": p_shard.n_bytes,
              "tag_compared_on_every_rank": True, "path": "the timed step's own call (%s)" % (
                  "agcm_stream_crypt" if world == 1 else "agcm_stream_crypt_peer_async + agcm_peer_join" if px is not None
                  else "agcm_stream_part + all_gather + agcm_stream_finish")}
    del dp_in, dp_out, p_pt, want_ct, got_ct

    # ---- headline: weak scaling, 2^30 B per GPU
    total = SHARD_BYTES * world
    shard = shard_plan(total, world)[rank]
    gen = torch.Generator(device=dev)
    gen.manual_seed(1 + rank)
    d_in = torch.randint(0, 256, (shard.n_bytes,), dtype=torch.uint8, device=dev, generator=gen)
    d_out = torch.empty_like(d_in)
    step = make_step(total, shard, d_in, d_out)

    def timed(step_fn, steps, warmup, sampler=None, timing=False):
        for _ in range(warmup):
            step_fn()
        join()
        barrier()
        if timing:
            eng.timing_enable(True)
        l0 = eng.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler:
            sampler.mark_start()
        ev0.record()
        for _ in range(steps):
            step_fn()
        join()            # every step's tag is finished inside the timed region
        ev1.record()
        barrier()
        if sampler:
            sampler.mark_stop()
        return allmax(ev0.elapsed_time(ev1)), eng.launch_count - l0

    sampler = ClockSampler(local_rank) if rank == 0 else None
    warm = max(args.warmup, 3)
    ms, launches = timed(step, args.steps, warm, sampler, timing=True)
    k_ms, k_n = eng.timing_read()
    eng.timing_enable(False)
    value = total * args.steps / (ms * 1e-3) / 1e9
    if px is not None:
        px.check()   # raises if any exchange failed closed
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, d_out, d_tag)   # before the strong-scaling steps reuse both

    # the work was real: the plaintext round-trips on this rank's shard (the tag was checked above)
    d_chk = torch.empty_like(d_in)
    eng.gctr_device(iv, shard.first_block, d_out, d_chk)
    torch.cuda.synchronize()
    assert torch.equal(d_chk, d_in), "round trip failed"
    del d_chk
    weak_tag = d_tag.cpu().numpy().tobytes()

    # ---- strong scaling: config 2 as SURVEY 8(d) writes it, ONE 2^30 B stream in 2^30/N B ranges
    strong = None
    if world > 1 and not args.no_extras:
        s_total = SHARD_BYTES
        s_shard = shard_plan(s_total, world)[rank]
        s_step = make_step(s_total, s_shard, d_in[:s_shard.n_bytes], d_out[:s_shard.n_bytes])
        s_steps = max(args.steps, 20)
        s_ms, _ = timed(s_step, s_steps, warm)
        strong = {"value": round(s_total * s_steps / (s_ms * 1e-3) / 1e9, 3), "unit": UNIT, "scaling": "strong",
                  "stream_bytes": s_total, "bytes_per_gpu": s_shard.n_bytes, "steps": s_steps,
                  "ms_per_step": round(s_ms / s_steps, 4),
                  "note": "BASELINE config 2 as specified: one 2^30 B stream, 2^30/N B per rank; same step, same exchange"}
        if px is not None:
            px.check()

    # ---- e2e: the same step through the host-buffer API, copies inside the timed region
    e2e_steps = max(3, min(args.steps, 10))
    h_in = torch.empty(shard.n_bytes, dtype=torch.uint8, pin_memory=True)
    h_in.copy_(d_in)
    h_out = torch.empty(shard.n_bytes, dtype=torch.uint8, pin_memory=True)

    def e2e_step():
        if world == 1:
            _, tag = eng.encrypt(iv, aad, h_in, out=h_out)
            return tag
        if px is not None:
            return px.crypt_host(0, iv, aad, shard, h_in, h_out, total)
        part = eng.stream_part_host(0, iv, shard.first_block, h_in, h_out, shard.blocks_after)
        d_part.copy_(torch.frombuffer(bytearray(part), dtype=torch.uint8))
        dist.all_gather_into_tensor(d_parts.view(-1), d_part)
        return eng.stream_finish_host(0, iv, d_parts.cpu().numpy(), aad, total)

    barrier()   # (pinning 2 x 1 GiB takes a different time on every rank)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        tag_e2e = e2e_step()
    barrier()
    e2e_s = allmax((time.perf_counter() - t0) / e2e_steps)
    assert tag_e2e == weak_tag, "host-buffer path and device path disagree on the tag"
    clocks = sampler.finish() if sampler else None
    del h_in, h_out, d_in, d_out
    torch.cuda.empty_cache()

    # ---- configs 3 and 4, messages split over the ranks
    batched = None
    if not args.no_extras:
        try:
            batched = batched_split(eng, torch, dist, dev, rank, world)
            if world > 1:
                batched += batched_split(eng, torch, dist, dev, rank, world, weak=True)
        except AssertionError:
            raise
        except Exception as ex:  # never lose the headline line over a secondary measurement
            batched = {"error": "%s: %s" % (type(ex).__name__, ex)}

    if rank == 0:
        peak, peak_src = peaks()
        # algorithmic bytes of ONE launch of the dominant kernel k_stream<14,ENC> (SURVEY 8d /
        # BASELINE.md 3): PT read + CT written + IV + key; AAD and tag belong to the finish
        alg = 2 * shard.n_bytes + 12 + 32
        k_avg_ms = k_ms / max(k_n, 1)
        achieved = alg / (k_avg_ms * 1e-3) / 1e9
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        # ncu-evidenced per-launch figures of the SAME kernel and size (profiles/ncu_traffic.json,
        # written by tools/make_profiles.py from the committed `ncu --set full` capture): DRAM bytes
        # and L1/shared data-pipe wavefronts.  They are read from that file, not measured in this run.
        traffic, wavefronts, src = None, None, None
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                tj = json.load(f)
            if tj.get("n_bytes") == shard.n_bytes:
                traffic = int(tj["dram_bytes_read"] + tj["dram_bytes_write"])
                wavefronts = tj.get("lsu_wavefronts_per_32_blocks")
                src = "profiles/ncu_traffic.json (%s)" % tj.get("source", "ncu --set full")
        except Exception:
            pass
        bound = None
        if wavefronts:
            # the L1/shared-memory data pipe retires 1 wavefront (128 B) per clock per SM
            smem_bound = eng.sm_count * sm_mhz * 1e6 / wavefronts * 32 * 16 / 1e9  # payload GB/s
            bound = {"payload_GBps_bound": round(smem_bound, 1), "sm_mhz_used": sm_mhz,
                     "lsu_wavefronts_per_32_blocks": wavefronts, "source": src,
                     "frac": round(shard.n_bytes / (k_avg_ms * 1e-3) / 1e9 / smem_bound, 4),
                     "note": "the binding roofline of this formulation is the 128 B/clk/SM L1/shared-memory data pipe "
                             "(ncu: l1tex__data_pipe_lsu_wavefronts), not HBM (DESIGN.md 4.1)"}
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world),
            "gpu_launches": int(launches),
            "parity_checked": True, "parity": parity,
            "e2e": {"value": round(total / e2e_s / 1e9, 3), "unit": UNIT,
                    "h2d_bytes_per_step": int(shard.n_bytes + AAD_BYTES),
                    "d2h_bytes_per_step": int(shard.n_bytes + 16), "steps": e2e_steps,
                    "api": "GcmEngine.encrypt (agcm_stream_crypt_host), pinned host buffers" if world == 1 else
                           ("PeerExchange.crypt_host (agcm_stream_crypt_peer_host), pinned host buffers" if px is not None else
                            "GcmEngine.stream_part_host + all_gather + stream_finish_host, pinned host buffers")},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": src,
                         "kernel": "k_stream<14,ENC>",
                         "kernel_ms": round(k_avg_ms, 4), "kernel_launches": int(k_n), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(alg)},
            "bound_smem_lookup": bound,
            "clocks": clocks,
        }
        if strong is not None:
            line["strong_scaling"] = strong
        if batched is not None:
            line["batched_split"] = batched
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            sample = calibrate_sample(cores, 4.0)
            v, dt = cpu_reference_rate(sample, cores, 3, 1)
            line["cpu_baseline"] = cpu_baseline_block(cores, sample, v, dt, 3, False)
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
    eng.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's tag and a fixed ciphertext sample as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm times a host-dependent sample")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under it
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
