#!/usr/bin/env python
"""Verify-then-release batch decrypt (agcm_batch_decrypt_verified*) against the releasing decrypt of the same inputs,
the two alternated in one run and timed with CUDA events; then, in a profiled run of its own, the kernel time per pass
(pass 1 = k_batch_verify / k_batch_warp_verify, pass 2 = k_batch_ctr_gated).  All tags valid, so both forms write
every message.  Prints one JSON line per shape and the card's name, power limit and SM clock.

Shapes: config 3 (2^20 x 1500 B at a 1504 B pitch, AES-192, 16 B AAD), config 4 (2^20 x 1500 B, a key per message,
AES-256), the config 1 shape (262144 x 4 KiB, AES-256), the 64 / 576 / 1500 B mix of tools/bench_ragged.py (2^20
messages packed by offsets, AES-128) and a few long messages (16 x 4 MiB, AES-256).  Every working set is larger than
the 126 MB L2 except the last one (64 MiB), which is read from L2 after the first pass."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.getcwd())
import numpy as np  # noqa: E402
import torch  # noqa: E402

import aesgcm_b200  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def shapes(eng, n_scale):
    rng = np.random.default_rng(5)
    g = torch.Generator(device="cuda").manual_seed(5)
    R = lambda k: torch.randint(0, 256, (k,), dtype=torch.uint8, device="cuda", generator=g)   # noqa: E731
    n = (1 << 20) // n_scale
    # config 3
    ivs, aad, buf = R(12 * n), R(16 * n), R(1504 * n)
    out, tags, ok = torch.empty_like(buf), torch.zeros(16 * n, dtype=torch.uint8, device="cuda"), torch.zeros(n, dtype=torch.uint8,
                                                                                                         device="cuda")
    key = R(24)
    yield ("config 3: 2^20 x 1500 B @ 1504, AES-192, 16 B AAD", 1500 * n, lambda: eng.set_key(key.cpu().numpy()),
           lambda: eng.batch_crypt_uniform_device(1, ivs, aad, 16, 16, buf, out, 1500, 1504, tags, ok),
           lambda: eng.batch_decrypt_verified_uniform_device(ivs, aad, 16, 16, buf, out, 1500, 1504, tags, ok),
           lambda: eng.batch_crypt_uniform_device(0, ivs, aad, 16, 16, buf, buf, 1500, 1504, tags))
    # config 4
    keys, buf4 = R(32 * n), R(1500 * n)
    out4 = torch.empty_like(buf4)
    yield ("config 4: 2^20 x 1500 B, a key per message, AES-256", 1500 * n, lambda: None,
           lambda: eng.batch_crypt_perkey_uniform_device(256, 1, keys, ivs, None, 0, 0, buf4, out4, 1500, 1500, tags, ok),
           lambda: eng.batch_decrypt_verified_perkey_uniform_device(256, keys, ivs, None, 0, 0, buf4, out4, 1500, 1500, tags, ok),
           lambda: eng.batch_crypt_perkey_uniform_device(256, 0, keys, ivs, None, 0, 0, buf4, buf4, 1500, 1500, tags))
    del buf4, out4, keys
    # config 1 shape
    n1 = 262144 // n_scale
    buf1 = R(4096 * n1)
    out1 = torch.empty_like(buf1)
    key32 = R(32)
    yield ("262144 x 4 KiB, AES-256", 4096 * n1, lambda: eng.set_key(key32.cpu().numpy()),
           lambda: eng.batch_crypt_uniform_device(1, ivs[:12 * n1], None, 0, 0, buf1, out1, 4096, 4096, tags, ok, n_msgs=n1),
           lambda: eng.batch_decrypt_verified_uniform_device(ivs[:12 * n1], None, 0, 0, buf1, out1, 4096, 4096, tags, ok, n_msgs=n1),
           lambda: eng.batch_crypt_uniform_device(0, ivs[:12 * n1], None, 0, 0, buf1, buf1, 4096, 4096, tags, n_msgs=n1))
    del buf1, out1
    # ragged mix
    lens = rng.choice([64, 576, 1500], n, p=[0.58, 0.33, 0.09])
    off = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)).cuda()
    total = int(lens.sum())
    bufr = R(total)
    outr = torch.empty_like(bufr)
    key16 = R(16)
    hint = int(lens.mean())
    yield ("IMIX 64 / 576 / 1500 B (58 / 33 / 9 %), 2^20 by offsets, AES-128", total, lambda: eng.set_key(key16.cpu().numpy()),
           lambda: eng.batch_crypt_device(1, ivs, None, None, bufr, off, outr, tags, ok, avg_len_hint=hint),
           lambda: eng.batch_decrypt_verified_device(ivs, None, None, bufr, off, outr, tags, ok, avg_len_hint=hint),
           lambda: eng.batch_crypt_device(0, ivs, None, None, bufr, off, bufr, tags, avg_len_hint=hint))
    del bufr, outr
    # a few long messages
    nl, L = 16, 4 << 20
    bufl = R(nl * L)
    outl = torch.empty_like(bufl)
    yield ("16 x 4 MiB, AES-256 (64 MiB: L2-resident)", nl * L, lambda: eng.set_key(key32.cpu().numpy()),
           lambda: eng.batch_crypt_uniform_device(1, ivs[:12 * nl], None, 0, 0, bufl, outl, L, L, tags, ok, n_msgs=nl),
           lambda: eng.batch_decrypt_verified_uniform_device(ivs[:12 * nl], None, 0, 0, bufl, outl, L, L, tags, ok, n_msgs=nl),
           lambda: eng.batch_crypt_uniform_device(0, ivs[:12 * nl], None, 0, 0, bufl, bufl, L, L, tags, n_msgs=nl))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--scale", type=int, default=1, help="divide the message counts (rehearsal runs)")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    eng = aesgcm_b200.GcmEngine(0)
    info = {"card": card()}
    print(json.dumps(info), flush=True)
    lines = [info]
    for name, nbytes, setup, rel, ver, enc in shapes(eng, a.scale):
        setup()
        enc()   # valid tags: both forms then write every message
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        for f in (rel, ver):
            f()
        torch.cuda.synchronize()
        t_rel = t_ver = 0.0
        for _ in range(a.reps):
            ev[0].record(); rel(); ev[1].record()
            ev[2].record(); ver(); ev[3].record()
            torch.cuda.synchronize()
            t_rel += ev[0].elapsed_time(ev[1])
            t_ver += ev[2].elapsed_time(ev[3])
        t_rel /= a.reps
        t_ver /= a.reps
        # kernel time per pass, profiled separately
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ver()
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if e.device_type == torch.autograd.DeviceType.CUDA and e.count:
                k = e.key.split("<")[0].split("(")[0]
                per[k] = per.get(k, 0.0) + e.device_time_total / 3 / 1000.0
        rec = {"shape": name, "bytes": nbytes, "release_ms": round(t_rel, 4), "verified_ms": round(t_ver, 4),
               "release_GBps": round(nbytes / t_rel / 1e6, 1), "verified_GBps": round(nbytes / t_ver / 1e6, 1),
               "verified_over_release": round(t_rel / t_ver, 3), "verified_kernel_ms": {k: round(v, 4) for k, v in per.items()}}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
