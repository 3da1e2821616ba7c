"""Batch cases for the emulator and GPU tests of the batch entry points: the host build of tests/host_emul.cu (the `emul`
fixture), ragged offsets batches with the oracle's output and tags, corruption of some of their messages, and thin
wrappers around the emulator's batch calls."""
import ctypes
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, u8p, u64p

SENTINEL = 0xA5
AG_DECRYPT_VERIFIED = 2   # `decrypt` of the tag-only pass, as in csrc/kernels.h
CSRC = os.path.join(ROOT, "aes-gcm-128-192-256-bits_b200", "csrc")


@pytest.fixture(scope="module")
def emul():
    """Host build of tests/host_emul.cu, rebuilt when it or any header under csrc/ is newer than the library."""
    # conftest's fixture of the same name, which this one overrides, misses perkey_core.cuh, host_sched.h and kernels.h
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    bdir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(bdir, exist_ok=True)
    so = os.path.join(bdir, "libhost_emul.so")
    src = os.path.join(ROOT, "tests", "host_emul.cu")
    deps = [src] + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h"))
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call([nvcc, "-w", "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-o", so, src])
    return ctypes.CDLL(so)


def u32p(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))


def expand_key(oracle, key):
    """-> (round keys, nr)"""
    rk = np.frombuffer(oracle.key_expand(key.tobytes()), dtype=np.uint8).copy()
    return rk, len(rk) // 16 - 1


def gf_inv(oracle, h):
    """h^(2^128 - 2) = h^-1 in GCM's field"""
    r, e = bytes([0x80]) + bytes(15), (1 << 128) - 2
    while e:
        if e & 1:
            r = oracle.gfmul(r, h)
        h = oracle.gfmul(h, h)
        e >>= 1
    return r


def iv_for_j0(oracle, h, h_inv, j0):
    """The 16-byte IV whose J0 = GHASH_H(IV || 0^64 || [128]_64) = IV.H^2 ^ L.H is `j0`: IV = ((J0.H^-1) ^ L).H^-1."""
    x = bytearray(oracle.gfmul(j0, h_inv))
    x[15] ^= 128   # L = [0]_64 || [128]_64
    iv = oracle.gfmul(bytes(x), h_inv)
    assert oracle.ghash_absorb(h, iv + bytes(8) + (128).to_bytes(8, "big")) == j0
    return iv


def wrap_at(i):
    """J0 counter field whose payload block i has counter 0 (inc32 wraps from 0xFFFFFFFF between blocks i-1 and i)"""
    return (0xFFFFFFFF - i) & 0xFFFFFFFF


def top_carry_at(i):
    """J0 counter field whose payload block i has counter 0x01000000 (carry into the counter's top byte)"""
    return 0x00FFFFFF - i


def byte13_carry_at(i):
    """J0 counter field whose payload block i has counter 0x00010000 (carry into byte 13 of the counter block)"""
    return 0x0000FFFF - i


def offsets_case(oracle, rng, n, kb, max_len=300, max_aad=300, lens=(), aad_lens=(), shift=0, perkey=False, decrypt=True,
                 j0_ctrs=None):
    """n messages in the offsets form under one key (perkey: a key per message) with the oracle's output and tags.
    Payload lengths start 0, 1, 15, 16, 17, 16*7+3; messages 6, 7, ... take `lens` and `aad_lens`; the rest are drawn.
    The batch starts `shift` bytes into `data`, which runs on past its end.
    j0_ctrs: message m gets a 16-byte IV whose J0 ends in the counter field j0_ctrs[m]; past its end, or where it holds
    None, an IV of a drawn length (12 bytes for some).  c["ivs"] then holds the J0 blocks (iv_is_j0), c["iv_raw"] and
    c["iv_off"] the IVs and their offsets, and the reference is the oracle's any-IV composition."""
    ln = rng.integers(0, max_len, n)
    ln[:6] = [0, 1, 15, 16, 17, 16 * 7 + 3][:min(6, n)]
    ln[6:6 + len(lens)] = lens
    alens = rng.integers(0, max_aad + 1, n)
    alens[6:6 + len(aad_lens)] = aad_lens
    in_off = (shift + np.concatenate([[0], np.cumsum(ln)])).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    data = rng.integers(0, 256, int(in_off[-1]) + 9, dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]) + 1, dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n, dtype=np.uint8)
    key = rng.integers(0, 256, kb * (n if perkey else 1), dtype=np.uint8)
    out, tags = oracle.gcm_batch(key, kb, not perkey, ivs, aad, aad_off, data, in_off, decrypt=decrypt, threads=8)
    c = dict(n=n, kb=kb, perkey=perkey, lens=ln, alens=alens, in_off=in_off, aad_off=aad_off, data=data, aad=aad, ivs=ivs,
             key=key, out=out, tags=tags)
    if j0_ctrs is not None:
        assert not perkey   # the per-key entry points take 96-bit IVs only
        h = oracle.aes_encrypt_block(oracle.key_expand(key.tobytes()), bytes(16))
        h_inv = gf_inv(oracle, h)
        c["ivs"], c["iv_is_j0"], raw = np.zeros(16 * n, np.uint8), 1, []
        for m in range(n):
            c0 = j0_ctrs[m] if m < len(j0_ctrs) else None
            if c0 is None:
                iv = rng.integers(0, 256, int(rng.choice([1, 8, 12, 16, 20, 33])), dtype=np.uint8).tobytes()
                j0 = iv + bytes([0, 0, 0, 1]) if len(iv) == 12 else oracle.ghash_absorb(
                    h, iv + bytes(-len(iv) % 16) + bytes(8) + (8 * len(iv)).to_bytes(8, "big"))
            else:
                j0 = rng.integers(0, 256, 12, dtype=np.uint8).tobytes() + int(c0).to_bytes(4, "big")
                iv = iv_for_j0(oracle, h, h_inv, j0)
            c["ivs"][16 * m:16 * m + 16] = np.frombuffer(j0, np.uint8)
            raw.append(iv)
            a, b = int(in_off[m]), int(in_off[m + 1])
            o_, t_ = oracle.gcm_crypt_any_iv(key.tobytes(), iv, aad[int(aad_off[m]):int(aad_off[m + 1])].tobytes(),
                                             data[a:b].tobytes(), decrypt=decrypt)
            out[a:b] = np.frombuffer(o_, np.uint8)
            tags[16 * m:16 * m + 16] = np.frombuffer(t_, np.uint8)
        c["iv_raw"] = np.frombuffer(b"".join(raw), np.uint8).copy()
        c["iv_off"] = np.concatenate([[0], np.cumsum([len(iv) for iv in raw])]).astype(np.int64)
    if not perkey:
        c["rk"], c["nr"] = expand_key(oracle, key)
    return c


def corrupt(rng, c, frac=0.1):
    """Flip a tag bit, a ciphertext byte or an AAD byte of about frac of case c's messages.  -> expected ok flags."""
    ok = np.ones(c["n"], np.uint8)
    for m in rng.choice(c["n"], max(1, int(frac * c["n"])), replace=False):
        kind = int(rng.integers(0, 3))
        if kind == 1 and c["lens"][m]:
            c["data"][int(c["in_off"][m]) + int(rng.integers(0, c["lens"][m]))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2 and c["alens"][m]:
            c["aad"][int(c["aad_off"][m]) + int(rng.integers(0, c["alens"][m]))] ^= 1 << int(rng.integers(0, 8))
        else:
            c["tags"][16 * m + int(rng.integers(0, 16))] ^= 1 << int(rng.integers(0, 8))
        ok[m] = 0
    return ok


def expect_offsets(c, ok):
    """A SENTINEL-filled buffer like c's data holding the oracle's output of the messages whose ok flag is set."""
    want = np.full_like(c["data"], SENTINEL)
    for m in np.nonzero(ok)[0]:
        a, b = int(c["in_off"][m]), int(c["in_off"][m + 1])
        want[a:b] = c["out"][a:b]
    return want


def _opt(conv, a):
    return None if a is None else conv(a)


def emul_batch(emul, c, decrypt, G=1, S=1):
    """emul_batch (emul_batch_perkey for a per-key case) on case c into a SENTINEL-filled output.  Without in_off, c is
    in the uniform (len, stride, aad_len, aad_stride) or the slots form (len_arr).  -> (out, tags, ok): the tags are
    the computed ones (encrypt) or c's expected ones (decrypt); ok starts as 7, so every flag must be written."""
    n, U64 = c["n"], ctypes.c_uint64
    out = np.full_like(c["data"], SENTINEL)
    tags = c["tags"].copy() if decrypt else np.zeros(16 * n, np.uint8)
    ok = np.full(n, 7, np.uint8)
    if c.get("perkey"):
        rc = emul.emul_batch_perkey(u8p(c["key"]), c["kb"], decrypt, u8p(c["ivs"]), u8p(c["aad"]), u64p(c["aad_off"]),
                                    u8p(c["data"]), u64p(c["in_off"]), u8p(out), u8p(tags), u8p(ok), U64(n))
    else:
        rc = emul.emul_batch(u8p(c["rk"]), c["nr"], decrypt, G, S, u8p(c["ivs"]), c.get("iv_is_j0", 0), u8p(c["aad"]),
                             _opt(u64p, c.get("aad_off")), U64(c.get("aad_len", 0)), U64(c.get("aad_stride", 0)),
                             u8p(c["data"]), _opt(u64p, c.get("in_off")), U64(c.get("len", 0)), U64(c.get("stride", 0)),
                             _opt(u32p, c.get("len_arr")), u8p(out), u8p(tags), u8p(ok), U64(n))
    assert rc == 0
    return out, tags, ok


def emul_ctr_gated(emul, c, ok, n_warps):
    """Pass 2 of the verify-then-release decrypt on case c (layout as in emul_batch) into a SENTINEL-filled output."""
    U64 = ctypes.c_uint64
    out = np.full_like(c["data"], SENTINEL)
    assert emul.emul_batch_ctr_gated(u8p(c["rk"]), c["nr"], u8p(c["ivs"]), c.get("iv_is_j0", 0), u8p(c["data"]),
                                     _opt(u64p, c.get("in_off")), U64(c.get("len", 0)), U64(c.get("stride", 0)),
                                     _opt(u32p, c.get("len_arr")), u8p(out), u8p(ok), U64(c["n"]), U64(n_warps)) == 0
    return out
