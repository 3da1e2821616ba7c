"""CPU check of the engine's per-thread device code (tests/host_emul.cu runs the
functions of csrc/gcm_core.cuh on the host) against the oracle: index arithmetic
of the strided Horner, table multiply, T-table AES, ragged last block."""
import ctypes

import numpy as np
import pytest

from batch_cases import emul, emul_batch, expect_offsets, offsets_case  # noqa: F401 (emul: the fixture)
from conftest import u8p, u64p


def test_sbox_and_key_expand(emul, oracle):
    sb = np.zeros(256, np.uint8)
    emul.emul_sbox(u8p(sb))
    assert (sb == oracle.sbox_table()).all()
    rng = np.random.default_rng(11)
    for kb in (16, 24, 32):
        for _ in range(8):
            k = rng.integers(0, 256, kb, dtype=np.uint8)
            out = np.zeros(240, np.uint8)
            nr = emul.emul_key_expand(u8p(k), kb, u8p(out))
            assert out[:16 * (nr + 1)].tobytes() == oracle.key_expand(k.tobytes())


def test_gf_multiplies(emul, oracle):
    rng = np.random.default_rng(12)
    out = np.zeros(16, np.uint8)
    cases = [rng.integers(0, 256, (2, 16), dtype=np.uint8) for _ in range(300)]
    edge = [np.zeros(16, np.uint8), np.full(16, 255, np.uint8), np.array([0x80] + [0] * 15, np.uint8),
            np.array([0] * 15 + [1], np.uint8)]
    cases += [np.stack([a, b]) for a in edge for b in edge]
    for ab in cases:
        a, b = np.ascontiguousarray(ab[0]), np.ascontiguousarray(ab[1])
        want = oracle.gfmul(a.tobytes(), b.tobytes())
        emul.emul_gf_mul(u8p(a), u8p(b), u8p(out))
        assert out.tobytes() == want
        emul.emul_gf_mul_table(u8p(a), u8p(b), u8p(out))  # Shoup-table path of the hot loop
        assert out.tobytes() == want
        emul.emul_gf_sqr(u8p(a), u8p(out))                 # linear squaring used by the key setup
        assert out.tobytes() == oracle.gfmul(a.tobytes(), a.tobytes())


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_stream_lanes(emul, oracle, kb):
    rng = np.random.default_rng(13 + kb)
    for n in (0, 1, 15, 16, 17, 31, 32, 100, 1000, 4096 + 5):
        for (ncta, nt) in ((1, 1), (1, 4), (3, 8), (2, 32)):
            for mode in (0, 1, 2):
                key = rng.integers(0, 256, kb, dtype=np.uint8).tobytes()
                iv = rng.integers(0, 256, 12, dtype=np.uint8)
                data = rng.integers(0, 256, max(n, 1), dtype=np.uint8)[:n].copy()
                rk = np.frombuffer(oracle.key_expand(key), dtype=np.uint8).copy()
                nr = len(rk) // 16 - 1
                out = np.zeros(max(n, 1), np.uint8)
                part = np.zeros(16, np.uint8)
                inp = data if n else np.zeros(1, np.uint8)
                ctr0 = int(rng.integers(2, 2 ** 32))  # includes wrap-around of the 32-bit counter
                rc = emul.emul_stream(u8p(rk), nr, u8p(iv), ctypes.c_uint32(ctr0), u8p(inp), u8p(out), ctypes.c_uint64(n),
                                      mode, ncta, nt, u8p(part))
                assert rc == 0
                h, _ = oracle.h_ej0(rk.tobytes(), iv.tobytes())
                if mode == 2:
                    assert part.tobytes() == oracle.ghash_absorb(h, data.tobytes())
                    continue
                exp_out = oracle.gctr(rk.tobytes(), iv.tobytes(), ctr0, data.tobytes())
                assert out[:n].tobytes() == exp_out, (kb, n, ncta, nt, mode)
                ct = data.tobytes() if mode == 1 else exp_out
                assert part.tobytes() == oracle.ghash_absorb(h, ct), (kb, n, ncta, nt, mode)


def _releasing(emul, c, dec, bad, G=1, S=1):
    """Encrypt or releasing decrypt of case c: every message is written, and a decrypt rejects message `bad` only."""
    if dec:
        c["tags"][16 * bad + 5] ^= 0x10
    out, tags, ok = emul_batch(emul, c, dec, G, S)
    assert (out == expect_offsets(c, np.ones(c["n"]))).all()
    if dec:
        assert list(ok) == [int(m != bad) for m in range(c["n"])]
    else:
        assert (tags == c["tags"]).all()


@pytest.mark.parametrize("G", [1, 2, 4, 8, 16, 32])
def test_batch_lanes(emul, oracle, G):
    """Lane groups of G lanes; the 16*600+3 B message carries the counter byte past 256 blocks."""
    rng = np.random.default_rng(17 + G)
    for kb in (16, 24, 32):
        for dec in (0, 1):
            c = offsets_case(oracle, rng, 9, kb, max_len=200, max_aad=70, lens=(1500, 16 * 600 + 3), aad_lens=(0, 16),
                             decrypt=bool(dec))
            _releasing(emul, c, dec, 7, G)


@pytest.mark.parametrize("S", [2, 4, 16])
def test_batch_split_segments(emul, oracle, S):
    """Messages cut into S counter-range segments (the split layout of k_batch_cta): AAD with
    segment 0, length block with segment S-1, partials scaled by H^after and XORed.  Includes
    messages shorter than S blocks (empty segments), ragged tails and empty payloads."""
    rng = np.random.default_rng(300 + S)
    for kb, G in ((16, 4), (32, 32), (24, 8)):
        for dec in (0, 1):
            c = offsets_case(oracle, rng, 10, kb, max_len=400, max_aad=70, lens=(16 * 300 + 5, 33, 16 * S * 7),
                             aad_lens=(0, 16), decrypt=bool(dec))
            _releasing(emul, c, dec, 6, G, S)


@pytest.mark.parametrize("n_warps", [1, 3, 7, 40])
def test_batch_balanced_partition(emul, oracle, n_warps):
    """k_batch_warp's balanced partition of uniform records over a virtual grid: cuts inside the AAD,
    inside the payload, inside one payload block's weight, inside the finish positions; more warps
    than messages and more messages than warps; ragged tails; every message closed exactly once."""
    rng = np.random.default_rng(500 + n_warps)
    for kb, nm, length, alen in ((16, 5, 16 * 37 + 5, 16 * 11 + 3), (32, 2, 16 * 200, 0), (24, 9, 100, 700), (16, 3, 0, 50),
                                 (32, 6, 16, 16), (24, 1, 16 * 129 + 1, 16 * 5)):
        for dec in (0, 1):
            stride, astride = length + 3, alen + 5
            buf = rng.integers(0, 256, nm * stride + 1, dtype=np.uint8)
            abuf = rng.integers(0, 256, nm * astride + 1, dtype=np.uint8)
            ivs = rng.integers(0, 256, 12 * nm, dtype=np.uint8)
            key = rng.integers(0, 256, kb, dtype=np.uint8)
            rk = np.frombuffer(oracle.key_expand(key.tobytes()), dtype=np.uint8).copy()
            nr = len(rk) // 16 - 1
            packed = buf[:nm * stride].reshape(nm, stride)[:, :length].reshape(-1).copy()
            apacked = abuf[:nm * astride].reshape(nm, astride)[:, :alen].reshape(-1).copy()
            in_off = (np.arange(nm + 1) * length).astype(np.uint64)
            aad_off = (np.arange(nm + 1) * alen).astype(np.uint64)
            eo, et = oracle.gcm_batch(key, kb, True, ivs, apacked if alen else None, aad_off if alen else None, packed, in_off,
                                      decrypt=bool(dec))
            out = np.zeros_like(buf)
            tag = np.zeros(16 * nm, np.uint8)
            ok = np.zeros(nm, np.uint8)
            if dec:
                tag[:] = et
                tag[16 * (nm - 1) + 2] ^= 0x40
            rc = emul.emul_batch_balanced(u8p(rk), nr, dec, n_warps, u8p(ivs), u8p(abuf), ctypes.c_uint64(alen),
                                          ctypes.c_uint64(astride), u8p(buf), u8p(out), ctypes.c_uint64(length),
                                          ctypes.c_uint64(stride), u8p(tag), u8p(ok), ctypes.c_uint64(nm))
            assert rc == 0
            got = out[:nm * stride].reshape(nm, stride)[:, :length].reshape(-1)
            assert (got == eo[:nm * length]).all(), (kb, nm, length, alen, dec)
            if dec:
                assert list(ok) == [1] * (nm - 1) + [0], (kb, nm, length, alen)
            else:
                assert (tag == et).all(), (kb, nm, length, alen)


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_perkey_messages(emul, oracle, kb):
    """One distinct key per message: on-the-fly key schedule + private 4-bit GHASH table."""
    rng = np.random.default_rng(23 + kb)
    for dec in (0, 1):
        c = offsets_case(oracle, rng, 12, kb, max_aad=80, lens=(1500,), aad_lens=(64, 0), perkey=True, decrypt=bool(dec))
        _releasing(emul, c, dec, 4)


def test_host_pipeline_granule_schedule(emul):
    """csrc/host_sched.h: the ramped granule list of the host-buffer pipeline covers the range exactly, keeps every
    granule but the last a whole number of counter blocks, never exceeds the stage buffer, starts and ends small, and
    falls back to equal granules when the list would not fit."""
    emul.emul_chunk_schedule.restype = ctypes.c_uint32
    MiB = 1 << 20
    cap = 1024
    sz = np.zeros(cap, np.uint64)

    def plan(n, peak, base, cap_=cap):
        k = emul.emul_chunk_schedule(ctypes.c_uint64(n), ctypes.c_uint64(peak), ctypes.c_uint64(base), u64p(sz), cap_)
        return [int(x) for x in sz[:k]]

    assert plan(0, 32 * MiB, 2 * MiB) == []
    rng = np.random.default_rng(5)
    sizes = [1, 15, 16, 17, MiB, 4 * MiB, 4 * MiB + 1, 8 * MiB, 8 * MiB + 5, 32 * MiB, 32 * MiB + 4097, 92 * MiB - 1, 92 * MiB,
             92 * MiB + 16, 1 << 30, (1 << 30) + 7, 3 << 30] + [int(x) for x in rng.integers(1, 1 << 31, 200)]
    for peak, base in ((32 * MiB, 2 * MiB), (32 * MiB, MiB), (24 * MiB, 2 * MiB), (64 * MiB, 4 * MiB), (32 * MiB, 0), (2 * MiB, 2 * MiB)):
        for n in sizes:
            p = plan(n, peak, base)
            if (n + peak - 1) // peak > cap:      # the caller grows the granule first (pick_chunk)
                assert p == []
                continue
            assert sum(p) == n and all(x > 0 for x in p), (n, peak, base)
            assert all(x % 16 == 0 for x in p[:-1])
            assert max(p) <= peak + 15
            if base and base < peak and n >= 3 * peak:
                assert p[0] == base and base <= p[-1] < base + 16          # ramps at both ends
                lmax = (peak // base).bit_length() - 1
                assert p[:lmax] == [base << i for i in range(lmax)]
                assert [x & ~15 for x in p[-lmax:]] == [base << i for i in reversed(range(lmax))]
                assert len(p) <= n // peak + 2 * 8 + 2
            if not base or base >= peak:
                assert p == [peak] * (n // peak) + ([n % peak] if n % peak else [])
    # one GiB at the defaults: 2, 4, 8, 16 MiB, the odd rest, 30 x 32 MiB ... and back down
    p = plan(1 << 30, 32 * MiB, 2 * MiB)
    assert p[:4] == [2 * MiB, 4 * MiB, 8 * MiB, 16 * MiB] and p[-4:] == [16 * MiB, 8 * MiB, 4 * MiB, 2 * MiB]
    # a short range shortens the ramp instead of dropping it
    assert plan(8 * MiB, 32 * MiB, 2 * MiB) == [2 * MiB, 4 * MiB, 2 * MiB]
    # does not fit the list: equal granules; cannot fit at all: 0
    assert plan(64 * MiB, 32 * MiB, 2 * MiB, 3) == [32 * MiB, 32 * MiB]
    assert plan(64 * MiB + 1, 32 * MiB, 2 * MiB, 2) == []
