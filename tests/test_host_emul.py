"""CPU check of the engine's per-thread device code (tests/host_emul.cu runs the
functions of csrc/gcm_core.cuh on the host) against the oracle: index arithmetic
of the strided Horner, table multiply, T-table AES, ragged last block."""
import ctypes

import numpy as np
import pytest

from batch_cases import (byte13_carry_at, emul, emul_batch, expect_offsets, gf_inv, iv_for_j0, offsets_case,  # noqa: F401
                         top_carry_at, wrap_at)
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
    """Block i has counter ctr0 + i (mod 2^32): the pinned ctr0 put the 32-bit wrap on block 0, on the first block of
    the second CTA and of the second grid row and on two blocks past a row's first, and the carries into the counter's
    top byte and into byte 13 on block 8; two more are drawn."""
    rng = np.random.default_rng(13 + kb)
    for n in (0, 1, 15, 16, 17, 31, 32, 100, 1000, 4096 + 5):
        for (ncta, nt) in ((1, 1), (1, 4), (3, 8), (2, 32)):
            gt = ncta * nt
            pinned = [wrap_at(0), wrap_at(nt), wrap_at(gt), wrap_at(gt // 2 + 1), wrap_at(2 * gt + 3), 0x00FFFFF8, 0x0000FFF8]
            for ctr0 in pinned + [int(x) for x in rng.integers(2, 2 ** 32, 2)]:
                for mode in (0, 1, 2):
                    key = rng.integers(0, 256, kb, dtype=np.uint8).tobytes()
                    iv = rng.integers(0, 256, 12, dtype=np.uint8)
                    data = rng.integers(0, 256, max(n, 1), dtype=np.uint8)[:n].copy()
                    rk = np.frombuffer(oracle.key_expand(key), dtype=np.uint8).copy()
                    nr = len(rk) // 16 - 1
                    out = np.zeros(max(n, 1), np.uint8)
                    part = np.zeros(16, np.uint8)
                    inp = data if n else np.zeros(1, np.uint8)
                    rc = emul.emul_stream(u8p(rk), nr, u8p(iv), ctypes.c_uint32(ctr0), u8p(inp), u8p(out), ctypes.c_uint64(n),
                                          mode, ncta, nt, u8p(part))
                    assert rc == 0
                    h, _ = oracle.h_ej0(rk.tobytes(), iv.tobytes())
                    if mode == 2:
                        assert part.tobytes() == oracle.ghash_absorb(h, data.tobytes())
                        continue
                    exp_out = oracle.gctr(rk.tobytes(), iv.tobytes(), ctr0, data.tobytes())
                    assert out[:n].tobytes() == exp_out, (kb, n, ncta, nt, mode, hex(ctr0))
                    ct = data.tobytes() if mode == 1 else exp_out
                    assert part.tobytes() == oracle.ghash_absorb(h, ct), (kb, n, ncta, nt, mode, hex(ctr0))


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


# J0 counter fields of the J0 cases below, one per message of offsets_case's fixed lengths 0, 1, 15, 16, 17, 16*7+3:
# the 32-bit wrap on block 0, 0, 1 (past the ragged end), 0 (of a whole block) and 1 (ragged), and the top-byte carry
# on block 3
J0_FIRST6 = [wrap_at(0), wrap_at(0), wrap_at(1), wrap_at(0), wrap_at(1), top_carry_at(3)]


@pytest.mark.parametrize("G", [1, 2, 4, 8, 16, 32])
def test_batch_lanes(emul, oracle, G):
    """Lane groups of G lanes; the 16*600+3 B message carries the counter byte past 256 blocks.  J0 cases: the 32-bit
    wrap and the carries into the counter's top byte and byte 13 on payload blocks 64 (a row boundary for every G) and
    37 (inside a row for G > 1)."""
    rng = np.random.default_rng(17 + G)
    for kb in (16, 24, 32):
        for dec in (0, 1):
            c = offsets_case(oracle, rng, 9, kb, max_len=200, max_aad=70, lens=(1500, 16 * 600 + 3), aad_lens=(0, 16),
                             decrypt=bool(dec))
            _releasing(emul, c, dec, 7, G)
            c = offsets_case(oracle, rng, 12, kb, max_len=200, max_aad=70, lens=(16 * 100 + 3, 16 * 50, 16 * 70 + 9, 100, 16 * 40),
                             aad_lens=(0, 16, 0, 33, 0), decrypt=bool(dec),
                             j0_ctrs=J0_FIRST6 + [wrap_at(64), wrap_at(37), top_carry_at(64), byte13_carry_at(5),
                                                  top_carry_at(37)])
            _releasing(emul, c, dec, 7, G)


@pytest.mark.parametrize("S", [2, 4, 16])
def test_batch_split_segments(emul, oracle, S):
    """Messages cut into S counter-range segments (the split layout of k_batch_cta): AAD with
    segment 0, length block with segment S-1, partials scaled by H^after and XORed.  Includes
    messages shorter than S blocks (empty segments), ragged tails and empty payloads."""
    rng = np.random.default_rng(300 + S)
    n_wrap = 16 * S * 7   # blocks of the J0 messages below, no AAD: S segments of 4 * n_wrap / S weight positions each
    seg1 = -(-4 * n_wrap // S) // 4   # ag_batch_segment: first payload block of segment 1
    for kb, G in ((16, 4), (32, 32), (24, 8)):
        for dec in (0, 1):
            c = offsets_case(oracle, rng, 10, kb, max_len=400, max_aad=70, lens=(16 * 300 + 5, 33, 16 * S * 7),
                             aad_lens=(0, 16), decrypt=bool(dec))
            _releasing(emul, c, dec, 6, G, S)
            # J0 cases: the wrap and the top-byte carry on the first block of segment 1, on its last block before that
            # and on a block inside it
            c = offsets_case(oracle, rng, 10, kb, max_len=400, max_aad=70, lens=(16 * n_wrap,) * 4, aad_lens=(0,) * 4,
                             decrypt=bool(dec), j0_ctrs=J0_FIRST6 + [wrap_at(seg1), top_carry_at(seg1), wrap_at(seg1 - 1),
                                                                     top_carry_at(seg1 + 3)])
            _releasing(emul, c, dec, 6, G, S)


@pytest.mark.parametrize("n_warps", [1, 3, 7, 40])
def test_batch_balanced_partition(emul, oracle, n_warps):
    """k_batch_warp's balanced partition of uniform records over a virtual grid: cuts inside the AAD,
    inside the payload, inside one payload block's weight, inside the finish positions; more warps
    than messages and more messages than warps; ragged tails; every message closed exactly once.
    The last three batches take J0 blocks (16-byte IVs) with the 32-bit wrap, the carry into the counter's top byte
    and the carry into byte 13 on the first, a middle and the last payload block."""
    rng = np.random.default_rng(500 + n_warps)
    edge = lambda nb: [wrap_at(0), wrap_at(nb // 2), top_carry_at(nb - 1), byte13_carry_at(1), top_carry_at(nb // 3),  # noqa: E731
                       wrap_at(nb - 1)]
    for kb, nm, length, alen, j0 in ((16, 5, 16 * 37 + 5, 16 * 11 + 3, False), (32, 2, 16 * 200, 0, False),
                                     (24, 9, 100, 700, False), (16, 3, 0, 50, False), (32, 6, 16, 16, False),
                                     (24, 1, 16 * 129 + 1, 16 * 5, False),
                                     (16, 6, 16 * 37 + 5, 16 * 11 + 3, True), (32, 5, 16 * 200, 0, True), (24, 6, 100, 70, True)):
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
            if j0:
                h = oracle.aes_encrypt_block(rk.tobytes(), bytes(16))
                h_inv = gf_inv(oracle, h)
                ivs = np.zeros(16 * nm, np.uint8)
                eo, et = np.zeros(nm * length, np.uint8), np.zeros(16 * nm, np.uint8)
                for m, c0 in enumerate(edge((length + 15) // 16)[:nm]):
                    j0b = rng.integers(0, 256, 12, dtype=np.uint8).tobytes() + c0.to_bytes(4, "big")
                    ivs[16 * m:16 * m + 16] = np.frombuffer(j0b, np.uint8)
                    p_, t_ = oracle.gcm_crypt_any_iv(key.tobytes(), iv_for_j0(oracle, h, h_inv, j0b),
                                                     apacked[m * alen:(m + 1) * alen].tobytes(),
                                                     packed[m * length:(m + 1) * length].tobytes(), decrypt=bool(dec))
                    eo[m * length:(m + 1) * length] = np.frombuffer(p_, np.uint8)
                    et[16 * m:16 * m + 16] = np.frombuffer(t_, np.uint8)
            else:
                eo, et = oracle.gcm_batch(key, kb, True, ivs, apacked if alen else None, aad_off if alen else None, packed,
                                          in_off, decrypt=bool(dec))
            out = np.zeros_like(buf)
            tag = np.zeros(16 * nm, np.uint8)
            ok = np.zeros(nm, np.uint8)
            if dec:
                tag[:] = et
                tag[16 * (nm - 1) + 2] ^= 0x40
            rc = emul.emul_batch_balanced(u8p(rk), nr, dec, n_warps, u8p(ivs), int(j0), u8p(abuf), ctypes.c_uint64(alen),
                                          ctypes.c_uint64(astride), u8p(buf), u8p(out), ctypes.c_uint64(length),
                                          ctypes.c_uint64(stride), u8p(tag), u8p(ok), ctypes.c_uint64(nm))
            assert rc == 0
            got = out[:nm * stride].reshape(nm, stride)[:, :length].reshape(-1)
            assert (got == eo[:nm * length]).all(), (kb, nm, length, alen, dec, j0)
            if dec:
                assert list(ok) == [1] * (nm - 1) + [0], (kb, nm, length, alen, j0)
            else:
                assert (tag == et).all(), (kb, nm, length, alen, j0)


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_perkey_messages(emul, oracle, kb):
    """One distinct key per message: on-the-fly key schedule + private 4-bit GHASH table."""
    rng = np.random.default_rng(23 + kb)
    for dec in (0, 1):
        c = offsets_case(oracle, rng, 12, kb, max_aad=80, lens=(1500,), aad_lens=(64, 0), perkey=True, decrypt=bool(dec))
        _releasing(emul, c, dec, 4)


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_counter_caches(emul, oracle, kb):
    """The per-lane counter caches against AES-ECB of the counter blocks: the batch lanes' sequential cache, the stream
    kernel's cache and the per-key kernels' copy of the sequential refill (schedule on the fly).  32-block windows
    across the carry into the counter's top byte, the carry into byte 13 and the wrap to 0; and steps that move one
    counter byte alone (2^24: the top byte only), which consecutive counters never do."""
    rng = np.random.default_rng(40 + kb)
    key = rng.integers(0, 256, kb, dtype=np.uint8)
    iv = rng.integers(0, 256, 12, dtype=np.uint8)
    rk = np.frombuffer(oracle.key_expand(key.tobytes()), dtype=np.uint8).copy()
    nr = len(rk) // 16 - 1
    U32, U64 = ctypes.c_uint32, ctypes.c_uint64
    for ctr0, stride, n in ((0x00FFFFF0, 1, 32), (0x0000FFF0, 1, 32), (0xFFFFFFF0, 1, 32), (0xFFFFFFF0, 3, 32),
                            (0x00FFFFF0, 256, 32), (0x12345678, 1 << 24, 300), (0x12345678, 1 << 16, 300),
                            (0x12345678, 1 << 8, 300), (0x12345678, 0x01010101, 300)):
        want = b"".join(oracle.aes_encrypt_block(rk.tobytes(), iv.tobytes() + ((ctr0 + k * stride) & 0xFFFFFFFF).to_bytes(4, "big"))
                        for k in range(n))
        out = np.zeros(16 * n, np.uint8)
        for which in (0, 1):
            assert emul.emul_ctr_cached(u8p(rk), nr, u8p(iv), U32(ctr0), U32(stride), U64(n), which, u8p(out)) == 0
            assert out.tobytes() == want, (kb, hex(ctr0), stride, which)
        out[:] = 0
        assert emul.emul_perkey_ctr(u8p(key), kb, u8p(iv), U32(ctr0), U32(stride), U64(n), u8p(out)) == 0
        assert out.tobytes() == want, (kb, hex(ctr0), stride, "perkey")


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
