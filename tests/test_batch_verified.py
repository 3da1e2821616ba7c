"""Verify-then-release batch decrypt (agcm_batch_decrypt_verified*): a message's plaintext is written only if its tag
matches, and no other byte of the output is ever written.

CPU: the tag-only flavour of the shared-key lane code, the gated GCTR slot mapping and the verified per-key message,
run on the host by tests/host_emul.cu, against the oracle.  GPU: all seven entry points on random batches with about
10 % of the messages corrupted, against the oracle, with the output prefilled by a sentinel."""
import numpy as np
import pytest

from batch_cases import (AG_DECRYPT_VERIFIED, SENTINEL, byte13_carry_at, corrupt, emul, emul_batch,  # noqa: F401 (emul)
                         emul_ctr_gated, expand_key, expect_offsets, offsets_case, top_carry_at, wrap_at)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kb", [16, 24, 32])
@pytest.mark.parametrize("G,S", [(1, 1), (2, 1), (4, 1), (32, 1), (32, 4), (32, 16)])
def test_emul_offsets_verify_then_gated(emul, oracle, kb, G, S):
    """The batch starts at byte 5 of its buffer: bytes before in_off[0] stay untouched.  The second batch holds J0 blocks
    whose counters wrap past 2^32 or carry into the counter's top byte or byte 13: on the first block of a segment of
    the tag-only pass, inside a lane-group row and on a row boundary; the gated pass then decrypts the same messages."""
    rng = np.random.default_rng(1000 + kb + 7 * G + S)
    c = offsets_case(oracle, rng, 40, kb, lens=(16 * 40 + 9,), shift=5)
    n = 16 * 9 + 5                      # blocks of the J0 messages (no AAD)
    seg1 = -(-n // S)                   # first block of segment 1 (ag_batch_segment, a payload block weighing 1)
    c_j0 = offsets_case(oracle, rng, 40, kb, lens=(16 * n,) * 7, aad_lens=(0,) * 7, shift=5,
                        j0_ctrs=[wrap_at(0), wrap_at(0), wrap_at(1), top_carry_at(0), wrap_at(1), byte13_carry_at(3),
                                 wrap_at(seg1), top_carry_at(seg1), wrap_at(5 * G + 3), wrap_at(4 * G), top_carry_at(64),
                                 byte13_carry_at(100), wrap_at(n - 1)])
    for c in (c, c_j0):
        want_ok = corrupt(rng, c)
        _, _, ok = emul_batch(emul, c, AG_DECRYPT_VERIFIED, G, S)
        assert (ok == want_ok).all(), (kb, G, S)
        for n_warps in (1, 3):
            assert (emul_ctr_gated(emul, c, ok, n_warps) == expect_offsets(c, want_ok)).all(), (kb, G, S, n_warps)


@pytest.mark.parametrize("kb", [16, 24, 32])
@pytest.mark.parametrize("form", ["uniform", "slots"])
def test_emul_fixed_pitch_verify_then_gated(emul, oracle, kb, form):
    rng = np.random.default_rng(2000 + kb + len(form))
    n, stride, astride = 37, 16 * 9 + 5, 70
    length = stride - 4 if form == "uniform" else stride
    lens = np.full(n, length) if form == "uniform" else rng.integers(0, stride + 20, n)   # slots: some past the pitch
    lens_cl = np.minimum(lens, stride)
    alen = 45
    buf = rng.integers(0, 256, n * stride, dtype=np.uint8)
    abuf = rng.integers(0, 256, n * astride, dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n, dtype=np.uint8)
    key = rng.integers(0, 256, kb, dtype=np.uint8)
    rk, nr = expand_key(oracle, key)
    rec = [buf[m * stride:m * stride + int(lens_cl[m])] for m in range(n)]
    in_off = np.concatenate([[0], np.cumsum(lens_cl)]).astype(np.uint64)
    packed = np.concatenate(rec) if in_off[-1] else np.zeros(0, np.uint8)
    apacked = np.concatenate([abuf[m * astride:m * astride + alen] for m in range(n)])
    aad_off = (np.arange(n + 1) * alen).astype(np.uint64)
    pt, tags = oracle.gcm_batch(key, kb, True, ivs, apacked, aad_off, packed, in_off, decrypt=True)
    want_ok = np.ones(n, np.uint8)
    for m in rng.choice(n, 5, replace=False):
        tags[16 * m + 3] ^= 0x20
        want_ok[m] = 0
    c = dict(n=n, rk=rk, nr=nr, ivs=ivs, aad=abuf, aad_len=alen, aad_stride=astride, data=buf, len=length, stride=stride,
             len_arr=lens.astype(np.uint32) if form == "slots" else None, tags=tags)
    _, _, ok = emul_batch(emul, c, AG_DECRYPT_VERIFIED, G=2)
    assert (ok == want_ok).all()
    want = np.full_like(buf, SENTINEL)
    for m in range(n):
        if want_ok[m]:
            want[m * stride:m * stride + int(lens_cl[m])] = pt[int(in_off[m]):int(in_off[m + 1])]
    assert (emul_ctr_gated(emul, c, ok, 2) == want).all(), (kb, form)


def test_emul_j0_forms(emul, oracle):
    """J0 blocks of IVs that are not 96 bits: the counter starts at inc32(J0), E_K(J0) masks the tag.  Through the
    releasing decrypt and through both passes of the verify-then-release decrypt."""
    rng = np.random.default_rng(31)
    n = 12
    c = offsets_case(oracle, rng, n, 16, max_len=100, max_aad=40)
    ivs = [rng.integers(0, 256, int(k), dtype=np.uint8).tobytes() for k in [1, 12, 16, 39] + list(rng.integers(1, 40, n - 4))]
    h, _ = oracle.h_ej0(c["rk"].tobytes(), bytes(12))
    c["ivs"], c["iv_is_j0"] = np.zeros(16 * n, np.uint8), 1
    for m, iv in enumerate(ivs):
        if len(iv) == 12:
            c["ivs"][16 * m:16 * m + 16] = np.frombuffer(iv + b"\0\0\0\1", np.uint8)
        else:
            blk = iv + bytes((-len(iv)) % 16) + bytes(8) + (8 * len(iv)).to_bytes(8, "big")
            c["ivs"][16 * m:16 * m + 16] = np.frombuffer(oracle.ghash_absorb(h, blk), np.uint8)
        a, b = int(c["in_off"][m]), int(c["in_off"][m + 1])
        aad = c["aad"][int(c["aad_off"][m]):int(c["aad_off"][m + 1])].tobytes()
        p_, t_ = oracle.gcm_crypt_any_iv(c["key"].tobytes(), iv, aad, c["data"][a:b].tobytes(), decrypt=True)
        c["out"][a:b] = np.frombuffer(p_, np.uint8)
        c["tags"][16 * m:16 * m + 16] = np.frombuffer(t_, np.uint8)
    c["tags"][16 * 4] ^= 1
    want_ok = [1] * 4 + [0] + [1] * 7
    out, _, ok = emul_batch(emul, c, 1, G=4)
    assert list(ok) == want_ok
    assert (out == expect_offsets(c, np.ones(n))).all()
    _, _, ok = emul_batch(emul, c, AG_DECRYPT_VERIFIED, G=4)
    assert list(ok) == want_ok
    assert (emul_ctr_gated(emul, c, ok, 1) == expect_offsets(c, ok)).all()


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_emul_perkey_verified(emul, oracle, kb):
    rng = np.random.default_rng(3000 + kb)
    c = offsets_case(oracle, rng, 30, kb, perkey=True)
    want_ok = corrupt(rng, c)
    out, _, ok = emul_batch(emul, c, AG_DECRYPT_VERIFIED)
    assert (ok == want_ok).all()
    assert (out == expect_offsets(c, want_ok)).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [0, 1, 2, 4, 8, 16, 32, 4097, 4100])
def test_offsets_verified(engine, oracle, lanes):
    import torch
    rng = np.random.default_rng(4000 + lanes)
    for kb in (16, 24, 32):
        c = offsets_case(oracle, rng, 1500, kb, shift=int(rng.integers(0, 16)))
        want_ok = corrupt(rng, c)
        engine.set_key(c["key"])
        out = torch.full((c["data"].size,), SENTINEL, dtype=torch.uint8, device="cuda")
        ok = torch.full((1500,), 9, dtype=torch.uint8, device="cuda")
        engine.batch_decrypt_verified_device(_t(c["ivs"]), _t(c["aad"]), _t(c["aad_off"].astype(np.int64)), _t(c["data"]),
                                             _t(c["in_off"].astype(np.int64)), out, _t(c["tags"]), ok, lanes=lanes,
                                             avg_len_hint=150)
        torch.cuda.synchronize()
        assert (ok.cpu().numpy() == want_ok).all(), (kb, lanes)
        assert (out.cpu().numpy() == expect_offsets(c, want_ok)).all(), (kb, lanes)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["few_long", "warp_units", "classes", "small_grid"])
def test_offsets_verified_layouts(engine, engine_small, oracle, shape):
    """Shapes that auto-select warp units, the three length classes, very long messages, and the odd 5 x 128 grid."""
    import torch
    rng = np.random.default_rng(4100 + len(shape))
    eng = engine_small if shape == "small_grid" else engine
    if shape == "few_long":
        c = offsets_case(oracle, rng, 8, 32, lens=(3 << 20, (1 << 20) + 5))
    elif shape == "warp_units":
        c = offsets_case(oracle, rng, 40, 16, max_len=200 << 10, max_aad=2000)
    elif shape == "classes":
        c = offsets_case(oracle, rng, 3000, 24, max_len=1600, lens=(40000, 70000, 20000))
    else:
        c = offsets_case(oracle, rng, 1200, 16, max_len=5000)
    n = len(c["lens"])
    want_ok = corrupt(rng, c)
    eng.set_key(c["key"])
    out = torch.full((c["data"].size,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    eng.batch_decrypt_verified_device(_t(c["ivs"]), _t(c["aad"]), _t(c["aad_off"].astype(np.int64)), _t(c["data"]),
                                      _t(c["in_off"].astype(np.int64)), out, _t(c["tags"]), ok,
                                      avg_len_hint=int(np.mean(c["lens"])))
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all(), shape
    assert (out.cpu().numpy() == expect_offsets(c, want_ok)).all(), shape


@pytest.mark.gpu
def test_offsets_verified_matches_releasing_and_in_place(engine, oracle):
    """All tags valid: output and ok identical to the releasing decrypt.  In place with corruption: failed messages keep
    their ciphertext."""
    import torch
    rng = np.random.default_rng(4200)
    c = offsets_case(oracle, rng, 2000, 32, max_len=2000)
    engine.set_key(c["key"])
    args = (_t(c["ivs"]), _t(c["aad"]), _t(c["aad_off"].astype(np.int64)))
    d_in, d_off, d_tags = _t(c["data"]), _t(c["in_off"].astype(np.int64)), _t(c["tags"])
    out_r = torch.full_like(d_in, SENTINEL)
    out_v = torch.full_like(d_in, SENTINEL)
    ok_r = torch.zeros(2000, dtype=torch.uint8, device="cuda")
    ok_v = torch.zeros(2000, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_device(1, *args, d_in, d_off, out_r, d_tags, ok_r)
    engine.batch_decrypt_verified_device(*args, d_in, d_off, out_v, d_tags, ok_v)
    torch.cuda.synchronize()
    assert torch.equal(out_r, out_v) and torch.equal(ok_r, ok_v) and int(ok_v.min()) == 1
    want_ok = corrupt(rng, c)
    buf = _t(c["data"])
    ok = torch.zeros(2000, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_device(_t(c["ivs"]), _t(c["aad"]), _t(c["aad_off"].astype(np.int64)), buf, d_off, buf,
                                         _t(c["tags"]), ok)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all()
    want = c["data"].copy()
    for m in np.nonzero(want_ok)[0]:
        a, b = int(c["in_off"][m]), int(c["in_off"][m + 1])
        want[a:b] = c["out"][a:b]
    assert (buf.cpu().numpy() == want).all()


@pytest.mark.gpu
def test_j0_forms_verified(engine, oracle):
    """IVs of other lengths through agcm_batch_derive_j0 and the _j0 forms (offsets and uniform)."""
    import torch
    rng = np.random.default_rng(4300)
    kb, n = 24, 300
    key = rng.integers(0, 256, kb, dtype=np.uint8)
    engine.set_key(key)
    iv_lens = rng.integers(1, 60, n)
    iv_off = np.concatenate([[0], np.cumsum(iv_lens)]).astype(np.int64)
    ivb = rng.integers(0, 256, int(iv_off[-1]), dtype=np.uint8)
    j0 = engine.batch_derive_j0_device(_t(ivb), iv_off=_t(iv_off))
    length, stride, alen = 333, 340, 20
    buf = rng.integers(0, 256, n * stride, dtype=np.uint8)
    abuf = rng.integers(0, 256, n * alen, dtype=np.uint8)
    pt = np.zeros_like(buf)
    tags = np.zeros(16 * n, np.uint8)
    for m in range(n):
        iv = ivb[iv_off[m]:iv_off[m + 1]].tobytes()
        p_, t_ = oracle.gcm_crypt_any_iv(key.tobytes(), iv, abuf[m * alen:(m + 1) * alen].tobytes(),
                                         buf[m * stride:m * stride + length].tobytes(), decrypt=True)
        pt[m * stride:m * stride + length] = np.frombuffer(p_, np.uint8)
        tags[16 * m:16 * m + 16] = np.frombuffer(t_, np.uint8)
    bad = rng.choice(n, 30, replace=False)
    want_ok = np.ones(n, np.uint8)
    want_ok[bad] = 0
    tags[16 * bad + 7] ^= 0x80
    # uniform
    out = torch.full((buf.size,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_uniform_device(j0, _t(abuf), alen, alen, _t(buf), out, length, stride, _t(tags), ok, j0=True)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all()
    want = np.full_like(buf, SENTINEL)
    for m in np.nonzero(want_ok)[0]:
        want[m * stride:m * stride + length] = pt[m * stride:m * stride + length]
    assert (out.cpu().numpy() == want).all()
    # offsets over the same records (the pitch padding counts as part of each message here: stride = message length)
    packed = buf.reshape(n, stride)[:, :length].reshape(-1).copy()
    in_off = (np.arange(n + 1) * length).astype(np.int64)
    aad_off = (np.arange(n + 1) * alen).astype(np.int64)
    out = torch.full((packed.size,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_device(j0, _t(abuf), _t(aad_off), _t(packed), _t(in_off), out, _t(tags), ok, j0=True)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all()
    assert (out.cpu().numpy() == want.reshape(n, stride)[:, :length].reshape(-1)).all()


def _uniform_case(oracle, rng, n, kb, length, stride, alen, astride, perkey=False):
    buf = rng.integers(0, 256, n * stride + 32, dtype=np.uint8)
    abuf = rng.integers(0, 256, n * astride + 32, dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n, dtype=np.uint8)
    keys = rng.integers(0, 256, kb * (n if perkey else 1), dtype=np.uint8)
    packed = buf[:n * stride].reshape(n, stride)[:, :length].reshape(-1).copy()
    apacked = abuf[:n * astride].reshape(n, astride)[:, :alen].reshape(-1).copy()
    in_off = (np.arange(n + 1) * length).astype(np.uint64)
    aad_off = (np.arange(n + 1) * alen).astype(np.uint64)
    pt, tags = oracle.gcm_batch(keys, kb, not perkey, ivs, apacked if alen else None, aad_off if alen else None, packed, in_off,
                                decrypt=True, threads=8)
    return buf, abuf, ivs, keys, pt, tags


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [0, 1, 2, 4, 8, 16, 32, 4097])
@pytest.mark.parametrize("layout", [(1500, 1504, 16, 16, 0), (4096, 4096, 0, 0, 0), (333, 341, 13, 21, 3), (40000, 40000, 64, 64, 0)])
def test_uniform_verified(engine, oracle, lanes, layout):
    """Records at aligned and odd pitches and buffer offsets; record and AAD padding stay untouched."""
    import torch
    length, stride, alen, astride, shift = layout
    rng = np.random.default_rng(4400 + lanes + length)
    n = 64 if length >= 40000 else 700
    kb = (16, 24, 32)[lanes % 3]
    buf, abuf, ivs, key, pt, tags = _uniform_case(oracle, rng, n, kb, length, stride, alen, astride)
    bad = rng.choice(n, n // 10, replace=False)
    want_ok = np.ones(n, np.uint8)
    want_ok[bad] = 0
    tags[16 * bad] ^= 4
    engine.set_key(key)
    d_buf = _t(np.concatenate([np.zeros(shift, np.uint8), buf]))   # the records start `shift` bytes into the allocation
    out = torch.full((buf.size + 16,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_uniform_device(_t(ivs), _t(abuf) if alen else None, alen, astride, d_buf[shift:],
                                                 out[shift:], length, stride, _t(tags), ok, lanes=lanes)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all(), (lanes, layout)
    want = np.full(buf.size + 16, SENTINEL, np.uint8)
    for m in np.nonzero(want_ok)[0]:
        want[shift + m * stride:shift + m * stride + length] = pt[m * length:(m + 1) * length]
    assert (out.cpu().numpy() == want).all(), (lanes, layout)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [0, 1, 4, 32, 4098])
def test_slots_verified(engine, engine_small, oracle, lanes):
    import torch
    rng = np.random.default_rng(4500 + lanes)
    n, stride, astride = 1300, 1504, 48
    lens = rng.integers(0, stride + 100, n)
    lens[:4] = [0, 1, stride, stride + 50]
    alens = rng.integers(0, astride + 1, n)
    lcl = np.minimum(lens, stride)
    buf = rng.integers(0, 256, n * stride, dtype=np.uint8)
    abuf = rng.integers(0, 256, n * astride, dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n, dtype=np.uint8)
    key = rng.integers(0, 256, 32, dtype=np.uint8)
    in_off = np.concatenate([[0], np.cumsum(lcl)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    packed = np.concatenate([buf[m * stride:m * stride + lcl[m]] for m in range(n)])
    apacked = np.concatenate([abuf[m * astride:m * astride + alens[m]] for m in range(n)])
    pt, tags = oracle.gcm_batch(key, 32, True, ivs, apacked, aad_off, packed, in_off, decrypt=True, threads=8)
    want_ok = np.ones(n, np.uint8)
    for m in rng.choice(n, n // 10, replace=False):
        want_ok[m] = 0
        if lcl[m] and m % 2:
            buf[m * stride + int(rng.integers(0, lcl[m]))] ^= 0x40
        else:
            tags[16 * m + 15] ^= 1
    for eng in (engine, engine_small):
        eng.set_key(key)
        out = torch.full((buf.size,), SENTINEL, dtype=torch.uint8, device="cuda")
        ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        eng.batch_decrypt_verified_slots_device(_t(ivs), _t(abuf), _t(alens.astype(np.uint32)).view(torch.int32), 0, astride,
                                                _t(buf), out, _t(lens.astype(np.uint32)).view(torch.int32), stride, _t(tags), ok,
                                                lanes=lanes)
        torch.cuda.synchronize()
        assert (ok.cpu().numpy() == want_ok).all(), lanes
        want = np.full_like(buf, SENTINEL)
        for m in np.nonzero(want_ok)[0]:
            want[m * stride:m * stride + lcl[m]] = pt[int(in_off[m]):int(in_off[m + 1])]
        assert (out.cpu().numpy() == want).all(), lanes


@pytest.mark.gpu
@pytest.mark.parametrize("kb", [16, 24, 32])
def test_perkey_verified(engine, oracle, kb):
    import torch
    rng = np.random.default_rng(4600 + kb)
    n = 2500
    c = offsets_case(oracle, rng, n, kb, max_len=1600, max_aad=100, shift=3, perkey=True)
    want_ok = corrupt(rng, c)
    out = torch.full((c["data"].size,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_perkey_device(kb * 8, _t(c["key"]), _t(c["ivs"]), _t(c["aad"]),
                                                _t(c["aad_off"].astype(np.int64)), _t(c["data"]),
                                                _t(c["in_off"].astype(np.int64)), out, _t(c["tags"]), ok)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all()
    assert (out.cpu().numpy() == expect_offsets(c, want_ok)).all()
    # uniform records, in place: failed records keep their ciphertext, padding untouched
    length, stride, alen = 1500, 1504, 16
    m_u = 3000
    buf, abuf, ivs, keys, pt, tags = _uniform_case(oracle, rng, m_u, kb, length, stride, alen, alen, perkey=True)
    bad = rng.choice(m_u, 300, replace=False)
    want_ok = np.ones(m_u, np.uint8)
    want_ok[bad] = 0
    tags[16 * bad + 1] ^= 2
    d = _t(buf)
    ok = torch.zeros(m_u, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_perkey_uniform_device(kb * 8, _t(keys), _t(ivs), _t(abuf), alen, alen, d, d, length, stride,
                                                        _t(tags), ok)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all()
    want = buf.copy()
    for m in np.nonzero(want_ok)[0]:
        want[m * stride:m * stride + length] = pt[m * length:(m + 1) * length]
    assert (d.cpu().numpy() == want).all()


@pytest.mark.gpu
def test_stream_order_on_side_stream(engine, oracle):
    """A releasing encrypt feeds the verified decrypt on a non-blocking side stream with no synchronise between them."""
    import torch
    rng = np.random.default_rng(4700)
    n, length, stride = 4000, 1500, 1504
    key = rng.integers(0, 256, 16, dtype=np.uint8)
    engine.set_key(key)
    s = torch.cuda.Stream()
    ptb = rng.integers(0, 256, n * stride, dtype=np.uint8)
    ivs = _t(rng.integers(0, 256, 12 * n, dtype=np.uint8))
    d_pt = _t(ptb)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        ct = torch.empty_like(d_pt)
        tags = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
        back = torch.full_like(d_pt, SENTINEL)
        ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_uniform_device(0, ivs, None, 0, 0, d_pt, ct, length, stride, tags, stream=s)
        engine.batch_decrypt_verified_uniform_device(ivs, None, 0, 0, ct, back, length, stride, tags, ok, stream=s)
    s.synchronize()
    assert int(ok.min()) == 1
    assert torch.equal(back.view(n, stride)[:, :length], d_pt.view(n, stride)[:, :length])
    assert int((back.view(n, stride)[:, length:] != SENTINEL).sum()) == 0


@pytest.mark.gpu
def test_error_codes(engine, engine_lib):
    import torch
    import aesgcm_b200
    from aesgcm_b200 import _lib
    L = engine_lib
    eng = aesgcm_b200.GcmEngine(0)   # no key yet
    n, length = 4, 64
    buf = torch.zeros(n * length, dtype=torch.uint8, device="cuda")
    ivs = torch.zeros(12 * n, dtype=torch.uint8, device="cuda")
    tags = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * length
    P = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
    ctx = eng._ctx
    uni = lambda lanes, t, o, ln=length, st=length, c=ctx: L.agcm_batch_decrypt_verified_uniform(   # noqa: E731
        c, lanes, P(ivs), None, 0, 0, P(buf), P(buf), ln, st, P(t), P(o), n, 0)
    assert uni(0, tags, ok) == _lib.E_NO_KEY
    eng.set_key(bytes(16))
    assert uni(0, tags, None) == _lib.E_BAD_ARG
    assert uni(0, None, ok) == _lib.E_BAD_ARG
    for lanes in (1024, 1025, 1028, 2048, 4096, 3):
        assert uni(lanes, tags, ok) == _lib.E_BAD_ARG, lanes
    over = uni(0, tags, ok, ln=length + 1)
    assert over == L.agcm_batch_crypt_uniform(ctx, 1, 0, P(ivs), None, 0, 0, P(buf), P(buf), length + 1, length, P(tags), P(ok), n, 0)
    assert over == _lib.E_BAD_LEN
    assert L.agcm_batch_decrypt_verified(ctx, 0, 0, P(ivs), None, None, P(buf), P(off), P(buf), P(tags), None, n, 0) == _lib.E_BAD_ARG
    assert L.agcm_batch_decrypt_verified(ctx, 2048, 0, P(ivs), None, None, P(buf), P(off), P(buf), P(tags), P(ok), n, 0) == _lib.E_BAD_ARG
    lens = torch.full((n,), length, dtype=torch.int32, device="cuda")
    assert L.agcm_batch_decrypt_verified_slots(ctx, 1024, P(ivs), None, None, 0, 0, P(buf), P(buf), P(lens), length, 0, P(tags),
                                               P(ok), n, 0) == _lib.E_BAD_ARG
    keys = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
    assert L.agcm_batch_decrypt_verified_perkey(ctx, 128, P(keys), P(ivs), None, None, P(buf), P(off), P(buf), None, P(ok), n,
                                                0) == _lib.E_BAD_ARG
    assert L.agcm_batch_decrypt_verified_perkey_uniform(ctx, 100, P(keys), P(ivs), None, 0, 0, P(buf), P(buf), length, length,
                                                        P(tags), P(ok), n, 0) == _lib.E_BAD_MODE
    before = eng.launch_count
    assert L.agcm_batch_decrypt_verified(ctx, 0, 0, P(ivs), None, None, P(buf), P(off), P(buf), P(tags), P(ok), 0, 0) == 0
    assert uni(0, tags, ok) == 0 and eng.launch_count > before
    before = eng.launch_count
    assert L.agcm_batch_decrypt_verified_uniform(ctx, 0, P(ivs), None, 0, 0, P(buf), P(buf), length, length, P(tags), P(ok), 0,
                                                 0) == 0
    assert L.agcm_batch_decrypt_verified_perkey_uniform(ctx, 128, P(keys), P(ivs), None, 0, 0, P(buf), P(buf), length, length,
                                                        P(tags), P(ok), 0, 0) == 0
    assert eng.launch_count == before
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("perkey", [False, True])
def test_full_size_config_shapes(engine, oracle, perkey):
    """2^20 x 1500 B: config 3 (one AES-192 key, 1504 B pitch, 16 B AAD) and config 4 (a key per message, AES-256), 0.1 %
    corrupted tags.  The ciphertext comes from the releasing encrypt; the oracle checks a sample of the authentic messages
    and every corrupted message's range holds the sentinel."""
    import torch
    n, length = 1 << 20, 1500
    stride, alen, kb = (1500, 0, 32) if perkey else (1504, 16, 24)
    rng = np.random.default_rng(4800 + perkey)
    g = torch.Generator(device="cuda").manual_seed(7)
    pt = torch.randint(0, 256, (n * stride,), dtype=torch.uint8, device="cuda", generator=g)
    ivs = torch.randint(0, 256, (12 * n,), dtype=torch.uint8, device="cuda", generator=g)
    aad = torch.randint(0, 256, (max(1, n * alen),), dtype=torch.uint8, device="cuda", generator=g) if alen else None
    keys = torch.randint(0, 256, (kb * (n if perkey else 1),), dtype=torch.uint8, device="cuda", generator=g)
    ct = torch.empty_like(pt)
    tags = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
    if perkey:
        engine.batch_crypt_perkey_uniform_device(kb * 8, 0, keys, ivs, None, 0, 0, pt, ct, length, stride, tags)
    else:
        engine.set_key(keys.cpu().numpy())
        engine.batch_crypt_uniform_device(0, ivs, aad, alen, alen, pt, ct, length, stride, tags)
    bad = torch.from_numpy(rng.choice(n, n // 1000, replace=False)).cuda()
    tags.view(n, 16)[bad, 5] ^= 0x10
    out = torch.full_like(pt, SENTINEL)
    ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    if perkey:
        engine.batch_decrypt_verified_perkey_uniform_device(kb * 8, keys, ivs, None, 0, 0, ct, out, length, stride, tags, ok)
    else:
        engine.batch_decrypt_verified_uniform_device(ivs, aad, alen, alen, ct, out, length, stride, tags, ok)
    torch.cuda.synchronize()
    want_ok = torch.ones(n, dtype=torch.uint8, device="cuda")
    want_ok[bad] = 0
    assert torch.equal(ok, want_ok)
    o2, p2 = out.view(n, stride), pt.view(n, stride)
    good = want_ok.bool()
    assert torch.equal(o2[good][:, :length], p2[good][:, :length])
    assert int((o2[bad] != SENTINEL).sum()) == 0
    if stride > length:
        assert int((o2[:, length:] != SENTINEL).sum()) == 0
    # oracle sample of authentic messages
    idx = [int(i) for i in rng.choice(n, 48, replace=False) if want_ok[int(i)]]
    ct_h, ivs_h, tags_h = ct.view(n, stride).cpu().numpy(), ivs.view(n, 12).cpu().numpy(), tags.view(n, 16).cpu().numpy()
    keys_h = keys.view(-1, kb).cpu().numpy()
    aad_h = aad.view(n, alen).cpu().numpy() if alen else None
    for m in idx:
        k = keys_h[m if perkey else 0].tobytes()
        p_, t_ = oracle.gcm_crypt(k, ivs_h[m].tobytes(), aad_h[m].tobytes() if alen else b"", ct_h[m, :length], decrypt=True)
        assert t_ == tags_h[m].tobytes()
        assert o2[m, :length].cpu().numpy().tobytes() == p_
