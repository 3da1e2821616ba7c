"""Counter edges on the GPU.  GCM steps only the low 32 bits of the counter block (inc32); with an IV that is not 96
bits, J0 = GHASH_H(IV || pad || len) can start the counter anywhere, so a legal message may wrap it from 0xFFFFFFFF to
0 or carry into its top byte (0x00FFFFFF -> 0x01000000) after a few blocks.  Here a 16-byte IV is built for a chosen
J0 (batch_cases.iv_for_j0), so the wrap or carry falls on a chosen block: a host granule, grid row, shard, segment,
keystream window or tile boundary.  Every stream, shared-key batch and per-key path against the oracle's any-IV
composition, which the counter-edge vectors of golden/long_iv_vectors.json pin to OpenSSL."""
import numpy as np
import pytest

from batch_cases import (SENTINEL, byte13_carry_at, emul, expect_offsets, gf_inv, iv_for_j0, offsets_case,  # noqa: F401
                         top_carry_at, u64p, wrap_at)

pytestmark = pytest.mark.gpu
MiB = 1 << 20


def _t(a):
    import torch
    return torch.from_numpy(np.array(a)).cuda()   # a copy: frombuffer views are read-only


def _h(t):
    return t.cpu().numpy().tobytes()


def _flip(tag):
    return bytes([tag[0] ^ 0x01]) + tag[1:]


class Edge:
    """A key, and 16-byte IVs under it whose J0 ends in a chosen counter field."""

    def __init__(self, oracle, rng, kb):
        self.oracle, self.rng = oracle, rng
        self.key = rng.integers(0, 256, kb, dtype=np.uint8).tobytes()
        self.rk = oracle.key_expand(self.key)
        self.h = oracle.aes_encrypt_block(self.rk, bytes(16))
        self.h_inv = gf_inv(oracle, self.h)

    def iv(self, c0):
        """-> (IV, J0)"""
        j0 = self.rng.integers(0, 256, 12, dtype=np.uint8).tobytes() + c0.to_bytes(4, "big")
        return iv_for_j0(self.oracle, self.h, self.h_inv, j0), j0

    def data(self, n):
        return self.rng.integers(0, 256, n, dtype=np.uint8).tobytes()

    def ref(self, iv, aad, pt):
        return self.oracle.gcm_crypt_any_iv(self.key, iv, aad, pt)


# ------------------------------------------------------------------------------------------------------------ stream
def test_stream_host_calls(engine, oracle, emul):
    """agcm_stream_crypt_iv_host: one-shot sizes, and sizes of several pipeline granules with the wrap on the first
    granule boundary and inside later granules.  The granules are the ones host_sched.h makes at the context's
    defaults (32 MiB steady granule, 1 MiB first and last)."""
    import ctypes
    rng = np.random.default_rng(7000)
    sz = np.zeros(64, np.uint64)
    n_multi = 4 * MiB + 53
    k = emul.emul_chunk_schedule(ctypes.c_uint64(n_multi), ctypes.c_uint64(32 * MiB), ctypes.c_uint64(MiB), u64p(sz), 64)
    bounds = [int(b) // 16 for b in np.cumsum(sz[:k])[:-1]]   # first block of granules 1, 2, ...
    assert len(bounds) >= 2
    cases = [(16 * 5000 + 7, 20, c0) for c0 in (wrap_at(0), wrap_at(1234), top_carry_at(77), byte13_carry_at(4999))]
    cases += [(n_multi, 16, wrap_at(bounds[0])), (n_multi, 0, wrap_at(bounds[-1] + 1000)), (n_multi, 33, top_carry_at(bounds[0] + 5)),
              (n_multi, 0, wrap_at(bounds[0] - 1))]
    for it, (n, alen, c0) in enumerate(cases):
        e = Edge(oracle, rng, (16, 24, 32)[it % 3])
        iv, _ = e.iv(c0)
        aad, pt = e.data(alen), e.data(n)
        want_ct, want_tag = e.ref(iv, aad, pt)
        engine.set_key(e.key)
        ct, tag = engine.encrypt(iv, aad, pt)
        assert ct == want_ct and tag == want_tag, (it, n, hex(c0))
        assert engine.decrypt(iv, aad, ct, tag) == pt, (it, n, hex(c0))
        assert engine.decrypt(iv, aad, ct, _flip(tag), raise_on_fail=False)[1] is False


def _device_case(eng, e, iv, aad, pt, in_place=False, out_shift=0):
    """Encrypt and decrypt through agcm_stream_crypt_iv with device buffers, and a flipped tag rejected."""
    import torch
    n = len(pt)
    want_ct, want_tag = e.ref(iv, aad, pt)
    d_aad = _t(np.frombuffer(aad, np.uint8)) if aad else None
    d_in = _t(np.frombuffer(pt, np.uint8))
    if in_place:
        d_out = d_in
    else:
        d_buf = torch.full((n + out_shift + 16,), SENTINEL, dtype=torch.uint8, device="cuda")
        d_out = d_buf[out_shift:out_shift + n]
    d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
    eng.stream_crypt_device(0, iv, d_aad, d_in, d_out, d_tag, n_bytes=n)
    torch.cuda.synchronize()
    assert _h(d_out) == want_ct and _h(d_tag) == want_tag
    if not in_place:
        assert bool((d_buf[:out_shift] == SENTINEL).all()) and bool((d_buf[out_shift + n:] == SENTINEL).all())
    d_ct = d_out.clone()
    d_back = torch.full_like(d_ct, SENTINEL) if not in_place else d_out
    d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
    eng.stream_crypt_device(1, iv, d_aad, d_ct if not in_place else d_out, d_back, d_tag, d_ok, n_bytes=n)
    torch.cuda.synchronize()
    assert _h(d_back) == pt and int(d_ok.item()) == 1
    eng.stream_crypt_device(1, iv, d_aad, d_ct, d_back, _t(np.frombuffer(_flip(want_tag), np.uint8)), d_ok, n_bytes=n)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 0


def test_stream_device_calls(engine, engine_small, oracle):
    """agcm_stream_crypt_iv on device buffers: one grid row, several rows with the wrap on a row boundary, the small
    grid (stride 640 blocks: the stream kernel's counter cache refills every block), in place, output at odd addresses
    (the warp's cooperative stores), AAD beyond the inline limit (the bulk-AAD finish)."""
    rng = np.random.default_rng(7001)
    row = engine.n_cta * engine.threads
    srow = engine_small.n_cta * engine_small.threads
    cases = [  # engine, payload bytes, AAD bytes, J0 counter field, in place, output offset
        (engine, 16 * 1000 + 3, 16, wrap_at(500), False, 0),
        (engine, 16 * 1000 + 3, 0, top_carry_at(999), False, 0),
        (engine, 16 * (2 * row + 100) + 7, 0, wrap_at(row), False, 0),
        (engine, 16 * (2 * row + 100) + 7, 20, wrap_at(2 * row), False, 0),
        (engine, 16 * (row + 50), 0, top_carry_at(row - 1), False, 0),
        (engine_small, 16 * srow * 5 + 7, 16, wrap_at(2 * srow), False, 0),
        (engine_small, 16 * srow * 5 + 7, 0, top_carry_at(1000), False, 0),
        (engine_small, 16 * srow * 5 + 7, 0, byte13_carry_at(3 * srow + 1), False, 0),
        (engine, 16 * 3000 + 5, 16, wrap_at(1500), True, 0),
        (engine_small, 16 * 3000 + 5, 0, top_carry_at(srow), True, 0),
        (engine, 16 * 3000 + 5, 16, wrap_at(1501), False, 1),
        (engine_small, 16 * 3000 + 9, 0, wrap_at(srow), False, 3),
        (engine, 16 * 2000 + 9, 5000, wrap_at(1000), False, 0),
        (engine_small, 16 * 900, 4097, top_carry_at(3), False, 0),
    ]
    for it, (eng, n, alen, c0, in_place, shift) in enumerate(cases):
        e = Edge(oracle, rng, (16, 24, 32)[it % 3])
        eng.set_key(e.key)
        iv, _ = e.iv(c0)
        try:
            _device_case(eng, e, iv, e.data(alen), e.data(n), in_place, shift)
        except AssertionError as x:
            raise AssertionError((it, n, alen, hex(c0), in_place, shift)) from x


def test_stream_shards_gctr_peer(engine, oracle):
    """agcm_stream_part_j0 / _finish_j0 over the shard plans of 1, 3 and 8 ranks with a shard boundary exactly at the
    wrap (and at a top-byte carry), agcm_gctr_j0 from a first block on either side of the wrap, agcm_stream_crypt_peer_j0
    with one rank."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(7002)
    n, alen = 16 * 3000 + 5, 20
    blocks = (n + 15) // 16
    for it, world in enumerate((1, 3, 8)):
        per = -(-blocks // world)
        for c0 in ((wrap_at(0), top_carry_at(1)) if world == 1 else (wrap_at(per), top_carry_at(2 * per))):
            e = Edge(oracle, rng, (16, 24, 32)[it])
            engine.set_key(e.key)
            iv, _ = e.iv(c0)
            aad, pt = e.data(alen), e.data(n)
            want_ct, want_tag = e.ref(iv, aad, pt)
            d_aad = _t(np.frombuffer(aad, np.uint8))
            for dec, src, want in ((0, pt, want_ct), (1, want_ct, pt)):
                d_in = _t(np.frombuffer(src, np.uint8))
                d_out = torch.full_like(d_in, SENTINEL)
                parts = torch.zeros((world, 16), dtype=torch.uint8, device="cuda")
                for sh in shard_plan(n, world):
                    sl = slice(sh.byte_offset, sh.byte_offset + sh.n_bytes)
                    engine.stream_part_device(dec, iv, sh.first_block, d_in[sl], d_out[sl], sh.blocks_after, parts[sh.rank],
                                              n_bytes=sh.n_bytes)
                d_tag = _t(np.frombuffer(want_tag, np.uint8)) if dec else torch.zeros(16, dtype=torch.uint8, device="cuda")
                d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
                engine.stream_finish_device(dec, iv, parts, world, d_aad, n, d_tag, d_ok if dec else None)
                torch.cuda.synchronize()
                assert _h(d_out) == want, (world, hex(c0), dec)
                if dec:
                    assert int(d_ok.item()) == 1, (world, hex(c0))
                    engine.stream_finish_device(1, iv, parts, world, d_aad, n, _t(np.frombuffer(_flip(want_tag), np.uint8)), d_ok)
                    torch.cuda.synchronize()
                    assert int(d_ok.item()) == 0, (world, hex(c0))
                else:
                    assert _h(d_tag) == want_tag, (world, hex(c0))
    # GCTR half: counters j0ctr + 1 + first_block + i, across the wrap
    e = Edge(oracle, rng, 32)
    engine.set_key(e.key)
    for c0, first_block in ((wrap_at(700), 690), (wrap_at(690), 690), (wrap_at(691), 690), (top_carry_at(50), 40)):
        iv, j0 = e.iv(c0)
        data = e.data(16 * 20 + 3)
        d_in = _t(np.frombuffer(data, np.uint8))
        d_out = torch.full_like(d_in, SENTINEL)
        engine.gctr_device(iv, first_block, d_in, d_out)
        torch.cuda.synchronize()
        assert _h(d_out) == oracle.gctr(e.rk, j0[:12], c0 + 1 + first_block, data), (hex(c0), first_block)
    # peer exchange, one rank
    buf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    engine.peer_setup(0, 1, [buf.data_ptr()])
    for c0 in (wrap_at(1000), top_carry_at(0)):
        iv, _ = e.iv(c0)
        aad, pt = e.data(16), e.data(n)
        want_ct, want_tag = e.ref(iv, aad, pt)
        d_in, d_aad = _t(np.frombuffer(pt, np.uint8)), _t(np.frombuffer(aad, np.uint8))
        d_out = torch.full_like(d_in, SENTINEL)
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_peer_device(0, iv, 0, d_in, d_out, 0, d_aad, n, d_tag)
        d_back = torch.full_like(d_in, SENTINEL)
        d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_peer_device(1, iv, 0, d_out, d_back, 0, d_aad, n, d_tag.clone(), d_ok)
        torch.cuda.synchronize()
        assert _h(d_out) == want_ct and _h(d_tag) == want_tag and _h(d_back) == pt and int(d_ok.item()) == 1, hex(c0)


def test_stream_decrypt_verified(engine, oracle):
    """agcm_stream_decrypt_verified and its host form: the GHASH-only pass, then the gated GCTR pass across the wrap; a
    flipped tag leaves the output as it was."""
    import torch
    rng = np.random.default_rng(7003)
    row = engine.n_cta * engine.threads
    for it, (n, alen, c0) in enumerate(((16 * 3000 + 5, 16, wrap_at(0)), (16 * 3000 + 5, 0, wrap_at(777)),
                                        (16 * (row + 10) + 1, 5000, wrap_at(row)), (100, 20, top_carry_at(2)))):
        e = Edge(oracle, rng, (16, 24, 32)[it % 3])
        engine.set_key(e.key)
        iv, _ = e.iv(c0)
        aad, pt = e.data(alen), e.data(n)
        ct, tag = e.ref(iv, aad, pt)
        assert engine.decrypt_verified(iv, aad, ct, tag) == pt, (it, hex(c0))
        out = np.full(n, SENTINEL, np.uint8)
        assert engine.decrypt_verified(iv, aad, ct, _flip(tag), out=out, raise_on_fail=False) == (None, False)
        assert (out == SENTINEL).all()
        d_ct, d_aad = _t(np.frombuffer(ct, np.uint8)), (_t(np.frombuffer(aad, np.uint8)) if alen else None)
        d_pt = torch.full_like(d_ct, SENTINEL)
        d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
        engine.stream_decrypt_verified_device(iv, d_aad, d_ct, d_pt, _t(np.frombuffer(_flip(tag), np.uint8)), d_ok)
        torch.cuda.synchronize()
        assert int(d_ok.item()) == 0 and bool((d_pt == SENTINEL).all()), (it, hex(c0))
        engine.stream_decrypt_verified_device(iv, d_aad, d_ct, d_pt, _t(np.frombuffer(tag, np.uint8)), d_ok)
        torch.cuda.synchronize()
        assert int(d_ok.item()) == 1 and _h(d_pt) == pt, (it, hex(c0))


@pytest.mark.parametrize("ed", ["enc", "dec"])
def test_gcm_adapter_keystream_window(oracle, ed):
    """The `gcm` adapter fetches keystream in windows of gcm_model._KS_WINDOW bytes from the block a callback needs:
    the wrap and a top-byte carry inside the second window, and the wrap on its first block."""
    from aesgcm_b200 import gcm_model
    rng = np.random.default_rng(7004 + len(ed))
    wb = gcm_model._KS_WINDOW // 16
    for kb, c0, n in ((16, wrap_at(wb + 100), 16 * (wb + 200) + 5), (32, top_carry_at(wb + 7), 16 * (wb + 20)),
                      (24, wrap_at(wb), 16 * (wb + 3) + 1)):
        e = Edge(oracle, rng, kb)
        iv, _ = e.iv(c0)
        aad, text = e.data(20), e.data(n)
        ct, tag = e.ref(iv, aad, text)
        m = gcm_model.gcm({'data': e.key.hex().upper(), 'n_bytes': kb}, {'data': iv.hex().upper(), 'n_bytes': 16}, ed)
        m.load_aad(aad)
        src, want = (text, ct) if ed == "enc" else (ct, text)
        for i in range(0, n, 16):
            (m.load_plain_text if ed == "enc" else m.load_cipher_text)(src[i:i + 16])
        m.get_tag(tag)
        assert b"".join(m.data_out) == want and m.tag == [tag], (kb, hex(c0))


# -------------------------------------------------------------------------------------------------- shared-key batch
# Messages 0..5 of offsets_case (0, 1, 15, 16, 17, 16*7+3 B): the wrap on block 0, 0, 1 (past the ragged end), 0 and
# 1 (ragged), the top-byte carry on block 3.  Messages 6..12 (16*2048+5 B, no AAD but the last): the wrap on block 512
# (a row boundary of every lane group and of the 512-thread CTA), 37 (inside a row) and 2048 (the ragged last block),
# on block 513 (the first of segment 1 of 4, lanes = 1028 / 4100) and the top-byte carry there and on block 1024, the
# byte-13 carry on block 100.  The other messages take IVs of drawn lengths (some 96-bit).
BATCH_J0 = [wrap_at(0), wrap_at(0), wrap_at(1), wrap_at(0), wrap_at(1), top_carry_at(3),
            wrap_at(512), wrap_at(37), wrap_at(513), top_carry_at(513), top_carry_at(1024), byte13_carry_at(100), wrap_at(2048)]


@pytest.fixture(scope="module")
def edge_batches(oracle):
    """An encrypt case and a decrypt case (three tags corrupted: bad_tags, want_ok) of 48 messages each."""
    rng = np.random.default_rng(7100)
    kw = dict(max_len=300, max_aad=40, lens=(16 * 2048 + 5,) * 7, aad_lens=(0,) * 6 + (33,), j0_ctrs=BATCH_J0)
    enc = offsets_case(oracle, rng, 48, 24, decrypt=False, **kw)
    dec = offsets_case(oracle, rng, 48, 24, decrypt=True, **kw)
    dec["bad_tags"], dec["want_ok"] = dec["tags"].copy(), np.ones(48, np.uint8)
    for m in (6, 12, 30):
        dec["bad_tags"][16 * m + 11] ^= 0x02
        dec["want_ok"][m] = 0
    return enc, dec


def _derive(engine, c):
    """k_batch_j0 on the case's raw IVs; the J0 blocks must be exactly the chosen ones."""
    d_j0 = engine.batch_derive_j0_device(_t(c["iv_raw"]), _t(c["iv_off"]))
    assert _h(d_j0) == c["ivs"].tobytes()
    return d_j0


@pytest.mark.parametrize("lanes", [0, 1, 2, 4, 8, 16, 32, 1024, 1028, 4097, 4100])
def test_batch_offsets(engine, edge_batches, lanes):
    """agcm_batch_derive_j0 + agcm_batch_crypt_j0 (encrypt, releasing decrypt) and agcm_batch_decrypt_verified_j0 on
    lane groups, whole CTAs, CTA segments, warps and warp units."""
    import torch
    for c in edge_batches:
        engine.set_key(c["key"])
        d_j0 = _derive(engine, c)
        d_aad, d_aad_off = _t(c["aad"]), _t(c["aad_off"].astype(np.int64))
        d_in, d_in_off = _t(c["data"]), _t(c["in_off"].astype(np.int64))
        n = c["n"]
        out = torch.full_like(d_in, SENTINEL)
        if "bad_tags" not in c:
            tags = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
            engine.batch_crypt_device(0, d_j0, d_aad, d_aad_off, d_in, d_in_off, out, tags, lanes=lanes, j0=True)
            torch.cuda.synchronize()
            assert (out.cpu().numpy() == expect_offsets(c, np.ones(n))).all() and (tags.cpu().numpy() == c["tags"]).all(), lanes
            continue
        ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(1, d_j0, d_aad, d_aad_off, d_in, d_in_off, out, _t(c["bad_tags"]), ok, lanes=lanes, j0=True)
        torch.cuda.synchronize()
        assert (out.cpu().numpy() == expect_offsets(c, np.ones(n))).all(), lanes
        assert (ok.cpu().numpy() == c["want_ok"]).all(), lanes
        if lanes in (1024, 1028):   # the verify-then-release decrypt has no CTA layouts
            continue
        out = torch.full_like(d_in, SENTINEL)
        ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
        engine.batch_decrypt_verified_device(d_j0, d_aad, d_aad_off, d_in, d_in_off, out, _t(c["bad_tags"]), ok, lanes=lanes,
                                             j0=True)
        torch.cuda.synchronize()
        assert (ok.cpu().numpy() == c["want_ok"]).all(), lanes
        assert (out.cpu().numpy() == expect_offsets(c, c["want_ok"])).all(), lanes


@pytest.mark.parametrize("lanes", [0, 2048])
def test_batch_uniform(engine, oracle, lanes):
    """agcm_batch_crypt_uniform_j0 on 1500 B records at a 1504 B pitch (lanes = 2048: the TMA-staged tile kernel) with
    the wrap and the top-byte carry on an even and on an odd block of the record, on its first and on its ragged last
    block; agcm_batch_decrypt_verified_uniform_j0 with corrupted tags."""
    import torch
    rng = np.random.default_rng(7200 + lanes)
    n, length, stride = 64, 1500, 1504
    ctrs = [wrap_at(40), wrap_at(41), top_carry_at(50), top_carry_at(51), wrap_at(0), wrap_at(93), byte13_carry_at(92),
            top_carry_at(0), wrap_at(64), wrap_at(1)]
    e = Edge(oracle, rng, 16)
    engine.set_key(e.key)
    ivs, j0s = zip(*[e.iv(c0) for c0 in ctrs])
    ivs = list(ivs) + [e.data(16) for _ in range(n - len(ctrs))]
    buf = np.frombuffer(e.data(n * stride), np.uint8).copy()
    recs = [buf[m * stride:m * stride + length].tobytes() for m in range(n)]
    want = [e.ref(iv, b"", r) for iv, r in zip(ivs, recs)]
    d_j0 = engine.batch_derive_j0_device(_t(np.frombuffer(b"".join(ivs), np.uint8)), None, 16)
    assert _h(d_j0)[:16 * len(ctrs)] == b"".join(j0s)
    out = torch.full((n * stride,), SENTINEL, dtype=torch.uint8, device="cuda")
    tags = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_uniform_device(0, d_j0, None, 0, 0, _t(buf), out, length, stride, tags, n_msgs=n, lanes=lanes, j0=True)
    torch.cuda.synchronize()
    got, got_tags = out.cpu().numpy().reshape(n, stride), _h(tags)
    for m in range(n):
        assert got[m, :length].tobytes() == want[m][0] and got_tags[16 * m:16 * m + 16] == want[m][1], (lanes, m)
    assert (got[:, length:] == SENTINEL).all()
    if lanes:   # no tile layout for the verify-then-release decrypt
        return
    ctb = np.full(n * stride, 0x3C, np.uint8).reshape(n, stride)
    for m in range(n):
        ctb[m, :length] = np.frombuffer(want[m][0], np.uint8)
    tagb = np.frombuffer(b"".join(w[1] for w in want), np.uint8).copy()
    want_ok = np.ones(n, np.uint8)
    for m in (0, 5, 9, 33):
        tagb[16 * m + 9] ^= 0x08
        want_ok[m] = 0
    out = torch.full((n * stride,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    engine.batch_decrypt_verified_uniform_device(d_j0, None, 0, 0, _t(ctb.reshape(-1)), out, length, stride, _t(tagb), ok,
                                                 n_msgs=n, j0=True)
    torch.cuda.synchronize()
    assert (ok.cpu().numpy() == want_ok).all()
    got = out.cpu().numpy().reshape(n, stride)
    for m in range(n):
        assert got[m, :length].tobytes() == (recs[m] if want_ok[m] else bytes([SENTINEL]) * length), m
    assert (got[:, length:] == SENTINEL).all()


# ------------------------------------------------------------------------------------------------------------ per-key
def test_perkey_byte13_carry(engine, oracle):
    """A per-key batch with a 16*65536+5 B message: its counter (2 + block for a 96-bit IV) carries into byte 13 on
    block 65534, inside one thread's run through the per-key kernel's own counter cache."""
    import torch
    rng = np.random.default_rng(7300)
    kb = 24
    lens = np.array([16 * 65536 + 5, 100, 0, 1500, 16 * 300 + 1])
    alens = np.array([16, 0, 5, 20, 0])
    nm = len(lens)
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    data = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * nm, dtype=np.uint8)
    keys = rng.integers(0, 256, kb * nm, dtype=np.uint8)
    ct, tags = oracle.gcm_batch(keys, kb, False, ivs, aad, aad_off, data, in_off, threads=8)
    out = torch.full((data.size,), SENTINEL, dtype=torch.uint8, device="cuda")
    d_tags = torch.zeros(16 * nm, dtype=torch.uint8, device="cuda")
    args = (_t(keys), _t(ivs), _t(aad), _t(aad_off.astype(np.int64)))
    d_off = _t(in_off.astype(np.int64))
    engine.batch_crypt_perkey_device(8 * kb, 0, *args, _t(data), d_off, out, d_tags)
    torch.cuda.synchronize()
    assert _h(out) == ct.tobytes() and _h(d_tags) == tags.tobytes()
    bad = tags.copy()
    bad[16 * 0 + 4] ^= 0x20
    back = torch.full((data.size,), SENTINEL, dtype=torch.uint8, device="cuda")
    ok = torch.full((nm,), 7, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_perkey_device(8 * kb, 1, *args, _t(ct), d_off, back, _t(bad), ok)
    torch.cuda.synchronize()
    assert _h(back) == data.tobytes() and list(ok.cpu().numpy()) == [0] + [1] * (nm - 1)
