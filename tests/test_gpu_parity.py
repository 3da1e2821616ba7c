"""Parity of the CUDA engine (through the C ABI) against the CPU oracle, the
committed golden fixtures and OpenSSL.  Everything here needs a B200."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def _rb(rng, n):
    return rng.integers(0, 256, n, dtype=np.uint8).tobytes()


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    return torch


def _dev(torch, b):
    a = np.frombuffer(bytes(b), dtype=np.uint8) if not isinstance(b, np.ndarray) else b
    if a.size == 0:
        return torch.empty(0, dtype=torch.uint8, device="cuda")
    return torch.from_numpy(a.copy()).cuda()


# --------------------------------------------------------------------------- keys
def test_key_expand_device_matches_reference_fixtures(engine, torch_mod):
    torch = torch_mod
    fx = _load("key_exp_vectors.json")
    for size, kb in (("128", 16), ("192", 24), ("256", 32)):
        cases = [c for c in fx["cases"] if c["size"] == size]
        keys = np.frombuffer(b"".join(bytes.fromhex(c["key"]) for c in cases), dtype=np.uint8)
        rks = engine.expand_keys_device(int(size), _dev(torch, keys))
        torch.cuda.synchronize()
        got = rks.cpu().numpy()
        for i, c in enumerate(cases):
            assert got[i].tobytes().hex() == c["expanded"], c["key"]
        # host convenience call + the key_exp.py drop-in
        assert engine.expand_key_host(bytes.fromhex(cases[0]["key"])).hex() == cases[0]["expanded"]


def test_key_exp_adapter_signature(engine):
    from aesgcm_b200 import key_exp
    fx = _load("key_exp_vectors.json")
    for c in fx["cases"][:6] + fx["cases"][-6:]:
        out = key_exp.aes_expand_key(c["key"], c["size"])
        assert isinstance(out, list) and bytes(out).hex() == c["expanded"]


def test_set_key_raw_and_preexpanded(engine, oracle):
    rng = np.random.default_rng(21)
    for kb in (16, 24, 32):
        key = _rb(rng, kb)
        engine.set_key(key)
        rk = engine.round_keys()
        assert rk == oracle.key_expand(key)
        h, _ = oracle.h_ej0(rk, bytes(12))
        assert engine.hash_subkey() == h
        engine.set_key(rk)  # pre-expanded stages, used as they are
        assert engine.round_keys() == rk and engine.hash_subkey() == h
        # the same key again keeps H and the tables (src/gcm_ghash.vhd:123-139): no kernel runs;
        # a different key, or the same bytes in the other format, is a new load
        n0 = engine.launch_count
        engine.set_key(rk)
        assert engine.launch_count == n0 and engine.hash_subkey() == h
        iv, pt = _rb(rng, 12), _rb(rng, 100)
        ct1, tag1 = engine.encrypt(iv, b"", pt)
        engine.set_key(key)
        assert engine.launch_count > n0
        ct2, tag2 = engine.encrypt(iv, b"", pt)
        assert (ct1, tag1) == (ct2, tag2) == oracle.gcm_crypt(key, iv, b"", pt)
        other = bytes(b ^ 1 for b in key)
        engine.set_key(other)
        assert engine.encrypt(iv, b"", pt) == oracle.gcm_crypt(other, iv, b"", pt)
    import aesgcm_b200
    with pytest.raises(aesgcm_b200.AgcmError):
        engine.set_key(b"x" * 17)


# --------------------------------------------------------------------------- KATs
def test_known_answer_vectors_host_api(engine):
    for v in _load("kat_vectors.json")["vectors"]:
        key, iv = bytes.fromhex(v["key"]), bytes.fromhex(v["iv"])
        pt, aad = bytes.fromhex(v["pt"]), bytes.fromhex(v["aad"])
        engine.set_key(key)
        ct, tag = engine.encrypt(iv, aad, pt)
        assert ct.hex() == v["ct"] and tag.hex() == v["tag"], v["name"]
        assert engine.decrypt(iv, aad, ct, tag) == pt


def test_committed_openssl_vectors_engine(engine):
    """The engine against the committed OpenSSL-generated fixtures directly (no oracle in the loop)."""
    for v in _load("openssl_random_vectors.json")["vectors"]:
        key, iv, aad, pt = (bytes.fromhex(v[k]) for k in ("key", "iv", "aad", "pt"))
        engine.set_key(key)
        ct, tag = engine.encrypt(iv, aad, pt)
        assert ct.hex() == v["ct"] and tag.hex() == v["tag"]
        assert engine.decrypt(iv, aad, ct, tag) == pt


def test_known_answer_vectors_device_api(engine, torch_mod):
    torch = torch_mod
    for v in _load("kat_vectors.json")["vectors"]:
        key, iv = bytes.fromhex(v["key"]), bytes.fromhex(v["iv"])
        pt, aad = bytes.fromhex(v["pt"]), bytes.fromhex(v["aad"])
        engine.set_key(key)
        d_in, d_aad = _dev(torch, pt), _dev(torch, aad)
        d_out = torch.empty_like(d_in)
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_device(0, iv, d_aad if len(aad) else None, d_in, d_out, d_tag)
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes().hex() == v["ct"], v["name"]
        assert d_tag.cpu().numpy().tobytes().hex() == v["tag"], v["name"]
        # batched path, every lane count
        for lanes in (1, 2, 4, 8, 16, 32):
            n = 3
            ivs = _dev(torch, iv * n)
            data = _dev(torch, pt * n)
            outb = torch.empty_like(data)
            tags = torch.zeros(16 * n, dtype=torch.uint8, device="cuda")
            aadb = _dev(torch, aad * n) if len(aad) else None
            engine.batch_crypt_uniform_device(0, ivs, aadb, len(aad), len(aad), data, outb, len(pt), len(pt), tags,
                                              n_msgs=n, lanes=lanes)
            torch.cuda.synchronize()
            assert outb.cpu().numpy().tobytes().hex() == v["ct"] * n, (v["name"], lanes)
            assert tags.cpu().numpy().tobytes().hex() == v["tag"] * n, (v["name"], lanes)


# ------------------------------------------------------------------- random messages
def _stream_case(eng, oracle, kb, n, alen, rng):
    key, iv, aad, pt = _rb(rng, kb), _rb(rng, 12), _rb(rng, alen), _rb(rng, n)
    eng.set_key(key)
    want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt, threads=8)
    ct, tag = eng.encrypt(iv, aad, pt)
    assert ct == want_ct, (kb, n, alen)
    assert tag == want_tag, (kb, n, alen)
    # decrypt + verify, then reject a flipped ciphertext bit and a flipped tag bit
    assert eng.decrypt(iv, aad, ct, tag) == pt
    if n:
        bad = bytearray(ct)
        bad[n // 2] ^= 0x01
        _, ok = eng.decrypt(iv, aad, bytes(bad), tag, raise_on_fail=False)
        assert not ok
    badtag = bytearray(tag)
    badtag[15] ^= 0x80
    _, ok = eng.decrypt(iv, aad, ct, bytes(badtag), raise_on_fail=False)
    assert not ok


def test_long_iv_vectors_engine(engine, oracle, torch_mod):
    """IVs that are not 96 bits long (agcm_stream_crypt_iv / _iv_host: J0 = GHASH_H(IV || pad || len)
    derived on the device): committed OpenSSL vectors incl. the published McGrew-Viega cases 5, 6,
    11, 12, 17, 18, through the host and the device entry points, decrypt and forged tag."""
    torch = torch_mod
    for v in _load("long_iv_vectors.json")["vectors"]:
        key, iv = bytes.fromhex(v["key"]), bytes.fromhex(v["iv"])
        pt, aad = bytes.fromhex(v["pt"]), bytes.fromhex(v["aad"])
        engine.set_key(key)
        ct, tag = engine.encrypt(iv, aad, pt)
        assert ct.hex() == v["ct"] and tag.hex() == v["tag"], v["name"]
        assert engine.decrypt(iv, aad, ct, tag) == pt
        bad = bytearray(tag)
        bad[0] ^= 1
        assert engine.decrypt(iv, aad, ct, bytes(bad), raise_on_fail=False)[1] is False
        d_in, d_aad = _dev(torch, pt), (_dev(torch, aad) if aad else None)
        d_out = torch.empty_like(d_in)
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_device(0, iv, d_aad, d_in, d_out, d_tag)
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes().hex() == v["ct"] and d_tag.cpu().numpy().tobytes().hex() == v["tag"], v["name"]


def test_long_iv_paths_vs_oracle(engine, engine_small, oracle, torch_mod):
    """IV lengths from 1 byte to several KB (the IV itself spans more than one GHASH row), J0
    counters that wrap 2^32 mid-message are whatever GHASH makes them; messages of several grid
    rows, AAD beyond the inline limit (part + finish path), in place, both directions, both grids.
    A 96-bit IV afterwards still gives the 96-bit result (the J0 counter does not leak)."""
    torch = torch_mod
    rng = np.random.default_rng(96)
    for it, (eng, ivl, n, alen) in enumerate(((engine, 1, 100, 0), (engine, 16, 16 * 151552 + 33, 20),
                                              (engine, 13, 70000, 5000), (engine_small, 60, 640 * 16 * 5 + 7, 16),
                                              (engine_small, 4096 + 5, 3000, 4097), (engine, 20000, 1 << 20, 64),
                                              (engine, 11, 0, 33))):
        kb = (16, 24, 32)[it % 3]
        key, iv, aad, pt = _rb(rng, kb), _rb(rng, ivl), _rb(rng, alen), _rb(rng, n)
        eng.set_key(key)
        want_ct, want_tag = oracle.gcm_crypt_any_iv(key, iv, aad, pt)
        ct, tag = eng.encrypt(iv, aad, pt)
        assert ct == want_ct and tag == want_tag, (it, "host")
        assert eng.decrypt(iv, aad, ct, tag) == pt
        d = _dev(torch, pt) if n else torch.zeros(1, dtype=torch.uint8, device="cuda")
        d_aad = _dev(torch, aad) if alen else None
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        eng.stream_crypt_device(0, iv, d_aad, d, d, d_tag, n_bytes=n)       # in place
        torch.cuda.synchronize()
        assert d[:n].cpu().numpy().tobytes() == want_ct and d_tag.cpu().numpy().tobytes() == want_tag, (it, "device")
        d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
        eng.stream_crypt_device(1, iv, d_aad, d, d, d_tag, d_ok, n_bytes=n)
        torch.cuda.synchronize()
        assert d[:n].cpu().numpy().tobytes() == pt and int(d_ok.item()) == 1, (it, "device dec")
        iv12 = _rb(rng, 12)
        assert eng.encrypt(iv12, aad, pt[:1000]) == oracle.gcm_crypt(key, iv12, aad, pt[:1000]), (it, "96-bit after")


def test_long_iv_shard_gctr_peer_and_batch_paths(engine, oracle, torch_mod):
    """SURVEY 8 f-4 remainder: IVs that are not 96 bits on the counter-range shard calls
    (agcm_stream_part_j0 / _finish_j0), the GCTR half, the peer exchange (world = 1 on this GPU) and
    the batch entry points (agcm_batch_derive_j0 + agcm_batch_crypt_j0), against the oracle."""
    torch = torch_mod
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(97)
    key = _rb(rng, 24)
    engine.set_key(key)
    for ivl, n, alen in ((8, 16 * 151552 * 2 + 5, 20), (33, 5000, 0), (1, 17, 7)):
        iv, aad, pt = _rb(rng, ivl), _rb(rng, alen), rng.integers(0, 256, n, dtype=np.uint8)
        want_ct, want_tag = oracle.gcm_crypt_any_iv(key, iv, aad, pt.tobytes())
        d_in, d_aad = _dev(torch, pt), (_dev(torch, aad) if alen else None)
        for world in (1, 3):
            d_out = torch.zeros_like(d_in)
            parts = torch.zeros((world, 16), dtype=torch.uint8, device="cuda")
            for sh in shard_plan(n, world):
                sl = slice(sh.byte_offset, sh.byte_offset + sh.n_bytes)
                engine.stream_part_device(0, iv, sh.first_block, d_in[sl], d_out[sl], sh.blocks_after, parts[sh.rank],
                                          n_bytes=sh.n_bytes)
            d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
            engine.stream_finish_device(0, iv, parts, world, d_aad, n, d_tag)
            torch.cuda.synchronize()
            assert d_out.cpu().numpy().tobytes() == want_ct and d_tag.cpu().numpy().tobytes() == want_tag, (ivl, world)
        d_back = torch.zeros_like(d_in)
        engine.gctr_device(iv, 0, _dev(torch, np.frombuffer(want_ct, dtype=np.uint8)), d_back)
        torch.cuda.synchronize()
        assert d_back.cpu().numpy().tobytes() == pt.tobytes(), ("gctr", ivl)
        buf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
        engine.peer_setup(0, 1, [buf.data_ptr()])
        d_out = torch.zeros_like(d_in)
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_peer_device(0, iv, 0, d_in, d_out, 0, d_aad, n, d_tag, defer=True)
        engine.peer_join()
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes() == want_ct and d_tag.cpu().numpy().tobytes() == want_tag, ("peer", ivl)
    # batch: every message its own IV length (1 .. 40 bytes, some exactly 12)
    n_msgs = 300
    ivlens = rng.integers(1, 41, n_msgs)
    ivlens[::7] = 12
    lens = rng.integers(0, 900, n_msgs)
    alens = rng.integers(0, 50, n_msgs)
    iv_off = np.concatenate([[0], np.cumsum(ivlens)]).astype(np.int64)
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.int64)
    ivs = rng.integers(0, 256, int(iv_off[-1]), dtype=np.uint8)
    data = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    want = [oracle.gcm_crypt_any_iv(key, ivs[iv_off[i]:iv_off[i + 1]].tobytes(), aad[aad_off[i]:aad_off[i + 1]].tobytes(),
                                    data[in_off[i]:in_off[i + 1]].tobytes()) for i in range(n_msgs)]
    d_j0 = engine.batch_derive_j0_device(_dev(torch, ivs), torch.from_numpy(iv_off).cuda())
    for lanes in (0, 1, 4, 32, 1024, 4097, 4100):
        d_out = torch.zeros(data.size, dtype=torch.uint8, device="cuda")
        d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(0, d_j0, _dev(torch, aad), torch.from_numpy(aad_off).cuda(), _dev(torch, data),
                                  torch.from_numpy(in_off).cuda(), d_out, d_tags, lanes=lanes, j0=True)
        torch.cuda.synchronize()
        out, tags = d_out.cpu().numpy(), d_tags.cpu().numpy()
        for i in range(n_msgs):
            assert out[in_off[i]:in_off[i + 1]].tobytes() == want[i][0], (lanes, i)
            assert tags[16 * i:16 * i + 16].tobytes() == want[i][1], (lanes, i)
    # uniform form with a fixed 16-byte IV
    n_u, length = 64, 1500
    ivs_u = rng.integers(0, 256, 16 * n_u, dtype=np.uint8)
    data_u = rng.integers(0, 256, n_u * length, dtype=np.uint8)
    d_j0 = engine.batch_derive_j0_device(_dev(torch, ivs_u), None, 16)
    d_out = torch.zeros(n_u * length, dtype=torch.uint8, device="cuda")
    d_tags = torch.zeros(16 * n_u, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_uniform_device(0, d_j0, None, 0, 0, _dev(torch, data_u), d_out, length, length, d_tags, n_msgs=n_u, j0=True)
    torch.cuda.synchronize()
    for i in (0, 17, n_u - 1):
        w = oracle.gcm_crypt_any_iv(key, ivs_u[16 * i:16 * i + 16].tobytes(), b"", data_u[i * length:(i + 1) * length].tobytes())
        assert d_out[i * length:(i + 1) * length].cpu().numpy().tobytes() == w[0]
        assert d_tags[16 * i:16 * i + 16].cpu().numpy().tobytes() == w[1]


def test_decrypt_verified_releases_nothing_on_a_bad_tag(engine, oracle, torch_mod):
    """agcm_stream_decrypt_verified(_host): GHASH + tag check first, GCTR gated by the flag.  An
    authentic message decrypts; with one flipped bit in the tag, the ciphertext or the AAD, ok = 0
    and the output buffer keeps its previous contents (device and host forms, chunked sizes, long
    AAD, a non-96-bit IV)."""
    torch = torch_mod
    rng = np.random.default_rng(98)
    for kb, ivl, n, alen in ((32, 12, (40 << 20) + 13, 16), (16, 12, 100, 5000), (24, 20, 16 * 151552 + 1, 0), (16, 12, 0, 9)):
        key, iv, aad, pt = _rb(rng, kb), _rb(rng, ivl), _rb(rng, alen), rng.integers(0, 256, n, dtype=np.uint8)
        engine.set_key(key)
        if n > (1 << 22):
            AESGCM = pytest.importorskip("cryptography.hazmat.primitives.ciphers.aead").AESGCM
            o = AESGCM(key).encrypt(iv, pt.tobytes(), aad)
            ct, tag = o[:-16], o[-16:]
        else:
            ct, tag = oracle.gcm_crypt_any_iv(key, iv, aad, pt.tobytes())
        # host form
        assert engine.decrypt_verified(iv, aad, ct, tag) == pt.tobytes()
        bad_tag = bytes([tag[0] ^ 0x80]) + tag[1:]
        out = np.full(max(n, 1), 0x5A, dtype=np.uint8)
        res, ok = engine.decrypt_verified(iv, aad, ct, bad_tag, out=out[:n], raise_on_fail=False)
        assert ok is False and res is None and (out == 0x5A).all()
        if n:
            bad_ct = bytearray(ct)
            bad_ct[n // 2] ^= 1
            res, ok = engine.decrypt_verified(iv, aad, bytes(bad_ct), tag, out=out[:n], raise_on_fail=False)
            assert ok is False and (out == 0x5A).all()
        with pytest.raises(ValueError):
            engine.decrypt_verified(iv, aad + b"x", ct, tag)
        # device form
        d_ct = _dev(torch, np.frombuffer(ct, dtype=np.uint8)) if n else torch.zeros(1, dtype=torch.uint8, device="cuda")
        d_aad = _dev(torch, aad) if alen else None
        d_pt = torch.full((max(n, 1),), 0x5A, dtype=torch.uint8, device="cuda")
        d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
        engine.stream_decrypt_verified_device(iv, d_aad, d_ct, d_pt, _dev(torch, np.frombuffer(bad_tag, dtype=np.uint8)), d_ok, n_bytes=n)
        torch.cuda.synchronize()
        assert int(d_ok.item()) == 0 and bool((d_pt == 0x5A).all())
        engine.stream_decrypt_verified_device(iv, d_aad, d_ct, d_pt, _dev(torch, np.frombuffer(tag, dtype=np.uint8)), d_ok, n_bytes=n)
        torch.cuda.synchronize()
        assert int(d_ok.item()) == 1 and d_pt[:n].cpu().numpy().tobytes() == pt.tobytes()
        if ivl != 12:
            # device form on a side stream, right behind the encryption that produced its ciphertext there (no
            # synchronise in between): the J0 of the long IV has to be derived in that stream's order
            d_src = _dev(torch, pt)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                d_ct2 = torch.empty_like(d_src)
                d_tag2 = torch.zeros(16, dtype=torch.uint8, device="cuda")
                engine.stream_crypt_device(0, iv, d_aad, d_src, d_ct2, d_tag2)
                d_back = torch.full_like(d_src, 0x5A)
                d_ok2 = torch.zeros(1, dtype=torch.uint8, device="cuda")
                engine.stream_decrypt_verified_device(iv, d_aad, d_ct2, d_back, d_tag2, d_ok2)
            side.synchronize()
            assert int(d_ok2.item()) == 1 and torch.equal(d_back, d_src)


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_stream_random_sizes_vs_oracle(engine, oracle, kb):
    """Default persistent grid (#SMs x 1024): empty, sub-block, ragged, one partial row, >1 row."""
    rng = np.random.default_rng(100 + kb)
    sizes = [0, 1, 15, 16, 17, 31, 32, 33, 1500, 4096, 65536 + 3, 1024 * 151552 // 64 + 7]
    if kb == 32:
        sizes.append(3 * 16 * 151552 + 16 * 5 + 9)   # three rows of the 148 x 1024 grid
    for n in sizes:
        for alen in (0, 16, 20):
            _stream_case(engine, oracle, kb, n, alen, rng)


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_stream_small_odd_grid_vs_oracle(engine_small, oracle, kb):
    """5 x 128 grid (stride 640 blocks): many rows, front padding, counter-cache refills."""
    rng = np.random.default_rng(200 + kb)
    row = 640 * 16
    for n in (1, row - 1, row, row + 1, 3 * row + 89, 17 * row + 5, 256 * row // 5 + 3):
        for alen in (0, 16, 4097):
            _stream_case(engine_small, oracle, kb, n, alen, rng)


@pytest.mark.parametrize("which", ["default", "small"])
def test_stream_unaligned_and_in_place_device_buffers(engine, engine_small, oracle, torch_mod, which):
    """Device pointers at byte offsets 1 / 4 / 8 (byte and 32-bit paths), different in/out
    alignments, and exact in-place operation."""
    torch = torch_mod
    rng = np.random.default_rng(61)
    key, iv, aad = _rb(rng, 32), _rb(rng, 12), _rb(rng, 16)
    if which == "small":
        engine = engine_small
    engine.set_key(key)
    d_aad = _dev(torch, aad)
    for n in ((1, 100, 16 * 151552 + 33) if which == "default" else (100, 640 * 16 * 3 + 5, 640 * 16 * 40 + 33)):
        pt = rng.integers(0, 256, n, dtype=np.uint8)
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt, threads=8)
        for off_in, off_out in ((1, 1), (4, 4), (8, 0), (0, 3), (16, 16)):
            buf_in = torch.zeros(n + 64, dtype=torch.uint8, device="cuda")
            buf_out = torch.full((n + 64,), 0xEE, dtype=torch.uint8, device="cuda")
            buf_in[off_in:off_in + n] = torch.from_numpy(pt).cuda()
            d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
            engine.stream_crypt_device(0, iv, d_aad, buf_in[off_in:off_in + n], buf_out[off_out:off_out + n], d_tag, n_bytes=n)
            torch.cuda.synchronize()
            out = buf_out.cpu().numpy()
            assert out[off_out:off_out + n].tobytes() == want_ct, (n, off_in, off_out)
            assert (out[:off_out] == 0xEE).all() and (out[off_out + n:] == 0xEE).all()   # nothing written outside
            assert d_tag.cpu().numpy().tobytes() == want_tag
        # in place
        buf = torch.from_numpy(pt).cuda()
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_device(0, iv, d_aad, buf, buf, d_tag)
        torch.cuda.synchronize()
        assert buf.cpu().numpy().tobytes() == want_ct and d_tag.cpu().numpy().tobytes() == want_tag
        d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
        engine.stream_crypt_device(1, iv, d_aad, buf, buf, d_tag, d_ok)
        torch.cuda.synchronize()
        assert int(d_ok.item()) == 1 and buf.cpu().numpy().tobytes() == pt.tobytes()


def test_stream_long_aad_paths(engine, oracle):
    # AAD > 4 KiB goes through the grid-wide GHASH-only kernel, AAD <= 4 KiB is folded in the finish kernel
    rng = np.random.default_rng(7)
    key, iv = _rb(rng, 16), _rb(rng, 12)
    engine.set_key(key)
    for alen in (1, 511, 512, 513, 4095, 4096, 4097, 100000 + 1, 16 * 151552 + 3):
        for n in (0, 64, 5000):
            aad, pt = _rb(rng, alen), _rb(rng, n)
            want = oracle.gcm_crypt(key, iv, aad, pt, threads=8)
            assert engine.encrypt(iv, aad, pt) == want, (alen, n)


def test_config1_aes128_4k_messages_vs_oracle_and_openssl(engine, oracle, torch_mod):
    """BASELINE config 1 (SURVEY 8d): AES-128, random 4096 B messages, AAD in {0,16,20,64}."""
    torch = torch_mod
    AESGCM = pytest.importorskip("cryptography.hazmat.primitives.ciphers.aead").AESGCM
    rng = np.random.default_rng(0)
    key = _rb(rng, 16)
    engine.set_key(key)
    n_msgs, length = 10000, 4096   # BASELINE.md 5 row 1: 10 k messages
    for alen in (0, 16, 20, 64):
        ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
        data = rng.integers(0, 256, n_msgs * length, dtype=np.uint8)
        aad = rng.integers(0, 256, max(1, n_msgs * alen), dtype=np.uint8)
        in_off = (np.arange(n_msgs + 1) * length).astype(np.uint64)
        aad_off = (np.arange(n_msgs + 1) * alen).astype(np.uint64)
        want_out, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), 16, True, ivs, aad, aad_off, data, in_off,
                                               threads=8)
        for lanes in ((0, 1, 8, 32) if alen in (0, 20) else (0,)):
            d_out = torch.empty(n_msgs * length, dtype=torch.uint8, device="cuda")
            d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
            engine.batch_crypt_uniform_device(0, _dev(torch, ivs), _dev(torch, aad) if alen else None, alen, alen,
                                              _dev(torch, data), d_out, length, length, d_tags, n_msgs=n_msgs, lanes=lanes)
            torch.cuda.synchronize()
            assert (d_out.cpu().numpy() == want_out).all(), (alen, lanes)
            assert (d_tags.cpu().numpy() == want_tags).all(), (alen, lanes)
        a = AESGCM(key)
        for i in (0, 1, n_msgs - 1):
            ref = a.encrypt(ivs[12 * i:12 * i + 12].tobytes(), data[i * length:(i + 1) * length].tobytes(),
                            aad[i * alen:(i + 1) * alen].tobytes() if alen else None)
            assert ref[:-16] == want_out[i * length:(i + 1) * length].tobytes()
            assert ref[-16:] == want_tags[16 * i:16 * i + 16].tobytes()


@pytest.mark.parametrize("kb", [16, 24, 32])
def test_batch_ragged_offsets_all_lane_counts(engine, oracle, torch_mod, kb):
    """Ragged, unaligned (contiguous) messages incl. empty ones; encrypt, decrypt, corrupted tags."""
    torch = torch_mod
    rng = np.random.default_rng(300 + kb)
    n_msgs = 700
    lens = rng.integers(0, 400, n_msgs)
    lens[:6] = [0, 1, 15, 16, 17, 1500]
    alens = rng.integers(0, 80, n_msgs)
    alens[:4] = [0, 16, 0, 64]
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    data = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    key = _rb(rng, kb)
    rk = oracle.key_expand(key)
    engine.set_key(rk)  # shared PRE-EXPANDED key (config 3 flavour)
    want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), kb, True, ivs, aad, aad_off, data, in_off, threads=8)
    d_ivs, d_aad, d_data = _dev(torch, ivs), _dev(torch, aad), _dev(torch, data)
    d_in_off, d_aad_off = torch.from_numpy(in_off.view(np.int64)).cuda(), torch.from_numpy(aad_off.view(np.int64)).cuda()
    for lanes in (1, 2, 4, 8, 16, 32, 0, 4097, 4099, 4104):
        d_ct = torch.zeros_like(d_data)
        d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(0, d_ivs, d_aad, d_aad_off, d_data, d_in_off, d_ct, d_tags, lanes=lanes, avg_len_hint=200)
        torch.cuda.synchronize()
        assert (d_ct.cpu().numpy() == want_ct).all(), lanes
        assert (d_tags.cpu().numpy() == want_tags).all(), lanes
        # decrypt + verify with 1% corrupted tags
        bad = rng.choice(n_msgs, n_msgs // 100 + 1, replace=False)
        tags_in = want_tags.copy().reshape(n_msgs, 16)
        tags_in[bad, rng.integers(0, 16)] ^= 0x04
        d_pt = torch.zeros_like(d_data)
        d_ok = torch.full((n_msgs,), 7, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(1, d_ivs, d_aad, d_aad_off, d_ct, d_in_off, d_pt, _dev(torch, tags_in.reshape(-1)), d_ok,
                                  lanes=lanes, avg_len_hint=200)
        torch.cuda.synchronize()
        assert (d_pt.cpu().numpy() == data).all(), lanes
        ok = d_ok.cpu().numpy()
        expect = np.ones(n_msgs, np.uint8)
        expect[bad] = 0
        assert (ok == expect).all(), lanes


def test_batch_cta_per_message(engine, oracle, torch_mod):
    """Few long messages: one CTA per message (lanes=1024) or per 1/S of a message (lanes=1024+S:
    counter-range segments, scaled partials XORed by k_batch_split_finish), ragged lengths, AAD
    longer than the payload, messages shorter than S blocks."""
    torch = torch_mod
    rng = np.random.default_rng(77)
    key = _rb(rng, 32)
    engine.set_key(key)
    lens = np.array([0, 5, 16 * 1024, 16 * 1024 * 3 + 7, 200000, 16 * 1024 * 16 + 1, 1 << 20])
    alens = np.array([70000, 0, 16, 20, 0, 64, 300000])
    n_msgs = len(lens)
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    data = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), 32, True, ivs, aad, aad_off, data, in_off, threads=8)
    d_in_off, d_aad_off = torch.from_numpy(in_off.view(np.int64)).cuda(), torch.from_numpy(aad_off.view(np.int64)).cuda()
    d_data, d_aad, d_ivs = _dev(torch, data), _dev(torch, aad), _dev(torch, ivs)
    for lanes in (1024, 0, 32, 1026, 1028, 1032, 1040, 4097, 4098, 4101, 4096 + 64, 4096 + 1000):
        d_ct = torch.zeros_like(d_data)
        d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(0, d_ivs, d_aad, d_aad_off, d_data, d_in_off, d_ct, d_tags, lanes=lanes,
                                  avg_len_hint=int(lens.mean()))
        torch.cuda.synchronize()
        assert (d_ct.cpu().numpy() == want_ct).all(), lanes
        assert (d_tags.cpu().numpy() == want_tags).all(), lanes
        d_pt = torch.zeros_like(d_data)
        d_ok = torch.zeros(n_msgs, dtype=torch.uint8, device="cuda")
        tags_in = want_tags.copy()
        tags_in[16 * 2] ^= 2
        engine.batch_crypt_device(1, d_ivs, d_aad, d_aad_off, d_ct, d_in_off, d_pt, _dev(torch, tags_in), d_ok, lanes=lanes,
                                  avg_len_hint=int(lens.mean()))
        torch.cuda.synchronize()
        assert (d_pt.cpu().numpy() == data).all(), lanes
        assert list(d_ok.cpu().numpy()) == [1, 1, 0, 1, 1, 1, 1], lanes


def test_batch_few_long_messages_auto_split(engine, oracle, torch_mod):
    """The shape the split layout exists for: more long messages than fit one round of CTAs but
    fewer than two (the library picks lanes = 1024 + S on its own).  Uniform layout, in place,
    sampled messages vs the oracle, full decrypt round trip with one corrupted tag."""
    torch = torch_mod
    rng = np.random.default_rng(78)
    key = _rb(rng, 16)
    engine.set_key(key)
    ncta = engine.n_cta
    n_msgs, length, alen = ncta + ncta // 2 + 3, 4 << 20, 48
    gen = torch.Generator(device="cuda")
    gen.manual_seed(78)
    d_pt = torch.randint(0, 256, (n_msgs * length,), dtype=torch.uint8, device="cuda", generator=gen)
    d_iv = torch.randint(0, 256, (n_msgs * 12,), dtype=torch.uint8, device="cuda", generator=gen)
    d_aad = torch.randint(0, 256, (n_msgs * alen,), dtype=torch.uint8, device="cuda", generator=gen)
    d_ct = torch.empty_like(d_pt)
    d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
    before = engine.launch_count
    engine.batch_crypt_uniform_device(0, d_iv, d_aad, alen, alen, d_pt, d_ct, length, length, d_tags, n_msgs=n_msgs)
    torch.cuda.synchronize()
    assert engine.launch_count - before == 1              # k_batch_warp: balanced units, combine and tags in one launch
    for i in (0, 1, n_msgs // 2, n_msgs - 1):
        pt = d_pt[i * length:(i + 1) * length].cpu().numpy().tobytes()
        iv = d_iv[12 * i:12 * i + 12].cpu().numpy().tobytes()
        aad = d_aad[alen * i:alen * (i + 1)].cpu().numpy().tobytes()
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt)
        assert d_ct[i * length:(i + 1) * length].cpu().numpy().tobytes() == want_ct, i
        assert d_tags[16 * i:16 * i + 16].cpu().numpy().tobytes() == want_tag, i
    # the same tags from the unsplit layout
    d_tags1 = torch.zeros_like(d_tags)
    d_ct1 = torch.empty_like(d_pt)
    engine.batch_crypt_uniform_device(0, d_iv, d_aad, alen, alen, d_pt, d_ct1, length, length, d_tags1, n_msgs=n_msgs, lanes=1024)
    torch.cuda.synchronize()
    assert torch.equal(d_tags, d_tags1) and torch.equal(d_ct, d_ct1)
    del d_ct1
    d_tags[16 * 5 + 2] ^= 0x08
    d_ok = torch.zeros(n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_uniform_device(1, d_iv, d_aad, alen, alen, d_ct, d_ct, length, length, d_tags, d_ok, n_msgs=n_msgs)
    torch.cuda.synchronize()
    assert torch.equal(d_ct, d_pt)
    ok = d_ok.cpu().numpy()
    assert ok[5] == 0 and int(ok.sum()) == n_msgs - 1


def test_config3_shape_strided_packets(engine, oracle, torch_mod):
    """BASELINE config 3 shape at reduced count: AES-192, 1500 B packets at a 1504 B stride,
    per-message IV, shared pre-expanded key, no AAD; plus the contiguous 1500 B layout."""
    torch = torch_mod
    rng = np.random.default_rng(2)
    key = _rb(rng, 24)
    engine.set_key(oracle.key_expand(key))
    n_msgs = 4096
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    for stride in (1504, 1500):
        buf = rng.integers(0, 256, n_msgs * stride, dtype=np.uint8)
        in_off = np.arange(n_msgs + 1, dtype=np.uint64) * 1500
        packed = buf.reshape(n_msgs, stride)[:, :1500].reshape(-1).copy()
        want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), 24, True, ivs, None, None, packed, in_off,
                                              threads=8)
        for lanes in (0, 1, 4):
            d_buf = _dev(torch, buf)
            d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
            engine.batch_crypt_uniform_device(0, _dev(torch, ivs), None, 0, 0, d_buf, d_buf, 1500, stride, d_tags,
                                              n_msgs=n_msgs, lanes=lanes)  # in place
            torch.cuda.synchronize()
            got = d_buf.cpu().numpy().reshape(n_msgs, stride)
            assert (got[:, :1500].reshape(-1) == want_ct).all(), (stride, lanes)
            assert (got[:, 1500:] == buf.reshape(n_msgs, stride)[:, 1500:]).all()  # padding untouched
            assert (d_tags.cpu().numpy() == want_tags).all(), (stride, lanes)


def test_batch_split_over_ranks_single_gpu(engine, oracle, torch_mod):
    """SURVEY 8(e) regime 1 (independent messages, no collective): parallel.batch_split hands each
    rank a contiguous message range; the ranks are played one after the other on this GPU, each on
    ITS slice of the buffers (shared-key batch and per-message-key batch, ragged lengths)."""
    torch = torch_mod
    from aesgcm_b200.parallel import batch_split
    rng = np.random.default_rng(77)
    key = _rb(rng, 24)
    n_msgs = 1003
    lens = rng.integers(0, 700, n_msgs)
    alens = rng.integers(0, 40, n_msgs)
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    data = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    keys = rng.integers(0, 256, 32 * n_msgs, dtype=np.uint8)
    want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), 24, True, ivs, aad, aad_off, data, in_off, threads=8)
    wk_ct, wk_tags = oracle.gcm_batch(keys, 32, False, ivs, aad, aad_off, data, in_off, threads=8)
    engine.set_key(key)
    for world in (1, 2, 3, 8):
        got_ct, got_tags = np.zeros_like(data), np.zeros(16 * n_msgs, dtype=np.uint8)
        gk_ct, gk_tags = np.zeros_like(data), np.zeros(16 * n_msgs, dtype=np.uint8)
        for rank in range(world):
            lo, hi = batch_split(n_msgs, world, rank)
            b0, b1 = int(in_off[lo]), int(in_off[hi])
            a0, a1 = int(aad_off[lo]), int(aad_off[hi])
            r_in = _dev(torch, data[b0:b1])
            r_aad = _dev(torch, aad[a0:a1]) if a1 > a0 else torch.zeros(1, dtype=torch.uint8, device="cuda")
            r_inoff = torch.from_numpy((in_off[lo:hi + 1] - in_off[lo]).astype(np.int64)).cuda()
            r_aadoff = torch.from_numpy((aad_off[lo:hi + 1] - aad_off[lo]).astype(np.int64)).cuda()
            r_iv = _dev(torch, ivs[12 * lo:12 * hi])
            r_out = torch.zeros(max(1, b1 - b0), dtype=torch.uint8, device="cuda")
            r_tags = torch.zeros(16 * (hi - lo), dtype=torch.uint8, device="cuda")
            engine.batch_crypt_device(0, r_iv, r_aad, r_aadoff, r_in if b1 > b0 else r_out, r_inoff, r_out, r_tags)
            torch.cuda.synchronize()
            got_ct[b0:b1] = r_out.cpu().numpy()[:b1 - b0]
            got_tags[16 * lo:16 * hi] = r_tags.cpu().numpy()
            r_out.zero_()
            engine.batch_crypt_perkey_device(256, 0, _dev(torch, keys[32 * lo:32 * hi]), r_iv, r_aad, r_aadoff,
                                             r_in if b1 > b0 else r_out, r_inoff, r_out, r_tags)
            torch.cuda.synchronize()
            gk_ct[b0:b1] = r_out.cpu().numpy()[:b1 - b0]
            gk_tags[16 * lo:16 * hi] = r_tags.cpu().numpy()
        assert (got_ct == want_ct).all() and (got_tags == want_tags).all(), world
        assert (gk_ct == wk_ct).all() and (gk_tags == wk_tags).all(), world


def test_batch_tile_tma_staged_records(engine, oracle, torch_mod):
    """k_batch_tile (lanes = 2048): fixed-size records staged through shared memory by 2-D TMA,
    a message per lane.  Record lengths around the 16- and 32-byte tile edges (the out-of-range
    bytes of a box must read as zeros and must not be written back), pitch > length with the
    padding left untouched, message counts that are not a multiple of the 32-message group, AAD,
    every key size, in place, decrypt with corrupted tags, and a non-96-bit IV batch (J0 form)."""
    torch = torch_mod
    rng = np.random.default_rng(123)
    # (key bytes, record length, record pitch, AAD length, AAD pitch, messages); an AAD pitch that is a multiple
    # of 16 sends the AAD through TMA tiles as well, any other pitch reads it in place
    cases = [(16, 1500, 1504, 0, 0, 1000), (24, 1500, 1504, 0, 0, 4097), (32, 1500, 1520, 64, 64, 333), (16, 16, 16, 0, 0, 70),
             (24, 5, 16, 20, 20, 65), (32, 33, 48, 0, 0, 31), (16, 4096, 4096, 16, 16, 129), (32, 31, 32, 7, 7, 200),
             (24, 64, 64, 0, 0, 32), (16, 100, 112, 20, 32, 77), (32, 48, 48, 1000, 1008, 45), (24, 16, 16, 33, 48, 64)]
    for kb, length, stride, alen, astride, n_msgs in cases:
        key = _rb(rng, kb)
        engine.set_key(key)
        ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
        buf = rng.integers(0, 256, n_msgs * stride, dtype=np.uint8)
        aad_buf = rng.integers(0, 256, max(1, n_msgs * astride), dtype=np.uint8)
        aad = aad_buf[:n_msgs * astride].reshape(n_msgs, max(astride, 1))[:, :alen].reshape(-1).copy() if alen else aad_buf
        packed = buf.reshape(n_msgs, stride)[:, :length].reshape(-1).copy()
        in_off = np.arange(n_msgs + 1, dtype=np.uint64) * length
        aad_off = np.arange(n_msgs + 1, dtype=np.uint64) * alen
        want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), kb, True, ivs, aad if alen else None,
                                              aad_off if alen else None, packed, in_off, threads=8)
        d_buf = _dev(torch, buf)
        d_aad = _dev(torch, aad_buf) if alen else None
        d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_uniform_device(0, _dev(torch, ivs), d_aad, alen, astride, d_buf, d_buf, length, stride, d_tags,
                                          n_msgs=n_msgs, lanes=2048)   # in place
        torch.cuda.synchronize()
        got = d_buf.cpu().numpy().reshape(n_msgs, stride)
        assert (got[:, :length].reshape(-1) == want_ct).all(), (kb, length, stride)
        assert (got[:, length:] == buf.reshape(n_msgs, stride)[:, length:]).all(), "padding between records was written"
        assert (d_tags.cpu().numpy() == want_tags).all(), (kb, length, stride)
        # decrypt into a second buffer, 1 tag in 16 corrupted
        tags = want_tags.copy()
        bad = np.arange(0, n_msgs, 16)
        tags[16 * bad + 3] ^= 0x20
        d_pt = torch.full((n_msgs * stride,), 0xEE, dtype=torch.uint8, device="cuda")
        d_ok = torch.full((n_msgs,), 7, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_uniform_device(1, _dev(torch, ivs), d_aad, alen, astride, d_buf, d_pt, length, stride, _dev(torch, tags),
                                          d_ok, n_msgs=n_msgs, lanes=2048)
        torch.cuda.synchronize()
        back = d_pt.cpu().numpy().reshape(n_msgs, stride)
        assert (back[:, :length] == buf.reshape(n_msgs, stride)[:, :length]).all()
        assert (back[:, length:] == 0xEE).all()
        ok = d_ok.cpu().numpy()
        assert (ok[bad] == 0).all() and int(ok.sum()) == n_msgs - bad.size
    # J0 form: 16-byte IVs
    key = _rb(rng, 16)
    engine.set_key(key)
    n_msgs, length = 100, 200
    ivs16 = rng.integers(0, 256, 16 * n_msgs, dtype=np.uint8)
    data = rng.integers(0, 256, n_msgs * 208, dtype=np.uint8)
    d_j0 = engine.batch_derive_j0_device(_dev(torch, ivs16), None, 16)
    d_out = torch.zeros(n_msgs * 208, dtype=torch.uint8, device="cuda")
    d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_uniform_device(0, d_j0, None, 0, 0, _dev(torch, data), d_out, length, 208, d_tags, n_msgs=n_msgs, lanes=2048,
                                      j0=True)
    torch.cuda.synchronize()
    for i in (0, 50, 99):
        w = oracle.gcm_crypt_any_iv(key, ivs16[16 * i:16 * i + 16].tobytes(), b"", data[i * 208:i * 208 + length].tobytes())
        assert d_out[i * 208:i * 208 + length].cpu().numpy().tobytes() == w[0]
        assert d_tags[16 * i:16 * i + 16].cpu().numpy().tobytes() == w[1]
    # an unaligned pitch cannot take this kernel
    with pytest.raises(Exception):
        engine.batch_crypt_uniform_device(0, d_j0, None, 0, 0, _dev(torch, data), d_out, 200, 204, d_tags, n_msgs=10, lanes=2048)


def test_perkey_tile_tma_staged_records(engine, oracle, torch_mod, monkeypatch):
    """k_batch_perkey_tile (distinct key per message, fixed-size records staged by TMA), forced on
    small batches: every key size, ragged record lengths, AAD, message counts off the 32-message
    group, decrypt with corrupted tags, output padding untouched; and the same inputs through the
    thread-per-message kernel give the same bytes."""
    torch = torch_mod
    rng = np.random.default_rng(124)
    for kb, length, stride, alen, n_msgs in ((32, 1500, 1504, 64, 1000), (16, 1500, 1504, 0, 67), (24, 40, 48, 20, 33),
                                             (32, 16, 16, 0, 64), (16, 7, 16, 5, 50), (32, 4096, 4096, 64, 40)):
        keys = rng.integers(0, 256, kb * n_msgs, dtype=np.uint8)
        ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
        buf = rng.integers(0, 256, n_msgs * stride, dtype=np.uint8)
        aad = rng.integers(0, 256, max(1, n_msgs * alen), dtype=np.uint8)
        packed = buf.reshape(n_msgs, stride)[:, :length].reshape(-1).copy()
        in_off = np.arange(n_msgs + 1, dtype=np.uint64) * length
        aad_off = np.arange(n_msgs + 1, dtype=np.uint64) * alen
        want_ct, want_tags = oracle.gcm_batch(keys, kb, False, ivs, aad if alen else None, aad_off if alen else None, packed,
                                              in_off, threads=8)
        d_keys, d_ivs, d_in = _dev(torch, keys), _dev(torch, ivs), _dev(torch, buf)
        d_aad = _dev(torch, aad) if alen else None
        outs = {}
        for tile in ("1", "0"):
            monkeypatch.setenv("AGCM_PERKEY_TILE", tile)
            d_out = torch.full((n_msgs * stride,), 0xEE, dtype=torch.uint8, device="cuda")
            d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
            engine.batch_crypt_perkey_uniform_device(8 * kb, 0, d_keys, d_ivs, d_aad, alen, alen, d_in, d_out, length, stride,
                                                     d_tags, n_msgs=n_msgs)
            torch.cuda.synchronize()
            got = d_out.cpu().numpy().reshape(n_msgs, stride)
            assert (got[:, :length].reshape(-1) == want_ct).all(), (tile, kb, length)
            assert (got[:, length:] == 0xEE).all(), (tile, "padding written")
            assert (d_tags.cpu().numpy() == want_tags).all(), (tile, kb, length)
            outs[tile] = d_out
        monkeypatch.setenv("AGCM_PERKEY_TILE", "1")
        tags = want_tags.copy()
        bad = np.arange(1, n_msgs, 9)
        tags[16 * bad] ^= 1
        d_back = torch.zeros(n_msgs * stride, dtype=torch.uint8, device="cuda")
        d_ok = torch.full((n_msgs,), 9, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_perkey_uniform_device(8 * kb, 1, d_keys, d_ivs, d_aad, alen, alen, outs["1"], d_back, length, stride,
                                                 _dev(torch, tags), d_ok, n_msgs=n_msgs)
        torch.cuda.synchronize()
        assert (d_back.cpu().numpy().reshape(n_msgs, stride)[:, :length] == buf.reshape(n_msgs, stride)[:, :length]).all()
        ok = d_ok.cpu().numpy()
        assert (ok[bad] == 0).all() and int(ok.sum()) == n_msgs - bad.size


def test_batch_bulk_aad_layouts(engine, oracle, torch_mod):
    """Bulk AAD per message (the AAD-heavy end of BASELINE config 5) through every batch layout:
    AAD-only rows run in their own loop with a two-row prefetch when the AAD is 16-byte aligned.
    Ragged AAD tails, AAD that ends mid-row, payload shorter than a row, unaligned AAD pitch,
    uniform (balanced warp units) and offset (ticketed segments) forms."""
    torch = torch_mod
    rng = np.random.default_rng(321)
    for kb, n_msgs, length, alen, astride in ((16, 37, 1000, 16 * 700 + 5, 16 * 701), (32, 9, 16 * 64, 100000, 100000),
                                              (24, 5, 0, 16 * 3000, 16 * 3000), (16, 12, 40, 16 * 96 + 1, 16 * 96 + 3),
                                              (32, 3, 16 * 5000 + 3, 16 * 20000 + 9, 16 * 20001)):
        key = _rb(rng, kb)
        engine.set_key(key)
        stride = (length + 15) & ~15
        ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
        buf = rng.integers(0, 256, max(1, n_msgs * stride), dtype=np.uint8)
        abuf = rng.integers(0, 256, n_msgs * astride, dtype=np.uint8)
        packed = buf[:n_msgs * stride].reshape(n_msgs, max(stride, 1))[:, :length].reshape(-1).copy() if length else np.zeros(0, np.uint8)
        apacked = abuf.reshape(n_msgs, astride)[:, :alen].reshape(-1).copy()
        in_off = np.arange(n_msgs + 1, dtype=np.uint64) * length
        aad_off = np.arange(n_msgs + 1, dtype=np.uint64) * alen
        want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), kb, True, ivs, apacked, aad_off, packed, in_off,
                                              threads=8)
        d_in, d_aad, d_iv = _dev(torch, buf), _dev(torch, abuf), _dev(torch, ivs)
        for lanes in (0, 4, 32, 1024, 1028, 4097, 4096 + 7):
            d_out = torch.zeros_like(d_in)
            d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
            engine.batch_crypt_uniform_device(0, d_iv, d_aad, alen, astride, d_in, d_out, length, stride, d_tags, n_msgs=n_msgs,
                                              lanes=lanes)
            torch.cuda.synchronize()
            if length:
                got = d_out.cpu().numpy()[:n_msgs * stride].reshape(n_msgs, stride)[:, :length].reshape(-1)
                assert (got == want_ct[:n_msgs * length]).all(), (kb, alen, lanes)
            assert (d_tags.cpu().numpy() == want_tags).all(), (kb, alen, lanes)
        # offset form (packed buffers): ticketed segments
        for lanes in (0, 4096 + 3):
            d_out = torch.zeros(max(1, packed.size), dtype=torch.uint8, device="cuda")
            d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
            engine.batch_crypt_device(0, d_iv, _dev(torch, apacked), torch.from_numpy(aad_off.astype(np.int64)).cuda(),
                                      _dev(torch, packed) if length else d_out, torch.from_numpy(in_off.astype(np.int64)).cuda(),
                                      d_out, d_tags, lanes=lanes, avg_len_hint=length + alen // 4)
            torch.cuda.synchronize()
            if length:
                assert (d_out.cpu().numpy()[:packed.size] == want_ct[:packed.size]).all(), (kb, alen, lanes, "offsets")
            assert (d_tags.cpu().numpy() == want_tags).all(), (kb, alen, lanes, "offsets")


def test_batch_ragged_length_sorted(engine, oracle, torch_mod):
    """Offset batches of >= 1024 messages are taken in length order (counting sort on the device, longest
    first) and handed out by ticket: an IMIX-like mix with a few jumbo messages, empty messages and AAD, every
    lane-group width, encrypt and decrypt with corrupted tags -- same bytes as the oracle, message by message."""
    torch = torch_mod
    rng = np.random.default_rng(4242)
    key = _rb(rng, 32)
    engine.set_key(key)
    n_msgs = 3001
    lens = rng.choice([0, 1, 64, 576, 1500, 9000], n_msgs, p=[0.02, 0.03, 0.5, 0.3, 0.13, 0.02])
    lens[7], lens[2999] = 70000, 16 * 4200 + 5          # beyond the last sort bucket
    alens = rng.choice([0, 13, 16, 200], n_msgs)
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    data = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), 32, True, ivs, aad, aad_off, data, in_off, threads=8)
    d_io, d_ao = torch.from_numpy(in_off.view(np.int64)).cuda(), torch.from_numpy(aad_off.view(np.int64)).cuda()
    d_data, d_aad, d_iv = _dev(torch, data), _dev(torch, aad), _dev(torch, ivs)
    for lanes in (0, 1, 2, 8, 32):
        d_out = torch.zeros_like(d_data)
        d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(0, d_iv, d_aad, d_ao, d_data, d_io, d_out, d_tags, lanes=lanes, avg_len_hint=int(lens.mean()))
        torch.cuda.synchronize()
        assert (d_out.cpu().numpy() == want_ct).all(), lanes
        assert (d_tags.cpu().numpy() == want_tags).all(), lanes
        tags_in = want_tags.copy()
        bad = np.arange(3, n_msgs, 97)
        tags_in[16 * bad + 1] ^= 0x04
        d_back = torch.zeros_like(d_data)
        d_ok = torch.full((n_msgs,), 5, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_device(1, d_iv, d_aad, d_ao, d_out, d_io, d_back, _dev(torch, tags_in), d_ok, lanes=lanes,
                                  avg_len_hint=int(lens.mean()))
        torch.cuda.synchronize()
        assert (d_back.cpu().numpy() == data).all(), lanes
        ok = d_ok.cpu().numpy()
        assert (ok[bad] == 0).all() and int(ok.sum()) == n_msgs - bad.size, lanes


def test_batch_slots_per_message_lengths(engine, oracle, torch_mod):
    """agcm_batch_crypt_slots: messages of different lengths in fixed-pitch slots (a packet ring), AAD in slots of its
    own with per-message lengths or one common length; small batches (arrival order) and large ones (length-sorted);
    a length beyond the pitch is clamped; the rest of every slot is left untouched; decrypt with corrupted tags.
    lanes = 2048 names the row-gathering TMA kernel (k_batch_tile<GATHER>: tile::gather4 / scatter4 over the sorted
    order), AGCM_GATHER=1 makes it the default choice for large batches (the last case)."""
    torch = torch_mod
    rng = np.random.default_rng(777)
    for kb, n_msgs, stride, astride, per_msg_aad in ((16, 300, 1504, 64, True), (32, 5000, 2048, 32, False), (24, 2000, 256, 0, False),
                                                     (32, 33, 48, 16, False), (16, 90000, 208, 32, True)):
        key = _rb(rng, kb)
        engine.set_key(key)
        lens = rng.choice([0, 1, 15, 16, 17, 31, 32, 33, 64, 100, 576, 1500, stride - 1, stride], n_msgs).astype(np.uint32)
        lens = np.minimum(lens, stride).astype(np.uint32)
        alens = (rng.integers(0, astride + 1, n_msgs) if per_msg_aad else np.full(n_msgs, astride // 2)).astype(np.uint32)
        ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
        buf = rng.integers(0, 256, n_msgs * stride, dtype=np.uint8)
        abuf = rng.integers(0, 256, max(1, n_msgs * astride), dtype=np.uint8)
        in_off = np.concatenate([[0], np.cumsum(lens.astype(np.int64))]).astype(np.uint64)
        aad_off = np.concatenate([[0], np.cumsum(alens.astype(np.int64))]).astype(np.uint64)
        packed = np.concatenate([buf[i * stride:i * stride + lens[i]] for i in range(n_msgs)] + [np.zeros(0, np.uint8)])
        apacked = np.concatenate([abuf[i * astride:i * astride + alens[i]] for i in range(n_msgs)] + [np.zeros(0, np.uint8)])
        want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), kb, True, ivs, apacked if astride else None,
                                              aad_off if astride else None, packed, in_off, threads=8)
        d_len = torch.from_numpy(lens.astype(np.int32)).cuda()
        d_len_over = d_len.clone()
        d_len_over[lens == stride] = stride + 999            # clamped to the pitch by the kernel
        d_alen = torch.from_numpy(alens.astype(np.int32)).cuda() if per_msg_aad else None
        d_in, d_aad = _dev(torch, buf), (_dev(torch, abuf) if astride else None)
        col = np.arange(stride)[None, :]
        inside = col < lens[:, None].astype(np.int64)
        want = np.full((n_msgs, stride), 0x3C, dtype=np.uint8)
        want[inside] = want_ct
        for lanes in (0, 1, 4, 32, 2048, "gather"):
            d_out = torch.full((n_msgs * stride,), 0x3C, dtype=torch.uint8, device="cuda")
            d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
            if lanes == "gather":
                os.environ["AGCM_GATHER"] = "1"      # the A/B switch: large aligned batches take the gathering kernel by default
            try:
                n0 = engine.launch_count
                engine.batch_crypt_slots_device(0, _dev(torch, ivs), d_aad, d_alen, astride // 2, astride, d_in, d_out, d_len_over, stride,
                                                d_tags, lanes=0 if lanes == "gather" else lanes, avg_len_hint=int(lens.mean()))
                n_launch = engine.launch_count - n0
            finally:
                os.environ.pop("AGCM_GATHER", None)
            torch.cuda.synchronize()
            if lanes == 2048 or (lanes == "gather" and n_msgs >= 148 * 512):
                assert n_launch == (4 if n_msgs >= 64 else 1), (lanes, n_launch)     # length sort (3) + one k_batch_tile<GATHER>
            got = d_out.cpu().numpy().reshape(n_msgs, stride)
            bad_rows = np.nonzero((got != want).any(axis=1))[0]
            assert bad_rows.size == 0, (kb, lanes, bad_rows[:5], lens[bad_rows[:5]])   # ciphertext, and the slot padding untouched
            assert (d_tags.cpu().numpy() == want_tags).all(), (kb, lanes)
        tags_in = want_tags.copy()
        bad = np.arange(1, n_msgs, 53)
        tags_in[16 * bad + 15] ^= 0x80
        d_back = torch.zeros(n_msgs * stride, dtype=torch.uint8, device="cuda")
        d_ok = torch.full((n_msgs,), 3, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_slots_device(1, _dev(torch, ivs), d_aad, d_alen, astride // 2, astride, d_out, d_back, d_len, stride,
                                        _dev(torch, tags_in), d_ok, avg_len_hint=int(lens.mean()))
        torch.cuda.synchronize()
        back = d_back.cpu().numpy().reshape(n_msgs, stride)
        for i in range(0, n_msgs, 7):
            assert back[i, :lens[i]].tobytes() == buf[i * stride:i * stride + lens[i]].tobytes(), i
        ok = d_ok.cpu().numpy()
        assert (ok[bad] == 0).all() and int(ok.sum()) == n_msgs - bad.size


def test_batch_host_api_roundtrip(engine, oracle):
    rng = np.random.default_rng(9)
    key = _rb(rng, 32)
    engine.set_key(key)
    n_msgs, length, stride, alen = 3000, 1500, 1504, 64
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    data = rng.integers(0, 256, n_msgs * stride, dtype=np.uint8)
    aad = rng.integers(0, 256, n_msgs * alen, dtype=np.uint8)
    out = data.copy()
    tags = np.zeros(16 * n_msgs, np.uint8)
    engine.crypt_batch_uniform_host(0, ivs, aad, alen, alen, data, out, length, stride, tags)
    in_off = np.arange(n_msgs + 1, dtype=np.uint64) * length
    aad_off = np.arange(n_msgs + 1, dtype=np.uint64) * alen
    packed = data.reshape(n_msgs, stride)[:, :length].reshape(-1).copy()
    want_ct, want_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), 32, True, ivs, aad, aad_off, packed, in_off, threads=8)
    assert (out.reshape(n_msgs, stride)[:, :length].reshape(-1) == want_ct).all()
    assert (tags == want_tags).all()
    back = out.copy()
    ok = np.zeros(n_msgs, np.uint8)
    tags[16 * 5] ^= 1
    engine.crypt_batch_uniform_host(1, ivs, aad, alen, alen, out, back, length, stride, tags, ok)
    assert (back.reshape(n_msgs, stride)[:, :length] == data.reshape(n_msgs, stride)[:, :length]).all()
    assert ok.sum() == n_msgs - 1 and ok[5] == 0
    # long records through the host pipeline: several chunks in flight on the library's streams at once, one CTA per
    # message inside each (the chunks must not share a work ticket)
    n_msgs, length = 700, 128 * 1024
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    data = rng.integers(0, 256, n_msgs * length, dtype=np.uint8)
    out = np.zeros_like(data)
    tags = np.zeros(16 * n_msgs, np.uint8)
    engine.crypt_batch_uniform_host(0, ivs, None, 0, 0, data, out, length, length, tags, lanes=1024)
    AESGCM = pytest.importorskip("cryptography.hazmat.primitives.ciphers.aead").AESGCM
    a = AESGCM(key)
    for i in list(range(0, n_msgs, 37)) + [n_msgs - 1]:
        ref = a.encrypt(ivs[12 * i:12 * i + 12].tobytes(), data[i * length:(i + 1) * length].tobytes(), None)
        assert ref[:-16] == out[i * length:(i + 1) * length].tobytes() and ref[-16:] == tags[16 * i:16 * i + 16].tobytes(), i


def test_perkey_ragged_length_sorted(engine, oracle, torch_mod):
    """A key per message AND a length per message (the reference's regression runs: every test has its own random key,
    IV, AAD and payload sizes, tb/gcm_testbench.py:25-39): from 1024 messages on the per-key kernel takes the messages
    in length order (perm[] from the device sort).  Encrypt vs the oracle, decrypt with corrupted tags, every key size;
    the unsorted order (AGCM_NO_LEN_SORT) gives the same bytes."""
    torch = torch_mod
    rng = np.random.default_rng(4242)
    for kb, nm in ((32, 3000), (16, 1024), (24, 1500)):
        lens = rng.choice([0, 1, 16, 64, 100, 576, 1500, 4000], nm)
        alens = rng.integers(0, 70, nm)
        in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
        msg = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
        aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
        ivs = rng.integers(0, 256, 12 * nm, dtype=np.uint8)
        keys = rng.integers(0, 256, kb * nm, dtype=np.uint8)
        w_ct, w_tags = oracle.gcm_batch(keys, kb, False, ivs, aad, aad_off, msg, in_off, decrypt=False, threads=8)
        d_io, d_ao = torch.from_numpy(in_off.view(np.int64)).cuda(), torch.from_numpy(aad_off.view(np.int64)).cuda()
        d_keys, d_iv, d_aad, d_msg = _dev(torch, keys), _dev(torch, ivs), _dev(torch, aad), _dev(torch, msg)
        for nosort in (False, True):
            if nosort:
                os.environ["AGCM_NO_LEN_SORT"] = "1"
            try:
                d_ct = torch.zeros(msg.size + 16, dtype=torch.uint8, device="cuda")
                d_tags = torch.zeros(16 * nm, dtype=torch.uint8, device="cuda")
                n0 = engine.launch_count
                engine.batch_crypt_perkey_device(kb * 8, 0, d_keys, d_iv, d_aad, d_ao, d_msg, d_io, d_ct, d_tags)
                torch.cuda.synchronize()
                assert engine.launch_count - n0 == (1 if nosort else 4)      # 3 sort launches + the kernel
            finally:
                os.environ.pop("AGCM_NO_LEN_SORT", None)
            assert (d_ct.cpu().numpy()[:msg.size] == w_ct).all(), (kb, nosort)
            assert (d_ct.cpu().numpy()[msg.size:] == 0).all()
            assert (d_tags.cpu().numpy() == w_tags).all(), (kb, nosort)
        tags_in = w_tags.copy()
        bad = np.arange(3, nm, 97)
        tags_in[16 * bad] ^= 1
        d_back = torch.zeros(msg.size, dtype=torch.uint8, device="cuda")
        d_ok = torch.full((nm,), 7, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_perkey_device(kb * 8, 1, d_keys, d_iv, d_aad, d_ao, d_ct[:msg.size], d_io, d_back, _dev(torch, tags_in), d_ok)
        torch.cuda.synchronize()
        assert (d_back.cpu().numpy() == msg).all()
        ok = d_ok.cpu().numpy()
        assert (ok[bad] == 0).all() and int(ok.sum()) == nm - bad.size


def test_config4_perkey_decrypt_verify(engine, oracle, torch_mod):
    """BASELINE config 4 semantics at reduced count: AES-256 decrypt+verify, a DISTINCT key per
    message expanded on the device, 64 B AAD, payload swept over {64, 256, 1500, 4096} B, some tags
    corrupted; plus the other key sizes and ragged offsets; encrypt leg vs the oracle."""
    torch = torch_mod
    rng = np.random.default_rng(3)
    for kb, length, alen, n_msgs in ((32, 1500, 64, 3000), (32, 64, 64, 2000), (32, 256, 64, 2000), (32, 4096, 64, 600),
                                     (16, 1500, 0, 1500), (24, 333, 20, 1500)):
        keys = rng.integers(0, 256, kb * n_msgs, dtype=np.uint8)
        ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
        pt = rng.integers(0, 256, n_msgs * length, dtype=np.uint8)
        aad = rng.integers(0, 256, max(1, n_msgs * alen), dtype=np.uint8)
        in_off = np.arange(n_msgs + 1, dtype=np.uint64) * length
        aad_off = np.arange(n_msgs + 1, dtype=np.uint64) * alen
        want_ct, want_tags = oracle.gcm_batch(keys, kb, False, ivs, aad, aad_off, pt, in_off, threads=8)
        d_keys, d_ivs, d_pt = _dev(torch, keys), _dev(torch, ivs), _dev(torch, pt)
        d_aad = _dev(torch, aad) if alen else None
        d_ct = torch.zeros_like(d_pt)
        d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_perkey_uniform_device(kb * 8, 0, d_keys, d_ivs, d_aad, alen, alen, d_pt, d_ct, length, length,
                                                 d_tags, n_msgs=n_msgs)
        torch.cuda.synchronize()
        assert (d_ct.cpu().numpy() == want_ct).all(), (kb, length)
        assert (d_tags.cpu().numpy() == want_tags).all(), (kb, length)
        bad = rng.choice(n_msgs, max(1, n_msgs // 1000 + 2), replace=False)
        tags_in = want_tags.copy().reshape(n_msgs, 16)
        tags_in[bad, 3] ^= 0x40
        d_back = torch.zeros_like(d_pt)
        d_ok = torch.full((n_msgs,), 9, dtype=torch.uint8, device="cuda")
        engine.batch_crypt_perkey_uniform_device(kb * 8, 1, d_keys, d_ivs, d_aad, alen, alen, d_ct, d_back, length, length,
                                                 _dev(torch, tags_in.reshape(-1)), d_ok, n_msgs=n_msgs)
        torch.cuda.synchronize()
        assert (d_back.cpu().numpy() == pt).all()
        expect = np.ones(n_msgs, np.uint8)
        expect[bad] = 0
        assert (d_ok.cpu().numpy() == expect).all()
    # ragged offsets
    n_msgs = 500
    lens = rng.integers(0, 300, n_msgs)
    alens = rng.integers(0, 70, n_msgs)
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
    keys = rng.integers(0, 256, 32 * n_msgs, dtype=np.uint8)
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    pt = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
    aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
    want_ct, want_tags = oracle.gcm_batch(keys, 32, False, ivs, aad, aad_off, pt, in_off, threads=8)
    d_ct = torch.zeros(pt.size, dtype=torch.uint8, device="cuda")
    d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_perkey_device(256, 0, _dev(torch, keys), _dev(torch, ivs), _dev(torch, aad),
                                     torch.from_numpy(aad_off.view(np.int64)).cuda(), _dev(torch, pt),
                                     torch.from_numpy(in_off.view(np.int64)).cuda(), d_ct, d_tags)
    torch.cuda.synchronize()
    assert (d_ct.cpu().numpy() == want_ct).all() and (d_tags.cpu().numpy() == want_tags).all()


def test_config4_full_size_roundtrip(engine, oracle, torch_mod):
    """BASELINE config 4 at full size: 2^20 messages x 1500 B, distinct AES-256 key each, 64 B AAD.
    Inputs for the decrypt come from the engine's own (parity-checked) encrypt; 0.1 % of the tags
    are corrupted and the ok flags must say exactly which; sampled messages vs the oracle."""
    torch = torch_mod
    n_msgs, length, alen = 1 << 20, 1500, 64
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    d_keys = torch.randint(0, 256, (n_msgs * 32,), dtype=torch.uint8, device="cuda", generator=gen)
    d_ivs = torch.randint(0, 256, (n_msgs * 12,), dtype=torch.uint8, device="cuda", generator=gen)
    d_aad = torch.randint(0, 256, (n_msgs * alen,), dtype=torch.uint8, device="cuda", generator=gen)
    d_pt = torch.randint(0, 256, (n_msgs * length,), dtype=torch.uint8, device="cuda", generator=gen)
    d_ct = torch.zeros_like(d_pt)
    d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_perkey_uniform_device(256, 0, d_keys, d_ivs, d_aad, alen, alen, d_pt, d_ct, length, length, d_tags,
                                             n_msgs=n_msgs)
    torch.cuda.synchronize()
    for i in (0, 7, 99999, n_msgs - 1):
        key = d_keys[32 * i:32 * i + 32].cpu().numpy().tobytes()
        iv = d_ivs[12 * i:12 * i + 12].cpu().numpy().tobytes()
        aad = d_aad[alen * i:alen * (i + 1)].cpu().numpy().tobytes()
        pt = d_pt[length * i:length * (i + 1)].cpu().numpy().tobytes()
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt)
        assert d_ct[length * i:length * (i + 1)].cpu().numpy().tobytes() == want_ct, i
        assert d_tags[16 * i:16 * i + 16].cpu().numpy().tobytes() == want_tag, i
    rng = np.random.default_rng(3)
    bad = np.sort(rng.choice(n_msgs, n_msgs // 1000, replace=False))
    d_tags_in = d_tags.clone()
    d_tags_in.view(n_msgs, 16)[torch.from_numpy(bad).cuda(), 0] ^= 1
    d_back = torch.zeros_like(d_pt)
    d_ok = torch.zeros(n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_perkey_uniform_device(256, 1, d_keys, d_ivs, d_aad, alen, alen, d_ct, d_back, length, length,
                                             d_tags_in, d_ok, n_msgs=n_msgs)
    torch.cuda.synchronize()
    assert torch.equal(d_back, d_pt)
    ok = d_ok.cpu().numpy()
    assert int(ok.sum()) == n_msgs - bad.size and (ok[bad] == 0).all()


# ------------------------------------------------------------ shards (one GPU, k parts)
def test_counter_range_shards_combine(engine, oracle, torch_mod):
    """SURVEY 8(e) regime 2 on one GPU: k counter-range shards + XOR of pre-scaled partials."""
    torch = torch_mod
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(31)
    key, iv, aad = _rb(rng, 32), _rb(rng, 12), _rb(rng, 16)
    engine.set_key(key)
    for n in (0, 100, 16 * 1000, 5 * 16 * 151552 + 11):
        pt = rng.integers(0, 256, n, dtype=np.uint8)
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt, threads=8)
        d_in = _dev(torch, pt)
        for world in (1, 2, 4, 8):
            d_out = torch.zeros_like(d_in)
            parts = torch.zeros((world, 16), dtype=torch.uint8, device="cuda")
            for s in shard_plan(n, world):
                sl = slice(s.byte_offset, s.byte_offset + s.n_bytes)
                engine.stream_part_device(0, iv, s.first_block, d_in[sl], d_out[sl], s.blocks_after, parts[s.rank],
                                          n_bytes=s.n_bytes)
            d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
            engine.stream_finish_device(0, iv, parts, world, _dev(torch, aad), n, d_tag)
            torch.cuda.synchronize()
            assert d_out.cpu().numpy().tobytes() == want_ct, (n, world)
            assert d_tag.cpu().numpy().tobytes() == want_tag, (n, world)


def test_peer_exchange_single_gpu_emulation(engine_lib, oracle, torch_mod):
    """agcm_stream_crypt_peer on ONE GPU: world = 1 (own buffer), and world = 2 emulated with two
    contexts, two exchange buffers and two streams on the same device.  The bulk kernels only POST;
    the one-warp finishes wait on the contexts' side streams.  Covers the synchronous and the
    deferred form, more messages than the ring holds, and an empty counter range."""
    torch = torch_mod
    import aesgcm_b200
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(88)
    key, iv, aad = _rb(rng, 32), _rb(rng, 12), _rb(rng, 20)
    d_aad = _dev(torch, aad)
    # world = 1
    e0 = aesgcm_b200.GcmEngine(0)
    e0.set_key(key)
    buf0 = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    e0.peer_setup(0, 1, [buf0.data_ptr()])
    for n in (5, 16 * 151552 + 3):
        pt = rng.integers(0, 256, n, dtype=np.uint8)
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt, threads=8)
        d_in = _dev(torch, pt)
        d_out = torch.zeros_like(d_in)
        d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
        for rep in range(11):   # epochs wrap the 8-deep ring
            e0.stream_crypt_peer_device(0, iv, 0, d_in, d_out, 0, d_aad, n, d_tag, defer=bool(rep & 1))
        e0.peer_join()
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes() == want_ct and d_tag.cpu().numpy().tobytes() == want_tag
        assert not e0.peer_timed_out()
    # world = 2 on one device
    e1 = aesgcm_b200.GcmEngine(0)
    e1.set_key(key)
    buf1 = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    ptrs = [buf0.data_ptr(), buf1.data_ptr()]
    e0.peer_setup(0, 2, ptrs)
    e1.peer_setup(1, 2, ptrs)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for n in (9, 16 * 100 + 7, 4 * 16 * 151552 + 11):   # 9 B: one block, rank 1's range is empty
        pt = rng.integers(0, 256, n, dtype=np.uint8)
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt, threads=8)
        d_in = _dev(torch, pt)
        for dec in (0, 1):
            for defer in (False, True):
                src = d_in if not dec else _dev(torch, np.frombuffer(want_ct, dtype=np.uint8))
                d_out = torch.zeros_like(d_in)
                tags = [torch.zeros(16, dtype=torch.uint8, device="cuda") for _ in range(2)]
                oks = [torch.zeros(1, dtype=torch.uint8, device="cuda") for _ in range(2)]
                if dec:
                    for t in tags:
                        t.copy_(torch.from_numpy(np.frombuffer(want_tag, dtype=np.uint8).copy()))
                torch.cuda.synchronize()
                plan = shard_plan(n, 2)
                for rep in range(3 if defer else 1):
                    for r, (eng, st) in enumerate(zip((e0, e1), streams)):
                        sh = plan[r]
                        sl = slice(sh.byte_offset, sh.byte_offset + sh.n_bytes)
                        eng.stream_crypt_peer_device(dec, iv, sh.first_block, src[sl] if sh.n_bytes else None,
                                                     d_out[sl] if sh.n_bytes else None, sh.blocks_after, d_aad, n, tags[r],
                                                     oks[r], n_bytes=sh.n_bytes, stream=st, defer=defer)
                for eng, st in zip((e0, e1), streams):
                    eng.peer_join(st)
                torch.cuda.synchronize()
                assert not e0.peer_timed_out() and not e1.peer_timed_out()
                assert d_out.cpu().numpy().tobytes() == (pt.tobytes() if dec else want_ct), (n, dec, defer)
                if dec:
                    assert int(oks[0].item()) == 1 and int(oks[1].item()) == 1
                else:
                    assert tags[0].cpu().numpy().tobytes() == want_tag and tags[1].cpu().numpy().tobytes() == want_tag
    e0.close()
    e1.close()


def test_peer_exchange_fails_closed_on_missing_rank(engine_lib, oracle, torch_mod, monkeypatch):
    """world = 2 but rank 1 never calls: rank 0's finish gives up after the timeout, ZEROES the tag
    (a tag built from an incomplete XOR must never leave the engine), clears ok, and every later
    peer call returns AGCM_E_PEER_TIMEOUT until the exchange is set up again."""
    torch = torch_mod
    import aesgcm_b200
    monkeypatch.setenv("AGCM_PEER_TIMEOUT_MS", "200")
    rng = np.random.default_rng(89)
    key, iv = _rb(rng, 16), _rb(rng, 12)
    e0 = aesgcm_b200.GcmEngine(0)
    e0.set_key(key)
    bufs = [torch.zeros(4096, dtype=torch.uint8, device="cuda") for _ in range(2)]
    e0.peer_setup(0, 2, [b.data_ptr() for b in bufs])
    n = 4096
    d_in = _dev(torch, rng.integers(0, 256, n, dtype=np.uint8))
    d_out = torch.zeros_like(d_in)
    d_tag = torch.full((16,), 0xAA, dtype=torch.uint8, device="cuda")
    d_ok = torch.ones(1, dtype=torch.uint8, device="cuda")
    e0.stream_crypt_peer_device(1, iv, 0, d_in, d_out, n // 16, None, 2 * n, d_tag, d_ok)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 0
    assert e0.peer_timed_out()
    with pytest.raises(aesgcm_b200.AgcmError) as ei:
        e0.stream_crypt_peer_device(0, iv, 0, d_in, d_out, n // 16, None, 2 * n, d_tag)
    assert ei.value.rc == aesgcm_b200._lib.E_PEER_TIMEOUT
    # encrypt side of the same failure: the tag that comes back is all zero, not a partial XOR
    e0.peer_setup(0, 2, [b.data_ptr() for b in bufs])
    e0.stream_crypt_peer_device(0, iv, 0, d_in, d_out, n // 16, None, 2 * n, d_tag)
    torch.cuda.synchronize()
    assert d_tag.cpu().numpy().tobytes() == bytes(16)
    assert e0.peer_timed_out()
    e0.close()


def _peer_worker(rank, world, port, q):
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    import aesgcm_b200
    from aesgcm_b200.parallel import PeerExchange, shard_plan
    from oracle import cpu_oracle as o
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    rng = np.random.default_rng(5)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    iv = rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
    aad = rng.integers(0, 256, 16, dtype=np.uint8)
    n = 3 * 16 * 151552 + 5
    pt = rng.integers(0, 256, n, dtype=np.uint8)
    eng = aesgcm_b200.GcmEngine(rank)
    eng.set_key(key)
    px = PeerExchange(eng)
    sh = shard_plan(n, world)[rank]
    dev = torch.device("cuda", rank)
    d_in = torch.from_numpy(pt[sh.byte_offset:sh.byte_offset + sh.n_bytes].copy()).to(dev)
    d_out = torch.zeros_like(d_in)
    d_tag = torch.zeros(16, dtype=torch.uint8, device=dev)
    d_aad = torch.from_numpy(aad).to(dev)
    for rep in range(12):
        px.crypt(0, iv, d_aad, sh, d_in, d_out, n, d_tag, defer=rep >= 4)
    px.join()
    torch.cuda.synchronize()
    want_ct, want_tag = o.gcm_crypt(key, iv, aad.tobytes(), pt, threads=4)
    ok = (d_out.cpu().numpy().tobytes() == want_ct[sh.byte_offset:sh.byte_offset + sh.n_bytes]
          and d_tag.cpu().numpy().tobytes() == want_tag and not eng.peer_timed_out())
    # host-buffer form of the same exchange
    h_out = np.zeros(sh.n_bytes, dtype=np.uint8)
    tag_h = px.crypt_host(0, iv, aad, sh, pt[sh.byte_offset:sh.byte_offset + sh.n_bytes].copy(), h_out, n)
    ok = ok and tag_h == want_tag and h_out.tobytes() == want_ct[sh.byte_offset:sh.byte_offset + sh.n_bytes]
    # regime 1: independent messages split over the ranks (parallel.batch_split), no collective
    from aesgcm_b200.parallel import batch_split
    n_msgs, length = 4001, 1500
    ivs = rng.integers(0, 256, 12 * n_msgs, dtype=np.uint8)
    msgs = rng.integers(0, 256, n_msgs * length, dtype=np.uint8)
    lo, hi = batch_split(n_msgs, world, rank)
    b_in = torch.from_numpy(msgs[lo * length:hi * length].copy()).to(dev)
    b_out = torch.zeros_like(b_in)
    b_tags = torch.zeros(16 * (hi - lo), dtype=torch.uint8, device=dev)
    eng.batch_crypt_uniform_device(0, torch.from_numpy(ivs[12 * lo:12 * hi].copy()).to(dev), None, 0, 0, b_in, b_out, length,
                                   length, b_tags, n_msgs=hi - lo)
    torch.cuda.synchronize()
    off = (np.arange(hi - lo + 1) * length).astype(np.uint64)
    w_ct, w_tags = o.gcm_batch(np.frombuffer(key, dtype=np.uint8), 32, True, ivs[12 * lo:12 * hi], None, None,
                               msgs[lo * length:hi * length], off, threads=4)
    ok = ok and (b_out.cpu().numpy() == w_ct).all() and (b_tags.cpu().numpy() == w_tags).all()
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


def test_peer_exchange_two_gpus(engine_lib, torch_mod):
    """Real NVLink peer-memory exchange: 2 processes, 2 GPUs, torch symmetric memory buffers."""
    torch = torch_mod
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_peer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
    assert res == [(0, True), (1, True)]


def test_gctr_and_ghash_halves(engine, oracle, torch_mod):
    torch = torch_mod
    rng = np.random.default_rng(41)
    key, iv = _rb(rng, 24), _rb(rng, 12)
    engine.set_key(key)
    rk = oracle.key_expand(key)
    h, _ = oracle.h_ej0(rk, iv)
    for n in (1, 16, 1000, 70000 + 5):
        data = _rb(rng, n)
        d_in = _dev(torch, data)
        d_out = torch.empty_like(d_in)
        for first_block in (0, 5, 2 ** 32 - 2 - (n + 15) // 16):
            engine.gctr_device(iv, first_block, d_in, d_out)
            torch.cuda.synchronize()
            assert d_out.cpu().numpy().tobytes() == oracle.gctr(rk, iv, 2 + first_block, data)
        y = torch.zeros(16, dtype=torch.uint8, device="cuda")
        engine.ghash_device(d_in, y)
        torch.cuda.synchronize()
        assert y.cpu().numpy().tobytes() == oracle.ghash_absorb(h, data)


def test_counter_overflow_rejected(engine, torch_mod):
    torch = torch_mod
    import aesgcm_b200
    engine.set_key(bytes(16))
    buf = torch.zeros(64, dtype=torch.uint8, device="cuda")
    part = torch.zeros(16, dtype=torch.uint8, device="cuda")
    with pytest.raises(aesgcm_b200.AgcmError) as ei:
        engine.stream_part_device(0, bytes(12), 2 ** 32 - 3, buf, buf, 0, part)  # 4 blocks from 2^32-3: past 2^32-2
    assert ei.value.rc == aesgcm_b200._lib.E_COUNTER_OVERFLOW
    with pytest.raises(aesgcm_b200.AgcmError):
        aesgcm_b200.GcmEngine(0).encrypt(bytes(12), b"", b"abc")  # no key


def test_fuzz_all_paths(engine, engine_small, oracle, torch_mod):
    """Seeded fuzz over every device entry point: random key size, direction, lengths, AAD lengths,
    byte alignment, lane counts, shard position (incl. counters that wrap 2^32)."""
    torch = torch_mod
    # soak runs: AGCM_FUZZ_SEED / AGCM_FUZZ_ITERS override the committed seed and length
    rng = np.random.default_rng(int(os.environ.get("AGCM_FUZZ_SEED", "2026")))
    for it in range(int(os.environ.get("AGCM_FUZZ_ITERS", "60"))):
        eng = engine if it % 2 else engine_small
        kb = int(rng.choice([16, 24, 32]))
        key, iv = _rb(rng, kb), _rb(rng, 12)
        eng.set_key(key if it % 3 else oracle.key_expand(key))
        rk = oracle.key_expand(key)
        h, _ = oracle.h_ej0(rk, iv)
        dec = int(rng.integers(0, 2))
        # --- one shard at a random position of a long message
        n = int(rng.choice([0, 1, 16, 17, 255, 4096, 40000, 640 * 16 * 3 + 7]))
        n -= n % 16 if it % 4 == 0 else 0
        first_block = int(rng.choice([0, 1, 255, 2 ** 24 - 3, 2 ** 32 - 2 - (n + 15) // 16 - 7]))
        after = 0 if n % 16 else int(rng.choice([0, 1, 5]))
        off = int(rng.integers(0, 9))
        data = rng.integers(0, 256, n, dtype=np.uint8)
        buf_in = torch.zeros(n + 32, dtype=torch.uint8, device="cuda")
        buf_in[off:off + n] = torch.from_numpy(data).cuda()
        buf_out = torch.zeros(n + 32, dtype=torch.uint8, device="cuda")
        part = torch.zeros(16, dtype=torch.uint8, device="cuda")
        eng.stream_part_device(dec, iv, first_block, buf_in[off:off + n], buf_out[off:off + n], after, part, n_bytes=n)
        torch.cuda.synchronize()
        want = oracle.gctr(rk, iv, 2 + first_block, data.tobytes())
        assert buf_out[off:off + n].cpu().numpy().tobytes() == want, (it, "gctr")
        ct = data.tobytes() if dec else want
        want_part = oracle.gfmul(oracle.gf_pow(h, after), oracle.ghash_absorb(h, ct))
        assert part.cpu().numpy().tobytes() == want_part, (it, "partial")
        # --- a small ragged batch
        nm = int(rng.integers(1, 40))
        lens = rng.integers(0, 5000, nm) if it % 5 else rng.integers(0, 40, nm)
        alens = rng.integers(0, 100, nm)
        in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        aad_off = np.concatenate([[0], np.cumsum(alens)]).astype(np.uint64)
        msg = rng.integers(0, 256, int(in_off[-1]), dtype=np.uint8)
        aad = rng.integers(0, 256, int(aad_off[-1]), dtype=np.uint8)
        ivs = rng.integers(0, 256, 12 * nm, dtype=np.uint8)
        w_out, w_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), kb, True, ivs, aad, aad_off, msg, in_off,
                                         decrypt=False, threads=8)
        lanes = int(rng.choice([0, 1, 2, 4, 8, 16, 32, 1024, 1026, 1032, 4097, 4098, 4096 + 5, 4096 + 64]))
        d_out = torch.zeros(max(1, msg.size), dtype=torch.uint8, device="cuda")
        d_tags = torch.zeros(16 * nm, dtype=torch.uint8, device="cuda")
        d_io, d_ao = torch.from_numpy(in_off.view(np.int64)).cuda(), torch.from_numpy(aad_off.view(np.int64)).cuda()
        src = _dev(torch, msg) if msg.size else torch.zeros(1, dtype=torch.uint8, device="cuda")
        d_aadb = _dev(torch, aad) if aad.size else torch.zeros(1, dtype=torch.uint8, device="cuda")
        eng.batch_crypt_device(0, _dev(torch, ivs), d_aadb, d_ao, src, d_io, d_out, d_tags, lanes=lanes, avg_len_hint=int(lens.mean()))
        torch.cuda.synchronize()
        assert (d_out.cpu().numpy()[:msg.size] == w_out).all(), (it, "batch ct", lanes)
        assert (d_tags.cpu().numpy() == w_tags).all(), (it, "batch tag", lanes)
        # --- the same messages, each under its own key, decrypt + verify
        keys = rng.integers(0, 256, kb * nm, dtype=np.uint8)
        p_out, p_tags = oracle.gcm_batch(keys, kb, False, ivs, aad, aad_off, msg, in_off, decrypt=False, threads=8)
        d_back = torch.zeros_like(d_out)
        d_ok = torch.zeros(nm, dtype=torch.uint8, device="cuda")
        bad = int(rng.integers(0, nm))
        tags_in = p_tags.copy()
        tags_in[16 * bad + 7] ^= 0x08
        eng.batch_crypt_perkey_device(kb * 8, 1, _dev(torch, keys), _dev(torch, ivs), d_aadb, d_ao,
                                      _dev(torch, p_out) if p_out.size else src, d_io, d_back, _dev(torch, tags_in), d_ok)
        torch.cuda.synchronize()
        assert (d_back.cpu().numpy()[:msg.size] == msg).all(), (it, "perkey pt")
        exp = np.ones(nm, np.uint8)
        exp[bad] = 0
        assert (d_ok.cpu().numpy() == exp).all(), (it, "perkey ok")
        # --- slots: a pitch (16-byte aligned or not), a length per message, AAD of one length or one per message; lane
        #     groups, the length-sorted classes (from 1024 messages) and the row-gathering TMA kernel
        nm = int(rng.choice([1, 3, 33, 200, 1100]))
        aligned = bool(it % 3)
        stride = int(rng.choice([16, 48, 208, 1504])) if aligned else int(rng.choice([1, 7, 100, 1500]))
        astride = int(rng.choice([0, 16, 48])) if aligned else int(rng.choice([0, 5, 20]))
        per_msg_aad = bool(astride and it % 2)
        lens = rng.integers(0, stride + 1, nm).astype(np.uint32)
        alens = (rng.integers(0, astride + 1, nm) if per_msg_aad else np.full(nm, astride // 2)).astype(np.uint32)
        ivs = rng.integers(0, 256, 12 * nm, dtype=np.uint8)
        buf = rng.integers(0, 256, nm * stride, dtype=np.uint8)
        abuf = rng.integers(0, 256, max(1, nm * astride), dtype=np.uint8)
        in_off = np.concatenate([[0], np.cumsum(lens.astype(np.int64))]).astype(np.uint64)
        aad_off = np.concatenate([[0], np.cumsum(alens.astype(np.int64))]).astype(np.uint64)
        inside = np.arange(stride)[None, :] < lens[:, None].astype(np.int64)
        ainside = np.arange(max(astride, 1))[None, :] < alens[:, None].astype(np.int64)
        packed = buf.reshape(nm, stride)[inside]
        apacked = abuf[:nm * astride].reshape(nm, astride)[ainside[:, :astride]] if astride else None
        s_ct, s_tags = oracle.gcm_batch(np.frombuffer(key, dtype=np.uint8), kb, True, ivs, apacked, aad_off if astride else None,
                                        packed, in_off, threads=8)
        want_slots = np.full((nm, stride), 0x5D, dtype=np.uint8)
        want_slots[inside] = s_ct
        lanes = int(rng.choice([0, 1, 2, 8, 2048] if aligned else [0, 1, 2, 8]))
        d_out = torch.full((nm * stride,), 0x5D, dtype=torch.uint8, device="cuda")
        d_tags = torch.zeros(16 * nm, dtype=torch.uint8, device="cuda")
        eng.batch_crypt_slots_device(0, _dev(torch, ivs), _dev(torch, abuf) if astride else None,
                                     torch.from_numpy(alens.astype(np.int32)).cuda() if per_msg_aad else None, astride // 2, astride,
                                     _dev(torch, buf), d_out, torch.from_numpy(lens.astype(np.int32)).cuda(), stride, d_tags, lanes=lanes)
        torch.cuda.synchronize()
        assert (d_out.cpu().numpy().reshape(nm, stride) == want_slots).all(), (it, "slots ct / padding", lanes, stride, astride, nm)
        assert (d_tags.cpu().numpy() == s_tags).all(), (it, "slots tag", lanes, stride, astride, nm)
        # --- fixed-size records: every uniform layout (lane groups, TMA tiles, balanced warp units, CTA segments),
        #     96-bit IVs or 1..40-byte IVs through the J0 form, shared key and key per message
        if eng is engine:
            nm = int(rng.integers(1, 150))
            length = int(rng.choice([1, 15, 16, 17, 100, 1500, 4096, 16 * 700 + 3]))
            alen = int(rng.choice([0, 0, 5, 16, 64, 16 * 300 + 9]))
            stride = ((length + 15) & ~15) + 16 * int(rng.integers(0, 3))
            astride = ((alen + 15) & ~15) if it % 2 else alen
            ivl = 12 if it % 3 else int(rng.integers(1, 41))
            ivs = rng.integers(0, 256, ivl * nm, dtype=np.uint8)
            buf = rng.integers(0, 256, nm * stride, dtype=np.uint8)
            abuf = rng.integers(0, 256, max(1, nm * astride), dtype=np.uint8)
            want = [oracle.gcm_crypt_any_iv(key, ivs[ivl * i:ivl * (i + 1)].tobytes(), abuf[astride * i:astride * i + alen].tobytes(),
                                            buf[stride * i:stride * i + length].tobytes()) for i in range(nm)]
            d_iv = _dev(torch, ivs) if ivl == 12 else eng.batch_derive_j0_device(_dev(torch, ivs), None, ivl)
            lanes = int(rng.choice([0, 2, 8, 2048, 4097, 1024, 1028]))
            d_out = torch.full((nm * stride,), 0x77, dtype=torch.uint8, device="cuda")
            d_tags = torch.zeros(16 * nm, dtype=torch.uint8, device="cuda")
            eng.batch_crypt_uniform_device(0, d_iv, _dev(torch, abuf) if alen else None, alen, astride, _dev(torch, buf), d_out, length,
                                           stride, d_tags, n_msgs=nm, lanes=lanes, j0=ivl != 12)
            torch.cuda.synchronize()
            got, tg = d_out.cpu().numpy().reshape(nm, stride), d_tags.cpu().numpy()
            for i in range(nm):
                assert got[i, :length].tobytes() == want[i][0], (it, "uniform ct", lanes, length, alen, ivl, i)
                assert tg[16 * i:16 * i + 16].tobytes() == want[i][1], (it, "uniform tag", lanes, length, alen, ivl, i)
            assert (got[:, length:] == 0x77).all(), (it, "uniform padding", lanes)
            if ivl == 12:   # key per message, thread-per-message and TMA-tiled kernels
                keys = rng.integers(0, 256, kb * nm, dtype=np.uint8)
                wantk = [oracle.gcm_crypt(keys[kb * i:kb * (i + 1)].tobytes(), ivs[12 * i:12 * i + 12].tobytes(),
                                          abuf[astride * i:astride * i + alen].tobytes(), buf[stride * i:stride * i + length].tobytes())
                         for i in range(nm)]
                for tile in ("0", "1"):
                    os.environ["AGCM_PERKEY_TILE"] = tile
                    try:
                        d_out.fill_(0x77)
                        eng.batch_crypt_perkey_uniform_device(kb * 8, 0, _dev(torch, keys), d_iv, _dev(torch, abuf) if alen else None, alen,
                                                              astride, _dev(torch, buf), d_out, length, stride, d_tags, n_msgs=nm)
                        torch.cuda.synchronize()
                    finally:
                        del os.environ["AGCM_PERKEY_TILE"]
                    got, tg = d_out.cpu().numpy().reshape(nm, stride), d_tags.cpu().numpy()
                    for i in range(nm):
                        assert got[i, :length].tobytes() == wantk[i][0], (it, "perkey uniform ct", tile, length, alen, i)
                        assert tg[16 * i:16 * i + 16].tobytes() == wantk[i][1], (it, "perkey uniform tag", tile, length, alen, i)
                    assert (got[:, length:] == 0x77).all(), (it, "perkey uniform padding", tile)


def test_plain_c_client(engine_lib, tmp_path):
    """tests/abi_example.c: a gcc-only C99 program drives the C ABI (802.1AE vector of README.md:251)."""
    import shutil
    import subprocess
    import aesgcm_b200
    from conftest import ROOT
    gcc = shutil.which("gcc")
    if not gcc:
        pytest.skip("gcc not available")
    pkg = os.path.dirname(aesgcm_b200._lib.SO_PATH)
    exe = str(tmp_path / "abi_example")
    subprocess.check_call([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "abi_example.c"), "-L", pkg, "-laesgcm_b200", "-Wl,-rpath," + pkg,
                           "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "abi_example ok" in out.stdout, out.stdout + out.stderr


def test_error_codes(engine_lib, torch_mod):
    """Return-code contract of the C ABI (include/aesgcm_b200.h): never throws, negative codes."""
    torch = torch_mod
    import ctypes
    import aesgcm_b200
    L = engine_lib
    E = aesgcm_b200._lib
    ctx = ctypes.c_void_p()
    assert L.agcm_ctx_create_ex(ctypes.byref(ctx), 0, 300, 1024) == E.E_BAD_ARG      # > 256 CTAs
    assert L.agcm_ctx_create_ex(ctypes.byref(ctx), 0, 8, 96) == E.E_BAD_ARG          # threads not a power of two
    assert L.agcm_ctx_create_ex(ctypes.byref(ctx), 99, 0, 0) == E.E_NO_DEVICE
    assert L.agcm_ctx_create(ctypes.byref(ctx), 0) == 0
    buf = torch.zeros(64, dtype=torch.uint8, device="cuda")
    iv = (ctypes.c_uint8 * 12)()
    ivp = ctypes.addressof(iv)
    # no key yet
    assert L.agcm_stream_crypt(ctx, 0, ivp, 0, 0, buf.data_ptr(), buf.data_ptr(), 64, buf.data_ptr(), 0, 0) == E.E_NO_KEY
    assert L.agcm_gctr(ctx, ivp, 0, buf.data_ptr(), buf.data_ptr(), 64, 0) == E.E_NO_KEY
    assert L.agcm_get_h(ctx, buf.data_ptr()) == E.E_NO_KEY
    key = (ctypes.c_uint8 * 32)()
    kp = ctypes.addressof(key)
    assert L.agcm_set_key(ctx, 200, 0, kp, 25) == E.E_BAD_MODE
    assert L.agcm_set_key(ctx, 256, 0, kp, 16) == E.E_BAD_MODE                        # key/mode mismatch
    assert L.agcm_set_key(ctx, 128, 1, kp, 16) == E.E_BAD_MODE                        # pre-expanded needs 176 B
    assert L.agcm_set_key(ctx, 256, 0, kp, 32) == 0
    assert L.agcm_key_expand(ctx, 100, buf.data_ptr(), 1, buf.data_ptr(), 0) == E.E_BAD_MODE
    # decrypt needs the ok flag; null data with a length; shard rules
    assert L.agcm_stream_crypt(ctx, 1, ivp, 0, 0, buf.data_ptr(), buf.data_ptr(), 64, buf.data_ptr(), 0, 0) == E.E_BAD_ARG
    assert L.agcm_stream_crypt(ctx, 0, ivp, 0, 0, 0, 0, 64, buf.data_ptr(), 0, 0) == E.E_BAD_ARG
    assert L.agcm_stream_crypt(ctx, 0, ivp, 0, 5, buf.data_ptr(), buf.data_ptr(), 64, buf.data_ptr(), 0, 0) == E.E_BAD_ARG
    assert L.agcm_stream_part(ctx, 0, ivp, 0, buf.data_ptr(), buf.data_ptr(), 60, 3, buf.data_ptr(), 0) == E.E_BAD_LEN   # ragged non-last shard
    assert L.agcm_stream_part(ctx, 0, ivp, 2 ** 32, buf.data_ptr(), buf.data_ptr(), 64, 0, buf.data_ptr(), 0) == E.E_COUNTER_OVERFLOW
    assert L.agcm_batch_crypt_uniform(ctx, 0, 3, buf.data_ptr(), 0, 0, 0, buf.data_ptr(), buf.data_ptr(), 16, 16,
                                      buf.data_ptr(), 0, 2, 0) == E.E_BAD_ARG                                         # lanes = 3
    assert L.agcm_batch_crypt_uniform(ctx, 0, 0, buf.data_ptr(), 0, 0, 0, buf.data_ptr(), buf.data_ptr(), 32, 16,
                                      buf.data_ptr(), 0, 2, 0) == E.E_BAD_LEN                                         # stride < len
    assert L.agcm_batch_crypt_perkey_uniform(ctx, 64, 0, buf.data_ptr(), buf.data_ptr(), 0, 0, 0, buf.data_ptr(),
                                             buf.data_ptr(), 16, 16, buf.data_ptr(), 0, 1, 0) == E.E_BAD_MODE
    # AAD blocks + payload blocks + the length block must fit the 32-bit index of the unified sequence
    big = 16 * (2 ** 31)
    assert L.agcm_batch_crypt_uniform(ctx, 0, 0, buf.data_ptr(), buf.data_ptr(), big, big, buf.data_ptr(), buf.data_ptr(), big, big,
                                      buf.data_ptr(), 0, 1, 0) == E.E_COUNTER_OVERFLOW
    assert L.agcm_batch_crypt_perkey_uniform(ctx, 256, 0, buf.data_ptr(), buf.data_ptr(), buf.data_ptr(), big, big, buf.data_ptr(),
                                             buf.data_ptr(), big, big, buf.data_ptr(), 0, 1, 0) == E.E_COUNTER_OVERFLOW
    assert L.agcm_peer_join(ctx, 0) == E.E_BAD_ARG                                                                     # no peer_setup yet
    assert L.agcm_strerror(E.E_NO_KEY) == b"no key set"
    assert b"peer" in L.agcm_strerror(E.E_PEER_TIMEOUT)
    torch.cuda.synchronize()
    L.agcm_ctx_destroy(ctx)


# ------------------------------------------------------- the gcm_model.py drop-in surface
@pytest.mark.parametrize("ed", ["enc", "dec"])
def test_gcm_model_adapter_streaming_callbacks(oracle, ed):
    """Drives the adapter exactly like tb/gcm_test.py:76-94 / tb/gcm_sequencer.py:137-231:
    <=16-byte callbacks, AAD first, output available right after each call, tag at the end."""
    from aesgcm_b200 import gcm_model
    rng = np.random.default_rng(55)
    for kb, n, alen in ((16, 48, 28), (32, 0, 68), (24, 1000 + 7, 5), (32, 70000, 0)):
        key, iv, aad, text = _rb(rng, kb), _rb(rng, 12), _rb(rng, alen), _rb(rng, n)
        want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, text)
        src = text if ed == "enc" else want_ct
        want_out = want_ct if ed == "enc" else text
        m = gcm_model.gcm({'data': key.hex().upper(), 'n_bytes': kb}, {'data': iv.hex().upper(), 'n_bytes': 12}, ed)
        for i in range(0, alen, 16):
            m.load_aad(aad[i:i + 16])
        for i in range(0, n, 16):
            blk = src[i:i + 16]
            (m.load_plain_text if ed == "enc" else m.load_cipher_text)(blk)
            assert m.data_out[-1] == want_out[i:i + 16]          # available immediately
        m.get_tag(want_tag)
        assert b"".join(m.data_out) == want_out
        assert m.tag == [want_tag]
    if ed == "dec":  # forced mismatch path (tb/gcm_model.py:47-51): inverted received tag is appended
        m = gcm_model.gcm({'data': key.hex(), 'n_bytes': kb}, {'data': iv.hex(), 'n_bytes': 12}, 'dec')
        m.load_cipher_text(want_ct[:16])
        wrong = bytes(16)
        m.get_tag(wrong)
        assert m.tag == [bytes([0xFF] * 16)]


def test_gcm_model_adapter_long_iv_and_shared_engine(oracle):
    """tb/gcm_model.py:14-18 passes icb['n_bytes'] bytes of nonce to pycryptodome, whatever the
    length: the adapter takes them too (prefetched keystream from inc32(J0)).  Two models with
    different keys interleave their callbacks on the module's shared engine."""
    from aesgcm_b200 import gcm_model
    rng = np.random.default_rng(56)
    cases = []
    for kb, ivl, n, alen in ((16, 8, 100, 20), (32, 64, 70000 + 3, 0)):
        key, iv, aad, text = _rb(rng, kb), _rb(rng, ivl), _rb(rng, alen), _rb(rng, n)
        want_ct, want_tag = oracle.gcm_crypt_any_iv(key, iv, aad, text)
        m = gcm_model.gcm({'data': key.hex().upper(), 'n_bytes': kb}, {'data': iv.hex().upper(), 'n_bytes': ivl}, 'enc')
        cases.append((m, aad, text, want_ct, want_tag))
    assert cases[0][0].model is cases[1][0].model          # one engine for both
    for m, aad, _, _, _ in cases:
        for i in range(0, len(aad), 16):
            m.load_aad(aad[i:i + 16])
    for i in range(0, max(len(c[2]) for c in cases), 16):    # interleaved, block by block
        for m, _, text, want_ct, _ in cases:
            if i < len(text):
                m.load_plain_text(text[i:i + 16])
                assert m.data_out[-1] == want_ct[i:i + 16]
    for m, _, _, want_ct, want_tag in cases:
        m.get_tag(want_tag)
        assert b"".join(m.data_out) == want_ct and m.tag == [want_tag]


def test_adapter_reproduces_reference_model_traces():
    """The drop-in `gcm` class against traces of the reference's own tb/gcm_model.py: identical
    data_out lists (element by element) and identical tag lists in all three flows."""
    from aesgcm_b200 import gcm_model
    for c in _load("gcm_model_traces.json")["cases"]:
        aad, pt = bytes.fromhex(c["aad"]), bytes.fromhex(c["pt"])
        m = gcm_model.gcm(c["key"], c["iv"], 'enc')
        for i in range(0, len(aad), 16):
            m.load_aad(aad[i:i + 16])
        for i in range(0, len(pt), 16):
            m.load_plain_text(pt[i:i + 16])
        m.get_tag(bytes(16))
        assert [x.hex() for x in m.data_out] == c["enc_data_out"] and [t.hex() for t in m.tag] == c["enc_tag"]
        ct = b"".join(m.data_out)
        for label in ("dec_good", "dec_bad"):
            d = gcm_model.gcm(c["key"], c["iv"], 'dec')
            for i in range(0, len(aad), 16):
                d.load_aad(aad[i:i + 16])
            for i in range(0, len(ct), 16):
                d.load_cipher_text(ct[i:i + 16])
            d.get_tag(bytes.fromhex(c[label]["rx_tag"]))
            assert [x.hex() for x in d.data_out] == c[label]["data_out"], label
            assert [t.hex() for t in d.tag] == c[label]["tag"], label


def test_adapter_without_prefetch_matches(oracle):
    """prefetch=False: every callback is its own device GCTR call (no host-side XOR); odd call sizes."""
    from aesgcm_b200 import gcm_model
    rng = np.random.default_rng(66)
    key, iv, aad, pt = _rb(rng, 24), _rb(rng, 12), _rb(rng, 30), _rb(rng, 200)
    want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt)
    for prefetch in (False, True):
        m = gcm_model.gcm({'data': key.hex(), 'n_bytes': 24}, {'data': iv.hex(), 'n_bytes': 12}, 'enc', prefetch=prefetch)
        m.load_aad(aad)
        pos = 0
        for step in (16, 16, 5, 11, 16, 1, 40, 95):          # byte-granular streaming like pycryptodome's encrypt()
            m.load_plain_text(pt[pos:pos + step])
            assert m.data_out[-1] == want_ct[pos:pos + step]
            pos += step
        assert pos == len(pt)
        m.get_tag(want_tag)
        assert m.tag == [want_tag]


def test_readme_vectors_through_adapter():
    """The two command lines of README.md:251,257 (802.1AE vectors), via the model surface."""
    from aesgcm_b200 import gcm_model
    v = [x for x in _load("kat_vectors.json")["vectors"] if "802.1AE" in x["name"]]
    assert len(v) == 2
    for x in v:
        key, pt, aad = x["key"], bytes.fromhex(x["pt"]), bytes.fromhex(x["aad"])
        m = gcm_model.gcm({'data': key, 'n_bytes': len(key) // 2}, {'data': x["iv"], 'n_bytes': 12}, 'enc')
        for i in range(0, len(aad), 16):
            m.load_aad(aad[i:i + 16])
        for i in range(0, len(pt), 16):
            m.load_plain_text(pt[i:i + 16])
        m.get_tag(bytes.fromhex(x["tag"]))
        assert b"".join(m.data_out).hex() == x["ct"] and m.tag[0].hex() == x["tag"]


def test_recorded_configs_replay_through_cuda_model(oracle):
    """SURVEY 8(f) row 2: reference test configurations (tb/tmp/<seed>.json shape) replayed against
    the CUDA-backed model with no cocotb, incl. RANDOM stimulus, the decrypt flow and the
    pre-expanded-key flow; outputs equal the oracle's."""
    from aesgcm_b200 import gcm_model, key_exp, stimulus as st
    cfg = {'seed': 1, 'aes_mode': '256', 'key': '691D3EE909D7F54167FD1CA0B5D769081F2BDE1AEE655FDBAB80BD5295AE6BE7',
           'iv': 'F0761E8DCD3D000176D457ED', 'data': 'EMPTY', 'enc_dec': 'enc', 'max_n_byte': 4095,
           'aad': 'E20106D7CD0DF0761E8DCD3D88E5400076D457ED08000F101112131415161718191A1B1C1D1E1F202122232425262728292A2B2C2D2E2F303132333435363738393A0003'}
    r = st.replay(cfg, gcm_model.gcm)
    assert r['tag'].hex().upper() == '35217C774BBC31B63166BCF9D4ABED07' and r['ct_words'] == []   # README.md:257
    for seed in range(6):
        c = {'seed': 100 + seed, 'aes_mode': 'ALL', 'key': 'RANDOM', 'iv': 'RANDOM', 'aad': 'RANDOM', 'data': 'RANDOM',
             'enc_dec': 'dec' if seed % 2 else 'enc', 'max_n_byte': 4095}
        r = st.replay(c, gcm_model.gcm, pre_expanded=(seed % 3 == 0), expand_key=key_exp.aes_expand_key)
        key = bytes.fromhex(r['data']['key']['data'])
        iv = bytes.fromhex(r['data']['iv']['data'])
        want_ct, want_tag = oracle.gcm_crypt(key, iv, b"".join(r['aad_words']), b"".join(r['pt_words']))
        assert b"".join(r['ct_words']) == want_ct and r['tag'] == want_tag
        if c['enc_dec'] == 'dec':
            assert b"".join(r['dec_words']) == b"".join(r['pt_words']) and r['dec_tag'] == want_tag


# --------------------------------------------------------------- full-size properties
def test_config2_full_size_stream_properties(engine, oracle, torch_mod):
    """BASELINE config 2 at full size (AES-256, 2^30 B, 16 B AAD, default_rng(1)): too big for the
    bit-serial oracle, so: (1) windows of CT vs the oracle's GCTR at the matching counter, (2) the
    tag vs the sharded combine (8 parts) -- two different decompositions must agree, (3) decrypt
    round-trips and verifies, a flipped bit is rejected, (4) OpenSSL computes the same tag."""
    torch = torch_mod
    rng = np.random.default_rng(1)
    key, iv, aad = _rb(rng, 32), _rb(rng, 12), _rb(rng, 16)
    n = 1 << 30
    engine.set_key(key)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    d_pt = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=gen)
    d_ct = torch.empty_like(d_pt)
    d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
    d_aad = _dev(torch, aad)
    engine.stream_crypt_device(0, iv, d_aad, d_pt, d_ct, d_tag)
    torch.cuda.synchronize()
    rk = oracle.key_expand(key)
    for off in (0, 16 * 151552 - 32, n // 2 - 48, n - 4096):
        w = 4096
        pt_w = d_pt[off:off + w].cpu().numpy().tobytes()
        assert d_ct[off:off + w].cpu().numpy().tobytes() == oracle.gctr(rk, iv, 2 + off // 16, pt_w), off
    from aesgcm_b200.parallel import shard_plan
    parts = torch.zeros((8, 16), dtype=torch.uint8, device="cuda")
    d_ct2 = torch.empty_like(d_pt)
    for s in shard_plan(n, 8):
        sl = slice(s.byte_offset, s.byte_offset + s.n_bytes)
        engine.stream_part_device(0, iv, s.first_block, d_pt[sl], d_ct2[sl], s.blocks_after, parts[s.rank])
    d_tag2 = torch.zeros(16, dtype=torch.uint8, device="cuda")
    engine.stream_finish_device(0, iv, parts, 8, d_aad, n, d_tag2)
    torch.cuda.synchronize()
    assert torch.equal(d_ct, d_ct2) and torch.equal(d_tag, d_tag2)
    del d_ct2
    d_back = torch.empty_like(d_pt)
    d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
    engine.stream_crypt_device(1, iv, d_aad, d_ct, d_back, d_tag, d_ok)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 1 and torch.equal(d_back, d_pt)
    d_ct[n // 3] ^= 0x20
    engine.stream_crypt_device(1, iv, d_aad, d_ct, d_back, d_tag, d_ok)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 0
    d_ct[n // 3] ^= 0x20
    try:
        from cryptography.hazmat.primitives.ciphers.aead import AESGCM
    except Exception:
        return
    ref = AESGCM(key).encrypt(iv, d_pt.cpu().numpy().tobytes(), aad)
    assert ref[-16:] == d_tag.cpu().numpy().tobytes()
    assert ref[:4096] == d_ct[:4096].cpu().numpy().tobytes() and ref[-16 - 4096:-16] == d_ct[-4096:].cpu().numpy().tobytes()


def test_large_stream_8GiB_properties(engine, oracle, torch_mod):
    """2^33 bytes under one IV (2^29 blocks: exercises the 64-bit addressing and the upper counter
    bytes): CT windows vs the oracle's GCTR at the matching counters, tag equal to the 8-shard
    combine, decrypt verifies, a flipped bit far into the stream is rejected."""
    torch = torch_mod
    free, _ = torch.cuda.mem_get_info()
    n = 1 << 33
    if free < 3 * n + (1 << 30):
        pytest.skip("not enough free HBM")
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(8)
    key, iv, aad = _rb(rng, 16), _rb(rng, 12), _rb(rng, 33)
    engine.set_key(key)
    rk = oracle.key_expand(key)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(8)
    d_pt = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=gen)
    d_ct = torch.empty_like(d_pt)
    d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
    d_aad = _dev(torch, aad)
    engine.stream_crypt_device(0, iv, d_aad, d_pt, d_ct, d_tag)
    torch.cuda.synchronize()
    for off in (0, (1 << 32) - 64, (1 << 32) + 16 * 75776 * 3, n - 1024):
        w = 1024
        pt_w = d_pt[off:off + w].cpu().numpy().tobytes()
        assert d_ct[off:off + w].cpu().numpy().tobytes() == oracle.gctr(rk, iv, 2 + off // 16, pt_w), off
    parts = torch.zeros((8, 16), dtype=torch.uint8, device="cuda")
    for s in shard_plan(n, 8):
        sl = slice(s.byte_offset, s.byte_offset + s.n_bytes)
        engine.stream_part_device(1, iv, s.first_block, d_ct[sl], d_pt[sl], s.blocks_after, parts[s.rank])  # decrypt in place over pt
    d_tag2 = torch.zeros(16, dtype=torch.uint8, device="cuda")
    d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
    d_tag2.copy_(d_tag)
    engine.stream_finish_device(1, iv, parts, 8, d_aad, n, d_tag2, d_ok)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 1                      # the sharded decrypt recomputes the same tag
    d_ct[(1 << 32) + 12345] ^= 0x02
    engine.stream_crypt_device(1, iv, d_aad, d_ct, d_pt, d_tag, d_ok)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 0
    del d_pt, d_ct
    torch.cuda.empty_cache()


def test_two_contexts_two_threads_no_crosstalk(engine_lib, oracle, torch_mod):
    """The boundary contract: no global mutable state, distinct contexts are independent.  Two
    host threads, each with its own context, key and CUDA stream, interleave stream and batch
    calls (ctypes drops the GIL during a call); every result must match the oracle."""
    import threading
    import aesgcm_b200
    torch = torch_mod
    errors = []

    def worker(seed, kb):
        try:
            rng = np.random.default_rng(seed)
            eng = aesgcm_b200.GcmEngine(0)
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                for it in range(12):
                    key = _rb(rng, kb)
                    eng.set_key(key)
                    iv, aad = _rb(rng, 12), _rb(rng, int(rng.integers(0, 40)))
                    n = int(rng.integers(1, 300000))
                    pt = _rb(rng, n)
                    d_pt, d_aad = _dev(torch, pt), (_dev(torch, aad) if aad else None)
                    d_ct = torch.empty_like(d_pt)
                    d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
                    eng.stream_crypt_device(0, iv, d_aad, d_pt, d_ct, d_tag, stream=st.cuda_stream)
                    # a batch of short messages under the same key on the same stream
                    m, ln = 257, 208
                    ivs = _rb(rng, 12 * m)
                    bpt = _rb(rng, m * ln)
                    d_iv, d_bpt = _dev(torch, ivs), _dev(torch, bpt)
                    d_bct = torch.empty_like(d_bpt)
                    d_tags = torch.zeros(16 * m, dtype=torch.uint8, device="cuda")
                    eng.batch_crypt_uniform_device(0, d_iv, None, 0, 0, d_bpt, d_bct, ln, ln, d_tags, n_msgs=m,
                                                   stream=st.cuda_stream)
                    st.synchronize()
                    want_ct, want_tag = oracle.gcm_crypt(key, iv, aad, pt)
                    assert d_ct.cpu().numpy().tobytes() == want_ct, (seed, it)
                    assert d_tag.cpu().numpy().tobytes() == want_tag, (seed, it)
                    got_ct, got_tags = d_bct.cpu().numpy().tobytes(), d_tags.cpu().numpy().tobytes()
                    for i in (0, 100, m - 1):
                        c, t = oracle.gcm_crypt(key, ivs[12 * i:12 * i + 12], b"", bpt[ln * i:ln * i + ln])
                        assert got_ct[ln * i:ln * i + ln] == c and got_tags[16 * i:16 * i + 16] == t, (seed, it, i)
            eng.close()
        except BaseException as e:   # noqa: BLE001 - reported by the main thread
            errors.append((seed, repr(e)))

    threads = [threading.Thread(target=worker, args=(900 + i, kb)) for i, kb in enumerate((16, 32, 24))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


def test_maximum_length_stream_in_place(engine, oracle, torch_mod):
    """The longest message the 32-bit counter allows (src/aes_icb.vhd:99-100,118: the counter
    halts at 0xFFFFFFFF): 2^32-2 blocks = 68 719 476 704 bytes, encrypted IN PLACE in HBM.  CT
    windows (including the very last block, counter 0xFFFFFFFF) vs the oracle's GCTR; the tag must
    equal the 8-shard combine; the sharded decrypt restores the plaintext (64-bit word checksum)."""
    torch = torch_mod
    n = ((1 << 32) - 2) * 16
    free, _ = torch.cuda.mem_get_info()
    if free < n + (6 << 30):
        pytest.skip("not enough free HBM")
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(64)
    key, iv, aad = _rb(rng, 32), _rb(rng, 12), _rb(rng, 20)
    engine.set_key(key)
    rk = oracle.key_expand(key)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(64)
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    step = 1 << 32
    for off in range(0, n, step):                      # fill by pieces: no 64 GiB temporaries
        m = min(step, n - off)
        d[off:off + m] = torch.randint(0, 256, (m,), dtype=torch.uint8, device="cuda", generator=gen)
    def checksum():
        v = d.view(torch.int64)
        return [int(v[i::4].sum().item()) for i in range(4)]   # wraps mod 2^64; any restore error shows
    before = checksum()
    offs = (0, (1 << 32) - 512, (1 << 35) + 16 * 1001, n - 1024)
    w = 1024
    keep = {off: d[off:off + w].cpu().numpy().tobytes() for off in offs}
    d_tag = torch.zeros(16, dtype=torch.uint8, device="cuda")
    d_aad = _dev(torch, aad)
    engine.stream_crypt_device(0, iv, d_aad, d, d, d_tag)
    torch.cuda.synchronize()
    for off in offs:
        assert d[off:off + w].cpu().numpy().tobytes() == oracle.gctr(rk, iv, 2 + off // 16, keep[off]), off
    assert checksum() != before
    parts = torch.zeros((8, 16), dtype=torch.uint8, device="cuda")
    for s in shard_plan(n, 8):
        sl = slice(s.byte_offset, s.byte_offset + s.n_bytes)
        engine.stream_part_device(1, iv, s.first_block, d[sl], d[sl], s.blocks_after, parts[s.rank])
    d_ok = torch.zeros(1, dtype=torch.uint8, device="cuda")
    engine.stream_finish_device(1, iv, parts, 8, d_aad, n, d_tag, d_ok)
    torch.cuda.synchronize()
    assert int(d_ok.item()) == 1
    assert checksum() == before
    # one more block does not fit the counter
    with pytest.raises(Exception):
        engine.stream_part_device(0, iv, 16, d, d, 0, parts[0])      # first_block 16 + 2^32-2 blocks
    del d
    torch.cuda.empty_cache()


def test_config3_full_size_roundtrip(engine, oracle, torch_mod):
    """BASELINE config 3 at full size: 2^20 x 1500 B at a 1504 B stride, AES-192, shared
    pre-expanded key.  Sampled messages vs the oracle; full decrypt round trip; ok flags all 1."""
    torch = torch_mod
    rng = np.random.default_rng(2)
    key = _rb(rng, 24)
    engine.set_key(oracle.key_expand(key))
    n_msgs, length, stride = 1 << 20, 1500, 1504
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2)
    d_pt = torch.randint(0, 256, (n_msgs * stride,), dtype=torch.uint8, device="cuda", generator=gen)
    d_iv = torch.randint(0, 256, (n_msgs * 12,), dtype=torch.uint8, device="cuda", generator=gen)
    d_ct = torch.zeros_like(d_pt)
    d_tags = torch.zeros(16 * n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_uniform_device(0, d_iv, None, 0, 0, d_pt, d_ct, length, stride, d_tags, n_msgs=n_msgs)
    torch.cuda.synchronize()
    for i in (0, 1, 12345, n_msgs // 2, n_msgs - 1):
        pt = d_pt[i * stride:i * stride + length].cpu().numpy().tobytes()
        iv = d_iv[12 * i:12 * i + 12].cpu().numpy().tobytes()
        want_ct, want_tag = oracle.gcm_crypt(key, iv, b"", pt)
        assert d_ct[i * stride:i * stride + length].cpu().numpy().tobytes() == want_ct, i
        assert d_tags[16 * i:16 * i + 16].cpu().numpy().tobytes() == want_tag, i
    d_back = torch.zeros_like(d_pt)
    d_ok = torch.zeros(n_msgs, dtype=torch.uint8, device="cuda")
    engine.batch_crypt_uniform_device(1, d_iv, None, 0, 0, d_ct, d_back, length, stride, d_tags, d_ok, n_msgs=n_msgs)
    torch.cuda.synchronize()
    assert int(d_ok.sum().item()) == n_msgs
    v = d_back.view(n_msgs, stride)[:, :length]
    assert torch.equal(v, d_pt.view(n_msgs, stride)[:, :length])


@pytest.mark.gpu
def test_host_pipeline_ramped_granules(engine, torch_mod):
    """Host-buffer calls long enough for the ramped granule schedule (csrc/host_sched.h: 1, 2, 4 ... MiB up, the odd
    rest, the steady granules, and back down): every byte and the tag against OpenSSL, encrypt and decrypt, pageable and
    pinned buffers, lengths around the one-shot limit (2 MiB) and off every granule boundary; then the same message
    as two counter-range shards through agcm_stream_part_host / agcm_stream_finish_host."""
    AESGCM = pytest.importorskip("cryptography.hazmat.primitives.ciphers.aead").AESGCM
    torch = torch_mod
    rng = np.random.default_rng(123)
    key, iv, aad = _rb(rng, 32), _rb(rng, 12), _rb(rng, 21)
    engine.set_key(key)
    ossl = AESGCM(key)
    MiB = 1 << 20
    for n in (2 * MiB, 2 * MiB + 1, 3 * MiB + 16, 8 * MiB, 37 * MiB + 4097, 95 * MiB - 5):
        pt = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        pt.random_(0, 256)
        want = ossl.encrypt(iv, pt.numpy().tobytes(), aad)
        out = torch.zeros(n, dtype=torch.uint8, pin_memory=True)
        _, tag = engine.encrypt(iv, aad, pt, out=out)
        assert tag == want[-16:], n
        assert out.numpy().tobytes() == want[:-16], n
        back = np.zeros(n, dtype=np.uint8)                       # pageable output
        engine.decrypt(iv, aad, out, tag, out=back)
        assert back.tobytes() == pt.numpy().tobytes(), n
        with pytest.raises(ValueError):
            engine.decrypt(iv, aad, out, bytes([tag[0] ^ 1]) + tag[1:], out=back)
    # two shards of the last message, cut off a granule boundary
    cut = (41 * MiB + 4096) & ~15
    o2 = np.zeros(n, dtype=np.uint8)
    src = pt.numpy()
    p0 = engine.stream_part_host(0, iv, 0, src[:cut], o2[:cut], ((n - cut) + 15) // 16)
    p1 = engine.stream_part_host(0, iv, cut // 16, src[cut:], o2[cut:], 0)
    assert o2.tobytes() == want[:-16]
    assert engine.stream_finish_host(0, iv, p0 + p1, aad, n) == want[-16:]
