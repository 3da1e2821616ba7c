"""Pins the CPU oracle: reference key schedule fixtures, published AES-GCM
known-answer vectors, and OpenSSL on random cases (SURVEY 8c)."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN


def _load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def test_sbox_matches_reference_table(oracle):
    fx = _load("key_exp_vectors.json")
    assert oracle.sbox_table().tobytes().hex() == fx["sbox"]


def test_key_expand_matches_reference_key_exp_py(oracle):
    fx = _load("key_exp_vectors.json")
    assert len(fx["cases"]) >= 80
    for c in fx["cases"]:
        got = oracle.key_expand(bytes.fromhex(c["key"]))
        assert got.hex() == c["expanded"], c


def test_fips197_last_round_keys(oracle):
    want = {16: "d014f9a8c9ee2589e13f0cc8b6630ca6", 24: "e98ba06f448c773c8ecc720401002202",
            32: "fe4890d1e6188d0b046df344706c631e"}
    keys = {16: "2b7e151628aed2a6abf7158809cf4f3c", 24: "8e73b0f7da0e6452c810f32b809079e562f8ead2522c6b7b",
            32: "603deb1015ca71be2b73aef0857d77811f352c073b6108d72d9810a30914dff4"}
    for n, k in keys.items():
        assert oracle.key_expand(bytes.fromhex(k))[-16:].hex() == want[n]


def test_fips197_example_block(oracle):
    # FIPS-197 App. C.1
    rk = oracle.key_expand(bytes.fromhex("000102030405060708090a0b0c0d0e0f"))
    ct = oracle.aes_encrypt_block(rk, bytes.fromhex("00112233445566778899aabbccddeeff"))
    assert ct.hex() == "69c4e0d86a7b0430d8cdb78070b4c55a"


def test_known_answer_vectors(oracle):
    for v in _load("kat_vectors.json")["vectors"]:
        key, iv = bytes.fromhex(v["key"]), bytes.fromhex(v["iv"])
        pt, aad = bytes.fromhex(v["pt"]), bytes.fromhex(v["aad"])
        ct, tag = oracle.gcm_crypt(key, iv, aad, pt)
        assert ct.hex() == v["ct"] and tag.hex() == v["tag"], v["name"]
        # decrypt direction + pre-expanded key (config/config_aes_kprexp.py:66-95)
        pt2, tag2 = oracle.gcm_crypt(oracle.key_expand(key), iv, aad, ct, decrypt=True)
        assert pt2 == pt and tag2 == tag, v["name"]


def test_committed_openssl_vectors(oracle):
    vs = _load("openssl_random_vectors.json")["vectors"]
    assert len(vs) == 30
    for v in vs:
        key, iv, aad, pt = (bytes.fromhex(v[k]) for k in ("key", "iv", "aad", "pt"))
        ct, tag = oracle.gcm_crypt(key, iv, aad, pt)
        assert ct.hex() == v["ct"] and tag.hex() == v["tag"]
        pt2, tag2 = oracle.gcm_crypt(key, iv, aad, ct, decrypt=True)
        assert pt2 == pt and tag2 == tag


def test_long_iv_vectors(oracle):
    """IVs that are not 96 bits (J0 by GHASH, SP 800-38D 7.1): the oracle's composition of its own
    primitives vs OpenSSL-generated vectors anchored on the published McGrew-Viega tags."""
    import json, os
    from conftest import GOLDEN
    with open(os.path.join(GOLDEN, "long_iv_vectors.json")) as f:
        vectors = json.load(f)["vectors"]
    assert len(vectors) == 213 and sum("j0" in v for v in vectors) == 168
    for v in vectors:
        key, iv = bytes.fromhex(v["key"]), bytes.fromhex(v["iv"])
        pt, aad = bytes.fromhex(v["pt"]), bytes.fromhex(v["aad"])
        if "j0" in v:   # counter-edge vectors: the IV was built to give this J0
            h = oracle.aes_encrypt_block(oracle.key_expand(key), bytes(16))
            assert oracle.ghash_absorb(h, iv + bytes(8) + (8 * len(iv)).to_bytes(8, "big")).hex() == v["j0"], v["name"]
        ct, tag = oracle.gcm_crypt_any_iv(key, iv, aad, pt)
        assert ct.hex() == v["ct"] and tag.hex() == v["tag"], v["name"]
        back, tag2 = oracle.gcm_crypt_any_iv(key, iv, aad, ct, decrypt=True)
        assert back == pt and tag2 == tag, v["name"]
    # a 96-bit IV takes the plain path and agrees with it
    k, iv, a, d = bytes(range(16)), bytes(range(12)), b"hdr", b"x" * 100
    assert oracle.gcm_crypt_any_iv(k, iv, a, d) == oracle.gcm_crypt(k, iv, a, d)


def test_reference_model_traces(oracle):
    """Traces recorded from the reference's own tb/gcm_model.py (tests/golden/make_model_traces.py):
    the oracle reproduces its per-call outputs and tags, and the forced-mismatch tag is the
    bitwise complement of the received one (tb/gcm_model.py:47-51)."""
    cases = _load("gcm_model_traces.json")["cases"]
    assert len(cases) == 15
    for c in cases:
        key = bytes.fromhex(c["key"]["data"])
        iv = bytes.fromhex(c["iv"]["data"])
        aad, pt = bytes.fromhex(c["aad"]), bytes.fromhex(c["pt"])
        ct, tag = oracle.gcm_crypt(key, iv, aad, pt)
        assert "".join(c["enc_data_out"]) == ct.hex() and c["enc_tag"] == [tag.hex()]
        assert all(len(x) <= 32 for x in c["enc_data_out"])            # one <=16-byte block per call
        assert "".join(c["dec_good"]["data_out"]) == pt.hex() and c["dec_good"]["tag"] == [tag.hex()]
        rx = bytes.fromhex(c["dec_bad"]["rx_tag"])
        assert c["dec_bad"]["tag"] == [bytes(b ^ 0xFF for b in rx).hex()]


def test_readme_intermediates(oracle):
    # SURVEY appendix: H and E_K(J0) of the 802.1AE vectors
    key = bytes.fromhex("AD7A2BD03EAC835A6F620FDCB506B345")
    h, ej0 = oracle.h_ej0(oracle.key_expand(key), bytes.fromhex("12153524C0895E81B2C28465"))
    assert h.hex().upper() == "73A23D80121DE2D5A850253FCF43120E"
    assert ej0.hex().upper() == "EB4E051CB548A6B5490F6F11A27CB7D0"
    h0, _ = oracle.h_ej0(oracle.key_expand(bytes(16)), bytes(12))
    assert h0.hex().upper() == "66E94BD4EF8A2C3B884CFA59CA342B2E"


def test_random_against_openssl(oracle):
    AESGCM = pytest.importorskip("cryptography.hazmat.primitives.ciphers.aead").AESGCM
    rng = np.random.default_rng(0)
    sizes = [0, 1, 15, 16, 17, 31, 32, 33, 60, 64, 255, 256, 1500, 4096]
    for kb in (16, 24, 32):
        for n in sizes:
            for alen in (0, 1, 16, 20, 64):
                key = rng.integers(0, 256, kb, dtype=np.uint8).tobytes()
                iv = rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
                aad = rng.integers(0, 256, alen, dtype=np.uint8).tobytes()
                pt = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
                ref = AESGCM(key).encrypt(iv, pt, aad)
                ct, tag = oracle.gcm_crypt(key, iv, aad, pt)
                assert ct + tag == ref
                pt2, tag2 = oracle.gcm_crypt(key, iv, aad, ct, decrypt=True)
                assert pt2 == pt and tag2 == tag


def test_gf_properties(oracle):
    rng = np.random.default_rng(5)
    one = bytes([0x80] + [0] * 15)
    for _ in range(50):
        a, b, c = (rng.integers(0, 256, 16, dtype=np.uint8).tobytes() for _ in range(3))
        assert oracle.gfmul(a, one) == a
        assert oracle.gfmul(a, b) == oracle.gfmul(b, a)
        bc = bytes(x ^ y for x, y in zip(b, c))
        lhs = oracle.gfmul(a, bc)
        rhs = bytes(x ^ y for x, y in zip(oracle.gfmul(a, b), oracle.gfmul(a, c)))
        assert lhs == rhs  # linearity used by the shard combine (src/gcm_ghash.vhd:317-344)
    h = rng.integers(0, 256, 16, dtype=np.uint8).tobytes()
    assert oracle.gf_pow(h, 0) == one and oracle.gf_pow(h, 1) == h
    assert oracle.gf_pow(h, 5) == oracle.gfmul(oracle.gf_pow(h, 2), oracle.gf_pow(h, 3))


def test_threaded_stream_equals_serial(oracle):
    rng = np.random.default_rng(6)
    for n in (0, 5, 16, 1000, 40000 + 3):
        key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
        iv = rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
        aad = rng.integers(0, 256, 16, dtype=np.uint8).tobytes()
        pt = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert oracle.gcm_crypt(key, iv, aad, pt) == oracle.gcm_crypt(key, iv, aad, pt, threads=5)


def test_counter_overflow_is_an_error(oracle):
    # > 2^32-2 blocks per IV (src/aes_icb.vhd:114): checked without allocating
    import ctypes
    rc = oracle.lib().oracle_gcm_crypt(None, 16, None, None, ctypes.c_uint64(0), None,
                                       ctypes.c_uint64(16 * 0xFFFFFFFF), 0, None, None)
    assert rc == -2
