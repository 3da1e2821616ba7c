#!/usr/bin/env python
"""Golden vectors for IVs that are NOT 96 bits long (SP 800-38D 7.1: J0 by GHASH).

  python tests/golden/make_long_iv_golden.py   ->  tests/golden/long_iv_vectors.json

The reference IP fixes the IV at 96 bits (src/gcm_pkg.vhd:17) and holds no vector for this
case; the reference MODEL calls pycryptodome (tb/gcm_model.py:18), which accepts such nonces
and computes the function OpenSSL computes.  Expected CT/TAG here come from OpenSSL through
`cryptography` (nonces of 8..128 bytes, its supported range); the published tags of the
McGrew-Viega test cases 5, 6, 11, 12, 17, 18 (8- and 60-byte IVs) are asserted as anchors.

The counter-edge section (appended after the random vectors, from its own RNG, so the earlier vectors stay as they
were) chooses J0 and builds the 16-byte IV that GHASHes to it (iv_for_j0, plain Python, independent of the oracle):
J0 counter fields at the 32-bit wrap, at the carries into the counter's top byte and into byte 13, and 0, with the
carry or wrap on block 0, block 1, mid-message and in a ragged last block.  Each such vector also stores its `j0`.
"""
import json
import os
import random

from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
from cryptography.hazmat.primitives.ciphers.aead import AESGCM

HERE = os.path.dirname(os.path.abspath(__file__))

K = "feffe9928665731c6d6a8f9467308308feffe9928665731c6d6a8f9467308308"
PT = ("d9313225f88406e5a55909c5aff5269a86a7a9531534f7da2e4c303d8a318a72"
      "1c3c0c95956809532fcf0e2449a6b525b16aedf5aa0de657ba637b39")
AAD = "feedfacedeadbeeffeedfacedeadbeefabaddad2"
IV8 = "cafebabefacedbad"
IV60 = ("9313225df88406e555909c5aff5269aa6a7a9538534f7da1e4c303d2a318a728"
        "c3c0c95156809539fcf0e2429a6b525416aedbf5a0de6a57a637b39b")
PUBLISHED_TAGS = {  # McGrew & Viega, "The Galois/Counter Mode of Operation", appendix B
    ("MV-TC5", 16, IV8): "3612d2e79e3b0785561be14aaca2fccb",
    ("MV-TC6", 16, IV60): "619cc5aefffe0bfa462af43c1699d050",
    ("MV-TC11", 24, IV8): "65dcc57fcf623a24094fcca40d3533f8",
    ("MV-TC12", 24, IV60): "dcf566ff291c25bbb8568fc3d376a6d9",
    ("MV-TC17", 32, IV8): "3a337dbf46a792c45e454913fe2ea8f2",
    ("MV-TC18", 32, IV60): "a44a8266ee1c8eb0c8b5d4cf5ae9f19a",
}


def case(name, key, iv, aad, pt):
    out = AESGCM(key).encrypt(iv, pt, aad)
    return {"name": name, "key": key.hex(), "iv": iv.hex(), "aad": aad.hex(), "pt": pt.hex(),
            "ct": out[:-16].hex(), "tag": out[-16:].hex()}


def aes_ecb(key, block):
    e = Cipher(algorithms.AES(key), modes.ECB()).encryptor()
    return e.update(block) + e.finalize()


def gf_mul(x, y):
    """Product in GCM's GF(2^128) (SP 800-38D 6.3) on blocks read as big-endian integers."""
    z, v = 0, y
    for i in range(128):
        if (x >> (127 - i)) & 1:
            z ^= v
        v = (v >> 1) ^ (0xE1 << 120) if v & 1 else v >> 1
    return z


def gf_inv(h):
    """h^(2^128 - 2) = h^-1"""
    r, e = 1 << 127, (1 << 128) - 2   # 1 << 127 is the field's one
    while e:
        if e & 1:
            r = gf_mul(r, h)
        h = gf_mul(h, h)
        e >>= 1
    return r


def iv_for_j0(key, j0):
    """The 16-byte IV whose J0 = GHASH_H(IV || 0^64 || [128]_64) = IV.H^2 ^ L.H is `j0`: IV = ((J0.H^-1) ^ L).H^-1."""
    h = int.from_bytes(aes_ecb(key, bytes(16)), "big")
    hi, ln = gf_inv(h), 128
    iv = gf_mul(gf_mul(int.from_bytes(j0, "big"), hi) ^ ln, hi)
    assert gf_mul(gf_mul(iv, h) ^ ln, h) == int.from_bytes(j0, "big")
    return iv.to_bytes(16, "big")


def inc32(block, k=1):
    return block[:12] + ((int.from_bytes(block[12:], "big") + k) & 0xFFFFFFFF).to_bytes(4, "big")


# J0 counter fields: the 32-bit wrap on payload block 0, block 1 and block 15; the carry into the counter's top byte
# (0x00FFFFFF -> 0x01000000) on block 0 and block 15; the carry into byte 13 on block 15; an ordinary start
EDGE_CTRS = (0xFFFFFFFF, 0xFFFFFFFE, 0xFFFFFFF0, 0x00FFFFFF, 0x00FFFFF0, 0x0000FFF0, 0)
EDGE_LENS = (1, 17, 33, 16 * 40 + 9)


def counter_edge_vectors():
    rnd = random.Random(20261020)
    rb = lambda n: bytes(rnd.getrandbits(8) for _ in range(n))
    vectors = []
    for kb in (16, 24, 32):
        for c0 in EDGE_CTRS:
            key = rb(kb)
            j0 = rb(12) + c0.to_bytes(4, "big")
            iv = iv_for_j0(key, j0)
            for n in EDGE_LENS:
                for al in (0, 20):
                    pt = rb(n)
                    v = case("edge-k%d-c%08x-n%d-a%d" % (8 * kb, c0, n, al), key, iv, rb(al), pt)
                    # the keystream of blocks 0 and 1 is E_K(inc32(J0)), E_K(inc32^2(J0)): the wrap really happens
                    ks = bytes(a ^ b for a, b in zip(bytes.fromhex(v["ct"]), pt))[:32]
                    want = aes_ecb(key, inc32(j0, 1)) + aes_ecb(key, inc32(j0, 2))
                    assert ks == want[:len(ks)], v["name"]
                    v["j0"] = j0.hex()
                    vectors.append(v)
    return vectors


def main():
    vectors = []
    for (name, kb, iv), tag in PUBLISHED_TAGS.items():
        v = case(name, bytes.fromhex(K[:2 * kb]), bytes.fromhex(iv), bytes.fromhex(AAD), bytes.fromhex(PT))
        assert v["tag"] == tag, (name, v["tag"])
        vectors.append(v)
    rnd = random.Random(20261018)
    rb = lambda n: bytes(rnd.getrandbits(8) for _ in range(n))
    for kb in (16, 24, 32):
        for ivl in (8, 9, 11, 13, 15, 16, 17, 31, 32, 33, 64, 100, 128):
            n = rnd.choice([0, 1, 15, 16, 17, 64, 333, 1500, 4096])
            al = rnd.choice([0, 1, 16, 20, 64, 100])
            vectors.append(case("rand-k%d-iv%d" % (8 * kb, ivl), rb(kb), rb(ivl), rb(al), rb(n)))
    vectors += counter_edge_vectors()
    with open(os.path.join(HERE, "long_iv_vectors.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_long_iv_golden.py (OpenSSL via cryptography; MV tags asserted)",
                   "vectors": vectors}, f, indent=1)
    print(len(vectors), "vectors")


if __name__ == "__main__":
    main()
