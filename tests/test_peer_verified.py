"""Verify-then-release decrypt of a message sharded over GPUs (agcm_stream_decrypt_verified_peer and its host form): every
rank's ok flag is 1 if and only if the whole message's tag matches, and no rank writes a plaintext byte otherwise.

The ranks are N contexts on one GPU, each with its own exchange buffer and stream; the last test runs two processes on two
GPUs.  Reference: OpenSSL (`cryptography`) where it takes the IV,
else the oracle's any-IV composition.  Every output buffer starts as a sentinel and runs 16 bytes past the shard."""
import numpy as np
import pytest

from batch_cases import gf_inv, iv_for_j0, wrap_at

pytestmark = pytest.mark.gpu
SENT = 0x5A
ROWS = 4 * 16 * 151552 + 11   # more than one grid row of the default 148 x 1024 grid


def _t(a):
    import torch
    return torch.from_numpy(np.frombuffer(bytes(a), np.uint8).copy()).cuda()


def _h(t):
    return t.cpu().numpy().tobytes()


def _flip(b, i=0, bit=0):
    b = bytearray(b)
    b[i] ^= 1 << bit
    return bytes(b)


def _ref(oracle, key, iv, aad, pt):
    """-> (ct, tag)"""
    if 8 <= len(iv) <= 128:
        from cryptography.hazmat.primitives.ciphers.aead import AESGCM
        out = AESGCM(key).encrypt(iv, pt, aad)
        return out[:-16], out[-16:]
    return oracle.gcm_crypt_any_iv(key, iv, aad, pt)


def _msg(oracle, rng, key, iv_len, aad_len, n):
    iv, aad, pt = (rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (iv_len, aad_len, n))
    ct, tag = _ref(oracle, key, iv, aad, pt)
    return iv, aad, pt, ct, tag


def _load_stream_kernels(eng):
    """Launches every stream-kernel variant the exchanges below use (GHASH-only, gated GCTR, fused decrypt; 16-byte
    aligned and not) once for the loaded key size.  The emulated ranks share one CUDA context, in which the first launch
    of a kernel loads it lazily and waits for the running kernels -- among them another rank's finish, which waits for
    this rank's post -- so an exchange that meets an unloaded kernel stalls until the timeout.  (Ranks in separate
    processes, as on a real node, do not wait for each other's kernels.)"""
    import torch
    buf = torch.zeros(80, dtype=torch.uint8, device="cuda")
    tag, ok = torch.zeros(16, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.uint8, device="cuda")
    for off in (0, 1):
        d = buf[off:off + 64]
        eng.stream_decrypt_verified_device(bytes(12), None, d, d, tag, ok)
        eng.stream_crypt_device(1, bytes(12), None, d, d, tag, ok)
    torch.cuda.synchronize()


class Ranks:
    """Contexts on GPU 0, each with its own exchange buffer and stream: the ranks of an emulated world."""

    def __init__(self, n):
        import torch
        import aesgcm_b200
        self.engs = [aesgcm_b200.GcmEngine(0) for _ in range(n)]
        self.bufs = [torch.zeros(4096, dtype=torch.uint8, device="cuda") for _ in range(n)]
        self.streams = [torch.cuda.Stream() for _ in range(n)]

    def setup(self, world, key):
        for e in self.engs[:world]:
            e.set_key(key)
        _load_stream_kernels(self.engs[0])
        ptrs = [b.data_ptr() for b in self.bufs[:world]]
        for r in range(world):
            self.engs[r].peer_setup(r, world, ptrs)

    def close(self):
        for e in self.engs:
            e.close()


@pytest.fixture(scope="module")
def ranks(engine_lib):
    r = Ranks(4)
    yield r
    r.close()


def _decrypt_world(ranks, world, iv, aad, ct, tag, shift=0, in_place=False, flip_rank=None):
    """Every rank of an emulated world decrypts its shard of `ct` with agcm_stream_decrypt_verified_peer (rank
    `flip_rank` with one ciphertext bit flipped).  -> [(output buffer, its bytes before the call, ok)] per rank; the
    shard sits `shift` bytes into its buffer (in place: the ciphertext buffer itself)."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    n = len(ct)
    d_aad, d_tag = (_t(aad) if aad else None), _t(tag)
    res = []
    for sh in shard_plan(n, world):
        src = ct[sh.byte_offset:sh.byte_offset + sh.n_bytes]
        if sh.rank == flip_rank:
            src = _flip(src, sh.n_bytes - 1, 7)   # the last byte: the ragged end of the last shard
        out = torch.full((shift + sh.n_bytes + 16,), SENT, dtype=torch.uint8, device="cuda")
        cbuf = out if in_place else torch.full_like(out, 0x33)
        cbuf[shift:shift + sh.n_bytes] = _t(src)
        ok = torch.full((1,), 7, dtype=torch.uint8, device="cuda")
        res.append((sh, out, cbuf[shift:shift + sh.n_bytes], ok))
    torch.cuda.synchronize()
    before = [_h(out) for _, out, _, _ in res]
    for sh, out, d_ct, ok in res:
        n_sh = sh.n_bytes
        ranks.engs[sh.rank].stream_decrypt_verified_peer_device(iv, sh.first_block, d_ct if n_sh else None,
                                                                out[shift:shift + n_sh] if n_sh else None, sh.blocks_after,
                                                                d_aad, n, d_tag, ok, n_bytes=n_sh,
                                                                stream=ranks.streams[sh.rank])
    torch.cuda.synchronize()
    for e in ranks.engs[:world]:
        assert not e.peer_timed_out()
    return [(sh, _h(out), b, int(ok.item())) for (sh, out, _, ok), b in zip(res, before)]


def _check(res, pt, authentic, shift, what):
    for sh, got, before, ok in res:
        want = bytearray(before)
        if authentic:
            want[shift:shift + sh.n_bytes] = pt[sh.byte_offset:sh.byte_offset + sh.n_bytes]
        assert ok == int(authentic), (what, sh.rank)
        assert got == bytes(want), (what, sh.rank)


# ------------------------------------------------------------------------------------------------------------ world = 1
def test_world1_matches_single_gpu_verified_decrypt(ranks, oracle):
    """world = 1 (the context's own exchange buffer): output bytes and ok equal agcm_stream_decrypt_verified's on the
    same inputs, authentic and with a flipped tag."""
    import torch
    rng = np.random.default_rng(9100)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    ranks.setup(1, key)
    eng = ranks.engs[0]
    for n in (0, 9, 4099, ROWS):
        for iv_len in (12, 1, 20):
            for aad_len in (0, 16, 4096):
                iv, aad, pt, ct, tag = _msg(oracle, rng, key, iv_len, aad_len, n)
                d_ct, d_aad = _t(ct), (_t(aad) if aad_len else None)
                for t in (tag, _flip(tag, 15, 3)):
                    outs = [torch.full((n + 16,), SENT, dtype=torch.uint8, device="cuda") for _ in range(2)]
                    oks = [torch.full((1,), 7, dtype=torch.uint8, device="cuda") for _ in range(2)]
                    d_tag = _t(t)
                    eng.stream_decrypt_verified_peer_device(iv, 0, d_ct, outs[0][:n], 0, d_aad, n, d_tag, oks[0], n_bytes=n)
                    eng.stream_decrypt_verified_device(iv, d_aad, d_ct, outs[1][:n], d_tag, oks[1], n_bytes=n)
                    torch.cuda.synchronize()
                    what = (n, iv_len, aad_len, t == tag)
                    assert _h(outs[0]) == _h(outs[1]) and int(oks[0].item()) == int(oks[1].item()), what
                    want = (pt if t == tag else bytes([SENT]) * n) + bytes([SENT]) * 16
                    assert _h(outs[0]) == want and int(oks[0].item()) == int(t == tag), what
    assert not eng.peer_timed_out()


# ----------------------------------------------------------------------------------------------- world = 2, 3, 4 on one GPU
@pytest.mark.parametrize("world", [2, 3, 4])
def test_emulated_world_authentic_and_forged(ranks, oracle, world):
    """The authentic message decrypts on every rank; a bit flipped in the tag, in the AAD or in any one rank's
    ciphertext (the ragged last shard included) clears ok on EVERY rank and leaves every output buffer as it was."""
    rng = np.random.default_rng(9200 + world)
    key = rng.integers(0, 256, 16 * (1 + world % 2), dtype=np.uint8).tobytes()
    ranks.setup(world, key)
    for n, iv_len in ((16 * 1000 + 7, 12), (ROWS, 20)):
        iv, aad, pt, ct, tag = _msg(oracle, rng, key, iv_len, 16, n)
        _check(_decrypt_world(ranks, world, iv, aad, ct, tag), pt, True, 0, (world, n, "authentic"))
        _check(_decrypt_world(ranks, world, iv, aad, ct, _flip(tag, 7, 1)), pt, False, 0, (world, n, "tag"))
        _check(_decrypt_world(ranks, world, iv, _flip(aad, 3, 5), ct, tag), pt, False, 0, (world, n, "aad"))
        for k in range(world):
            _check(_decrypt_world(ranks, world, iv, aad, ct, tag, flip_rank=k), pt, False, 0, (world, n, "ct", k))


def test_emulated_world_layouts_and_edges(ranks, oracle):
    """Buffers 1 and 4 bytes off alignment, in place (a failed shard keeps its ciphertext), an empty counter range (a
    one-block message at world 4: ranks 1-3 hold nothing but still post) and total_len = 0 (GMAC only)."""
    rng = np.random.default_rng(9300)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    ranks.setup(3, key)
    iv, aad, pt, ct, tag = _msg(oracle, rng, key, 12, 20, 16 * 5000 + 3)
    for shift, in_place in ((1, False), (4, False), (0, True), (3, True)):
        what = (shift, in_place)
        _check(_decrypt_world(ranks, 3, iv, aad, ct, tag, shift, in_place), pt, True, shift, what)
        _check(_decrypt_world(ranks, 3, iv, aad, ct, _flip(tag)), pt, False, 0, what)
        _check(_decrypt_world(ranks, 3, iv, aad, ct, tag, shift, in_place, flip_rank=1), pt, False, shift, what)
    ranks.setup(4, key)
    for n in (9, 0):
        iv, aad, pt, ct, tag = _msg(oracle, rng, key, 12, 16, n)
        _check(_decrypt_world(ranks, 4, iv, aad, ct, tag), pt, True, 0, (n, "authentic"))
        _check(_decrypt_world(ranks, 4, iv, _flip(aad, 15, 2), ct, tag), pt, False, 0, (n, "aad"))
        _check(_decrypt_world(ranks, 4, iv, aad, ct, _flip(tag)), pt, False, 0, (n, "tag"))
        if n:
            _check(_decrypt_world(ranks, 4, iv, aad, ct, tag, flip_rank=0), pt, False, 0, (n, "ct"))


def test_counter_wrap_inside_a_shard(ranks, oracle):
    """A 16-byte IV whose J0 makes the 32-bit counter wrap inside rank 1's shard, and on its first block."""
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(9400)
    key = rng.integers(0, 256, 24, dtype=np.uint8).tobytes()
    ranks.setup(3, key)
    h = oracle.aes_encrypt_block(oracle.key_expand(key), bytes(16))
    h_inv = gf_inv(oracle, h)
    n = 16 * 6000 + 9
    fb1 = shard_plan(n, 3)[1].first_block
    for c0 in (wrap_at(fb1 + 777), wrap_at(fb1)):
        j0 = rng.integers(0, 256, 12, dtype=np.uint8).tobytes() + c0.to_bytes(4, "big")
        iv = iv_for_j0(oracle, h, h_inv, j0)
        aad, pt = rng.integers(0, 256, 16, dtype=np.uint8).tobytes(), rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        ct, tag = _ref(oracle, key, iv, aad, pt)
        _check(_decrypt_world(ranks, 3, iv, aad, ct, tag), pt, True, 0, hex(c0))


def test_ring_interleaves_verified_and_releasing_calls(ranks, oracle):
    """11 messages on one exchange (the 8-deep ring wraps), alternating the verified, the releasing and the deferred
    releasing decrypt; message 3 carries a forged tag.  Every result is that message's own."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(9500)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    world = 2
    ranks.setup(world, key)
    msgs = []
    for i in range(11):
        n = 16 * (2000 + 37 * i) + i
        iv, aad, pt, ct, tag = _msg(oracle, rng, key, 12, 16, n)
        if i == 3:
            tag = _flip(tag, 2, 6)
        plan = shard_plan(n, world)
        outs = [torch.full((sh.n_bytes + 16,), SENT, dtype=torch.uint8, device="cuda") for sh in plan]
        oks = [torch.full((1,), 7, dtype=torch.uint8, device="cuda") for _ in plan]
        msgs.append((i % 3, n, iv, _t(aad), pt, _t(ct), _t(tag), plan, outs, oks))
    torch.cuda.synchronize()
    for kind, n, iv, d_aad, pt, d_ct, d_tag, plan, outs, oks in msgs:
        for sh, out, ok in zip(plan, outs, oks):
            eng, st = ranks.engs[sh.rank], ranks.streams[sh.rank]
            src, dst = d_ct[sh.byte_offset:sh.byte_offset + sh.n_bytes], out[:sh.n_bytes]
            if kind == 0:
                eng.stream_decrypt_verified_peer_device(iv, sh.first_block, src, dst, sh.blocks_after, d_aad, n, d_tag, ok,
                                                        stream=st)
            else:
                eng.stream_crypt_peer_device(1, iv, sh.first_block, src, dst, sh.blocks_after, d_aad, n, d_tag, ok,
                                             stream=st, defer=kind == 2)
    for eng, st in zip(ranks.engs[:world], ranks.streams[:world]):
        eng.peer_join(st)
    torch.cuda.synchronize()
    for i, (kind, n, iv, d_aad, pt, d_ct, d_tag, plan, outs, oks) in enumerate(msgs):
        for sh, out, ok in zip(plan, outs, oks):
            authentic = i != 3
            shard_pt = pt[sh.byte_offset:sh.byte_offset + sh.n_bytes]
            want = (shard_pt if authentic else bytes([SENT]) * sh.n_bytes) + bytes([SENT]) * 16
            assert int(ok.item()) == int(authentic) and _h(out) == want, (i, kind, sh.rank)
    assert not any(e.peer_timed_out() for e in ranks.engs[:world])


# ---------------------------------------------------------------------------------------------------------- host form
def test_host_form_emulated(engine_lib, oracle, monkeypatch):
    """agcm_stream_decrypt_verified_peer_host at world 2 on one GPU, with 1 MiB granules so that each 3 MiB shard takes
    several: one rank calls the host form, the other the device form of the same exchange, and then the other way
    round (the host form on the first and on the ragged last shard).  Authentic, then a bit flipped in rank 1's
    ciphertext and in the tag: both ranks refuse, and neither output is touched."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    monkeypatch.setenv("AGCM_CHUNK_MB", "1")
    rng = np.random.default_rng(9600)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    world, n = 2, 6 * (1 << 20) + 5
    plan = shard_plan(n, world)
    iv, aad, pt, ct, tag = _msg(oracle, rng, key, 12, 16, n)
    # Both ranks live in one process here.  Two host threads each inside a synchronous call stall each other in the
    # driver until the timeout (ranks in separate processes, as on a real node, do not), so the other rank takes the
    # device form, which only enqueues.  The host rank must not wait for the whole device before it posts either: its
    # buffers are pinned and its staging buffers are grown beforehand (growing frees the old buffer, which waits for
    # every running kernel -- among them the other rank's finish, which waits for this rank's post).
    keep = []

    def pinned(b):
        t = torch.from_numpy(np.frombuffer(bytes(b), np.uint8).copy()).pin_memory()
        keep.append(t)
        return t.numpy()

    r = Ranks(world)
    try:
        r.setup(world, key)
        for e in r.engs:
            assert e.decrypt_verified(iv, aad, ct, tag) == pt
        h_aad, d_aad = pinned(aad), _t(aad)
        for host_rank in (0, 1):
            for what, cts, t in (("authentic", [ct, ct], tag), ("ct", [ct, _flip(ct, n - 1, 4)], tag),
                                 ("tag", [ct, ct], _flip(tag, 9))):
                shards = [cts[sh.rank][sh.byte_offset:sh.byte_offset + sh.n_bytes] for sh in plan]
                hs, ds = plan[host_rank], plan[1 - host_rank]
                h_ct, h_out, h_tag = pinned(shards[hs.rank]), pinned(bytes([SENT]) * hs.n_bytes), pinned(t)
                d_ct, d_tag = _t(shards[ds.rank]), _t(t)
                d_out = torch.full((ds.n_bytes + 16,), SENT, dtype=torch.uint8, device="cuda")
                d_ok = torch.full((1,), 7, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                r.engs[ds.rank].stream_decrypt_verified_peer_device(iv, ds.first_block, d_ct, d_out[:ds.n_bytes],
                                                                    ds.blocks_after, d_aad, n, d_tag, d_ok,
                                                                    stream=r.streams[ds.rank])
                ok_host = r.engs[hs.rank].stream_decrypt_verified_peer_host(iv, hs.first_block, h_ct, h_out,
                                                                            hs.blocks_after, h_aad, n, h_tag)
                torch.cuda.synchronize()
                authentic = what == "authentic"
                case = (host_rank, what)
                assert ok_host == authentic and int(d_ok.item()) == int(authentic), case
                want = pt[hs.byte_offset:hs.byte_offset + hs.n_bytes] if authentic else bytes([SENT]) * hs.n_bytes
                assert h_out.tobytes() == want, case
                want = pt[ds.byte_offset:ds.byte_offset + ds.n_bytes] if authentic else bytes([SENT]) * ds.n_bytes
                assert _h(d_out) == want + bytes([SENT]) * 16, case
        assert not any(e.peer_timed_out() for e in r.engs)
    finally:
        r.close()


# ------------------------------------------------------------------------------------------------------- fails closed
def test_fails_closed_on_missing_rank(engine_lib, monkeypatch):
    """world = 2 but rank 1 never calls: the device form clears ok, writes nothing, and the next peer call raises
    E_PEER_TIMEOUT; after a fresh setup the host form returns E_PEER_TIMEOUT with its output untouched."""
    import torch
    import aesgcm_b200
    monkeypatch.setenv("AGCM_PEER_TIMEOUT_MS", "200")
    rng = np.random.default_rng(9700)
    key, iv = rng.integers(0, 256, 16, dtype=np.uint8).tobytes(), rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
    n = 4096
    e0 = aesgcm_b200.GcmEngine(0)
    try:
        e0.set_key(key)
        bufs = [torch.zeros(4096, dtype=torch.uint8, device="cuda") for _ in range(2)]
        e0.peer_setup(0, 2, [b.data_ptr() for b in bufs])
        d_ct = _t(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
        d_pt = torch.full((n + 16,), SENT, dtype=torch.uint8, device="cuda")
        d_tag, d_ok = _t(bytes(16)), torch.ones(1, dtype=torch.uint8, device="cuda")
        e0.stream_decrypt_verified_peer_device(iv, 0, d_ct, d_pt[:n], n // 16, None, 2 * n, d_tag, d_ok)
        torch.cuda.synchronize()
        assert int(d_ok.item()) == 0 and _h(d_pt) == bytes([SENT]) * (n + 16)
        assert e0.peer_timed_out()
        with pytest.raises(aesgcm_b200.AgcmError) as ei:
            e0.stream_decrypt_verified_peer_device(iv, 0, d_ct, d_pt[:n], n // 16, None, 2 * n, d_tag, d_ok)
        assert ei.value.rc == aesgcm_b200._lib.E_PEER_TIMEOUT
        e0.peer_setup(0, 2, [b.data_ptr() for b in bufs])
        h_pt = np.full(n, SENT, np.uint8)
        with pytest.raises(aesgcm_b200.AgcmError) as ei:
            e0.stream_decrypt_verified_peer_host(iv, 0, _h(d_ct), h_pt, n // 16, b"", 2 * n, bytes(16))
        assert ei.value.rc == aesgcm_b200._lib.E_PEER_TIMEOUT
        assert h_pt.tobytes() == bytes([SENT]) * n
    finally:
        e0.close()


# ------------------------------------------------------------------------------------------------------------- errors
def test_error_codes(engine_lib):
    """Argument checks of both forms, through the C ABI."""
    import ctypes
    import torch
    import aesgcm_b200
    E = aesgcm_b200._lib
    L = engine_lib
    dev = torch.zeros(8192, dtype=torch.uint8, device="cuda")
    d, iv, tag = dev.data_ptr(), (ctypes.c_uint8 * 12)(), (ctypes.c_uint8 * 16)()
    h_buf = (ctypes.c_uint8 * 4096)()
    ok = ctypes.c_int(0)

    def dev_call(e, tag_p=d, ok_p=d + 16, aad_len=0, blocks_after=0, first_block=0, n=64, total=64):
        return L.agcm_stream_decrypt_verified_peer(e._ctx, ctypes.addressof(iv), 12, first_block, d + 64, d + 4096, n,
                                                   blocks_after, d + 32, aad_len, total, tag_p, ok_p, 0)

    def host_call(e, tag_p=True, ok_p=True, aad_len=0, blocks_after=0, n=64, total=64):
        return L.agcm_stream_decrypt_verified_peer_host(e._ctx, ctypes.addressof(iv), 12, 0, ctypes.addressof(h_buf),
                                                        ctypes.addressof(h_buf), n, blocks_after, ctypes.addressof(h_buf),
                                                        aad_len, total, ctypes.addressof(tag) if tag_p else None,
                                                        ctypes.byref(ok) if ok_p else None)

    xbuf = torch.zeros(4096, dtype=torch.uint8, device="cuda")   # exchange buffer of a world of one
    e = aesgcm_b200.GcmEngine(0)
    try:
        assert dev_call(e) == E.E_NO_KEY
        e.peer_setup(0, 1, [xbuf.data_ptr()])   # the host form checks the setup first
        assert host_call(e) == E.E_NO_KEY
        e.close()
        e = aesgcm_b200.GcmEngine(0)
        e.set_key(bytes(16))
        assert dev_call(e) == E.E_BAD_ARG and host_call(e) == E.E_BAD_ARG        # no agcm_peer_setup
        e.peer_setup(0, 1, [xbuf.data_ptr()])
        assert dev_call(e, tag_p=None) == E.E_BAD_ARG and dev_call(e, ok_p=None) == E.E_BAD_ARG
        assert host_call(e, tag_p=False) == E.E_BAD_ARG and host_call(e, ok_p=False) == E.E_BAD_ARG
        assert dev_call(e, aad_len=4097) == E.E_BAD_LEN and host_call(e, aad_len=4097) == E.E_BAD_LEN
        assert dev_call(e, blocks_after=1) == E.E_BAD_LEN and host_call(e, blocks_after=1) == E.E_BAD_LEN
        assert dev_call(e, first_block=2, n=64, total=64) == E.E_BAD_LEN
        assert dev_call(e, n=20, total=40, blocks_after=1) == E.E_BAD_LEN   # only the last shard may be ragged
        assert dev_call(e) == E.OK and host_call(e) == E.OK                 # the same arguments, consistent
        torch.cuda.synchronize()
        assert not e.peer_timed_out()
    finally:
        e.close()


# ------------------------------------------------------------------------------------------------------ two real GPUs
def _two_gpu_worker(rank, world, port, q):
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    import aesgcm_b200
    from aesgcm_b200.parallel import PeerExchange, shard_plan
    from cryptography.hazmat.primitives.ciphers.aead import AESGCM
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    rng = np.random.default_rng(9800)
    key, iv, aad = (rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (32, 20, 16))
    n = 3 * 16 * 151552 + 5
    pt = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    out = AESGCM(key).encrypt(iv, pt, aad)
    ct, tag = out[:-16], out[-16:]
    eng = aesgcm_b200.GcmEngine(rank)
    eng.set_key(key)
    px = PeerExchange(eng)
    sh = shard_plan(n, world)[rank]
    dev = torch.device("cuda", rank)
    my_ct, my_pt = ct[sh.byte_offset:sh.byte_offset + sh.n_bytes], pt[sh.byte_offset:sh.byte_offset + sh.n_bytes]
    d_ct = torch.from_numpy(np.frombuffer(my_ct, np.uint8).copy()).to(dev)
    d_aad = torch.from_numpy(np.frombuffer(aad, np.uint8).copy()).to(dev)
    good = True
    for t in (tag, _flip(tag, 5)):
        d_pt = torch.full((sh.n_bytes,), SENT, dtype=torch.uint8, device=dev)
        d_ok = torch.full((1,), 7, dtype=torch.uint8, device=dev)
        px.decrypt_verified(iv, d_aad, sh, d_ct, d_pt, n, torch.from_numpy(np.frombuffer(t, np.uint8).copy()).to(dev), d_ok)
        torch.cuda.synchronize()
        authentic = t == tag
        good = good and int(d_ok.item()) == int(authentic)
        good = good and d_pt.cpu().numpy().tobytes() == (my_pt if authentic else bytes([SENT]) * sh.n_bytes)
    for forged in (False, True):
        h_ct = _flip(my_ct, 0) if forged and rank == 0 else my_ct   # rank 0's ciphertext forged: rank 1 must refuse too
        h_pt = np.full(sh.n_bytes, SENT, np.uint8)
        okh = px.decrypt_verified_host(iv, aad, sh, np.frombuffer(h_ct, np.uint8), h_pt, n, tag)
        good = good and okh == (not forged) and h_pt.tobytes() == (bytes([SENT]) * sh.n_bytes if forged else my_pt)
    good = good and not eng.peer_timed_out()
    q.put((rank, bool(good)))
    dist.barrier()
    dist.destroy_process_group()
    eng.close()


def test_two_gpus(engine_lib):
    """PeerExchange.decrypt_verified / decrypt_verified_host between 2 processes on 2 GPUs: one authentic and one forged
    message through each form."""
    import socket
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
    assert res == [(0, True), (1, True)]
