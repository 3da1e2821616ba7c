"""The peer exchange set up through the C ABI alone: agcm_peer_export / agcm_peer_import / agcm_peer_close.

One process: worlds of 1, 2 and 4 contexts on GPU 0 whose exchange buffers the library allocated and handed over as
handles (a context of the exporting process uses the buffer at its own address), checked byte for byte against OpenSSL
(`cryptography`).  Two processes: the gcc-only client tests/peer_ipc_example.c as rank 0 and rank 1, on one GPU and, where
there are two, on two, mapping each other's buffers with CUDA IPC.  Every output buffer starts as a sentinel."""
import ctypes
import os
import shutil
import subprocess
import time

import numpy as np
import pytest

from conftest import ROOT

SENT = 0x5A


def _compile_client(out_dir):
    import aesgcm_b200
    gcc = shutil.which("gcc")
    if not gcc:
        pytest.skip("gcc not available")
    pkg = os.path.dirname(aesgcm_b200._lib.SO_PATH)
    exe = os.path.join(str(out_dir), "peer_ipc_example")
    subprocess.check_call([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "peer_ipc_example.c"), "-L", pkg, "-laesgcm_b200",
                           "-Wl,-rpath," + pkg, "-o", exe])
    return exe


def test_client_compiles(engine_lib, tmp_path):
    """tests/peer_ipc_example.c is plain C99 against the header and links against the library."""
    assert os.path.exists(_compile_client(tmp_path))


# ------------------------------------------------------------------------------------------------------ helpers (GPU)
def _aesgcm(key, iv, aad, pt):
    """-> (ct, tag) from OpenSSL"""
    from cryptography.hazmat.primitives.ciphers.aead import AESGCM
    out = AESGCM(key).encrypt(iv, pt, aad)
    return out[:-16], out[-16:]


def _t(b):
    import torch
    return torch.from_numpy(np.frombuffer(bytes(b), np.uint8).copy()).cuda()


def _h(t):
    return t.cpu().numpy().tobytes()


def _flip(b, i, bit=0):
    b = bytearray(b)
    b[i] ^= 1 << bit
    return bytes(b)


def _load_stream_kernels(eng):
    """Launches every stream-kernel variant the exchanges below use (encrypt, decrypt, GHASH-only, gated GCTR; 16-byte
    aligned and not) once for the loaded key size.  The ranks of an emulated world share one CUDA context, in which the
    first launch of a kernel loads it lazily and waits for the running kernels -- among them another rank's finish, which
    waits for this rank's post -- so an exchange that met an unloaded kernel would stall until the timeout."""
    import torch
    buf = torch.zeros(80, dtype=torch.uint8, device="cuda")
    tag, ok = torch.zeros(16, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.uint8, device="cuda")
    for off in (0, 1):
        d = buf[off:off + 64]
        eng.stream_crypt_device(0, bytes(12), None, d, d, tag)
        eng.stream_crypt_device(1, bytes(12), None, d, d, tag, ok)
        eng.stream_decrypt_verified_device(bytes(12), None, d, d, tag, ok)
    torch.cuda.synchronize()


class World:
    """`world` contexts on GPU 0, each with its own stream, set up only through peer_export / peer_import."""

    def __init__(self, world, key):
        import torch
        import aesgcm_b200
        self.world = world
        self.engs = [aesgcm_b200.GcmEngine(0) for _ in range(world)]
        for e in self.engs:
            e.set_key(key)
        _load_stream_kernels(self.engs[0])
        self.streams = [torch.cuda.Stream() for _ in range(world)]
        self.handles = [e.peer_export() for e in self.engs]
        self.imp()

    def imp(self):
        for r, e in enumerate(self.engs):
            e.peer_import(r, self.world, self.handles)

    def close(self):
        for e in self.engs:
            e.peer_close()
        for e in self.engs:
            e.close()


@pytest.fixture
def make_world(engine_lib):
    made = []

    def make(world, key):
        made.append(World(world, key))
        return made[-1]
    yield make
    for w in made:
        w.close()


# ----------------------------------------------------------------------------------------------- one process, 1-4 ranks
@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
def test_crypt_peer_device(make_world, world):
    """stream_crypt_peer_device, encrypt and decrypt, synchronous and deferred in turn, 11 messages per direction (the
    8-deep ring wraps), among them one of 9 bytes (ranks with an empty counter range) and one over a grid row."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    rng = np.random.default_rng(9900 + world)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    w = make_world(world, key)
    msgs = []
    for i in range(11):
        n = (9, 2 * 16 * 151552 + 5)[i] if i < 2 else 16 * (3000 + 101 * i) + i
        iv, aad, pt = (rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (12, 20, n))
        ct, tag = _aesgcm(key, iv, aad, pt)
        msgs.append((n, iv, aad, pt, ct, tag))
    for dec in (0, 1):
        runs = []
        for i, (n, iv, aad, pt, ct, tag) in enumerate(msgs):
            src = _t(ct if dec else pt)
            out = torch.full((n + 16,), SENT, dtype=torch.uint8, device="cuda")
            tags = [_t(tag) if dec else torch.zeros(16, dtype=torch.uint8, device="cuda") for _ in range(world)]
            oks = [torch.full((1,), 7, dtype=torch.uint8, device="cuda") for _ in range(world)]
            runs.append((src, out, tags, oks, _t(aad)))
        torch.cuda.synchronize()
        for i, ((n, iv, aad, pt, ct, tag), (src, out, tags, oks, d_aad)) in enumerate(zip(msgs, runs)):
            for sh in shard_plan(n, world):
                sl = slice(sh.byte_offset, sh.byte_offset + sh.n_bytes)
                w.engs[sh.rank].stream_crypt_peer_device(dec, iv, sh.first_block, src[sl] if sh.n_bytes else None,
                                                         out[sl] if sh.n_bytes else None, sh.blocks_after, d_aad, n,
                                                         tags[sh.rank], oks[sh.rank], n_bytes=sh.n_bytes,
                                                         stream=w.streams[sh.rank], defer=bool(i & 1))
        for e, st in zip(w.engs, w.streams):
            e.peer_join(st)
        torch.cuda.synchronize()
        assert not any(e.peer_timed_out() for e in w.engs)
        for i, ((n, iv, aad, pt, ct, tag), (src, out, tags, oks, d_aad)) in enumerate(zip(msgs, runs)):
            what = (world, dec, i, n)
            assert _h(out) == (pt if dec else ct) + bytes([SENT]) * 16, what
            for r in range(world):
                if dec:
                    assert int(oks[r].item()) == 1, what + (r,)
                else:
                    assert _h(tags[r]) == tag, what + (r,)


def _verified_world(w, iv, aad, ct, tag, flip_rank=None):
    """Every rank decrypts its shard with stream_decrypt_verified_peer_device (rank `flip_rank` with one ciphertext bit
    flipped).  -> [(shard, output bytes, ok)]"""
    import torch
    from aesgcm_b200.parallel import shard_plan
    n = len(ct)
    d_aad, d_tag = _t(aad), _t(tag)
    res = []
    for sh in shard_plan(n, w.world):
        src = ct[sh.byte_offset:sh.byte_offset + sh.n_bytes]
        if sh.rank == flip_rank:
            src = _flip(src, sh.n_bytes // 2, 3)
        out = torch.full((sh.n_bytes + 16,), SENT, dtype=torch.uint8, device="cuda")
        res.append((sh, _t(src) if sh.n_bytes else None, out, torch.full((1,), 7, dtype=torch.uint8, device="cuda")))
    torch.cuda.synchronize()
    for sh, d_ct, out, ok in res:
        w.engs[sh.rank].stream_decrypt_verified_peer_device(iv, sh.first_block, d_ct, out[:sh.n_bytes] if sh.n_bytes else None,
                                                            sh.blocks_after, d_aad, n, d_tag, ok, n_bytes=sh.n_bytes,
                                                            stream=w.streams[sh.rank])
    torch.cuda.synchronize()
    assert not any(e.peer_timed_out() for e in w.engs)
    return [(sh, _h(out), int(ok.item())) for sh, _, out, ok in res]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
def test_decrypt_verified_peer_device(make_world, world):
    """stream_decrypt_verified_peer_device: the authentic message decrypts on every rank; one bit flipped in any one
    rank's ciphertext gives ok = 0 on every rank and leaves every output buffer as it was."""
    rng = np.random.default_rng(9910 + world)
    key = rng.integers(0, 256, 16, dtype=np.uint8).tobytes()
    w = make_world(world, key)
    n = 16 * 151552 + 16 * 777 + 3
    iv, aad, pt = (rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (12, 16, n))
    ct, tag = _aesgcm(key, iv, aad, pt)
    for sh, got, ok in _verified_world(w, iv, aad, ct, tag):
        assert ok == 1 and got == pt[sh.byte_offset:sh.byte_offset + sh.n_bytes] + bytes([SENT]) * 16, sh.rank
    for k in range(world):
        for sh, got, ok in _verified_world(w, iv, aad, ct, tag, flip_rank=k):
            assert ok == 0 and got == bytes([SENT]) * (sh.n_bytes + 16), (k, sh.rank)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
def test_host_forms_against_device_forms(make_world, monkeypatch, world):
    """stream_crypt_peer_host (encrypt) and stream_decrypt_verified_peer_host (authentic, then a flipped tag) on one
    rank, the device forms on the others, each rank taking the host form in turn; 1 MiB granules, so each 3 MiB shard
    takes several."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    monkeypatch.setenv("AGCM_CHUNK_MB", "1")
    rng = np.random.default_rng(9920 + world)
    key = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    w = make_world(world, key)
    n = world * 3 * (1 << 20) - 11
    plan = shard_plan(n, world)
    iv, aad, pt = (rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (12, 16, n))
    ct, tag = _aesgcm(key, iv, aad, pt)
    # In one process, a synchronous host call must not wait for the whole device before it posts (the other ranks'
    # finishes wait for this rank): its host buffers are pinned, and its staging buffers are grown beforehand by the
    # single-GPU host calls (growing frees the old buffer, which waits for every running kernel).
    keep = []

    def pinned(b):
        t = torch.from_numpy(np.frombuffer(bytes(b), np.uint8).copy()).pin_memory()
        keep.append(t)
        return t.numpy()

    for e, sh in zip(w.engs, plan):
        c, t = e.encrypt(iv, aad, pt[:sh.n_bytes])
        assert e.decrypt_verified(iv, aad, c, t) == pt[:sh.n_bytes]
    d_aad, h_aad = _t(aad), pinned(aad)
    for host_rank in range(world):
        hs = plan[host_rank]
        shard = lambda b, sh: b[sh.byte_offset:sh.byte_offset + sh.n_bytes]   # noqa: E731
        # encrypt
        outs = {sh.rank: torch.full((sh.n_bytes + 16,), SENT, dtype=torch.uint8, device="cuda") for sh in plan}
        tags = {sh.rank: torch.zeros(16, dtype=torch.uint8, device="cuda") for sh in plan}
        srcs = {sh.rank: _t(shard(pt, sh)) for sh in plan}
        h_in, h_out = pinned(shard(pt, hs)), pinned(bytes([SENT]) * hs.n_bytes)
        torch.cuda.synchronize()
        for sh in plan:
            if sh.rank != host_rank:
                w.engs[sh.rank].stream_crypt_peer_device(0, iv, sh.first_block, srcs[sh.rank], outs[sh.rank][:sh.n_bytes],
                                                         sh.blocks_after, d_aad, n, tags[sh.rank], stream=w.streams[sh.rank])
        got_tag = w.engs[host_rank].stream_crypt_peer_host(0, iv, hs.first_block, h_in, h_out, hs.blocks_after, h_aad, n)
        torch.cuda.synchronize()
        assert got_tag == tag and h_out.tobytes() == shard(ct, hs), (world, host_rank, "encrypt")
        for sh in plan:
            if sh.rank != host_rank:
                assert _h(tags[sh.rank]) == tag, (world, host_rank, sh.rank)
                assert _h(outs[sh.rank]) == shard(ct, sh) + bytes([SENT]) * 16, (world, host_rank, sh.rank)
        # verify-then-release decrypt
        for t in (tag, _flip(tag, 11, 6)):
            authentic = t == tag
            outs = {sh.rank: torch.full((sh.n_bytes + 16,), SENT, dtype=torch.uint8, device="cuda") for sh in plan}
            oks = {sh.rank: torch.full((1,), 7, dtype=torch.uint8, device="cuda") for sh in plan}
            srcs = {sh.rank: _t(shard(ct, sh)) for sh in plan}
            h_ct, h_pt, h_tag, d_tag = pinned(shard(ct, hs)), pinned(bytes([SENT]) * hs.n_bytes), pinned(t), _t(t)
            torch.cuda.synchronize()
            for sh in plan:
                if sh.rank != host_rank:
                    w.engs[sh.rank].stream_decrypt_verified_peer_device(iv, sh.first_block, srcs[sh.rank],
                                                                        outs[sh.rank][:sh.n_bytes], sh.blocks_after, d_aad,
                                                                        n, d_tag, oks[sh.rank], stream=w.streams[sh.rank])
            ok_host = w.engs[host_rank].stream_decrypt_verified_peer_host(iv, hs.first_block, h_ct, h_pt, hs.blocks_after,
                                                                          h_aad, n, h_tag)
            torch.cuda.synchronize()
            case = (world, host_rank, authentic)
            assert ok_host == authentic, case
            assert h_pt.tobytes() == (shard(pt, hs) if authentic else bytes([SENT]) * hs.n_bytes), case
            for sh in plan:
                if sh.rank != host_rank:
                    assert int(oks[sh.rank].item()) == int(authentic), case + (sh.rank,)
                    want = shard(pt, sh) if authentic else bytes([SENT]) * sh.n_bytes
                    assert _h(outs[sh.rank]) == want + bytes([SENT]) * 16, case + (sh.rank,)
    assert not any(e.peer_timed_out() for e in w.engs)


def _encrypt_ok(w, rng, key):
    """One 2-rank encrypt through the current set-up, checked against OpenSSL."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    n = 16 * 5000 + 9
    iv, aad, pt = (rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (12, 16, n))
    ct, tag = _aesgcm(key, iv, aad, pt)
    src, out, d_aad = _t(pt), torch.zeros(n, dtype=torch.uint8, device="cuda"), _t(aad)
    tags = [torch.zeros(16, dtype=torch.uint8, device="cuda") for _ in range(w.world)]
    for sh in shard_plan(n, w.world):
        sl = slice(sh.byte_offset, sh.byte_offset + sh.n_bytes)
        w.engs[sh.rank].stream_crypt_peer_device(0, iv, sh.first_block, src[sl], out[sl], sh.blocks_after, d_aad, n,
                                                 tags[sh.rank], stream=w.streams[sh.rank])
    torch.cuda.synchronize()
    return _h(out) == ct and all(_h(t) == tag for t in tags) and not any(e.peer_timed_out() for e in w.engs)


@pytest.mark.gpu
def test_handle_checks_and_teardown(make_world):
    """A handle with a wrong magic or version, a buffer under 2560 bytes, a duplicated handle, an entry `rank` that
    belongs to another context, no export yet, null pointers and bad rank / world: AGCM_E_BAD_ARG.  Export is stable.
    After peer_close a peer call gives AGCM_E_BAD_ARG; re-import, a second import and agcm_peer_setup in between work."""
    import torch
    import aesgcm_b200
    E, L = aesgcm_b200._lib, aesgcm_b200._lib.lib()
    rng = np.random.default_rng(9930)
    key = rng.integers(0, 256, 16, dtype=np.uint8).tobytes()
    w = make_world(2, key)
    e0, e1 = w.engs
    h0, h1 = w.handles
    assert len(h0) == E.PEER_HANDLE_BYTES and e0.peer_export() == h0 and h0 != h1
    assert _encrypt_ok(w, rng, key)

    def rc_import(e, rank, handles):
        with pytest.raises(aesgcm_b200.AgcmError) as ei:
            e.peer_import(rank, len(handles), handles)
        return ei.value.rc

    def patched(h, off, value, size=4):
        b = bytearray(h)
        b[off:off + size] = int(value).to_bytes(size, "little")
        return bytes(b)

    assert rc_import(e0, 0, [h0, _flip(h1, 0)]) == E.E_BAD_ARG                       # magic
    assert rc_import(e0, 0, [h0, patched(h1, 4, 2)]) == E.E_BAD_ARG                  # version
    assert rc_import(e0, 0, [h0, patched(h1, 24, 2559, 8)]) == E.E_BAD_ARG          # size under AG_PEER_BYTES
    assert rc_import(e0, 0, [h0, h0]) == E.E_BAD_ARG                                 # duplicated handle
    assert rc_import(e1, 1, [h1, h1]) == E.E_BAD_ARG
    assert rc_import(e0, 0, [h1, h0]) == E.E_BAD_ARG                                 # entry `rank` is another context's
    assert rc_import(e0, 1, [h0, h1]) == E.E_BAD_ARG
    fresh = aesgcm_b200.GcmEngine(0)
    try:
        assert rc_import(fresh, 0, [h0]) == E.E_BAD_ARG                              # nothing exported yet
    finally:
        fresh.close()
    blob = (ctypes.c_uint8 * (2 * E.PEER_HANDLE_BYTES)).from_buffer_copy(h0 + h1)
    for rank, world in ((2, 2), (-1, 2), (0, 0), (0, 17)):
        assert L.agcm_peer_import(e0._ctx, rank, world, ctypes.addressof(blob)) == E.E_BAD_ARG, (rank, world)
    assert L.agcm_peer_import(e0._ctx, 0, 2, None) == E.E_BAD_ARG
    assert L.agcm_peer_export(e0._ctx, None) == E.E_BAD_ARG
    assert L.agcm_peer_import(None, 0, 2, ctypes.addressof(blob)) == E.E_BAD_ARG
    assert L.agcm_peer_close(None) == E.E_BAD_ARG
    # the refused imports left the world as it was
    assert _encrypt_ok(w, rng, key)

    # after peer_close a peer call is refused as before any set-up
    e0.peer_close()
    d = torch.zeros(64, dtype=torch.uint8, device="cuda")
    with pytest.raises(aesgcm_b200.AgcmError) as ei:
        e0.stream_crypt_peer_device(0, bytes(12), 0, d, d, 0, None, 64, d[:16])
    assert ei.value.rc == E.E_BAD_ARG
    with pytest.raises(aesgcm_b200.AgcmError) as ei:
        e0.peer_join()
    assert ei.value.rc == E.E_BAD_ARG
    with pytest.raises(aesgcm_b200.AgcmError) as ei:
        e0.stream_crypt_peer_host(0, bytes(12), 0, bytes(64), np.zeros(64, np.uint8), 0, b"", 64)
    assert ei.value.rc == E.E_BAD_ARG
    w.imp()                                                                          # re-import after close
    assert _encrypt_ok(w, rng, key)
    w.imp()                                                                          # a second import, no close
    assert _encrypt_ok(w, rng, key)
    bufs = [torch.zeros(4096, dtype=torch.uint8, device="cuda") for _ in range(2)]   # caller-owned buffers in between
    for r, e in enumerate(w.engs):
        e.peer_setup(r, 2, [b.data_ptr() for b in bufs])
    assert _encrypt_ok(w, rng, key)
    w.imp()
    assert _encrypt_ok(w, rng, key)
    assert w.engs[0].peer_export() == h0


# ------------------------------------------------------------------------------------------------------ two processes
def _splitmix_bytes(seed, n):
    """The client's input stream: splitmix64 outputs from `seed`, little-endian, cut to n bytes."""
    k = np.arange(1, (n + 7) // 8 + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + k * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return z.astype("<u8").tobytes()[:n]


CLIENT_SEED, CLIENT_N, CLIENT_AAD = 0x5EED5EED, (1 << 20) + 7, 20


def _exclusive_compute_mode(device):
    """True if `device` admits one process only (cudaComputeModeExclusiveProcess or Prohibited): a second process then
    gets cudaErrorDevicesUnavailable."""
    try:
        cudart = ctypes.CDLL("libcudart.so.12")
        v = ctypes.c_int(-1)
        return cudart.cudaDeviceGetAttribute(ctypes.byref(v), 20, int(device)) == 0 and v.value in (2, 3)
    except OSError:
        return False


def _run_ranks(exe, workdir, devices, timeout=300):
    """Runs the client as rank r on devices[r]; kills and reaps every child on a failure or on the timeout.
    -> [(returncode, output)]"""
    procs = []
    try:
        for r, d in enumerate(devices):
            procs.append(subprocess.Popen([exe, str(workdir), str(r), str(len(devices)), str(d)], stdout=subprocess.PIPE,
                                          stderr=subprocess.STDOUT, text=True))
        deadline = time.monotonic() + timeout
        while time.monotonic() < deadline:
            codes = [p.poll() for p in procs]
            if all(c is not None for c in codes) or any(c not in (None, 0) for c in codes):
                break
            time.sleep(0.05)
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
        outs = [p.communicate()[0] for p in procs]
    return [(p.returncode, o) for p, o in zip(procs, outs)]


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [(0, 0), (0, 1)], ids=["one_gpu", "two_gpus"])
def test_two_processes_plain_c(engine_lib, tmp_path, devices):
    """Two processes of the gcc-only client map each other's exchange buffers by CUDA IPC handle and shard one
    1 MiB + 7 B AES-256 message: ciphertext of both shards and the tag on both ranks; the releasing decrypt gives ok = 1
    with the good tag and ok = 0 with a flipped one; the verified decrypt releases the plaintext with the good tag and,
    with the flipped one, gives ok = 0 on both ranks and writes nothing."""
    import torch
    from aesgcm_b200.parallel import shard_plan
    if torch.cuda.device_count() <= max(devices):
        pytest.skip("needs %d GPUs" % (max(devices) + 1))
    exe = _compile_client(tmp_path)
    work = tmp_path / "xchg"
    work.mkdir()
    res = _run_ranks(exe, work, devices)
    if any(rc == 3 for rc, _ in res) and any(_exclusive_compute_mode(d) for d in devices):
        pytest.skip("cudaErrorDevicesUnavailable: the device is in an exclusive-process compute mode, a second process "
                    "cannot create a context on it")
    assert all(rc == 0 for rc, _ in res), res

    raw = _splitmix_bytes(CLIENT_SEED, 64 + CLIENT_N)
    key, iv, aad, pt = raw[:32], raw[32:44], raw[44:64], raw[64:]
    ct, tag = _aesgcm(key, iv, aad, pt)
    read = lambda name, r: (work / ("%s.%d" % (name, r))).read_bytes()   # noqa: E731
    for sh in shard_plan(CLIENT_N, len(devices)):
        r, sl = sh.rank, slice(sh.byte_offset, sh.byte_offset + sh.n_bytes)
        assert read("ct", r) == ct[sl], r
        assert read("tag", r) == tag, r
        assert read("released", r) == pt[sl], r
        assert read("verified", r) == pt[sl], r
        assert read("forged", r) == bytes([SENT]) * sh.n_bytes, r
        assert list(read("ok", r)) == [1, 0, 1, 0], r
