"""Host-side engine over the C ABI (include/aesgcm_b200.h).

`GcmEngine` owns one `agcm_ctx` on one GPU.  Two families of calls:

* host-buffer calls (`encrypt`, `decrypt`, `crypt_batch_uniform_host`, `stream_part_host`, ...) take
  bytes / numpy arrays / pinned torch CPU tensors and go through the library's
  chunked H2D -> kernel -> D2H pipeline: this is the call a user of the reference
  model makes (tb/gcm_model.py:8-51 semantics, whole message at a time);
* device calls (`stream_crypt_device`, `batch_crypt_*_device`, `stream_part_device`,
  `stream_finish_device`) take torch CUDA uint8 tensors already resident in HBM.

All arithmetic runs in the CUDA library; nothing here computes AES or GHASH.

A context owns scratch buffers (per-CTA partials, tickets, the cached H^n): issue the calls of one
engine on ONE CUDA stream at a time; use one engine per concurrently active stream.
"""
import ctypes

import numpy as np

from . import _lib

MODES = {128: 16, 192: 24, 256: 32}
EXPANDED = {176: 128, 208: 192, 240: 256}


class AuthenticationError(ValueError):
    """Tag mismatch on decrypt (pycryptodome raises ValueError: tb/gcm_model.py:46)."""


def _np_u8(b):
    if isinstance(b, np.ndarray):
        a = b if (b.dtype == np.uint8 and b.flags["C_CONTIGUOUS"]) else np.ascontiguousarray(b, dtype=np.uint8)
        return a.reshape(-1)
    if b is None:
        return np.zeros(0, dtype=np.uint8)
    if hasattr(b, "numpy") and hasattr(b, "is_cuda"):  # torch CPU tensor (shares memory, keeps pinning)
        if b.is_cuda:
            raise TypeError("host-buffer call got a CUDA tensor; use the *_device methods")
        return b.contiguous().view(-1).numpy()
    return np.frombuffer(bytes(b), dtype=np.uint8)


def _addr(a):
    return a.ctypes.data if a.size else 0


def _dptr(t):
    """torch CUDA uint8 tensor (or None) -> device address."""
    if t is None:
        return 0
    if not t.is_cuda or not t.is_contiguous():
        raise TypeError("expected a contiguous CUDA tensor")
    return t.data_ptr()


class GcmEngine:
    def __init__(self, device=0, n_cta=0, threads=0):
        self._L = _lib.lib()
        self._j0_cache = {}
        self._ctx = ctypes.c_void_p()
        rc = self._L.agcm_ctx_create_ex(ctypes.byref(self._ctx), int(device), int(n_cta), int(threads))
        if rc:
            self._ctx = ctypes.c_void_p()
            raise _lib.AgcmError(rc)
        self.device = int(device)
        self.mode = None
        a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        self._L.agcm_get_info(self._ctx, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        self.n_cta, self.threads, self.sm_count = a.value, b.value, c.value

    # -- lifetime ------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._L.agcm_ctx_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, rc):
        return _lib.check(rc, self._ctx)

    @property
    def launch_count(self):
        return int(self._L.agcm_launch_count(self._ctx))

    # -- keys ----------------------------------------------------------------
    def set_key(self, key, pre_expanded=None):
        """Raw 16/24/32-byte key (expanded on the device) or 176/208/240-byte
        pre-expanded stages (tb/gcm_gctr.py:144-214)."""
        k = _np_u8(key)
        n = k.size
        if pre_expanded is None:
            pre_expanded = n in EXPANDED
        mode = EXPANDED.get(n) if pre_expanded else {v: m for m, v in MODES.items()}.get(n)
        if mode is None:
            raise _lib.AgcmError(_lib.E_BAD_MODE, "key of %d bytes" % n)
        self._ck(self._L.agcm_set_key(self._ctx, mode, int(bool(pre_expanded)), _addr(k), n))
        self.mode = mode
        kb = (bool(pre_expanded), k.tobytes())
        if kb != getattr(self, "_key_loaded", None):   # the library itself keeps H when the same key is loaded again
            self._key_loaded = kb
            self._j0_cache = {}
        return self

    def derive_j0(self, iv):
        """The pre-counter block J0 of an IV of any length (SP 800-38D 7.1), computed on the device;
        96-bit IVs give IV || 00000001.  Cached per (key, IV)."""
        ivb = bytes(_np_u8(iv).tobytes())
        j0 = getattr(self, "_j0_cache", {}).get(ivb)
        if j0 is None:
            a = np.frombuffer(ivb, dtype=np.uint8)
            out = np.zeros(16, dtype=np.uint8)
            if a.size == 0:
                raise _lib.AgcmError(_lib.E_BAD_LEN, "empty IV")
            self._ck(self._L.agcm_derive_j0(self._ctx, _addr(a), a.size, _addr(out)))
            j0 = out.tobytes()
            if len(self._j0_cache) > 64:
                self._j0_cache.clear()
            self._j0_cache[ivb] = j0
        return j0

    def _iv_or_j0(self, iv):
        """(array, is_j0): the 12 IV bytes for the plain entry points, else J0 for the *_j0 forms."""
        ivb = _np_u8(iv)
        if ivb.size == 12:
            return ivb, False
        return np.frombuffer(self.derive_j0(ivb), dtype=np.uint8), True

    def round_keys(self):
        out = np.zeros(240, dtype=np.uint8)
        n = self._ck(self._L.agcm_get_round_keys(self._ctx, _addr(out), 240))
        return out[:n].tobytes()

    def hash_subkey(self):
        out = np.zeros(16, dtype=np.uint8)
        self._ck(self._L.agcm_get_h(self._ctx, _addr(out)))
        return out.tobytes()

    def expand_key_host(self, key):
        """tb/key_exp.py:118 for one key, on the device; returns bytes (176/208/240)."""
        k = _np_u8(key)
        mode = {v: m for m, v in MODES.items()}.get(k.size)
        if mode is None:
            raise _lib.AgcmError(_lib.E_BAD_MODE, "key of %d bytes" % k.size)
        out = np.zeros(240, dtype=np.uint8)
        self._ck(self._L.agcm_key_expand_host(self._ctx, mode, _addr(k), _addr(out)))
        return out[: 4 * MODES[mode] + 112].tobytes()

    def expand_keys_device(self, mode, keys, round_keys=None, stream=None):
        """keys: CUDA uint8 [n, mode/8] -> round_keys CUDA uint8 [n, (Nr+1)*16]."""
        import torch
        kb = MODES[mode]
        n = keys.numel() // kb
        if round_keys is None:
            round_keys = torch.empty((n, 4 * kb + 112), dtype=torch.uint8, device=keys.device)
        self._ck(self._L.agcm_key_expand(self._ctx, mode, _dptr(keys), n, _dptr(round_keys), _stream(stream)))
        return round_keys

    # -- host-buffer whole-message calls ---------------------------------------
    def encrypt(self, iv, aad, pt, out=None):
        """-> (ct, tag).  `out`: optional preallocated uint8 numpy array / pinned tensor."""
        return self._crypt_host(0, iv, aad, pt, None, out)

    def decrypt(self, iv, aad, ct, tag, out=None, raise_on_fail=True):
        """-> pt; raises AuthenticationError on tag mismatch (or returns (pt, ok))."""
        pt, ok = self._crypt_host(1, iv, aad, ct, tag, out)
        if raise_on_fail:
            if not ok:
                raise AuthenticationError("MAC check failed")
            return pt
        return pt, ok

    def decrypt_verified(self, iv, aad, ct, tag, out=None, raise_on_fail=True):
        """Verify-then-release: GHASH + tag check first, GCTR only when the tag matches; on a
        mismatch no plaintext byte is produced (`out` untouched).  -> pt, or (pt | None, ok)."""
        ivb, a, d, tb = _np_u8(iv), _np_u8(aad), _np_u8(ct), _np_u8(tag)
        if tb.size != 16:
            raise _lib.AgcmError(_lib.E_BAD_LEN, "tag must be 16 bytes")
        ret_bytes = out is None
        o = np.zeros(d.size, dtype=np.uint8) if out is None else _np_u8(out)
        if o.size < d.size:
            raise _lib.AgcmError(_lib.E_BAD_LEN, "output buffer too small")
        ok = ctypes.c_int(0)
        self._ck(self._L.agcm_stream_decrypt_verified_host(self._ctx, _addr(ivb), ivb.size, _addr(a), a.size, _addr(d),
                                                           _addr(o), d.size, _addr(tb), ctypes.byref(ok)))
        if not ok.value:
            if raise_on_fail:
                raise AuthenticationError("MAC check failed")
            return None, False
        res = o[: d.size].tobytes() if ret_bytes else o[: d.size]
        return res if raise_on_fail else (res, True)

    def _crypt_host(self, decrypt, iv, aad, data, tag, out):
        ivb = _np_u8(iv)   # 96 bits as in the reference IP (src/gcm_pkg.vhd:17), or any other length (SP 800-38D J0)
        if ivb.size == 0:
            raise _lib.AgcmError(_lib.E_BAD_LEN, "empty IV")
        a = _np_u8(aad)
        d = _np_u8(data)
        ret_bytes = out is None
        o = np.empty(d.size, dtype=np.uint8) if out is None else _np_u8(out)
        if o.size < d.size:
            raise _lib.AgcmError(_lib.E_BAD_LEN, "output buffer too small")
        t = np.zeros(16, dtype=np.uint8)
        if decrypt:
            tb = _np_u8(tag)
            if tb.size != 16:
                raise _lib.AgcmError(_lib.E_BAD_LEN, "tag must be 16 bytes")
            t[:] = tb
        ok = ctypes.c_int(1)
        self._ck(self._L.agcm_stream_crypt_iv_host(self._ctx, decrypt, _addr(ivb), ivb.size, _addr(a), a.size, _addr(d),
                                                   _addr(o), d.size, _addr(t), ctypes.byref(ok)))
        res = o[: d.size].tobytes() if ret_bytes else o[: d.size]
        if decrypt:
            return res, bool(ok.value)
        return res, t.tobytes()

    def stream_part_host(self, decrypt, iv, first_block, data, out, blocks_after):
        """One rank's counter-range shard, host buffers -> 16-byte partial (bytes)."""
        ivb, d, o = _np_u8(iv), _np_u8(data), _np_u8(out)
        part = np.zeros(16, dtype=np.uint8)
        self._ck(self._L.agcm_stream_part_host(self._ctx, int(decrypt), _addr(ivb), int(first_block), _addr(d), _addr(o),
                                               d.size, int(blocks_after), _addr(part)))
        return part.tobytes()

    def stream_finish_host(self, decrypt, iv, partials, aad, ct_len, tag=None):
        """partials: bytes / array of n x 16.  -> tag (encrypt) or ok flag (decrypt)."""
        ivb, p, a = _np_u8(iv), _np_u8(partials), _np_u8(aad)
        t = np.zeros(16, dtype=np.uint8)
        if decrypt:
            t[:] = _np_u8(tag)
        ok = ctypes.c_int(1)
        self._ck(self._L.agcm_stream_finish_host(self._ctx, int(decrypt), _addr(ivb), _addr(p), p.size // 16, _addr(a),
                                                 a.size, int(ct_len), _addr(t), ctypes.byref(ok)))
        return bool(ok.value) if decrypt else t.tobytes()

    def stream_crypt_peer_host(self, decrypt, iv, first_block, data, out, blocks_after, aad, total_len, tag=None):
        """One rank's shard in HOST memory + peer-memory exchange + finish.  -> tag (encrypt) / ok (decrypt)."""
        ivb, d, o, a = _np_u8(iv), _np_u8(data), _np_u8(out), _np_u8(aad)
        t = np.zeros(16, dtype=np.uint8)
        if decrypt:
            t[:] = _np_u8(tag)
        ok = ctypes.c_int(1)
        self._ck(self._L.agcm_stream_crypt_peer_host(self._ctx, int(decrypt), _addr(ivb), int(first_block), _addr(d), _addr(o),
                                                     d.size, int(blocks_after), _addr(a), a.size, int(total_len), _addr(t),
                                                     ctypes.byref(ok)))
        return bool(ok.value) if decrypt else t.tobytes()

    def stream_decrypt_verified_peer_host(self, iv, first_block, ct, pt, blocks_after, aad, total_len, tag):
        """Verify-then-release form of stream_crypt_peer_host(1, ...): `pt` is written only if the whole message's tag
        matches on every rank.  IV of any length.  -> ok."""
        ivb, d, o, a, tb = _np_u8(iv), _np_u8(ct), _np_u8(pt), _np_u8(aad), _np_u8(tag)
        if tb.size != 16:
            raise _lib.AgcmError(_lib.E_BAD_LEN, "tag must be 16 bytes")
        if o.size < d.size:
            raise _lib.AgcmError(_lib.E_BAD_LEN, "output buffer too small")
        ok = ctypes.c_int(0)
        self._ck(self._L.agcm_stream_decrypt_verified_peer_host(self._ctx, _addr(ivb), ivb.size, int(first_block), _addr(d),
                                                                _addr(o), d.size, int(blocks_after), _addr(a), a.size,
                                                                int(total_len), _addr(tb), ctypes.byref(ok)))
        return bool(ok.value)

    def timing_enable(self, on=True):
        self._ck(self._L.agcm_timing_enable(self._ctx, int(bool(on))))

    def timing_read(self):
        """(total_ms, launches) of the fused stream kernel since timing_enable."""
        ms, n = ctypes.c_double(), ctypes.c_uint64()
        self._ck(self._L.agcm_timing_read(self._ctx, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, int(n.value)

    def crypt_batch_uniform_host(self, decrypt, ivs, aad, aad_len, aad_stride, data, out, length, stride, tags, ok=None,
                                 lanes=0):
        """Fixed-size records in host memory (numpy / pinned tensors); in-place allowed."""
        ivs, a, d, o, t = _np_u8(ivs), _np_u8(aad), _np_u8(data), _np_u8(out), _np_u8(tags)
        n = ivs.size // 12
        okb = _np_u8(ok) if ok is not None else np.zeros(0, dtype=np.uint8)
        self._ck(self._L.agcm_batch_crypt_uniform_host(self._ctx, int(decrypt), int(lanes), _addr(ivs), _addr(a),
                                                       int(aad_len), int(aad_stride), _addr(d), _addr(o), int(length),
                                                       int(stride), _addr(t), _addr(okb), n))

    # -- device-resident calls ---------------------------------------------------
    def stream_crypt_device(self, decrypt, iv, aad, data_in, data_out, tag, ok=None, n_bytes=None, stream=None):
        ivb = _np_u8(iv)
        n = data_in.numel() if n_bytes is None else int(n_bytes)
        self._ck(self._L.agcm_stream_crypt_iv(self._ctx, int(decrypt), _addr(ivb), ivb.size, _dptr(aad),
                                              0 if aad is None else aad.numel(), _dptr(data_in), _dptr(data_out), n,
                                              _dptr(tag), _dptr(ok), _stream(stream)))

    def stream_decrypt_verified_device(self, iv, aad, ct, pt, tag, ok, n_bytes=None, stream=None):
        """Device form of decrypt_verified: `pt` is written only if `tag` matches (then ok[0] = 1)."""
        ivb = _np_u8(iv)
        n = ct.numel() if n_bytes is None else int(n_bytes)
        self._ck(self._L.agcm_stream_decrypt_verified(self._ctx, _addr(ivb), ivb.size, _dptr(aad),
                                                      0 if aad is None else aad.numel(), _dptr(ct), _dptr(pt), n, _dptr(tag),
                                                      _dptr(ok), _stream(stream)))

    def stream_part_device(self, decrypt, iv, first_block, data_in, data_out, blocks_after, partial16, n_bytes=None,
                           stream=None):
        ivb, j0 = self._iv_or_j0(iv)
        n = data_in.numel() if n_bytes is None else int(n_bytes)
        fn = self._L.agcm_stream_part_j0 if j0 else self._L.agcm_stream_part
        self._ck(fn(self._ctx, int(decrypt), _addr(ivb), int(first_block), _dptr(data_in), _dptr(data_out), n,
                    int(blocks_after), _dptr(partial16), _stream(stream)))

    def stream_finish_device(self, decrypt, iv, partials16, n_parts, aad, ct_len, tag, ok=None, stream=None):
        ivb, j0 = self._iv_or_j0(iv)
        fn = self._L.agcm_stream_finish_j0 if j0 else self._L.agcm_stream_finish
        self._ck(fn(self._ctx, int(decrypt), _addr(ivb), _dptr(partials16), int(n_parts), _dptr(aad),
                    0 if aad is None else aad.numel(), int(ct_len), _dptr(tag), _dptr(ok), _stream(stream)))

    def peer_setup(self, rank, world, peer_ptrs):
        """peer_ptrs: device addresses (ints) of every rank's exchange buffer, mapped in this process."""
        arr = (ctypes.c_uint64 * world)(*[int(p) for p in peer_ptrs])
        self._ck(self._L.agcm_peer_setup(self._ctx, int(rank), int(world), arr))

    def peer_export(self):
        """-> the handle (bytes) of this context's exchange buffer, allocated on the first call; every rank hands its
        handle to every other rank (any transport) for peer_import."""
        out = np.zeros(_lib.PEER_HANDLE_BYTES, dtype=np.uint8)
        self._ck(self._L.agcm_peer_export(self._ctx, _addr(out)))
        return out.tobytes()

    def peer_import(self, rank, world, handles):
        """handles: the world's peer_export() results in rank order (entry `rank` is this engine's own).  Maps the
        other ranks' buffers and sets up the exchange; barrier the ranks before the first peer call."""
        if len(handles) != int(world) or any(len(h) != _lib.PEER_HANDLE_BYTES for h in handles):
            raise _lib.AgcmError(_lib.E_BAD_ARG, "expected %d handles of %d bytes" % (int(world), _lib.PEER_HANDLE_BYTES))
        arr = np.frombuffer(b"".join(bytes(h) for h in handles), dtype=np.uint8)
        self._ck(self._L.agcm_peer_import(self._ctx, int(rank), int(world), _addr(arr)))

    def peer_close(self):
        """Unmap the other ranks' buffers and leave the world (every rank, then a barrier, then close())."""
        self._ck(self._L.agcm_peer_close(self._ctx))

    def peer_timed_out(self):
        v = ctypes.c_int()
        self._ck(self._L.agcm_peer_status(self._ctx, ctypes.byref(v)))
        return bool(v.value)

    def stream_crypt_peer_device(self, decrypt, iv, first_block, data_in, data_out, blocks_after, aad, total_len, tag, ok=None,
                                 n_bytes=None, stream=None, defer=False):
        """One rank's shard + peer-memory exchange + tag finish (every rank calls it).  defer=True:
        do not make `stream` wait for the finish -- call peer_join() before reading tag / ok."""
        ivb, j0 = self._iv_or_j0(iv)
        n = (0 if data_in is None else data_in.numel()) if n_bytes is None else int(n_bytes)
        args = (self._ctx, int(decrypt), _addr(ivb), int(first_block), _dptr(data_in), _dptr(data_out), n, int(blocks_after),
                _dptr(aad), 0 if aad is None else aad.numel(), int(total_len), _dptr(tag), _dptr(ok), _stream(stream))
        if j0:
            self._ck(self._L.agcm_stream_crypt_peer_j0(*args, int(bool(defer))))
        else:
            self._ck((self._L.agcm_stream_crypt_peer_async if defer else self._L.agcm_stream_crypt_peer)(*args))

    def stream_decrypt_verified_peer_device(self, iv, first_block, ct, pt, blocks_after, aad, total_len, tag, ok, n_bytes=None,
                                            stream=None):
        """Verify-then-release form of stream_crypt_peer_device(1, ...): ok[0] = 1 on every rank if and only if the whole
        message's tag matches, and only then is this rank's `pt` written.  IV of any length; no deferred form."""
        ivb = _np_u8(iv)
        n = (0 if ct is None else ct.numel()) if n_bytes is None else int(n_bytes)
        self._ck(self._L.agcm_stream_decrypt_verified_peer(self._ctx, _addr(ivb), ivb.size, int(first_block), _dptr(ct),
                                                           _dptr(pt), n, int(blocks_after), _dptr(aad),
                                                           0 if aad is None else aad.numel(), int(total_len), _dptr(tag),
                                                           _dptr(ok), _stream(stream)))

    def peer_join(self, stream=None):
        """`stream` waits for every deferred peer finish issued so far (no host synchronisation)."""
        self._ck(self._L.agcm_peer_join(self._ctx, _stream(stream)))

    def gctr_device(self, iv, first_block, data_in, data_out, n_bytes=None, stream=None):
        ivb, j0 = self._iv_or_j0(iv)
        n = data_in.numel() if n_bytes is None else int(n_bytes)
        fn = self._L.agcm_gctr_j0 if j0 else self._L.agcm_gctr
        self._ck(fn(self._ctx, _addr(ivb), int(first_block), _dptr(data_in), _dptr(data_out), n, _stream(stream)))

    def ghash_device(self, data_in, y16, n_bytes=None, stream=None):
        n = data_in.numel() if n_bytes is None else int(n_bytes)
        self._ck(self._L.agcm_ghash(self._ctx, _dptr(data_in), n, _dptr(y16), _stream(stream)))

    def batch_derive_j0_device(self, ivs, iv_off=None, iv_len=0, n_msgs=None, j0=None, stream=None):
        """n IVs of any lengths (iv_off: CUDA int64 [n+1] byte offsets, or fixed iv_len) -> CUDA uint8 [n, 16] J0 blocks
        for batch_crypt_device(..., j0=True)."""
        import torch
        n = (iv_off.numel() - 1) if iv_off is not None else (ivs.numel() // int(iv_len) if n_msgs is None else int(n_msgs))
        if j0 is None:
            j0 = torch.empty((n, 16), dtype=torch.uint8, device=ivs.device)
        self._ck(self._L.agcm_batch_derive_j0(self._ctx, _dptr(ivs), _dptr(iv_off), int(iv_len), n, _dptr(j0), _stream(stream)))
        return j0

    def batch_crypt_device(self, decrypt, ivs, aad, aad_off, data_in, in_off, data_out, tags, ok=None, lanes=0,
                           avg_len_hint=0, stream=None, j0=False):
        """ivs: [n, 12] IVs, or (j0=True) the [n, 16] J0 blocks of batch_derive_j0_device."""
        n = in_off.numel() - 1
        fn = self._L.agcm_batch_crypt_j0 if j0 else self._L.agcm_batch_crypt
        self._ck(fn(self._ctx, int(decrypt), int(lanes), int(avg_len_hint), _dptr(ivs), _dptr(aad), _dptr(aad_off),
                    _dptr(data_in), _dptr(in_off), _dptr(data_out), _dptr(tags), _dptr(ok), n, _stream(stream)))

    def batch_crypt_uniform_device(self, decrypt, ivs, aad, aad_len, aad_stride, data_in, data_out, length, stride, tags,
                                   ok=None, n_msgs=None, lanes=0, stream=None, j0=False):
        n = ivs.numel() // (16 if j0 else 12) if n_msgs is None else int(n_msgs)
        fn = self._L.agcm_batch_crypt_uniform_j0 if j0 else self._L.agcm_batch_crypt_uniform
        self._ck(fn(self._ctx, int(decrypt), int(lanes), _dptr(ivs), _dptr(aad), int(aad_len), int(aad_stride), _dptr(data_in),
                    _dptr(data_out), int(length), int(stride), _dptr(tags), _dptr(ok), n, _stream(stream)))

    def batch_crypt_slots_device(self, decrypt, ivs, aad, aad_lens, aad_len, aad_stride, data_in, data_out, lens, stride, tags,
                                 ok=None, n_msgs=None, lanes=0, avg_len_hint=0, stream=None):
        """Fixed-pitch slots, per-message lengths: `lens` / `aad_lens` are CUDA int32/uint32 tensors [n] (aad_lens may be
        None: `aad_len` for all; aad None: no AAD)."""
        n = lens.numel() if n_msgs is None else int(n_msgs)
        self._ck(self._L.agcm_batch_crypt_slots(self._ctx, int(decrypt), int(lanes), _dptr(ivs), _dptr(aad), _dptr(aad_lens),
                                                int(aad_len), int(aad_stride), _dptr(data_in), _dptr(data_out), _dptr(lens),
                                                int(stride), int(avg_len_hint), _dptr(tags), _dptr(ok), n, _stream(stream)))

    # Verify-then-release forms of the batch decrypts above: message i's plaintext is written only if ok[i] == 1, and no
    # other byte of data_out is touched (failed messages, gaps, slot and record padding).  data_out may be data_in.
    def batch_decrypt_verified_device(self, ivs, aad, aad_off, data_in, in_off, data_out, tags, ok, lanes=0, avg_len_hint=0,
                                      stream=None, j0=False):
        n = in_off.numel() - 1
        fn = self._L.agcm_batch_decrypt_verified_j0 if j0 else self._L.agcm_batch_decrypt_verified
        self._ck(fn(self._ctx, int(lanes), int(avg_len_hint), _dptr(ivs), _dptr(aad), _dptr(aad_off), _dptr(data_in),
                    _dptr(in_off), _dptr(data_out), _dptr(tags), _dptr(ok), n, _stream(stream)))

    def batch_decrypt_verified_uniform_device(self, ivs, aad, aad_len, aad_stride, data_in, data_out, length, stride, tags, ok,
                                              n_msgs=None, lanes=0, stream=None, j0=False):
        n = ivs.numel() // (16 if j0 else 12) if n_msgs is None else int(n_msgs)
        fn = self._L.agcm_batch_decrypt_verified_uniform_j0 if j0 else self._L.agcm_batch_decrypt_verified_uniform
        self._ck(fn(self._ctx, int(lanes), _dptr(ivs), _dptr(aad), int(aad_len), int(aad_stride), _dptr(data_in),
                    _dptr(data_out), int(length), int(stride), _dptr(tags), _dptr(ok), n, _stream(stream)))

    def batch_decrypt_verified_slots_device(self, ivs, aad, aad_lens, aad_len, aad_stride, data_in, data_out, lens, stride, tags,
                                            ok, n_msgs=None, lanes=0, avg_len_hint=0, stream=None):
        n = lens.numel() if n_msgs is None else int(n_msgs)
        self._ck(self._L.agcm_batch_decrypt_verified_slots(self._ctx, int(lanes), _dptr(ivs), _dptr(aad), _dptr(aad_lens),
                                                           int(aad_len), int(aad_stride), _dptr(data_in), _dptr(data_out),
                                                           _dptr(lens), int(stride), int(avg_len_hint), _dptr(tags), _dptr(ok),
                                                           n, _stream(stream)))

    def batch_decrypt_verified_perkey_device(self, mode, keys, ivs, aad, aad_off, data_in, in_off, data_out, tags, ok,
                                             stream=None):
        n = in_off.numel() - 1
        self._ck(self._L.agcm_batch_decrypt_verified_perkey(self._ctx, int(mode), _dptr(keys), _dptr(ivs), _dptr(aad),
                                                            _dptr(aad_off), _dptr(data_in), _dptr(in_off), _dptr(data_out),
                                                            _dptr(tags), _dptr(ok), n, _stream(stream)))

    def batch_decrypt_verified_perkey_uniform_device(self, mode, keys, ivs, aad, aad_len, aad_stride, data_in, data_out, length,
                                                     stride, tags, ok, n_msgs=None, stream=None):
        n = ivs.numel() // 12 if n_msgs is None else int(n_msgs)
        self._ck(self._L.agcm_batch_decrypt_verified_perkey_uniform(self._ctx, int(mode), _dptr(keys), _dptr(ivs), _dptr(aad),
                                                                    int(aad_len), int(aad_stride), _dptr(data_in),
                                                                    _dptr(data_out), int(length), int(stride), _dptr(tags),
                                                                    _dptr(ok), n, _stream(stream)))

    def batch_crypt_perkey_device(self, mode, decrypt, keys, ivs, aad, aad_off, data_in, in_off, data_out, tags, ok=None,
                                  stream=None):
        """One distinct raw key per message (keys: CUDA uint8 [n, mode/8]); BASELINE config 4."""
        n = in_off.numel() - 1
        self._ck(self._L.agcm_batch_crypt_perkey(self._ctx, int(mode), int(decrypt), _dptr(keys), _dptr(ivs), _dptr(aad),
                                                 _dptr(aad_off), _dptr(data_in), _dptr(in_off), _dptr(data_out),
                                                 _dptr(tags), _dptr(ok), n, _stream(stream)))

    def batch_crypt_perkey_uniform_device(self, mode, decrypt, keys, ivs, aad, aad_len, aad_stride, data_in, data_out,
                                          length, stride, tags, ok=None, n_msgs=None, stream=None):
        n = ivs.numel() // 12 if n_msgs is None else int(n_msgs)
        self._ck(self._L.agcm_batch_crypt_perkey_uniform(self._ctx, int(mode), int(decrypt), _dptr(keys), _dptr(ivs),
                                                         _dptr(aad), int(aad_len), int(aad_stride), _dptr(data_in),
                                                         _dptr(data_out), int(length), int(stride), _dptr(tags),
                                                         _dptr(ok), n, _stream(stream)))


def _stream(stream):
    if stream is None:
        try:
            import torch
            if torch.cuda.is_available():
                return torch.cuda.current_stream().cuda_stream
        except Exception:
            pass
        return 0
    return getattr(stream, "cuda_stream", stream)
