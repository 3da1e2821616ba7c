"""ctypes loader for libaesgcm_b200.so (C ABI: include/aesgcm_b200.h).

The shared library is the product.  It is built in-tree by ``make -C csrc`` (see
``__graft_entry__.build()``) and there is NO fallback: if it is missing or no
sm_100 device is present, every entry point raises.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("AGCM_LIB_PATH") or os.path.join(_HERE, "libaesgcm_b200.so")  # env: development builds only
CSRC = os.path.join(_HERE, "csrc")

OK = 0
E_BAD_MODE, E_BAD_LEN, E_COUNTER_OVERFLOW, E_CUDA, E_NO_KEY, E_BAD_ARG, E_NO_DEVICE, E_PEER_TIMEOUT = -1, -2, -3, -4, -5, -6, -7, -8
PEER_HANDLE_BYTES = 128   # AGCM_PEER_HANDLE_BYTES

c_u8p = ctypes.c_void_p  # raw addresses (host or device) are passed as integers
c_u64 = ctypes.c_uint64
c_sz = ctypes.c_size_t
c_int = ctypes.c_int
c_vp = ctypes.c_void_p

# name -> (restype, argtypes); one entry per symbol declared in include/aesgcm_b200.h
SIGNATURES = {
    "agcm_ctx_create": (c_int, [ctypes.POINTER(c_vp), c_int]),
    "agcm_ctx_create_ex": (c_int, [ctypes.POINTER(c_vp), c_int, c_int, c_int]),
    "agcm_ctx_destroy": (None, [c_vp]),
    "agcm_strerror": (ctypes.c_char_p, [c_int]),
    "agcm_last_cuda_error": (c_int, [c_vp]),
    "agcm_last_cuda_error_string": (ctypes.c_char_p, [c_vp]),
    "agcm_get_info": (c_int, [c_vp, ctypes.POINTER(c_int), ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "agcm_launch_count": (c_u64, [c_vp]),
    "agcm_timing_enable": (c_int, [c_vp, c_int]),
    "agcm_timing_read": (c_int, [c_vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(c_u64)]),
    "agcm_key_expand": (c_int, [c_vp, c_int, c_u8p, c_sz, c_u8p, c_vp]),
    "agcm_key_expand_host": (c_int, [c_vp, c_int, c_u8p, c_u8p]),
    "agcm_set_key": (c_int, [c_vp, c_int, c_int, c_u8p, c_sz]),
    "agcm_get_round_keys": (c_int, [c_vp, c_u8p, c_sz]),
    "agcm_get_h": (c_int, [c_vp, c_u8p]),
    "agcm_stream_crypt": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u8p, c_u8p, c_vp]),
    "agcm_stream_crypt_iv": (c_int, [c_vp, c_int, c_u8p, c_sz, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u8p, c_u8p, c_vp]),
    "agcm_stream_part": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_vp]),
    "agcm_stream_finish": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_int, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_vp]),
    "agcm_peer_export": (c_int, [c_vp, c_u8p]),
    "agcm_peer_import": (c_int, [c_vp, c_int, c_int, c_u8p]),
    "agcm_peer_close": (c_int, [c_vp]),
    "agcm_peer_setup": (c_int, [c_vp, c_int, c_int, ctypes.POINTER(c_u64)]),
    "agcm_peer_status": (c_int, [c_vp, ctypes.POINTER(c_int)]),
    "agcm_stream_crypt_peer": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u64, c_u64, c_u8p,
                                       c_u8p, c_vp]),
    "agcm_stream_decrypt_verified": (c_int, [c_vp, c_u8p, c_sz, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u8p, c_u8p, c_vp]),
    "agcm_stream_decrypt_verified_host": (c_int, [c_vp, c_u8p, c_sz, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u8p,
                                                  ctypes.POINTER(c_int)]),
    "agcm_stream_decrypt_verified_peer": (c_int, [c_vp, c_u8p, c_sz, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u64, c_u64,
                                                  c_u8p, c_u8p, c_vp]),
    "agcm_stream_decrypt_verified_peer_host": (c_int, [c_vp, c_u8p, c_sz, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u64,
                                                       c_u64, c_u8p, ctypes.POINTER(c_int)]),
    "agcm_derive_j0": (c_int, [c_vp, c_u8p, c_sz, c_u8p]),
    "agcm_gctr_j0": (c_int, [c_vp, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_vp]),
    "agcm_stream_part_j0": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_vp]),
    "agcm_stream_finish_j0": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_int, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_vp]),
    "agcm_stream_crypt_peer_j0": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u64, c_u64,
                                          c_u8p, c_u8p, c_vp, c_int]),
    "agcm_batch_crypt_slots": (c_int, [c_vp, c_int, c_int, c_u8p, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u8p, c_u64, c_u64,
                                       c_u8p, c_u8p, c_sz, c_vp]),
    "agcm_batch_derive_j0": (c_int, [c_vp, c_u8p, c_u8p, c_u64, c_sz, c_u8p, c_vp]),
    "agcm_batch_crypt_j0": (c_int, [c_vp, c_int, c_int, c_u64, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                    c_sz, c_vp]),
    "agcm_batch_crypt_uniform_j0": (c_int, [c_vp, c_int, c_int, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u64, c_u64,
                                            c_u8p, c_u8p, c_sz, c_vp]),
    "agcm_peer_join": (c_int, [c_vp, c_vp]),
    "agcm_stream_crypt_peer_async": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u64, c_u64,
                                             c_u8p, c_u8p, c_vp]),
    "agcm_batch_crypt": (c_int, [c_vp, c_int, c_int, c_u64, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                 c_sz, c_vp]),
    "agcm_batch_crypt_uniform": (c_int, [c_vp, c_int, c_int, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u64, c_u64,
                                         c_u8p, c_u8p, c_sz, c_vp]),
    "agcm_batch_crypt_perkey": (c_int, [c_vp, c_int, c_int, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                        c_sz, c_vp]),
    "agcm_batch_crypt_perkey_uniform": (c_int, [c_vp, c_int, c_int, c_u8p, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p,
                                                c_u64, c_u64, c_u8p, c_u8p, c_sz, c_vp]),
    "agcm_batch_decrypt_verified": (c_int, [c_vp, c_int, c_u64, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz,
                                            c_vp]),
    "agcm_batch_decrypt_verified_j0": (c_int, [c_vp, c_int, c_u64, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_sz,
                                               c_vp]),
    "agcm_batch_decrypt_verified_uniform": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p,
                                                    c_u8p, c_sz, c_vp]),
    "agcm_batch_decrypt_verified_uniform_j0": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p,
                                                       c_u8p, c_sz, c_vp]),
    "agcm_batch_decrypt_verified_slots": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u8p, c_u64,
                                                  c_u64, c_u8p, c_u8p, c_sz, c_vp]),
    "agcm_batch_decrypt_verified_perkey": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p, c_u8p,
                                                   c_sz, c_vp]),
    "agcm_batch_decrypt_verified_perkey_uniform": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u64,
                                                           c_u64, c_u8p, c_u8p, c_sz, c_vp]),
    "agcm_stream_crypt_host": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u8p,
                                       ctypes.POINTER(c_int)]),
    "agcm_stream_crypt_iv_host": (c_int, [c_vp, c_int, c_u8p, c_sz, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u8p,
                                          ctypes.POINTER(c_int)]),
    "agcm_stream_part_host": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p]),
    "agcm_stream_finish_host": (c_int, [c_vp, c_int, c_u8p, c_u8p, c_int, c_u8p, c_u64, c_u64, c_u8p,
                                        ctypes.POINTER(c_int)]),
    "agcm_stream_crypt_peer_host": (c_int, [c_vp, c_int, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u64, c_u64, c_u8p,
                                            ctypes.POINTER(c_int)]),
    "agcm_batch_crypt_uniform_host": (c_int, [c_vp, c_int, c_int, c_u8p, c_u8p, c_u64, c_u64, c_u8p, c_u8p, c_u64,
                                              c_u64, c_u8p, c_u8p, c_sz]),
    "agcm_host_alloc": (c_int, [ctypes.POINTER(c_vp), c_sz]),
    "agcm_host_free": (None, [c_vp]),
    "agcm_gctr": (c_int, [c_vp, c_u8p, c_u64, c_u8p, c_u8p, c_u64, c_vp]),
    "agcm_ghash": (c_int, [c_vp, c_u8p, c_u64, c_u8p, c_vp]),
}

_lib = None


def build(verbose=False):
    """Compile the CUDA library for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-j", str(min(4, os.cpu_count() or 1)), "-C", CSRC], stdout=out)
    return SO_PATH


def lib():
    """Load the library; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                "libaesgcm_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C %s`. There is no CPU fallback." % (SO_PATH, CSRC))
        L = ctypes.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the ABI and the header drifted apart
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class AgcmError(RuntimeError):
    def __init__(self, rc, detail=""):
        self.rc = rc
        msg = lib().agcm_strerror(rc).decode()
        super().__init__("aesgcm_b200: %s (rc=%d)%s" % (msg, rc, (": " + detail) if detail else ""))


def check(rc, ctx=None):
    if rc < 0:
        detail = ""
        if rc == E_CUDA and ctx:
            detail = lib().agcm_last_cuda_error_string(ctx).decode()
        raise AgcmError(rc, detail)
    return rc
