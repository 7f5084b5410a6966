"""ctypes binding of libmpvss_b200.so (include/mpvss_b200.h).

The CUDA library is the product; this module only marshals buffers.  It fails
loudly when the library is missing or no CUDA device can be opened -- there is no
CPU fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPVSS_B200_LIB") or os.path.join(_HERE, "libmpvss_b200.so")  # override: tuning builds only

GROUP_MODP, GROUP_SECP256K1, GROUP_RISTRETTO255 = 0, 1, 2
GROUP_IDS = {"modp": GROUP_MODP, "secp256k1": GROUP_SECP256K1, "ristretto255": GROUP_RISTRETTO255}
GEN_MAIN, GEN_SUBGROUP = 0, 1
OK, ERR_CUDA, ERR_ARG, ERR_ENCODING, ERR_UNSUPPORTED, ERR_NOT_INVERTIBLE, ERR_COMM = 0, -1, -2, -3, -4, -5, -6

_u8p = ctypes.POINTER(ctypes.c_uint8)
_i64p = ctypes.POINTER(ctypes.c_int64)
_intp = ctypes.POINTER(ctypes.c_int)
_sz = ctypes.c_size_t
_ctxp = ctypes.c_void_p

# name -> (restype, argtypes); kept in the order of include/mpvss_b200.h
SIGNATURES = {
    "mpvss_ctx_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.POINTER(_ctxp)]),
    "mpvss_ctx_destroy": (None, [_ctxp]),
    "mpvss_last_error": (ctypes.c_char_p, [_ctxp]),
    "mpvss_ctx_set_int": (ctypes.c_int, [_ctxp, ctypes.c_char_p, ctypes.c_int]),
    "mpvss_element_bytes": (_sz, [_ctxp]),
    "mpvss_scalar_bytes": (_sz, [_ctxp]),
    "mpvss_last_kernel_ms": (ctypes.c_float, [_ctxp]),
    "mpvss_last_kernel_launches": (ctypes.c_int, [_ctxp]),
    "mpvss_last_horner_products": (ctypes.c_uint64, [_ctxp, ctypes.c_int]),
    "mpvss_last_phase_ms": (ctypes.c_float, [_ctxp, ctypes.c_int]),
    "mpvss_batch_exp": (ctypes.c_int, [_ctxp, _u8p, _sz, _u8p, _sz, _u8p]),
    "mpvss_fixed_base_exp": (ctypes.c_int, [_ctxp, ctypes.c_int, _u8p, _sz, _u8p]),
    "mpvss_batch_mul": (ctypes.c_int, [_ctxp, _u8p, _u8p, _sz, _u8p]),
    "mpvss_poly_eval_exp": (ctypes.c_int, [_ctxp, _u8p, _sz, _i64p, _sz, _u8p]),
    "mpvss_scalar_poly_eval": (ctypes.c_int, [_ctxp, _u8p, _sz, _i64p, _sz, _u8p]),
    "mpvss_dleq_verify_commit": (ctypes.c_int, [_ctxp, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _sz, _sz, _u8p, _u8p]),
    "mpvss_dleq_prove_commit": (ctypes.c_int, [_ctxp, _u8p, _u8p, _u8p, _sz, _u8p, _u8p]),
    "mpvss_multi_exp": (ctypes.c_int, [_ctxp, _u8p, _u8p, _sz, _u8p]),
    "mpvss_verify_distribution": (ctypes.c_int, [_ctxp, _sz, _sz, _u8p, _i64p, _u8p, _u8p, _u8p, _u8p, _intp,
                                                 _u8p, _u8p, _u8p, _u8p]),
    "mpvss_verify_distribution_stage": (ctypes.c_int, [_ctxp, _sz, _sz, _u8p, _i64p, _u8p, _u8p, _u8p, _u8p]),
    "mpvss_verify_distribution_run": (ctypes.c_int, [_ctxp, _intp, _u8p, _u8p, _u8p, _u8p]),
    "mpvss_verify_distributions": (ctypes.c_int, [_ctxp, _sz, ctypes.POINTER(_sz), ctypes.POINTER(_sz), _u8p, _i64p,
                                                  _u8p, _u8p, _u8p, _u8p, _intp, _u8p]),
    "mpvss_distribute": (ctypes.c_int, [_ctxp, _sz, _sz, _u8p, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p,
                                        _u8p, _u8p]),
    "mpvss_distribute_secrets": (ctypes.c_int, [_ctxp, _sz, ctypes.POINTER(_sz), ctypes.POINTER(_sz), _u8p, _u8p, _u8p,
                                                _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _intp]),
    "mpvss_extract_shares": (ctypes.c_int, [_ctxp, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _intp]),
    "mpvss_verify_shares": (ctypes.c_int, [_ctxp, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _intp]),
    "mpvss_reconstruct": (ctypes.c_int, [_ctxp, _sz, _i64p, _u8p, _u8p, _u8p, _u8p]),
    "mpvss_reconstruct_secrets": (ctypes.c_int, [_ctxp, _sz, ctypes.POINTER(_sz), _i64p, _u8p, _u8p, _u8p, _u8p,
                                                 _intp]),
    "mpvss_comm_unique_id": (ctypes.c_int, [_u8p, _sz]),
    "mpvss_comm_init": (ctypes.c_int, [_ctxp, _u8p, _sz, ctypes.c_int, ctypes.c_int]),
    "mpvss_comm_destroy": (ctypes.c_int, [_ctxp]),
    "mpvss_comm_size": (ctypes.c_int, [_ctxp]),
    "mpvss_comm_rank": (ctypes.c_int, [_ctxp]),
    "mpvss_transcript_digest": (ctypes.c_int, [ctypes.c_int, _u8p, _sz, ctypes.c_int, _u8p]),
}
COMM_ID_BYTES = 128

_lib = None


def load():
    """dlopen the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `make` (or __graft_entry__.build()); "
                               "mpvss_rs_b200 has no CPU fallback")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class MpvssError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"mpvss status {status}: {message}")
        self.status = status


def buf(data=None, size=None):
    """ctypes byte buffer from bytes (copy) or of a given size."""
    if data is not None:
        return (ctypes.c_uint8 * len(data)).from_buffer_copy(data)
    return (ctypes.c_uint8 * size)()


def ptr(b):
    return ctypes.cast(b, _u8p) if b is not None else None


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the library (rank 0 calls it and hands the bytes to the other ranks)."""
    b = buf(size=COMM_ID_BYTES)
    st = load().mpvss_comm_unique_id(ptr(b), COMM_ID_BYTES)
    if st != OK:
        raise MpvssError(st, "mpvss_comm_unique_id failed (libnccl.so.2 not loadable?)")
    return bytes(b)


def transcript_digest(group: str, gathered_rows: bytes, n_total: int, nranks: int) -> bytes:
    """SHA-256 of the framed transcript rows in participant order, from the all-gather layout
    [rank][ceil(n_total / nranks)][4 x (8 + element bytes)] (host only: needs no device)."""
    out = buf(size=32)
    st = load().mpvss_transcript_digest(GROUP_IDS[group], ptr(buf(gathered_rows)), n_total, nranks, ptr(out))
    if st != OK:
        raise MpvssError(st, "mpvss_transcript_digest: bad arguments")
    return bytes(out)


class Context:
    """Owns one `mpvss_ctx` (one group on one CUDA device)."""

    def __init__(self, group="modp", device=0):
        self.lib = load()
        self.group = group
        h = _ctxp()
        st = self.lib.mpvss_ctx_create(GROUP_IDS[group], device, ctypes.byref(h))
        if st != OK:
            raise MpvssError(st, "mpvss_ctx_create failed (no CUDA device? there is no CPU fallback)")
        self.h = h
        self.eb = self.lib.mpvss_element_bytes(h)
        self.sb = self.lib.mpvss_scalar_bytes(h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.mpvss_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, st):
        if st != OK:
            raise MpvssError(st, self.lib.mpvss_last_error(self.h).decode())

    def set_int(self, key, value):
        self.check(self.lib.mpvss_ctx_set_int(self.h, key.encode(), value))

    @property
    def last_kernel_ms(self):
        return float(self.lib.mpvss_last_kernel_ms(self.h))

    def last_phase_ms(self, phase):
        return float(self.lib.mpvss_last_phase_ms(self.h, phase))

    def last_horner_products(self):
        """(squarings, multiplications) executed by the last X_i launch on this context"""
        return (int(self.lib.mpvss_last_horner_products(self.h, 0)), int(self.lib.mpvss_last_horner_products(self.h, 1)))

    # ---- multi-GPU: one context per GPU, joined by an NCCL communicator inside the library ----
    def comm_init(self, unique_id: bytes, nranks: int, rank: int):
        self.check(self.lib.mpvss_comm_init(self.h, ptr(buf(unique_id)), len(unique_id), nranks, rank))

    def comm_destroy(self):
        self.check(self.lib.mpvss_comm_destroy(self.h))

    @property
    def comm_size(self):
        return int(self.lib.mpvss_comm_size(self.h))

    @property
    def comm_rank(self):
        return int(self.lib.mpvss_comm_rank(self.h))

    @property
    def last_kernel_launches(self):
        return int(self.lib.mpvss_last_kernel_launches(self.h))
