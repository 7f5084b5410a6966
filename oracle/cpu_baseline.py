"""ctypes driver for oracle/cpu_baseline.c (OpenSSL proxy for the reference's CPU path).
TEST + BENCH INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "cpu_baseline.c")
SO = os.path.join(HERE, "_build", "libcpu_baseline.so")


def _stale(so):
    return not os.path.exists(so) or os.path.getmtime(SRC) > os.path.getmtime(so)


def build(force=False, so=SO):
    os.makedirs(os.path.dirname(so), exist_ok=True)
    if force or _stale(so):
        subprocess.check_call(["gcc", "-O2", "-Wno-deprecated-declarations", "-shared", "-fPIC", "-pthread", "-o", so, SRC, "-lcrypto"])
    return so


def _runtime_so():
    """The library built into the tree; when it is missing or stale and the tree cannot be written (a read-only
    checkout), a private copy in the temporary directory instead."""
    out_dir = os.path.dirname(SO)
    if not _stale(SO) or os.access(out_dir if os.path.isdir(out_dir) else HERE, os.W_OK):
        return build()
    return build(so=os.path.join(tempfile.gettempdir(), f"mpvss_cpu_baseline_{os.getuid()}", "libcpu_baseline.so"))


def load():
    lib = ctypes.CDLL(_runtime_so())
    p, sz = ctypes.c_char_p, ctypes.c_size_t
    lib.cpu_modp_verify.argtypes = [p, p, sz, ctypes.POINTER(ctypes.c_int64), p, p, p, p, sz, ctypes.c_int,
                                    ctypes.c_int, p, p, p]
    lib.cpu_modp_verify.restype = ctypes.c_int
    lib.cpu_secp_verify.argtypes = [p, sz, ctypes.POINTER(ctypes.c_int64), p, p, p, p, sz, ctypes.c_int, ctypes.c_int,
                                    p, p, p]
    lib.cpu_secp_verify.restype = ctypes.c_int
    lib.cpu_modp_exp.argtypes = [p, p, sz, p, sz, ctypes.c_int, p]
    lib.cpu_modp_exp.restype = ctypes.c_int
    lib.cpu_secp_mul.argtypes = [p, p, sz, p]
    lib.cpu_secp_mul.restype = ctypes.c_int
    return lib


def be(x):
    return int(x).to_bytes(256, "big")


def modp_verify(q, commitments, positions, pks, ys, rs, c, nthreads=1, schedule=0):
    """Returns (X, a1, a2) lists of ints for the given participants."""
    lib = load()
    s = len(positions)
    xo, a1o, a2o = (ctypes.create_string_buffer(256 * s) for _ in range(3))
    lib.cpu_modp_verify(be(q), b"".join(be(v) for v in commitments), len(commitments),
                        (ctypes.c_int64 * s)(*positions), b"".join(be(v) for v in pks), b"".join(be(v) for v in ys),
                        b"".join(be(v) for v in rs), be(c), s, nthreads, schedule, xo, a1o, a2o)
    dec = lambda b: [int.from_bytes(b.raw[i * 256:(i + 1) * 256], "big") for i in range(s)]
    return dec(xo), dec(a1o), dec(a2o)


def secp_verify(commitments, positions, pks, ys, rs, c, nthreads=1, schedule=0):
    """Inputs: 33-byte SEC1 points, integer scalars.  Returns (X, a1, a2) lists of 33-byte encodings."""
    lib = load()
    s = len(positions)
    xo, a1o, a2o = (ctypes.create_string_buffer(33 * s) for _ in range(3))
    lib.cpu_secp_verify(b"".join(commitments), len(commitments), (ctypes.c_int64 * s)(*positions), b"".join(pks),
                        b"".join(ys), b"".join(int(v).to_bytes(32, "big") for v in rs), int(c).to_bytes(32, "big"),
                        s, nthreads, schedule, xo, a1o, a2o)
    dec = lambda b: [b.raw[i * 33:(i + 1) * 33] for i in range(s)]
    return dec(xo), dec(a1o), dec(a2o)


def modp_exp(q, bases, exps, nthreads=1):
    """[b^e mod q]; `bases` may be one int (shared base)."""
    lib = load()
    n = len(exps)
    shared = isinstance(bases, int)
    out = ctypes.create_string_buffer(256 * n)
    lib.cpu_modp_exp(be(q), be(bases) if shared else b"".join(be(v) for v in bases), 0 if shared else 256,
                     b"".join(be(v) for v in exps), n, nthreads, out)
    return [int.from_bytes(out.raw[i * 256:(i + 1) * 256], "big") for i in range(n)]


def secp_mul(points, scalars):
    """[k * P]; points None = the generator.  33-byte encodings."""
    lib = load()
    n = len(scalars)
    out = ctypes.create_string_buffer(33 * n)
    lib.cpu_secp_mul(None if points is None else b"".join(points), b"".join(int(k).to_bytes(32, "big") for k in scalars),
                     n, out)
    return [out.raw[i * 33:(i + 1) * 33] for i in range(n)]
