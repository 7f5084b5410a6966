"""CPU execution of the multi-box elliptic-curve Horner body (ec_kernels.cuh: horner_boxes_body, the source
nvcc compiles for mpvss_verify_distributions) through tests/emu/emu_multibox.cpp, bit-exact against the
oracle's Horner schedule for boxes of different t, positions and chunk counts."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import emu_util as eu
from oracle import pvss
from oracle.groups import ED_L, SECP_N, Ristretto255Group, Secp256k1Group

SRC = os.path.join(eu.HERE, "emu_multibox.cpp")
SO = os.path.join(eu.HERE, "libemu_multibox.so")


@pytest.fixture(scope="module")
def L():
    deps = [SRC] + [os.path.join(eu.CSRC, f) for f in ("simt.h", "fp256.cuh", "fpspecial.cuh", "secp.cuh", "rist.cuh",
                                                       "ec_kernels.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-DMPVSS_SIMT_EMU", "-shared", "-fPIC", "-pthread",
                               "-o", SO, SRC])
    return ctypes.CDLL(SO)


CURVES = {
    "secp": (Secp256k1Group, eu.secp_consts, SECP_N),
    "rist": (Ristretto255Group, eu.rist_consts, ED_L),
}

# (t, positions) per box: different t (one box shorter than K, so its upper chunks are empty), dense and
# scattered positions, one above 2^17
BOXES = [
    (1, [1, 2]),
    (5, [1, 2, 3, 4, 5, 6]),
    (9, [7, 300, 1 << 17 | 5, 65536]),
]


@pytest.mark.parametrize("cv", ["secp", "rist"])
@pytest.mark.parametrize("K", [1, 3, 4])
def test_multibox_horner_equals_horner_schedule(L, cv, K):
    Gc, consts, order = CURVES[cv]
    G = Gc()
    C = consts()
    rng = random.Random(100 + K)
    comms, pos, coff, ct = [], [], [], []
    for t, ps in BOXES:
        box = [G.exp(G.generator(), rng.randrange(1, order)) for _ in range(t)]
        if t == 5:
            box[2] = G.identity()                     # identity commitment inside a box
        for p in ps:
            pos.append(p)
            coff.append(sum(len(b) for b in comms))
            ct.append(t)
        comms.append(box)
    flat = [c for box in comms for c in box]
    eb = len(G.element_to_bytes(flat[0]))
    cb = (ctypes.c_uint8 * (eb * len(flat))).from_buffer_copy(b"".join(G.element_to_bytes(c) for c in flat))
    n = len(pos)
    u32 = lambda v: np.array(v, dtype=np.uint32)
    P, O, T = u32(pos), u32(coff), u32(ct)
    out = (ctypes.c_uint8 * (eb * n))()
    assert getattr(L, f"emu_{cv}_horner_boxes")(eu.P(C), cb, len(flat), eu.P(P), eu.P(O), eu.P(T), n, K, out) == 0
    i = 0
    for j, (t, ps) in enumerate(BOXES):
        for p in ps:
            want = G.element_to_bytes(pvss.x_horner_schedule(G, comms[j], p))
            assert bytes(out)[eb * i:eb * (i + 1)] == want, (cv, K, j, p)
            i += 1
