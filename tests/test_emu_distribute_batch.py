"""CPU execution of the kernel bodies of mpvss_distribute_secrets (modp_kernels.cuh / ec_kernels.cuh:
poly_boxes_body, and modp_kernels.cuh: resp_body with one challenge per instance -- the source nvcc compiles)
through tests/emu/emu_distribute_batch.cpp, bit-exact against Python integers, box by box."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import emu_util as eu
from oracle.groups import ED_L, SECP_N, ModpGroup

SRC = os.path.join(eu.HERE, "emu_distribute_batch.cpp")
SO = os.path.join(eu.HERE, "libemu_distribute_batch.so")
ORDER = ModpGroup().q - 1

# (n, t): t = 1 in a box of one and of several participants, t = n, and mixed t across the boxes
BOXES = [(1, 1), (3, 1), (4, 4), (9, 5), (17, 9), (6, 2), (33, 33)]


@pytest.fixture(scope="module")
def L():
    deps = [SRC] + [os.path.join(eu.CSRC, f) for f in ("simt.h", "modp_arith.cuh", "modp_sqr.cuh", "modp_kernels.cuh",
                                                       "fp256.cuh", "fpspecial.cuh", "secp.cuh", "rist.cuh",
                                                       "ec_kernels.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-DMPVSS_SIMT_EMU", "-shared", "-fPIC", "-pthread",
                               "-o", SO, SRC])
    return ctypes.CDLL(SO)


def _layout(boxes):
    """positions 1..n_b per box, then per instance its box's first coefficient row, t_b and first instance row"""
    pos, coff, bt, ioff = [], [], [], []
    t0 = 0
    for n, t in boxes:
        ioff += [len(pos)] * n
        coff += [t0] * n
        bt += [t] * n
        pos += list(range(1, n + 1))
        t0 += t
    return np.array(pos + coff + bt + ioff, dtype=np.uint32)


def _coeffs(rng, boxes, order, top):
    """per box t_b coefficients below `top`, each box's a_0 = order - 1 and every coefficient of box 2 (t = n = 4)
    order - 1"""
    co = []
    for b, (n, t) in enumerate(boxes):
        c = [rng.randrange(top) for _ in range(t)]
        c[0] = order - 1
        if b == 2:
            c = [order - 1] * t
        co.append(c)
    return co


def _want(co, x, order):
    return sum(a * x ** j for j, a in enumerate(co)) % order


def test_modp_poly_boxes(L):
    """P_b(i) mod (q-1) for every instance of every box; coefficients of order - 1 and up to 2^2048 - 1 (the kernel
    takes them unreduced, as distribute uploads them) run the overflow fold"""
    rng = random.Random(3)
    co = _coeffs(rng, BOXES, ORDER, 1 << 2048)
    co[3][1] = (1 << 2048) - 1
    idx = _layout(BOXES)
    n = sum(nb for nb, _ in BOXES)
    flat = np.concatenate([eu.to_limbs(a) for c in co for a in c])
    out = np.zeros(64 * n, dtype=np.uint32)
    assert L.emu_modp_poly_boxes(eu.P(flat), eu.P(eu.to_limbs(ORDER)), eu.P(idx), n, eu.P(out)) == 0
    i = 0
    for (nb, t), c in zip(BOXES, co):
        for x in range(1, nb + 1):
            assert eu.from_limbs(out[64 * i:64 * i + 64]) == _want(c, x, ORDER), (nb, t, x)
            i += 1


@pytest.mark.parametrize("order", [SECP_N, ED_L])
def test_ec_poly_boxes(L, order):
    """P_b(i) mod the group order for every instance of every box (coefficients below the order, as scalars_in
    delivers them)"""
    rng = random.Random(4)
    co = _coeffs(rng, BOXES, order, order)
    idx = _layout(BOXES)
    n = sum(nb for nb, _ in BOXES)
    flat = np.concatenate([eu.to_limbs(a, 8) for c in co for a in c])
    out = np.zeros(8 * n, dtype=np.uint32)
    assert L.emu_ec_poly_boxes(eu.P(eu.modulus_words(order)), eu.P(flat), eu.P(idx), n, eu.P(out)) == 0
    i = 0
    for (nb, t), c in zip(BOXES, co):
        for x in range(1, nb + 1):
            assert eu.from_limbs(out[8 * i:8 * i + 8]) == _want(c, x, order), (nb, t, x)
            i += 1


def test_modp_responses_per_instance_challenge(L):
    """r_i = (w_i - p_i c_b) mod (q-1) with c_stride = 64: every instance reads its own box's challenge, and no
    instance reads another box's"""
    rng = random.Random(5)
    boxes = [3, 1, 7, 2]
    n = sum(boxes)
    cs = [rng.randrange(1 << 256) for _ in boxes]
    cs[1] = (1 << 256) - 1
    chal = [c for c, k in zip(cs, boxes) for _ in range(k)]
    p = [rng.randrange(ORDER) for _ in range(n)]
    w = [rng.randrange(1 << 2048) for _ in range(n)]
    p[0], w[0] = ORDER - 1, 0
    w[1] = ORDER - 1
    w[2] = (1 << 2048) - 1
    rows = lambda v: np.concatenate([eu.to_limbs(x) for x in v])
    out = np.zeros(64 * n, dtype=np.uint32)
    assert L.emu_modp_resp(eu.P(eu.to_limbs(ORDER)), eu.P(rows(p)), eu.P(rows(w)), eu.P(rows(chal)), 64, n,
                           eu.P(out)) == 0
    for i in range(n):
        assert eu.from_limbs(out[64 * i:64 * i + 64]) == (w[i] - p[i] * chal[i]) % ORDER, i
