"""CPU execution of the kernel bodies of mpvss_reconstruct_secrets (modp_kernels.cuh: lagrange_boxes_body,
mul_rows_body with product_tree_level; ec_kernels.cuh: lagrange_boxes_body, sum_boxes_body with sum_boxes_level --
the source nvcc compiles) through tests/emu/emu_reconstruct_batch.cpp, bit-exact against Python integers and the
oracle, box by box."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import emu_util as eu
from oracle.groups import ED_L, SECP_N, ModpGroup, Ristretto255Group, Secp256k1Group, lagrange_coefficient

SRC = os.path.join(eu.HERE, "emu_reconstruct_batch.cpp")
SO = os.path.join(eu.HERE, "libemu_reconstruct_batch.so")
Q = ModpGroup().q
TOP = (1 << 31) - 1

# k = 1, 5 and 11: a lone position, small positions the oracle's util.rs restatement can take, positions near 2^31
BOXES = [[7], [1, 3, 4, 9, 200], [TOP, 5, (1 << 30) + 3, 17, TOP - 8, 2, 1, 99, 100, TOP - 1, 65537]]


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
    """concatenated positions, and per position its box's first row and its box's k"""
    pos, boff, bk = [], [], []
    for box in boxes:
        boff += [len(pos)] * len(box)
        bk += [len(box)] * len(box)
        pos += box
    u32 = lambda v: np.array(v, dtype=np.uint32)
    return u32(pos), u32(boff), u32(bk)


def _exact(x, box):
    """prod x_j and prod (x_j - x_i) over the other positions of the box"""
    num = den = 1
    for y in box:
        if y != x:
            num, den = num * y, den * (y - x)
    return num, den


@pytest.mark.parametrize("parts", [1, 8])
def test_modp_lagrange_boxes(L, parts):
    """num_i, den_i mod (q-1) and the sign of every position, over its own box only; parts = 8 leaves empty ranges
    in every box (their product is 1)."""
    order = Q - 1
    pos, boff, bk = _layout(BOXES)
    n = len(pos)
    num, den = np.zeros(64 * n * parts, dtype=np.uint32), np.zeros(64 * n * parts, dtype=np.uint32)
    neg = np.zeros(n * parts, dtype=np.uint32)
    assert L.emu_modp_lagrange_boxes(eu.P(eu.to_limbs(order)), eu.P(pos), eu.P(boff), eu.P(bk), n, eu.P(num), eu.P(den),
                                     eu.P(neg), parts) == 0
    i = 0
    for box in BOXES:
        for x in box:
            pn = pd = 1
            sign = 0
            for p in range(parts):
                r = p * n + i
                pn = pn * eu.from_limbs(num[64 * r:64 * r + 64]) % order
                pd = pd * eu.from_limbs(den[64 * r:64 * r + 64]) % order
                sign ^= int(neg[r])
            full_n, full_d = _exact(x, box)
            assert (pn, pd) == (full_n % order, abs(full_d) % order), (box, x)
            assert bool(sign) == (full_d < 0)
            if max(box) < 1 << 16:
                n_, d_ = lagrange_coefficient(x, box)
                assert full_n * d_ == full_d * n_            # the rational number util.rs returns
            i += 1


@pytest.mark.parametrize("order", [SECP_N, ED_L])
def test_ec_lagrange_boxes(L, order):
    """lambda_i over its own box, with a box that holds a duplicate position: both copies get lambda = 0
    (inv(0) = 0, as the single-box kernel), the others keep the repeated factor."""
    boxes = BOXES + [[4, 9, 4, 11, 30]]
    pos, boff, bk = _layout(boxes)
    n = len(pos)
    out = np.zeros(8 * n, dtype=np.uint32)
    assert L.emu_ec_lagrange_boxes(eu.P(eu.modulus_words(order)), eu.P(pos), eu.P(boff), eu.P(bk), n, eu.P(out)) == 0
    i = 0
    for box in boxes:
        for j, x in enumerate(box):
            num = den = 1
            for m, y in enumerate(box):
                if m != j:
                    num, den = num * y % order, den * (y - x) % order
            want = num * pow(den, -1, order) % order if den else 0
            assert eu.from_limbs(out[8 * i:8 * i + 8]) == want, (box, x)
            if len(set(box)) == len(box) and max(box) < 1 << 16:
                n_, d_ = lagrange_coefficient(x, box)
                assert want == n_ * pow(d_, -1, order) % order
            i += 1
    assert eu.from_limbs(out[8 * (n - 5):8 * (n - 4)]) == 0 == eu.from_limbs(out[8 * (n - 3):8 * (n - 2)])


def test_modp_segmented_product_tree(L):
    """boxes of 1, 2, 3 and 17 values, each reduced to its product mod q at its first row; no level pairs rows of
    two boxes (ceil(log2 17) = 5 levels)"""
    rng = random.Random(5)
    sizes = [1, 2, 3, 17]
    vals = [[rng.randrange(Q) for _ in range(k)] for k in sizes]
    vals[3][4] = Q - 1
    vals[3][5] = 1
    flat = [x for v in vals for x in v]
    v = np.concatenate([eu.to_limbs(x) for x in flat])
    start = np.array(np.cumsum([0] + sizes[:-1]), dtype=np.uint32)
    cnt = np.array(sizes, dtype=np.uint32)
    assert L.emu_modp_tree(eu.P(eu.consts_block(Q)), eu.P(v), eu.P(start), eu.P(cnt), len(sizes), len(flat)) == 5
    for b, k in enumerate(sizes):
        want = 1
        for x in vals[b]:
            want = want * x % Q
        s = int(start[b])
        assert eu.from_limbs(v[64 * s:64 * s + 64]) == want, k


CURVES = {"secp": (Secp256k1Group, eu.secp_consts, SECP_N), "rist": (Ristretto255Group, eu.rist_consts, ED_L)}


@pytest.mark.parametrize("cv", ["secp", "rist"])
def test_ec_segmented_sum(L, cv):
    """boxes of 1, 63, 64, 65 and 130 points (one, one, one, two and three groups of the first 64-way level, and a
    second level for the last two), against the oracle: point i is (i + 1) G, so box b sums to (sum e_i (i + 1)) G"""
    Gc, consts, order = CURVES[cv]
    G = Gc()
    rng = random.Random(11)
    sizes = [1, 63, 64, 65, 130]
    n = sum(sizes)
    pts, p = [], G.generator()
    for _ in range(n):
        pts.append(G.element_to_bytes(p))
        p = G.mul(p, G.generator())
    e = [rng.randrange(1, order) for _ in range(n)]
    eb = len(pts[0])
    start = np.array(np.cumsum([0] + sizes[:-1]), dtype=np.uint32)
    cnt = np.array(sizes, dtype=np.uint32)
    out = (ctypes.c_uint8 * (eb * len(sizes)))()
    assert getattr(L, f"emu_{cv}_sum_boxes")(eu.P(consts()), (ctypes.c_uint8 * (eb * n)).from_buffer_copy(b"".join(pts)),
                                             eu.P(np.concatenate([eu.to_limbs(x, 8) for x in e])), n, eu.P(start),
                                             eu.P(cnt), len(sizes), out) == 0
    for b, k in enumerate(sizes):
        s = int(start[b])
        scalar = sum(e[i] * (i + 1) for i in range(s, s + k)) % order
        assert bytes(out)[eb * b:eb * (b + 1)] == G.element_to_bytes(G.exp(G.generator(), scalar)), k
