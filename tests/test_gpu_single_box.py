"""The single calls that run the batch code: mpvss_reconstruct is mpvss_reconstruct_secrets over one box, and
mpvss_multi_exp folds through the same segmented product tree (ModpGroup) / 64-way sum (curves) with one segment.

Pinned here: the single reconstruct's failure statuses, its untouched outputs and error text on failure, and the
launch counts of reconstruct and multi_exp.  Also the curves' X_i and Horner product counts at (n, t) =
(1024, 683), a shape where the one-wave chunk rule (42 chunks) leaves 683 / 42 coefficients per chunk: the single
calls round it to 41 chunks of 17, the mpvss_verify_distributions batch launches 42 with the last one empty for
this box.  The counts were recorded on an NVIDIA B200 with the library as it was before the single calls ran the
batch code.  The chunk rule reads the SM count, so the Horner figures are checked on 148-SM devices only."""
import ctypes
import random

import pytest

import mpvss_rs_b200 as m
from mpvss_rs_b200 import lib as L
from mpvss_rs_b200 import synth
from mpvss_rs_b200.lib import buf, ptr
from oracle import pvss
from oracle.groups import GROUPS

pytestmark = pytest.mark.gpu
GNAMES = ["modp", "secp256k1", "ristretto255"]
SECRET = pvss.string_to_secret("single box")
RECONSTRUCT_KS = (1, 2, 43, 683, 2731)  # ModpGroup: direct below msm_threshold = 512, buckets from there on
MULTI_EXP_KS = (1, 2, 3, 64, 700)
N_H, T_H = 1024, 683

# mpvss_last_kernel_launches of the calls below, by k (multi_exp: by (modp_msm, k); the curves have no modp_msm)
RECONSTRUCT_LAUNCHES = {
    "modp": {1: 3, 2: 7, 43: 27, 683: 43, 2731: 49},
    "secp256k1": {1: 3, 2: 3, 43: 3, 683: 4, 2731: 4},
    "ristretto255": {1: 3, 2: 3, 43: 3, 683: 4, 2731: 4},
}
MULTI_EXP_LAUNCHES = {
    "modp": {(0, 1): 1, (0, 2): 2, (0, 3): 3, (0, 64): 7, (0, 700): 11,
             (1, 1): 5, (1, 2): 5, (1, 3): 5, (1, 64): 5, (1, 700): 5,
             (2, 1): 1, (2, 2): 2, (2, 3): 3, (2, 64): 7, (2, 700): 5},
    "secp256k1": {(None, 1): 2, (None, 2): 2, (None, 3): 2, (None, 64): 2, (None, 700): 3},
    "ristretto255": {(None, 1): 2, (None, 2): 2, (None, 3): 2, (None, 64): 2, (None, 700): 3},
}
# mpvss_last_horner_products (squarings, multiplications) of poly_eval_exp, the staged verify and a batch
HORNER_PRODUCTS = {
    "secp256k1": {"poly_eval_exp": (106895580, 89293590), "staged": (106895580, 89293590),
                  "batch": (109140606, 91047237)},
    "ristretto255": {"poly_eval_exp": (64380688, 121717696), "staged": (64380688, 121717696),
                     "batch": (65797096, 124007242)},
}


@pytest.fixture(scope="module", params=GNAMES)
def pair(request):
    return m.Group(request.param), GROUPS[request.param]()


def reconstruct_inputs(g, og, positions, seed):
    """decrypted shares S_i = G^P(i) of a polynomial with as many coefficients as positions, and
    U = mask(G^P(0)) xor SECRET"""
    co = synth.coefficients(seed, len(positions), og.order())
    c = g.codec
    shares = c.enc_elems(g.fixed_base_exp(g.scalar_poly_eval(co, positions)))
    u = (og.mask_of(og.exp(og.generator(), co[0])) ^ SECRET).to_bytes(c.eb, "big")
    return shares, u


def reconstruct(g, positions, shares, u, with_gs=True):
    """(status, secret_out, gs_out) of one mpvss_reconstruct; the output buffers start as 0xa5 bytes"""
    eb, k = g.codec.eb, len(positions)
    sec, gs = buf(b"\xa5" * eb), buf(b"\xa5" * eb)
    st = g.ctx.lib.mpvss_reconstruct(g.ctx.h, k, (ctypes.c_int64 * k)(*positions), ptr(buf(shares)), ptr(buf(u)),
                                     ptr(sec), ptr(gs) if with_gs else None)
    return st, bytes(sec), bytes(gs)


def reconstruct_launch_counts(g, og):
    rng = random.Random(3)
    counts = {}
    for k in RECONSTRUCT_KS:
        positions = sorted(rng.sample(range(1, 3 * k + 1), k))
        shares, u = reconstruct_inputs(g, og, positions, 100 + k)
        st, sec, gs = reconstruct(g, positions, shares, u)
        assert st == L.OK and int.from_bytes(sec, "big") == SECRET, k
        counts[k] = g.ctx.last_kernel_launches
        assert reconstruct(g, positions, shares, u, with_gs=False)[:2] == (st, sec), k
    return counts


def multi_exp_launch_counts(g, og):
    """bases G^a_i (fixed-base table) and scalars e_i with 0, 1 and order - 1 among them: the product is
    G^(sum a_i e_i), one exponentiation for the oracle"""
    rng = random.Random(4)
    order = og.order()
    counts = {}
    try:
        for msm in (0, 1, 2) if og.name == "modp" else (None,):
            if msm is not None:
                g.ctx.set_int("modp_msm", msm)
            for k in MULTI_EXP_KS:
                a = [rng.randrange(1, order) for _ in range(k)]
                e = [rng.randrange(order) for _ in range(k)]
                e[:3] = [0, 1, order - 1][:k]
                want = og.exp(og.generator(), sum(x * y for x, y in zip(a, e)) % order)
                got = g.multi_exp(g.fixed_base_exp(a), e)
                assert got == (want if og.name == "modp" else og.element_to_bytes(want)), (msm, k)
                counts[(msm, k)] = g.ctx.last_kernel_launches
    finally:
        if og.name == "modp":
            g.ctx.set_int("modp_msm", 2)  # the default, for the other tests on this context
    return counts


def horner_counts(g, og):
    """X_i = G^P(i) at (n, t) = (N_H, T_H) from poly_eval_exp and the staged verify, against P(i) by
    mpvss_scalar_poly_eval and G^P(i) by the fixed-base table; the same box in a mpvss_verify_distributions batch
    with a smaller one verifies with the staged call's digest.  Returns the Horner product counts of the three."""
    order = og.order()
    p = m.Participant(g)
    counts = {}
    boxes = []
    for seed, (n, t) in ((200, (N_H, T_H)), (201, (64, 43))):
        pks = g.fixed_base_exp(synth.private_keys(seed, n, og.name, order))
        co = synth.coefficients(seed, t, order)
        box = p.distribute_secret(SECRET, pks, t, coeffs=co, witnesses=synth.witnesses(seed, n, order))
        boxes.append((box, co))
    box, co = boxes[0]
    positions = list(range(1, N_H + 1))
    want = g.fixed_base_exp(g.scalar_poly_eval(co, positions))
    assert g.poly_eval_exp(box.commitments, positions) == want
    counts["poly_eval_exp"] = g.ctx.last_horner_products()
    tr = {}
    assert p.verify_distribution_shares(box, trace=tr) and tr["X"] == want
    counts["staged"] = g.ctx.last_horner_products()
    trs = [{}, {}]
    assert p.verify_distributions([b for b, _ in boxes], traces=trs) == [True, True]
    assert trs[0]["digest"] == tr["digest"]
    counts["batch"] = g.ctx.last_horner_products()
    return counts


def test_reconstruct_failures(pair):
    """A rejected single call keeps its status per group and failure kind, writes neither output and records an
    error.  The curves accept a repeated position (its Lagrange coefficient is 0)."""
    g, og = pair
    lib, h, eb = g.ctx.lib, g.ctx.h, g.codec.eb
    positions = [1, 2, 3, 4]
    shares, u = reconstruct_inputs(g, og, positions, 10)
    cases = [([1, 2, 1 << 40, 4], shares, L.ERR_ARG), ([0, 2, 3, 4], shares, L.ERR_ARG),
             ([1, 2, 2, 4], shares, L.ERR_ARG if og.name == "modp" else L.OK)]
    if og.name != "modp":
        bad = (b"\x05" + b"\x11" * 32) if og.name == "secp256k1" else b"\xff" * 32
        cases.append((positions, shares[:eb] + bad + shares[2 * eb:], L.ERR_ENCODING))
    for pos, sh, want in cases:
        lib.mpvss_ctx_set_int(h, b"no such tunable", 0)       # an error text of its own
        before = lib.mpvss_last_error(h)
        st, sec, gs = reconstruct(g, pos, sh, u)
        assert st == want, (pos, want)
        if want != L.OK:
            assert (sec, gs) == (b"\xa5" * eb, b"\xa5" * eb), pos
            assert lib.mpvss_last_error(h) not in (b"", before), pos
        st, sec, gs = reconstruct(g, positions, shares, u)    # a good call in between
        assert st == L.OK and int.from_bytes(sec, "big") == SECRET
    sec = buf(size=eb)
    one = (ctypes.c_int64 * 1)(1)
    assert lib.mpvss_reconstruct(h, 0, one, ptr(buf(shares)), ptr(buf(u)), ptr(sec), None) == L.ERR_ARG
    assert b"bad arguments" in lib.mpvss_last_error(h)
    assert lib.mpvss_reconstruct(h, 1, one, ptr(buf(shares)), ptr(buf(u)), None, None) == L.ERR_ARG


def test_reconstruct_launches(pair):
    g, og = pair
    assert reconstruct_launch_counts(g, og) == RECONSTRUCT_LAUNCHES[og.name]


def test_multi_exp_launches(pair):
    g, og = pair
    assert multi_exp_launch_counts(g, og) == MULTI_EXP_LAUNCHES[og.name]


@pytest.mark.parametrize("gname", ["secp256k1", "ristretto255"])
def test_curve_x_and_horner_products_at_n1024_t683(gname):
    import torch
    if torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the Horner product counts were recorded with 148 SMs")
    g, og = m.Group(gname), GROUPS[gname]()
    assert horner_counts(g, og) == HORNER_PRODUCTS[gname]
