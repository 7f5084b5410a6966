"""mpvss_reconstruct_secrets: many secrets in one call.  Every box's secret, G^s and status equal what
mpvss_reconstruct gives for the box alone (and the oracle for tiny boxes); a failing box fails on its own with zero
rows; argument errors are status codes; every MODP multi-exponentiation path gives the same bytes; the staged
single-box verify state survives a batch call in between."""
import copy
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
SECRET = pvss.string_to_secret("reconstruct batch")
GNAMES = ["modp", "secp256k1", "ristretto255"]
TOP = (1 << 31) - 1


@pytest.fixture(scope="module", params=GNAMES)
def pair(request):
    return m.Group(request.param), GROUPS[request.param]()


def make_box(g, og, seed, positions, t=None):
    """the raw inputs of one reconstruct: the decrypted shares S_i = G^P(i) of a polynomial of t coefficients
    (default: as many as positions) and U = mask(G^P(0)) xor SECRET"""
    t = t or len(positions)
    co = synth.coefficients(seed, t, og.order())
    c = g.codec
    shares = g.fixed_base_exp(g.scalar_poly_eval(co, positions))
    u = og.mask_of(og.exp(og.generator(), co[0])) ^ SECRET
    return dict(k=len(positions), pos=list(positions), s=c.enc_elems(shares), u=u.to_bytes(c.eb, "big"), co=co)


def batch(g, boxes, with_gs=True):
    nb, eb = len(boxes), g.codec.eb
    pos = [p for b in boxes for p in b["pos"]]
    sec, gs, st = buf(size=nb * eb), buf(size=nb * eb), (ctypes.c_int * nb)()
    rc = g.ctx.lib.mpvss_reconstruct_secrets(
        g.ctx.h, nb, (ctypes.c_size_t * nb)(*[b["k"] for b in boxes]), (ctypes.c_int64 * len(pos))(*pos),
        ptr(buf(b"".join(b["s"] for b in boxes))), ptr(buf(b"".join(b["u"] for b in boxes))), ptr(sec),
        ptr(gs) if with_gs else None, st)
    rows = lambda x: [bytes(x)[i * eb:(i + 1) * eb] for i in range(nb)]
    return rc, list(zip(rows(sec), rows(gs), list(st)))


def single(g, b):
    eb = g.codec.eb
    sec, gs = buf(size=eb), buf(size=eb)
    st = g.ctx.lib.mpvss_reconstruct(g.ctx.h, b["k"], (ctypes.c_int64 * b["k"])(*b["pos"]), ptr(buf(b["s"])),
                                     ptr(buf(b["u"])), ptr(sec), ptr(gs))
    return (bytes(sec), bytes(gs), st) if st == L.OK else (bytes(eb), bytes(eb), st)


def secret_of(row):
    return int.from_bytes(row[0], "big")


def test_mixed_shapes_equal_the_single_call(pair):
    """k from 1 to 2731: for ModpGroup the single call takes the bucket method at 2731 (msm_threshold), the batch
    keeps the box in its direct launch"""
    g, og = pair
    rng = random.Random(1)
    ks = [1, 2, 3, 43, 171, 683, 2731]
    boxes = [make_box(g, og, 10 + i, sorted(rng.sample(range(1, 3 * k + 1), k))) for i, k in enumerate(ks)]
    rc, rows = batch(g, boxes)
    assert rc == L.OK
    for b, row in zip(boxes, rows):
        assert row == single(g, b), b["k"]
        assert row[2] == L.OK and secret_of(row) == SECRET, b["k"]


def test_tiny_boxes_equal_the_oracle(pair):
    """dense, scattered above 2^17 and (oracle permitting) near 2^31 - 1; a box with more shares than coefficients"""
    g, og = pair
    c = g.codec
    shapes = [([1, 2, 3], 3), ([131073, 200003, 150001, 140009], 4), ([2, 4, 6, 8, 10], 3)]
    if og.name != "modp":                      # the oracle's util.rs restatement scans 1..max(position) for MODP
        shapes.append(([TOP, 5, (1 << 30) + 3, TOP - 2], 4))
    boxes, want = [], []
    for seed, (positions, t) in enumerate(shapes):
        co = synth.coefficients(seed + 20, t, og.order())
        ss = [og.exp(og.generator(), pvss.poly_get_value(co, x) % og.order()) for x in positions]
        obox = pvss.DistributionSharesBox(commitments=[None] * t, U=og.mask_of(og.exp(og.generator(), co[0])) ^ SECRET,
                                          positions={og.element_to_bytes(s): x for s, x in zip(ss, positions)})
        tr = {}
        sec = pvss.reconstruct(og, [pvss.ShareBox(publickey=s, share=s) for s in ss], obox, trace=tr)
        assert sec == SECRET
        want.append((sec, tr["G_s"]))
        enc = [s if og.name == "modp" else og.element_to_bytes(s) for s in ss]
        boxes.append(dict(k=len(positions), pos=positions, s=c.enc_elems(enc), u=obox.U.to_bytes(c.eb, "big")))
    if og.name == "modp":
        boxes.append(make_box(g, og, 29, [TOP, 5, (1 << 30) + 3, TOP - 2]))
    rc, rows = batch(g, boxes)
    assert rc == L.OK
    for (sec, gs), row in zip(want, rows):
        assert row[2] == L.OK and secret_of(row) == sec
        assert row[1] == c.enc_elem(gs if og.name == "modp" else og.element_to_bytes(gs))
    if og.name == "modp":
        assert rows[-1] == single(g, boxes[-1]) and secret_of(rows[-1]) == SECRET


@pytest.mark.parametrize("gname", GNAMES)
def test_failures_stay_in_their_box(gname):
    g, og = m.Group(gname), GROUPS[gname]()
    eb = g.codec.eb
    boxes = [make_box(g, og, 30 + i, [1, 2, 3, 4]) for i in range(5)]
    boxes[1] = dict(boxes[1], pos=[1, 2, 1 << 40, 4])           # out of range
    boxes[2] = dict(boxes[2], pos=[1, 2, 2, 4])                 # duplicate
    want_status = [L.OK, L.ERR_ARG, L.ERR_ARG if gname == "modp" else L.OK, L.OK, L.OK]
    if gname != "modp":                                         # a share that does not decode
        bad = (b"\x05" + b"\x11" * 32) if gname == "secp256k1" else b"\xff" * 32
        boxes[3] = dict(boxes[3], s=boxes[3]["s"][:eb] + bad + boxes[3]["s"][2 * eb:])
        want_status[3] = L.ERR_ENCODING
    rc, rows = batch(g, boxes)
    assert rc == L.OK and [r[2] for r in rows] == want_status
    assert g.ctx.lib.mpvss_last_error(g.ctx.h) == b""
    for b, row, st in zip(boxes, rows, want_status):
        assert row == single(g, b)
        if st != L.OK:
            assert row[:2] == (bytes(eb), bytes(eb))
    assert secret_of(rows[0]) == secret_of(rows[4]) == SECRET


def test_argument_errors(pair):
    g, og = pair
    b = make_box(g, og, 40, [1, 2, 3])
    lib, h, eb = g.ctx.lib, g.ctx.h, g.codec.eb
    sec, gs, st = buf(size=2 * eb), buf(size=2 * eb), (ctypes.c_int * 2)()
    pos = (ctypes.c_int64 * 6)(*(b["pos"] * 2))
    sh, u = ptr(buf(b["s"] * 2)), ptr(buf(b["u"] * 2))
    ks = lambda *v: (ctypes.c_size_t * len(v))(*v)
    assert lib.mpvss_reconstruct_secrets(h, 2, ks(3, 3), pos, sh, u, ptr(sec), None, st) == L.OK and list(st) == [0, 0]
    assert lib.mpvss_reconstruct_secrets(h, 0, ks(3, 3), pos, sh, u, ptr(sec), ptr(gs), st) == L.ERR_ARG
    assert lib.mpvss_reconstruct_secrets(h, 2, ks(3, 0), pos, sh, u, ptr(sec), ptr(gs), st) == L.ERR_ARG
    for i in range(7):
        args = [ks(3, 3), pos, sh, u, ptr(sec), ptr(gs), st]
        if i == 5:
            continue                                            # gs_out is optional
        args[i] = None
        assert lib.mpvss_reconstruct_secrets(h, 2, *args) == L.ERR_ARG, i


def test_modp_paths_agree():
    g, og = m.Group("modp"), GROUPS["modp"]()
    boxes = [make_box(g, og, 50 + i, list(range(1, k + 1))) for i, k in enumerate((3, 43, 700))]
    _, want = batch(g, boxes)
    assert [secret_of(r) for r in want] == [SECRET] * 3
    for msm in (0, 1, 2):
        for tpi in (4, 8, 16):
            g.ctx.set_int("modp_msm", msm)
            g.ctx.set_int("modp_tpi", tpi)
            assert batch(g, boxes) == (L.OK, want), (msm, tpi)


def test_staged_state_survives_a_batch(pair):
    g, og = pair
    c = g.codec
    n, t, seed = 9, 5, 60
    kb = getattr(og, "q", og.order())
    sks = synth.private_keys(seed, n, og.name, og.order(), getattr(og, "q", None))
    box = m.Participant(g).distribute_secret(SECRET, g.fixed_base_exp(sks), t,
                                             coeffs=synth.coefficients(seed, t, og.order()),
                                             witnesses=synth.witnesses(seed, n, kb))
    pos, ys, rs = m.Participant(g)._flatten(box)
    args = (n, t, ptr(buf(c.enc_elems(box.commitments))), (ctypes.c_int64 * n)(*pos),
            ptr(buf(c.enc_elems(box.publickeys))), ptr(buf(c.enc_elems(ys))), ptr(buf(c.enc_scalars(rs))),
            ptr(buf(c.enc_scalar(box.challenge))))
    lib, h = g.ctx.lib, g.ctx.h

    def run():
        ok, dig = ctypes.c_int(0), buf(size=32)
        assert lib.mpvss_verify_distribution_run(h, ctypes.byref(ok), None, None, None, ptr(dig)) == L.OK
        return bool(ok.value), bytes(dig)

    assert lib.mpvss_verify_distribution_stage(h, *args) == L.OK
    want = run()
    assert want[0]
    rc, rows = batch(g, [make_box(g, og, 61, list(range(1, 44))), make_box(g, og, 62, [3, 1, 2])])
    assert rc == L.OK and [secret_of(r) for r in rows] == [SECRET] * 2
    assert run() == want


def test_participant_reconstruct_secrets(pair):
    g, og = pair
    c = g.codec
    p = m.Participant(g)
    kb = getattr(og, "q", og.order())
    jobs = []
    for i, (n, t) in enumerate(((5, 3), (7, 4), (6, 6), (4, 2), (5, 5), (6, 3))):
        seed = 70 + i
        sks = synth.private_keys(seed, n, og.name, og.order(), getattr(og, "q", None))
        ws = synth.witnesses(seed, n, kb)
        co = synth.coefficients(seed, t, og.order())
        box = p.distribute_secret(SECRET, g.fixed_base_exp(sks), t, coeffs=co, witnesses=ws)
        sbs = p.extract_secret_shares(box, sks, ws)
        if i == 0:  # the decrypted shares are G^P(i), as make_box computes them
            assert [sb.share for sb in sbs] == g.fixed_base_exp(g.scalar_poly_eval(co, list(range(1, n + 1))))
        jobs.append((sbs[:t + (i % 2)], box))
    jobs[2] = (jobs[2][0][:-1], jobs[2][1])                      # fewer share boxes than t: None, not sent
    stranger = copy.copy(jobs[3][0][0])
    stranger.publickey = jobs[0][0][0].publickey                 # a key that is not in the box: None, not sent
    jobs[3] = ([stranger] + jobs[3][0][1:], jobs[3][1])
    bad = copy.copy(jobs[4][1])
    bad.positions = dict(bad.positions)
    bad.positions[c.key(jobs[4][0][0].publickey)] = 1 << 40      # rejected by the library: None (the single call raises)
    jobs[4] = (jobs[4][0], bad)
    traces = [{} for _ in jobs]
    got = p.reconstruct_secrets(jobs, traces=traces)
    assert got == [SECRET, SECRET, None, None, None, SECRET]
    for j in (0, 1, 5):
        one = {}
        assert p.reconstruct(*jobs[j], trace=one) == got[j]
        assert traces[j]["G_s"] == one["G_s"]
    assert p.reconstruct(*jobs[2]) is None and p.reconstruct(*jobs[3]) is None
    with pytest.raises(m.MpvssError):
        p.reconstruct(*jobs[4])
    assert traces[2] == traces[3] == traces[4] == {}
