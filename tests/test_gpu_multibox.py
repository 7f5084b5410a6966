"""mpvss_verify_distributions: many boxes in one call.  Every verdict and digest equals what
mpvss_verify_distribution gives for the box alone (and the oracle for tiny boxes); tampered or malformed
boxes are false on their own without disturbing the rest; argument errors are status codes; the staged
single-box state survives a batch call in between."""
import copy
import ctypes
import hashlib

import pytest

import mpvss_rs_b200 as m
from mpvss_rs_b200 import lib as L
from mpvss_rs_b200 import synth
from mpvss_rs_b200.lib import buf, ptr
from oracle import pvss
from oracle.groups import GROUPS, SECP_N

pytestmark = pytest.mark.gpu
SECRET = pvss.string_to_secret("multibox")
GNAMES = ["modp", "secp256k1", "ristretto255"]


@pytest.fixture(scope="module", params=GNAMES)
def pair(request):
    return m.Group(request.param), GROUPS[request.param]()


def _keys(og, seed, n):
    return synth.private_keys(seed, n, og.name, og.order(), getattr(og, "q", None))


def deal(g, og, seed, n, t):
    """(box, secret keys, coefficients, witnesses) dealt by the library from synth seeds"""
    kb = getattr(og, "q", og.order())
    sks = _keys(og, seed, n)
    co, ws = synth.coefficients(seed, t, og.order()), synth.witnesses(seed, n, kb)
    box = m.Participant(g).distribute_secret(SECRET, g.fixed_base_exp(sks), t, coeffs=co, witnesses=ws)
    return box, sks, co, ws


def raw(g, box):
    """the boundary bytes of one box, as mpvss_verify_distribution takes them"""
    c = g.codec
    pos, ys, rs = m.Participant(g)._flatten(box)
    return dict(n=len(pos), t=len(box.commitments), comm=c.enc_elems(box.commitments), pos=list(pos),
                pk=c.enc_elems(box.publickeys), y=c.enc_elems(ys), r=c.enc_scalars(rs), ch=c.enc_scalar(box.challenge))


def batch(g, rb):
    k = len(rb)
    ok, dig = (ctypes.c_int * k)(), buf(size=32 * k)
    allpos = [p for r in rb for p in r["pos"]]
    cat = lambda key: ptr(buf(b"".join(r[key] for r in rb)))
    st = g.ctx.lib.mpvss_verify_distributions(
        g.ctx.h, k, (ctypes.c_size_t * k)(*[r["n"] for r in rb]), (ctypes.c_size_t * k)(*[r["t"] for r in rb]),
        cat("comm"), (ctypes.c_int64 * len(allpos))(*allpos), cat("pk"), cat("y"), cat("r"), cat("ch"), ok, ptr(dig))
    return st, [bool(v) for v in ok], [bytes(dig)[32 * i:32 * i + 32] for i in range(k)]


def single(g, r):
    ok, dig = ctypes.c_int(0), buf(size=32)
    st = g.ctx.lib.mpvss_verify_distribution(
        g.ctx.h, r["n"], r["t"], ptr(buf(r["comm"])), (ctypes.c_int64 * r["n"])(*r["pos"]), ptr(buf(r["pk"])),
        ptr(buf(r["y"])), ptr(buf(r["r"])), ptr(buf(r["ch"])), ctypes.byref(ok), None, None, None, ptr(dig))
    assert st == L.OK
    return bool(ok.value), bytes(dig)


def test_mixed_shapes_agree_with_the_single_box_call(pair):
    g, og = pair
    shapes = [(3, 3), (17, 9), (256, 171), (1024, 683)] + ([] if og.name == "modp" else [(4096, 2731)])
    rb = [raw(g, deal(g, og, 40 + i, n, t)[0]) for i, (n, t) in enumerate(shapes)]
    st, ok, dig = batch(g, rb)
    assert st == L.OK and ok == [True] * len(shapes)
    for i, r in enumerate(rb):
        assert (True, dig[i]) == single(g, r), shapes[i]


def _oracle_digest(og, obox, otr):
    """the transcript restated: SHA-256 over F(X) F(Y) F(a1) F(a2) per participant (dleq.rs:58-61, 87-99)"""
    h = hashlib.sha256()
    for j, pk in enumerate(obox.publickeys):
        pvss.append_transcript(og, otr["X"][j], obox.shares[og.element_to_bytes(pk)], otr["a1"][j], otr["a2"][j], h)
    return h.digest()


def test_tiny_boxes_agree_with_the_oracle(pair):
    """The second box's positions are scattered and above 2^17 (sliding-window chains): it verifies as false
    against its challenge, but its digest is still the transcript of the recomputed values."""
    g, og = pair
    host = lambda e: e if og.name == "modp" else og.element_to_bytes(e)
    boxes, oboxes = [], []
    for seed, n, t, scattered in ((60, 5, 3, None), (61, 4, 2, [131073, 200003, (1 << 20) | 7, 999999])):
        box, sks, co, ws = deal(g, og, seed, n, t)
        obox = pvss.distribute_secret(og, SECRET, [og.generate_public_key(s) for s in sks], t, co, ws)
        assert box.commitments == [host(c) for c in obox.commitments]
        if scattered:
            box.positions = {g.codec.key(pk): p for pk, p in zip(box.publickeys, scattered)}
            obox.positions = {og.element_to_bytes(pk): p for pk, p in zip(obox.publickeys, scattered)}
        boxes.append(box)
        oboxes.append(obox)
    rb = [raw(g, b) for b in boxes]
    st, ok, dig = batch(g, rb)
    assert st == L.OK and ok == [True, False]
    for i, obox in enumerate(oboxes):
        otr = {}
        assert pvss.verify_distribution_shares(og, obox, trace=otr) == ok[i]
        assert dig[i] == _oracle_digest(og, obox, otr) == single(g, rb[i])[1]


def test_tampering_stays_confined_to_its_box(pair):
    g, og = pair
    rb = [raw(g, deal(g, og, 70 + i, 6, 4)[0]) for i in range(6)]
    r1 = bytearray(rb[1]["r"])
    r1[g.codec.sb // 2] ^= 1                                    # one response of box 1
    rb[1]["r"] = bytes(r1)
    rb[2]["ch"], rb[3]["ch"] = rb[3]["ch"], rb[2]["ch"]          # challenges of boxes 2 and 3 swapped
    eb = g.codec.eb
    rb[4]["comm"] = rb[4]["comm"][:eb] + rb[0]["comm"][eb:2 * eb] + rb[4]["comm"][2 * eb:]   # one commitment of box 4
    st, ok, _ = batch(g, rb)
    assert st == L.OK and ok == [True, False, False, False, False, True]


@pytest.mark.parametrize("gname", ["secp256k1", "ristretto255"])
def test_malformed_contents_stay_confined(gname):
    og, g = GROUPS[gname](), m.Group(gname)
    eb = g.codec.eb
    rb = [raw(g, deal(g, og, 80 + i, 5, 3)[0]) for i in range(6)]
    bad_point = (b"\x05" + b"\x11" * 32) if gname == "secp256k1" else b"\xff" * 32
    rb[1]["y"] = rb[1]["y"][:eb] + bad_point + rb[1]["y"][2 * eb:]              # a share that does not decode
    rb[2]["comm"] = rb[2]["comm"][:eb] + bad_point + rb[2]["comm"][2 * eb:]     # a commitment that does not decode
    rb[3]["pos"][2] = 1 << 40                                                   # a position out of range
    if gname == "secp256k1":                                                    # a response >= n (not a k256 Scalar)
        rb[4]["r"] = rb[4]["r"][:32] + SECP_N.to_bytes(32, "big") + rb[4]["r"][64:]
    st, ok, dig = batch(g, rb)
    want = [True, False, False, False, gname != "secp256k1", True]
    assert st == L.OK and ok == want
    assert g.ctx.lib.mpvss_last_error(g.ctx.h) == b""           # a rejected box is no context error
    for i in (1, 2, 3) + ((4,) if gname == "secp256k1" else ()):
        assert dig[i] == bytes(32)
    for i in (0, 5):
        assert (True, dig[i]) == single(g, rb[i])


def test_modp_malformed_and_invalid_elements_stay_confined():
    og, g = GROUPS["modp"](), m.Group("modp")
    rb = [raw(g, deal(g, og, 90 + i, 5, 3)[0]) for i in range(4)]
    rb[1]["pos"][0] = 1 << 40
    st, ok, dig = batch(g, rb)
    assert st == L.OK and ok == [True, False, True, True] and dig[1] == bytes(32)
    g.ctx.set_int("validate", 1)
    rb[2]["y"] = rb[2]["y"][:256] + (og.q + 1).to_bytes(256, "little") + rb[2]["y"][512:]   # element >= q
    rb[3]["comm"] = (og.q - 1).to_bytes(256, "little") + rb[3]["comm"][256:]              # -1: outside the subgroup
    st, ok, dig = batch(g, rb)
    assert st == L.OK and ok == [True, False, False, False]
    assert dig[2] == dig[3] == bytes(32) and (True, dig[0]) == single(g, rb[0])


def test_modp_lone_live_box_runs_unchunked():
    """A batch in which one box is left to plan -- a one-box call, or every other box rejected -- is still
    planned as a batch (K = 1, results at the box's own rows), also at n = 2048, t = 1366 where the single-box
    plan cuts the polynomial into chunks, and when "modp_chunks" asks for chunks.  Every placement of a2
    gives the same verdicts and digests."""
    og, g = GROUPS["modp"](), m.Group("modp")
    big = raw(g, deal(g, og, 130, 2048, 1366)[0])
    small = raw(g, deal(g, og, 131, 5, 3)[0])
    want = single(g, big)
    assert want[0]
    for ov in (3, 0, 2):
        g.ctx.set_int("modp_overlap", ov)
        assert batch(g, [big]) == (L.OK, [True], [want[1]]), ov
        small_bad = dict(small, pos=[1, 2, 1 << 40, 4, 5])
        assert batch(g, [small_bad, big]) == (L.OK, [False, True], [bytes(32), want[1]]), ov
    g.ctx.set_int("modp_overlap", 3)
    mid = raw(g, deal(g, og, 132, 300, 200)[0])
    g.ctx.set_int("modp_chunks", 4)
    st, ok, dig = batch(g, [mid])
    assert st == L.OK and ok == [True]
    g.ctx.set_int("modp_chunks", 0)
    assert (True, dig[0]) == single(g, mid)


def test_argument_errors(pair):
    g, og = pair
    r = raw(g, deal(g, og, 100, 3, 2)[0])
    lib, h = g.ctx.lib, g.ctx.h
    ok, dig = (ctypes.c_int * 2)(), buf(size=64)
    args = lambda: (ptr(buf(r["comm"] * 2)), None, ptr(buf(r["pk"] * 2)), ptr(buf(r["y"] * 2)), ptr(buf(r["r"] * 2)),
                    ptr(buf(r["ch"] * 2)), ok, ptr(dig))
    sz = lambda *v: (ctypes.c_size_t * len(v))(*v)
    assert lib.mpvss_verify_distributions(h, 2, sz(3, 3), sz(2, 2), *args()) == L.OK and list(ok) == [1, 1]
    assert lib.mpvss_verify_distributions(h, 0, sz(3, 3), sz(2, 2), *args()) == L.ERR_ARG
    assert lib.mpvss_verify_distributions(h, 2, None, sz(2, 2), *args()) == L.ERR_ARG
    assert lib.mpvss_verify_distributions(h, 2, sz(3, 3), None, *args()) == L.ERR_ARG
    assert lib.mpvss_verify_distributions(h, 2, sz(3, 0), sz(2, 2), *args()) == L.ERR_ARG
    assert lib.mpvss_verify_distributions(h, 2, sz(3, 3), sz(0, 2), *args()) == L.ERR_ARG


def test_staged_state_survives_a_batch(pair):
    g, og = pair
    a, b, c = (raw(g, deal(g, og, 110 + i, n, t)[0]) for i, (n, t) in enumerate(((9, 5), (12, 7), (4, 4))))
    want = single(g, a)
    assert want[0]
    lib, h = g.ctx.lib, g.ctx.h
    assert lib.mpvss_verify_distribution_stage(h, a["n"], a["t"], ptr(buf(a["comm"])), (ctypes.c_int64 * a["n"])(*a["pos"]),
                                               ptr(buf(a["pk"])), ptr(buf(a["y"])), ptr(buf(a["r"])),
                                               ptr(buf(a["ch"]))) == L.OK
    st, ok, _ = batch(g, [b, c])
    assert st == L.OK and ok == [True, True]
    res, dig = ctypes.c_int(0), buf(size=32)
    assert lib.mpvss_verify_distribution_run(h, ctypes.byref(res), None, None, None, ptr(dig)) == L.OK
    assert (bool(res.value), bytes(dig)) == want


def test_participant_verify_distributions(pair):
    g, og = pair
    boxes = [deal(g, og, 120 + i, n, t)[0] for i, (n, t) in enumerate(((5, 3), (8, 6), (7, 2), (6, 6)))]
    boxes[1] = copy.copy(boxes[1])
    boxes[1].responses = dict(boxes[1].responses)
    boxes[1].responses.pop(g.codec.key(boxes[1].publickeys[0]))            # a map miss: false, not sent
    boxes[2] = copy.copy(boxes[2])
    boxes[2].challenge = boxes[2].challenge + 1
    p = m.Participant(g)
    traces = [{} for _ in boxes]
    got = p.verify_distributions(boxes, traces=traces)
    assert got == [p.verify_distribution_shares(b) for b in boxes] == [True, False, False, True]
    for b, tr in zip((0, 3), (traces[0], traces[3])):
        one = {}
        p.verify_distribution_shares(boxes[b], trace=one)
        assert tr["digest"] == one["digest"]
    assert "digest" not in traces[1]
