"""mpvss_distribute_secrets: many dealings in one call.  Every output row of every box equals what mpvss_distribute
gives for the box alone (and the oracle for tiny boxes); the dealt boxes verify and reconstruct through the batch
calls; a rejected box fails on its own with zero rows; argument errors are status codes; no launch runs per box;
the staged single-box verify state survives a batch call in between."""
import ctypes
import threading

import pytest

import mpvss_rs_b200 as m
from mpvss_rs_b200 import lib as L
from mpvss_rs_b200 import synth
from mpvss_rs_b200.lib import buf, ptr
from oracle import pvss
from oracle.groups import GROUPS, SECP_N

pytestmark = pytest.mark.gpu
SECRET = pvss.string_to_secret("distribute batch")
GNAMES = ["modp", "secp256k1", "ristretto255"]
OUTS = ("comm", "shares", "chal", "resp", "u", "x")


@pytest.fixture(scope="module", params=GNAMES)
def pair(request):
    return m.Group(request.param), GROUPS[request.param]()


def job(g, og, seed, n, t, secret=SECRET):
    """the boundary bytes of one dealing from synth seeds, as mpvss_distribute takes them"""
    c = g.codec
    sks = synth.private_keys(seed, n, og.name, og.order(), getattr(og, "q", None))
    co, ws = synth.coefficients(seed, t, og.order()), synth.witnesses(seed, n, getattr(og, "q", og.order()))
    return dict(n=n, t=t, s=secret.to_bytes(max(1, (secret.bit_length() + 7) // 8), "big"), co=c.enc_scalars(co),
                w=c.enc_scalars(ws), pk=c.enc_elems(g.fixed_base_exp(sks)), sks=sks, cos=co, ws=ws)


def batch(g, jobs, with_x=True):
    """(return code, per box {comm, shares, chal, resp, u, x, st})"""
    c, k = g.codec, len(jobs)
    N, T = sum(j["n"] for j in jobs), sum(j["t"] for j in jobs)
    comm, shares, resp, x = buf(size=T * c.eb), buf(size=N * c.eb), buf(size=N * c.sb), buf(size=N * c.eb)
    chal, u, st = buf(size=k * c.sb), buf(size=k * c.eb), (ctypes.c_int * k)()
    cat = lambda key: ptr(buf(b"".join(j[key] for j in jobs)))
    rc = g.ctx.lib.mpvss_distribute_secrets(
        g.ctx.h, k, (ctypes.c_size_t * k)(*[j["n"] for j in jobs]), (ctypes.c_size_t * k)(*[j["t"] for j in jobs]),
        ptr(buf(b"".join(j["s"].rjust(c.eb, b"\0") for j in jobs))), cat("co"), cat("w"), cat("pk"), ptr(comm),
        ptr(shares), ptr(chal), ptr(resp), ptr(u), ptr(x) if with_x else None, st)
    rows, n0, t0 = [], 0, 0
    for b, j in enumerate(jobs):
        n, t = j["n"], j["t"]
        rows.append(dict(comm=bytes(comm)[t0 * c.eb:(t0 + t) * c.eb], shares=bytes(shares)[n0 * c.eb:(n0 + n) * c.eb],
                         chal=bytes(chal)[b * c.sb:(b + 1) * c.sb], resp=bytes(resp)[n0 * c.sb:(n0 + n) * c.sb],
                         u=bytes(u)[b * c.eb:(b + 1) * c.eb], x=bytes(x)[n0 * c.eb:(n0 + n) * c.eb], st=st[b]))
        n0, t0 = n0 + n, t0 + t
    return rc, rows


def single(g, j):
    """mpvss_distribute for one box, with the secret as its minimal big-endian bytes; zero rows when it fails"""
    c, n, t = g.codec, j["n"], j["t"]
    o = dict(comm=buf(size=t * c.eb), shares=buf(size=n * c.eb), chal=buf(size=c.sb), resp=buf(size=n * c.sb),
             u=buf(size=c.eb), x=buf(size=n * c.eb))
    st = g.ctx.lib.mpvss_distribute(g.ctx.h, n, t, ptr(buf(j["s"])), len(j["s"]), ptr(buf(j["co"])), ptr(buf(j["w"])),
                                    ptr(buf(j["pk"])), *(ptr(o[k]) for k in OUTS))
    return dict({k: bytes(v) if st == L.OK else bytes(len(v)) for k, v in o.items()}, st=st)


def test_mixed_shapes_equal_the_single_call(pair):
    g, og = pair
    shapes = [(1, 1), (3, 3), (17, 9), (256, 171), (1024, 683)]
    if og.name != "modp":
        shapes.append((4096, 2731))
    jobs = [job(g, og, 100 + i, n, t) for i, (n, t) in enumerate(shapes)]
    rc, rows = batch(g, jobs)
    assert rc == L.OK
    for j, row in zip(jobs, rows):
        assert row == single(g, j), (j["n"], j["t"])
        assert row["st"] == L.OK


def test_tiny_boxes_equal_the_oracle(pair):
    g, og = pair
    enc = (lambda e: e) if og.name == "modp" else og.element_to_bytes
    jobs = [job(g, og, 110 + i, n, t) for i, (n, t) in enumerate(((1, 1), (3, 2), (5, 5), (4, 1)))]
    got = m.Participant(g).distribute_secrets([(SECRET, g.codec.dec_elems(j["pk"], j["n"]), j["t"], j["cos"], j["ws"])
                                               for j in jobs])
    for j, box in zip(jobs, got):
        pks = [og.generate_public_key(s) for s in j["sks"]]
        obox = pvss.distribute_secret(og, SECRET, pks, j["t"], j["cos"], j["ws"])
        assert box.commitments == [enc(e) for e in obox.commitments]
        assert box.shares == {k: enc(v) for k, v in obox.shares.items()}
        assert (box.challenge, box.responses, box.U) == (obox.challenge, obox.responses, obox.U)


def test_round_trip_through_the_batch_calls(pair):
    """the dealt boxes verify in one mpvss_verify_distributions call with the single verify's digests, and the
    extracted shares give every box's secret back in one mpvss_reconstruct_secrets call"""
    g, og = pair
    p = m.Participant(g)
    shapes = ((5, 3), (7, 4), (9, 9), (1, 1))
    jobs = [job(g, og, 120 + i, n, t, secret=SECRET + i) for i, (n, t) in enumerate(shapes)]
    boxes = p.distribute_secrets([(SECRET + i, g.codec.dec_elems(j["pk"], j["n"]), j["t"], j["cos"], j["ws"])
                                  for i, j in enumerate(jobs)])
    traces = [{} for _ in boxes]
    assert p.verify_distributions(boxes, traces=traces) == [True] * len(boxes)
    for box, tr in zip(boxes, traces):
        one = {}
        assert p.verify_distribution_shares(box, trace=one) and one["digest"] == tr["digest"]
    shares = [p.extract_secret_shares(box, j["sks"], j["ws"]) for box, j in zip(boxes, jobs)]
    assert p.reconstruct_secrets(list(zip(shares, boxes))) == [SECRET + i for i in range(len(boxes))]


@pytest.mark.parametrize("gname", ["secp256k1", "ristretto255"])
def test_rejection_stays_in_its_box(gname):
    g, og = m.Group(gname), GROUPS[gname]()
    eb, sb = g.codec.eb, g.codec.sb
    jobs = [job(g, og, 130 + i, 6, 4) for i in range(4)]
    bad = (b"\x05" + b"\x11" * 32) if gname == "secp256k1" else b"\xff" * 32
    jobs[1]["pk"] = jobs[1]["pk"][:2 * eb] + bad + jobs[1]["pk"][3 * eb:]        # an undecodable public key
    want = [L.OK, L.ERR_ENCODING, L.OK, L.OK]
    if gname == "secp256k1":                                                   # a witness not below the order
        jobs[2]["w"] = jobs[2]["w"][:sb] + SECP_N.to_bytes(32, "big") + jobs[2]["w"][2 * sb:]
        want[2] = L.ERR_ENCODING
    rc, rows = batch(g, jobs)
    assert rc == L.OK and [r["st"] for r in rows] == want
    assert g.ctx.lib.mpvss_last_error(g.ctx.h) == b""
    for j, row, st in zip(jobs, rows, want):
        assert row == single(g, j)
        if st != L.OK:
            assert all(v == bytes(len(v)) for k, v in row.items() if k != "st")


def test_argument_errors(pair):
    g, og = pair
    j = job(g, og, 140, 3, 2)
    c, lib, h = g.codec, g.ctx.lib, g.ctx.h
    ks = lambda *v: (ctypes.c_size_t * len(v))(*v)
    outs = [ptr(buf(size=4 * c.eb)), ptr(buf(size=6 * c.eb)), ptr(buf(size=2 * c.sb)), ptr(buf(size=6 * c.sb)),
            ptr(buf(size=2 * c.eb)), ptr(buf(size=6 * c.eb))]
    ins = [ptr(buf(j["s"].rjust(c.eb, b"\0") * 2)), ptr(buf(j["co"] * 2)), ptr(buf(j["w"] * 2)), ptr(buf(j["pk"] * 2))]
    st = (ctypes.c_int * 2)()
    call = lambda nb, n, t, args: lib.mpvss_distribute_secrets(h, nb, n, t, *args)
    full = ins + outs + [st]
    assert call(2, ks(3, 3), ks(2, 2), full[:9] + [None, st]) == L.OK and list(st) == [0, 0]   # x_out is optional
    assert call(0, ks(3, 3), ks(2, 2), full) == L.ERR_ARG
    for n, t in (((3, 0), (2, 2)), ((3, 3), (2, 0)), ((3, 3), (2, 4))):
        assert call(2, ks(*n), ks(*t), full) == L.ERR_ARG, (n, t)
    assert call(2, None, ks(2, 2), full) == L.ERR_ARG and call(2, ks(3, 3), None, full) == L.ERR_ARG
    for i in range(len(full)):
        if i == 9:
            continue
        args = list(full)
        args[i] = None
        assert call(2, ks(3, 3), ks(2, 2), args) == L.ERR_ARG, i


def test_no_launch_per_box(pair):
    g, og = pair
    jobs = [job(g, og, 150 + i, 5, 3) for i in range(8)]
    assert batch(g, jobs[:1])[0] == L.OK
    one = g.ctx.last_kernel_launches
    assert batch(g, jobs)[0] == L.OK
    assert g.ctx.last_kernel_launches == one > 0


def test_staged_state_survives_a_batch(pair):
    g, og = pair
    c = g.codec
    n, t = 9, 5
    j = job(g, og, 160, n, t)
    box = m.Participant(g).distribute_secret(SECRET, c.dec_elems(j["pk"], n), t, coeffs=j["cos"], witnesses=j["ws"])
    pos, ys, rs = m.Participant(g)._flatten(box)
    args = (n, t, ptr(buf(c.enc_elems(box.commitments))), (ctypes.c_int64 * n)(*pos), ptr(buf(j["pk"])),
            ptr(buf(c.enc_elems(ys))), ptr(buf(c.enc_scalars(rs))), ptr(buf(c.enc_scalar(box.challenge))))
    lib, h = g.ctx.lib, g.ctx.h

    def run():
        ok, dig = ctypes.c_int(0), buf(size=32)
        assert lib.mpvss_verify_distribution_run(h, ctypes.byref(ok), None, None, None, ptr(dig)) == L.OK
        return bool(ok.value), bytes(dig)

    assert lib.mpvss_verify_distribution_stage(h, *args) == L.OK
    want = run()
    assert want[0]
    rc, rows = batch(g, [job(g, og, 161, 43, 29), job(g, og, 162, 3, 2)])
    assert rc == L.OK and [r["st"] for r in rows] == [L.OK, L.OK]
    assert run() == want


def test_participant_distribute_secrets(pair):
    g, og = pair
    c = g.codec
    p = m.Participant(g)
    jobs = []
    for i, (n, t) in enumerate(((5, 3), (7, 4), (6, 6), (4, 1))):
        j = job(g, og, 170 + i, n, t)
        jobs.append((SECRET + i, c.dec_elems(j["pk"], n), t, j["cos"], j["ws"]))
    got = p.distribute_secrets(jobs)
    for jb, box in zip(jobs, got):
        assert box == p.distribute_secret(*jb)
    if og.name != "modp":                                   # a box the library rejects is None
        bad = (b"\x05" + b"\x11" * 32) if og.name == "secp256k1" else b"\xff" * 32
        jobs[1] = (jobs[1][0], jobs[1][1][:2] + [bad] + jobs[1][1][3:]) + jobs[1][2:]
        got2 = p.distribute_secrets(jobs)
        assert got2[1] is None and [got2[i] for i in (0, 2, 3)] == [got[i] for i in (0, 2, 3)]
        with pytest.raises(m.MpvssError):
            p.distribute_secret(*jobs[1])
    fresh = p.distribute_secrets([(SECRET, jobs[0][1], 3)])  # coefficients and witnesses drawn by the library side
    assert p.verify_distribution_shares(fresh[0])
    with pytest.raises(AssertionError):                     # threshold > n, as distribute_secret
        p.distribute_secrets([(SECRET, jobs[0][1], 6)])


def test_not_collective():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from mpvss_rs_b200.lib import comm_unique_id
    og = GROUPS["modp"]()
    uid, groups, out = comm_unique_id(), [m.Group("modp", device=r) for r in range(2)], [None, None]
    j = job(groups[0], og, 180, 3, 2)

    def worker(r):
        groups[r].ctx.comm_init(uid, 2, r)
        out[r] = batch(groups[r], [j])[0]
    th = [threading.Thread(target=worker, args=(r,)) for r in range(2)]
    for x in th:
        x.start()
    for x in th:
        x.join(300)
    assert out == [L.ERR_UNSUPPORTED, L.ERR_UNSUPPORTED]
