"""Time one mpvss_verify_distributions call against the B single mpvss_verify_distribution calls it replaces.

For each group, B boxes of n participants and t = ceil(2n/3) commitments are dealt by the library
(mpvss_distribute, synth seeds).  Both forms read the same host buffers and are timed as host wall time that
ends in the call's own synchronise, after one warm-up of each; the two alternate, and the median and the
spread of the repetitions are reported with the kernel time and launch count the library reports.  For
ModpGroup the batch is also timed with a2 forced onto a side stream beside the X_i launch ("modp_overlap" 2),
the alternative to the placement the library picks.  The device name and power limit are read in the same
run.

    python tools/multibox_timing.py [--reps 3] [--out profiles/multibox_r03.json]
"""
import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mpvss_rs_b200 as m  # noqa: E402
from mpvss_rs_b200 import lib as L  # noqa: E402
from mpvss_rs_b200 import synth  # noqa: E402
from mpvss_rs_b200.lib import buf  # noqa: E402
from oracle.groups import GROUPS  # noqa: E402

SHAPES = {
    "modp": [(256, 64), (64, 256), (16, 1024), (4, 4096)],
    "secp256k1": [(64, 256), (16, 1024), (4, 4096)],
    "ristretto255": [(64, 256), (16, 1024), (4, 4096)],
}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def deal_boxes(g, og, B, n, t, seed0):
    c = g.codec
    kb = getattr(og, "q", og.order())
    parts = {k: [] for k in ("comm", "pk", "y", "r", "ch")}
    for b in range(B):
        seed = seed0 + b
        pks = g.fixed_base_exp(synth.private_keys(seed, n, og.name, og.order(), getattr(og, "q", None)))
        box = m.Participant(g).distribute_secret(1, pks, t, coeffs=synth.coefficients(seed, t, og.order()),
                                                 witnesses=synth.witnesses(seed, n, kb))
        parts["comm"].append(c.enc_elems(box.commitments))
        parts["pk"].append(c.enc_elems(pks))
        parts["y"].append(c.enc_elems([box.shares[c.key(pk)] for pk in pks]))
        parts["r"].append(c.enc_scalars([box.responses[c.key(pk)] for pk in pks]))
        parts["ch"].append(c.enc_scalar(box.challenge))
    return {k: buf(b"".join(v)) for k, v in parts.items()}


def at(b, off, typ=ctypes.c_uint8):
    return ctypes.cast(ctypes.addressof(b) + off, ctypes.POINTER(typ))


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "all": xs}


def time_shape(g, B, n, t, H, reps):
    lib, h, eb, sb = g.ctx.lib, g.ctx.h, g.codec.eb, g.codec.sb
    pos = (ctypes.c_int64 * (B * n))(*([p for _ in range(B) for p in range(1, n + 1)]))
    ns, ts = (ctypes.c_size_t * B)(*[n] * B), (ctypes.c_size_t * B)(*[t] * B)
    ok, dig = (ctypes.c_int * B)(), buf(size=32 * B)

    def batch():
        t0 = time.perf_counter()
        st = lib.mpvss_verify_distributions(h, B, ns, ts, at(H["comm"], 0), pos, at(H["pk"], 0), at(H["y"], 0),
                                            at(H["r"], 0), at(H["ch"], 0), ok, at(dig, 0))
        ms = (time.perf_counter() - t0) * 1e3
        assert st == L.OK and all(ok), (st, list(ok))
        return ms, g.ctx.last_kernel_ms, g.ctx.last_kernel_launches

    def singles():
        one, kms, launches = ctypes.c_int(0), 0.0, 0
        t0 = time.perf_counter()
        for b in range(B):
            st = lib.mpvss_verify_distribution(h, n, t, at(H["comm"], b * t * eb), at(pos, 8 * b * n, ctypes.c_int64),
                                               at(H["pk"], b * n * eb), at(H["y"], b * n * eb), at(H["r"], b * n * sb),
                                               at(H["ch"], b * sb), ctypes.byref(one), None, None, None, None)
            assert st == L.OK and one.value == 1
            kms += g.ctx.last_kernel_ms
            launches += g.ctx.last_kernel_launches
        return (time.perf_counter() - t0) * 1e3, kms, launches

    def batch_side():  # MODP: a2 forced onto the side stream beside the X_i launch ("modp_overlap" = 2)
        g.ctx.set_int("modp_overlap", 2)
        try:
            return batch()
        finally:
            g.ctx.set_int("modp_overlap", 3)

    side = g.name == "modp"
    batch()
    singles()
    if side:
        batch_side()
    rb, rs, rside = [], [], []
    for _ in range(reps):
        rb.append(batch())
        rs.append(singles())
        if side:
            rside.append(batch_side())
    bm, sm = spread([r[0] for r in rb]), spread([r[0] for r in rs])
    out = {"boxes": B, "n": n, "t": t, "batch_ms": bm, "single_ms": sm, "speedup": sm["median"] / bm["median"],
           "batch_kernel_ms": statistics.median(r[1] for r in rb), "batch_launches": rb[-1][2],
           "single_kernel_ms": statistics.median(r[1] for r in rs), "single_launches": rs[-1][2]}
    if side:
        out["batch_a2_side_ms"] = spread([r[0] for r in rside])
        out["batch_a2_side_kernel_ms"] = statistics.median(r[1] for r in rside)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "multibox_r03.json"))
    ap.add_argument("--groups", default=",".join(SHAPES))
    a = ap.parse_args()
    assert a.reps >= 3
    res = {"tool": "tools/multibox_timing.py", "gpu": gpu_info(), "reps": a.reps,
           "timing": "host wall time ending in the call's synchronise; batch and singles alternate", "shapes": []}
    for gname in a.groups.split(","):
        g, og = m.Group(gname), GROUPS[gname]()
        for B, n in SHAPES[gname]:
            t = math.ceil(2 * n / 3)
            H = deal_boxes(g, og, B, n, t, 1000 + B)
            r = dict(group=gname, **time_shape(g, B, n, t, H, a.reps))
            print(json.dumps({k: (v["median"] if isinstance(v, dict) else v) for k, v in r.items()}), flush=True)
            res["shapes"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
