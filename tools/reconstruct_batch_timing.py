"""Time one mpvss_reconstruct_secrets call against the B single mpvss_reconstruct calls it replaces.

For each group, B boxes of k = ceil(2n/3) decrypted shares at positions 1..k are made from synth coefficients
(S_i = G^P(i) by mpvss_fixed_base_exp of mpvss_scalar_poly_eval, which is what extract_shares decrypts to).  Both
forms read the same host buffers and are timed as host wall time that ends in the call's own synchronise, after
one warm-up of each; they alternate, and the median and the spread of the repetitions are reported with the kernel
time and launch count the library reports.  For ModpGroup the batch is also timed with every box forced into the
direct launch ("modp_msm" 0) and onto the bucket method ("modp_msm" 1), the two sides of the batch's bucket rule.
Every form's secrets and G^s are checked byte for byte against the single calls.  The device name and power limit
are read in the same run.

    python tools/reconstruct_batch_timing.py [--reps 3] [--out profiles/reconstruct_batch_r03.json]
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

SECRET = 0x5EC12E7
# (B, n): B boxes of k = ceil(2n/3) shares; the MODP shapes reach past the batch's bucket threshold
SHAPES = {
    "modp": [(256, 64), (64, 256), (16, 1024), (4, 4096), (2, 8192), (2, 16384)],
    "secp256k1": [(64, 256), (16, 1024), (4, 4096)],
    "ristretto255": [(64, 256), (16, 1024), (4, 4096)],
}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def make_boxes(g, og, B, k, seed0):
    c = g.codec
    pos = list(range(1, k + 1))
    s, u = [], []
    for b in range(B):
        co = synth.coefficients(seed0 + b, k, og.order())
        s.append(c.enc_elems(g.fixed_base_exp(g.scalar_poly_eval(co, pos))))
        u.append((og.mask_of(og.exp(og.generator(), co[0])) ^ SECRET).to_bytes(c.eb, "big"))
    return {"s": buf(b"".join(s)), "u": buf(b"".join(u))}


def at(b, off, typ=ctypes.c_uint8):
    return ctypes.cast(ctypes.addressof(b) + off, ctypes.POINTER(typ))


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "all": xs}


def time_shape(g, B, k, H, reps):
    lib, h, eb = g.ctx.lib, g.ctx.h, g.codec.eb
    pos = (ctypes.c_int64 * (B * k))(*([p for _ in range(B) for p in range(1, k + 1)]))
    ks = (ctypes.c_size_t * B)(*[k] * B)
    sec, gs, st = buf(size=B * eb), buf(size=B * eb), (ctypes.c_int * B)()
    one_sec, one_gs = buf(size=B * eb), buf(size=B * eb)

    def batch(msm=None):
        if msm is not None:
            g.ctx.set_int("modp_msm", msm)
        try:
            t0 = time.perf_counter()
            rc = lib.mpvss_reconstruct_secrets(h, B, ks, pos, at(H["s"], 0), at(H["u"], 0), at(sec, 0), at(gs, 0), st)
            ms = (time.perf_counter() - t0) * 1e3
        finally:
            if msm is not None:
                g.ctx.set_int("modp_msm", 2)
        assert rc == L.OK and list(st) == [L.OK] * B, (rc, list(st))
        assert bytes(sec) == bytes(one_sec) and bytes(gs) == bytes(one_gs), "batch differs from the single calls"
        return ms, g.ctx.last_kernel_ms, g.ctx.last_kernel_launches

    def singles():
        kms, launches = 0.0, 0
        t0 = time.perf_counter()
        for b in range(B):
            rc = lib.mpvss_reconstruct(h, k, at(pos, 8 * b * k, ctypes.c_int64), at(H["s"], b * k * eb),
                                       at(H["u"], b * eb), at(one_sec, b * eb), at(one_gs, b * eb))
            assert rc == L.OK
            kms += g.ctx.last_kernel_ms
            launches += g.ctx.last_kernel_launches
        return (time.perf_counter() - t0) * 1e3, kms, launches

    singles()
    assert all(int.from_bytes(bytes(one_sec)[b * eb:(b + 1) * eb], "big") == SECRET for b in range(B))
    forced = (0, 1) if g.name == "modp" else ()
    batch()
    for f in forced:
        batch(f)
    rb, rs, rf = [], [], {f: [] for f in forced}
    for _ in range(reps):
        rb.append(batch())
        rs.append(singles())
        for f in forced:
            rf[f].append(batch(f))
    bm, sm = spread([r[0] for r in rb]), spread([r[0] for r in rs])
    out = {"boxes": B, "k": k, "batch_ms": bm, "single_ms": sm, "speedup": sm["median"] / bm["median"],
           "batch_kernel_ms": statistics.median(r[1] for r in rb), "batch_launches": rb[-1][2],
           "single_kernel_ms": statistics.median(r[1] for r in rs), "single_launches": rs[-1][2]}
    for f, name in ((0, "direct"), (1, "buckets")):
        if f in rf:
            out[f"batch_{name}_ms"] = spread([r[0] for r in rf[f]])
            out[f"batch_{name}_kernel_ms"] = statistics.median(r[1] for r in rf[f])
            out[f"batch_{name}_launches"] = rf[f][-1][2]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reconstruct_batch_r03.json"))
    ap.add_argument("--groups", default=",".join(SHAPES))
    a = ap.parse_args()
    assert a.reps >= 3
    res = {"tool": "tools/reconstruct_batch_timing.py", "gpu": gpu_info(), "reps": a.reps,
           "timing": "host wall time ending in the call's synchronise; batch and singles alternate", "shapes": []}
    for gname in a.groups.split(","):
        g, og = m.Group(gname), GROUPS[gname]()
        for B, n in SHAPES[gname]:
            k = math.ceil(2 * n / 3)
            H = make_boxes(g, og, B, k, 2000 + B)
            r = dict(group=gname, n=n, **time_shape(g, B, k, H, a.reps))
            print(json.dumps({key: (v["median"] if isinstance(v, dict) else v) for key, v in r.items()}), flush=True)
            res["shapes"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
