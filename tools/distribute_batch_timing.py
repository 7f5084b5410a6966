"""Time one mpvss_distribute_secrets call against the B single mpvss_distribute calls it replaces.

For each group, B boxes of n participants and t = ceil(2n/3) coefficients are dealt to the same n public keys (the
participants of one round), each box with its own synth coefficients, witnesses and secret.  Both forms read the
same host buffers and are timed as host wall time that ends in the call's own synchronise, after one warm-up of
each; they alternate, and the median and the spread of the repetitions are reported with the kernel time and launch
count the library reports.  Every output row of the batch is checked byte for byte against the single calls.  The
device name and power limit are read in the same run.

    python tools/distribute_batch_timing.py [--reps 3] [--out profiles/distribute_batch_r03.json]
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

# (B, n): B boxes of n participants
SHAPES = {
    "modp": [(256, 64), (64, 256), (16, 1024), (4, 4096)],
    "secp256k1": [(64, 256), (16, 1024), (4, 4096)],
    "ristretto255": [(64, 256), (16, 1024), (4, 4096)],
}
OUTS = ("comm", "shares", "chal", "resp", "u", "x")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def make_inputs(g, og, B, n, t, seed0):
    c = g.codec
    pks = g.fixed_base_exp(synth.private_keys(seed0, n, og.name, og.order(), getattr(og, "q", None)))
    kb = getattr(og, "q", og.order())
    co = [synth.coefficients(seed0 + b, t, og.order()) for b in range(B)]
    ws = [synth.witnesses(seed0 + b, n, kb) for b in range(B)]
    return {"s": buf(b"".join((0x5EC12E7 + b).to_bytes(c.eb, "big") for b in range(B))),
            "co": buf(b"".join(c.enc_scalars(x) for x in co)), "w": buf(b"".join(c.enc_scalars(x) for x in ws)),
            "pk": buf(c.enc_elems(pks) * B)}


def at(b, off):
    return ctypes.cast(ctypes.addressof(b) + off, ctypes.POINTER(ctypes.c_uint8))


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "all": xs}


def time_shape(g, B, n, t, H, reps):
    lib, h, eb, sb = g.ctx.lib, g.ctx.h, g.codec.eb, g.codec.sb
    # bytes per box of every output
    sizes = {"comm": t * eb, "shares": n * eb, "chal": sb, "resp": n * sb, "u": eb, "x": n * eb}
    bo = {k: buf(size=B * v) for k, v in sizes.items()}
    so = {k: buf(size=B * v) for k, v in sizes.items()}
    ns, ts, st = (ctypes.c_size_t * B)(*[n] * B), (ctypes.c_size_t * B)(*[t] * B), (ctypes.c_int * B)()

    def batch():
        t0 = time.perf_counter()
        rc = lib.mpvss_distribute_secrets(h, B, ns, ts, at(H["s"], 0), at(H["co"], 0), at(H["w"], 0), at(H["pk"], 0),
                                          *(at(bo[k], 0) for k in OUTS), st)
        ms = (time.perf_counter() - t0) * 1e3
        assert rc == L.OK and list(st) == [L.OK] * B, (rc, list(st))
        assert all(bytes(bo[k]) == bytes(so[k]) for k in OUTS), "batch differs from the single calls"
        return ms, g.ctx.last_kernel_ms, g.ctx.last_kernel_launches

    def singles():
        kms, launches = 0.0, 0
        t0 = time.perf_counter()
        for b in range(B):
            # the secret as its minimal big-endian bytes (the batch rows are left-padded to element size)
            rc = lib.mpvss_distribute(h, n, t, at(H["s"], (b + 1) * eb - 4), 4, at(H["co"], b * t * sb),
                                      at(H["w"], b * n * sb), at(H["pk"], b * n * eb),
                                      *(at(so[k], b * sizes[k]) for k in OUTS))
            assert rc == L.OK
            kms += g.ctx.last_kernel_ms
            launches += g.ctx.last_kernel_launches
        return (time.perf_counter() - t0) * 1e3, kms, launches

    singles()
    batch()
    rb, rs = [], []
    for _ in range(reps):
        rb.append(batch())
        rs.append(singles())
    bm, sm = spread([r[0] for r in rb]), spread([r[0] for r in rs])
    return {"boxes": B, "t": t, "batch_ms": bm, "single_ms": sm, "speedup": sm["median"] / bm["median"],
            "batch_kernel_ms": statistics.median(r[1] for r in rb), "batch_launches": rb[-1][2],
            "single_kernel_ms": statistics.median(r[1] for r in rs), "single_launches": rs[-1][2]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "distribute_batch_r03.json"))
    ap.add_argument("--groups", default=",".join(SHAPES))
    a = ap.parse_args()
    assert a.reps >= 3
    res = {"tool": "tools/distribute_batch_timing.py", "gpu": gpu_info(), "reps": a.reps,
           "timing": "host wall time ending in the call's synchronise; batch and singles alternate", "shapes": []}
    for gname in a.groups.split(","):
        g, og = m.Group(gname), GROUPS[gname]()
        for B, n in SHAPES[gname]:
            t = math.ceil(2 * n / 3)
            H = make_inputs(g, og, B, n, t, 3000 + B)
            r = dict(group=gname, n=n, **time_shape(g, B, n, t, H, a.reps))
            print(json.dumps({key: (v["median"] if isinstance(v, dict) else v) for key, v in r.items()}), flush=True)
            res["shapes"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
