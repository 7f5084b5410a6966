#!/usr/bin/env python
"""bench.py -- verified DLEQ shares/sec on B200 (BASELINE.json metric).

A "step" is one pass of Participant::verify_distribution_shares (participant.rs:399-455)
over one synthetic DistributionSharesBox: for every participant recompute
X_i = prod_j C_j^(i^j) from the t commitments, a1 = g^r X^c, a2 = y^r Y^c, then hash the
framed transcript on the host and compare the challenge.  Workload at N=1: the headline
configuration of the metric, ModpGroup n=4096 t=2731.  With N GPUs (one process per GPU) the
library shards the participants of ONE box of N*4096 participants round robin over the ranks
(rank r verifies participants r, r+N, ...; weak scaling, t fixed), gathers the transcript rows
with one ncclAllGather issued by the library on its own stream, and every rank hashes them.
torch.distributed is used only for the NCCL-id hand-off, the barrier and the max-over-ranks.

`value`: the box is RESIDENT in HBM (staged once before the timed loop; kernels + all-gather +
D2H + host SHA-256 are timed).  `e2e`: the full mpvss_verify_distribution call from pinned host
buffers, host->device copies and position planning inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n N] [--t T] [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step returned (verdict, transcript digest and, on one GPU, the
X_i / a1 / a2 rows) as DIR/<name>.npy; the box is synthesised from --seed, so two builds run with the same
arguments can be compared output for output.

`--impl reference` times the reference's CPU schedule (oracle/cpu_baseline.c, an OpenSSL
proxy for num-bigint since the Rust reference cannot be built here) on all host cores; it never
touches the GPU library (its box is synthesised with OpenSSL and Python integers).
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRICS = {"modp": "verified DLEQ shares/sec (MODP n=4096 t=2731, verify_distribution_shares)",
           "secp256k1": "verified DLEQ shares/sec (secp256k1 n=4096 t=2731, verify_distribution_shares)",
           "ristretto255": "verified DLEQ shares/sec (ristretto255 n=4096 t=2731, verify_distribution_shares)"}
CPU_PROXY = {"modp": "OpenSSL BN_mod_exp_mont (proxy for num-bigint 0.2)",
             "secp256k1": "OpenSSL EC_POINT_mul on secp256k1 (proxy for k256 0.13; OpenSSL has no specialised "
                          "secp256k1 code, so this under-states k256)"}
DTYPE = {"modp": "u32 limbs (2048-bit integers)", "secp256k1": "u32 limbs (256-bit prime fields)",
         "ristretto255": "u32 limbs (255-bit prime field)"}
SQR_MACS, MUL_MACS = 6240, 8256          # SURVEY.md 8d: 2048-bit Montgomery sqr / mul, 32x32->64 MACs
# 256-bit fields, plain representation with special-form reduction (DESIGN.md section 4): 8x8 limb
# product + fold; a squaring needs 36 distinct limb products
EC_MUL_MACS = {"secp256k1": 64 + 8, "ristretto255": 64 + 8}
EC_SQR_MACS = {"secp256k1": 36 + 8, "ristretto255": 36 + 8}
SEED = 0x6D70767373
RFC3526_2048 = int(
    "ffffffffffffffffc90fdaa22168c234c4c6628b80dc1cd129024e088a67cc74020bbea63b139b22514a08798e3404dd"
    "ef9519b3cd3a431b302b0a6df25f14374fe1356d6d51c245e485b576625e7ec6f44c42e9a637ed6b0bff5cb6f406b7ed"
    "ee386bfb5a899fa5ae9f24117c4b1fe649286651ece45b3dc2007cb8a163bf0598da48361c55d39a69163fa8fd24cf5f"
    "83655d23dca3ad961c62f356208552bb9ed529077096966d670c354e4abc9804f1746c08ca18217c32905e462e36ce3b"
    "e39e772c180e86039b2783a2ec07a28fb5c55df06f4c52c9de2bcbf6955817183995497cea956ae515d2261898fa0510"
    "15728e5a8aacaa68ffffffffffffffff", 16)
SECP_N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
DUMP_BYTES = 64_000_000                  # --dump-outputs: all .npy files together stay below this


def env_int(k, d):
    return int(os.environ.get(k, d))


# ------------------------------------------------------------------ clocks ----
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v == "Active":
                    reasons.add(name)
        load = [x for x in sm if x > 200]
        return {"sm_mhz": statistics.median(load) if load else (statistics.median(sm) if sm else None),
                "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------- workload ----
def build_box(group, n_total, t, seed):
    """Synthetic DistributionSharesBox (SURVEY.md 8d) made with the library's own dealer path
    (mpvss_distribute; collective and sharded when the group's context has a communicator: every rank
    receives the same box).  Returns flat boundary-encoded arrays in publickeys order."""
    from mpvss_rs_b200 import synth
    from mpvss_rs_b200.lib import buf, ptr
    c = group.codec
    eb, sb = c.eb, c.sb
    sks = synth.private_keys(seed, n_total, c.name, c.order, c.key_bound)
    coeffs = synth.coefficients(seed, t, c.order)
    ws = synth.witnesses(seed, n_total, c.key_bound)
    pks = group.fixed_base_exp(sks)
    pk_b = c.enc_elems(pks)
    comm, shares = buf(size=t * eb), buf(size=n_total * eb)
    chal, resp, u, x = buf(size=sb), buf(size=n_total * sb), buf(size=eb), buf(size=n_total * eb)
    secret = b"Hello MPVSS Example."
    group.ctx.check(group.ctx.lib.mpvss_distribute(
        group.ctx.h, n_total, t, ptr(buf(secret)), len(secret), ptr(buf(c.enc_scalars(coeffs))),
        ptr(buf(c.enc_scalars(ws))), ptr(buf(pk_b)), ptr(comm), ptr(shares), ptr(chal), ptr(resp), ptr(u), ptr(x)))
    return {"commitments": bytes(comm), "publickeys": pk_b, "shares": bytes(shares), "responses": bytes(resp),
            "challenge": bytes(chal), "x_dealer": bytes(x), "n": n_total, "t": t, "eb": eb, "sb": sb,
            "group": c.name, "U": int.from_bytes(bytes(u), "big")}


def other_phases(group, box, seed, reps=2):
    """The other four entry points of the path at the box's (n, t) -- distribute_secret, extract_secret_share x t,
    verify_share x t, reconstruct from the first t shares (SURVEY.md 8d asks for them beside the verify metric).
    Each figure is one C-ABI call with host buffers (copies inside); wall_ms by the host clock around the call,
    kernel_ms by CUDA events on the library's stream; one untimed call first.  Results are checked: the shares
    verify and the secret comes back."""
    from mpvss_rs_b200 import synth
    from mpvss_rs_b200.lib import buf, ptr
    c, lib, h = group.codec, group.ctx.lib, group.ctx.h
    n, t, eb, sb = box["n"], box["t"], c.eb, c.sb
    secret = b"Hello MPVSS Example."
    sks = buf(c.enc_scalars(synth.private_keys(seed, n, c.name, c.order, c.key_bound)[:t]))
    ws_all = synth.witnesses(seed, n, c.key_bound)
    ws, wt = buf(c.enc_scalars(ws_all)), buf(c.enc_scalars(ws_all[:t]))
    coeffs = buf(c.enc_scalars(synth.coefficients(seed, t, c.order)))
    pk, ys = buf(box["publickeys"]), buf(box["shares"][:t * eb])
    comm, shares, chal, resp, u = buf(size=t * eb), buf(size=n * eb), buf(size=sb), buf(size=n * sb), buf(size=eb)
    pko, so, co, ro = buf(size=t * eb), buf(size=t * eb), buf(size=t * sb), buf(size=t * sb)
    st, ok = (ctypes.c_int * t)(), (ctypes.c_int * t)()
    pos = (ctypes.c_int64 * t)(*range(1, t + 1))
    ub, sec = buf(box["U"].to_bytes(eb, "big")), buf(size=eb)
    calls = [
        ("distribute_secret", n, lambda: lib.mpvss_distribute(h, n, t, ptr(buf(secret)), len(secret), ptr(coeffs), ptr(ws), ptr(pk),
                                                             ptr(comm), ptr(shares), ptr(chal), ptr(resp), ptr(u), None)),
        ("extract_secret_share", t, lambda: lib.mpvss_extract_shares(h, t, ptr(sks), ptr(wt), ptr(ys), ptr(pko), ptr(so), ptr(co),
                                                                     ptr(ro), st)),
        ("verify_share", t, lambda: lib.mpvss_verify_shares(h, t, ptr(pko), ptr(so), ptr(ys), ptr(co), ptr(ro), ok)),
        ("reconstruct", t, lambda: lib.mpvss_reconstruct(h, t, pos, ptr(so), ptr(ub), ptr(sec), None)),
    ]
    out = {}
    for name, units, fn in calls:
        group.ctx.check(fn())
        wall, kern = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            group.ctx.check(fn())
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(group.ctx.last_kernel_ms)
        out[name] = {"units": units, "wall_ms": statistics.mean(wall), "kernel_ms": statistics.mean(kern),
                     "units_per_s": units / (statistics.mean(wall) * 1e-3)}
    assert bytes(shares) == box["shares"] and bytes(chal) == box["challenge"], "dealer is not deterministic"
    assert all(x == 0 for x in st) and all(x == 1 for x in ok), "extracted shares do not verify"
    assert bytes(sec).lstrip(b"\0") == secret, "reconstruct did not return the secret"
    out["note"] = (f"one C-ABI call each with host buffers at n={n}, t={t}: distribute over n participants; extract / "
                   "verify_share / reconstruct over the first t; outputs checked (shares verify, secret recovered)")
    return out


def participant_box(group, box):
    """The flat box as the reference-shaped DistributionSharesBox (tests)."""
    import mpvss_rs_b200 as m
    c, n = group.codec, box["n"]
    b = m.DistributionSharesBox()
    b.commitments = c.dec_elems(box["commitments"], box["t"])
    b.publickeys = c.dec_elems(box["publickeys"], n)
    ys, rs = c.dec_elems(box["shares"], n), c.dec_scalars(box["responses"], n)
    for i, pk in enumerate(b.publickeys):
        k = c.key(pk)
        b.positions[k], b.shares[k], b.responses[k] = i + 1, ys[i], rs[i]
    b.challenge = c.dec_scalar(box["challenge"])
    b.U = box["U"]
    return b


def reference_box(group_name, n_total, t, sample_idx, seed, threads):
    """A box for the CPU reference arm, built WITHOUT the GPU library: commitments with OpenSSL
    (oracle/cpu_baseline.c), the sampled participants' keys / shares / responses with OpenSSL and Python
    integers.  The transcript challenge would need all n_total participants; a pseudo-challenge of the same
    size stands in (the DLEQ relations a1 = g^w, a2 = y^w hold for any challenge and are asserted)."""
    from mpvss_rs_b200 import synth       # pure Python (SHA-256 counter mode), no library call
    from oracle import cpu_baseline as cb
    from oracle import pvss
    modp = group_name == "modp"
    order = RFC3526_2048 - 1 if modp else SECP_N
    bound = RFC3526_2048 if modp else SECP_N
    sks = synth.private_keys(seed, n_total, group_name, order, bound)
    coeffs = synth.coefficients(seed, t, order)
    ws = synth.witnesses(seed, n_total, bound)
    chal = int.from_bytes(hashlib.sha256(b"bench pseudo-challenge %d" % seed).digest(), "big") % \
        ((RFC3526_2048 - 1) // 2 if modp else SECP_N)
    ps = [pvss.poly_eval_mod(coeffs, i + 1, order) for i in sample_idx]
    rs = [(ws[i] - p * chal) % order for i, p in zip(sample_idx, ps)]
    if modp:
        q = RFC3526_2048
        comm = cb.modp_exp(q, 4, coeffs, threads)
        pks = cb.modp_exp(q, 2, [sks[i] for i in sample_idx], threads)
        ys = cb.modp_exp(q, pks, ps, threads)
        a1 = cb.modp_exp(q, 4, [ws[i] for i in sample_idx], threads)
        a2 = cb.modp_exp(q, pks, [ws[i] for i in sample_idx], threads)
        le = lambda v: int(v).to_bytes(256, "little")
        enc_e = enc_s = le
    else:
        comm = cb.secp_mul(None, coeffs)
        pks = cb.secp_mul(None, [sks[i] for i in sample_idx])
        ys = cb.secp_mul(pks, ps)
        a1 = cb.secp_mul(None, [ws[i] for i in sample_idx])
        a2 = cb.secp_mul(pks, [ws[i] for i in sample_idx])
        enc_e = bytes
        enc_s = lambda v: int(v).to_bytes(32, "big")
    eb, sb = (256, 256) if modp else (33, 32)
    rows = lambda vals, enc, w: {i: enc(v) for i, v in zip(sample_idx, vals)}
    return {"commitments": b"".join(enc_e(v) for v in comm), "pk_rows": rows(pks, enc_e, eb), "y_rows": rows(ys, enc_e, eb),
            "r_rows": rows(rs, enc_s, sb), "challenge": enc_s(chal), "n": n_total, "t": t, "eb": eb, "sb": sb,
            "group": group_name, "expect_a1": [enc_e(v) for v in a1], "expect_a2": [enc_e(v) for v in a2]}


def dleq_macs(n, rwin=512, cwin=64):
    """Algorithmic MACs of the two DLEQ commitment launches (DESIGN.md section 2)."""
    def win4(w):        # variable base, fixed 4-bit windows: 14 table products + to-Montgomery, 4 sqr + 1 mul per window
        return 4 * (w - 1) * SQR_MACS + (15 + (w - 1)) * MUL_MACS
    comb = ((rwin + 1) // 2 - 1) * MUL_MACS            # g^r from the 8-bit fixed-base table: one product per byte
    a1 = comb + win4(cwin) + 2 * MUL_MACS              # * X^c, leave Montgomery form
    a2 = win4(rwin) + win4(cwin) + 2 * MUL_MACS
    return n * (a1 + a2)


def measure_imad_peak():
    """Measured 32-bit integer multiply-add issue peak of this GPU (tools/imad_peak.cu)."""
    exe = os.path.join(ROOT, "tools", "imad_peak")
    try:
        if os.environ.get("MPVSS_SKIP_PEAK"):
            raise RuntimeError("skipped (profiling run)")
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout
        j = json.loads(out)
        lo = max(v["tera_per_s"] for k, v in j.items() if k.startswith("imad_lo_"))
        wide = max(v["tera_per_s"] for k, v in j.items() if k.startswith("imad_wide"))
        return lo, wide, "measured live (tools/imad_peak)"
    except Exception:
        for name in ("imad_peak_r02.json", "imad_peak_r01.json"):
            try:
                j = json.load(open(os.path.join(ROOT, "profiles", name)))
                lo = max(v["tera_per_s"] for k, v in j.items() if k.startswith("imad_lo_"))
                wide = max(v["tera_per_s"] for k, v in j.items() if k.startswith("imad_wide"))
                return lo, wide, f"profiles/{name} (measured on this pool)"
            except Exception:
                continue
        return 18.4, 7.7, "fallback constant (round-1 measurement)"


# ------------------------------------------------------------ CPU baseline ----
def cpu_reference_step(box, sample_idx, threads, schedule=0):
    """One bounded sample of the workload on the host cores: X_i, a1, a2 of the sampled participants
    with the reference's loop structure, then their framed SHA-256 transcript.  Accepts the GPU arm's flat
    box or reference_box().  Returns (seconds, X rows, a1 rows, a2 rows) as boundary bytes."""
    from oracle import cpu_baseline
    lib = cpu_baseline.load()
    s = len(sample_idx)
    t, eb, sb = box["t"], box["eb"], box["sb"]
    pos = (ctypes.c_int64 * s)(*[i + 1 for i in sample_idx])

    def row(key, w):
        sparse = {"publickeys": "pk_rows", "shares": "y_rows", "responses": "r_rows"}[key]
        if sparse in box:                                   # reference_box(): only the sampled rows exist
            return [box[sparse][i] for i in sample_idx]
        return [box[key][i * w:(i + 1) * w] for i in sample_idx]
    xo, a1o, a2o = (ctypes.create_string_buffer(eb * s) for _ in range(3))
    if box["group"] == "modp":
        be = lambda b: bytes(reversed(b))
        comm = b"".join(be(box["commitments"][j * 256:(j + 1) * 256]) for j in range(t))
        sel = lambda key: b"".join(be(r) for r in row(key, 256))
        pk, y, r, c = sel("publickeys"), sel("shares"), sel("responses"), be(box["challenge"])
        q = RFC3526_2048.to_bytes(256, "big")
        t0 = time.perf_counter()
        lib.cpu_modp_verify(q, comm, t, pos, pk, y, r, c, s, threads, schedule, xo, a1o, a2o)
        h = hashlib.sha256()       # dleq.rs:58-61, 87-99: len_u64_be || minimal big-endian bytes
        for i in range(s):
            for blob in (xo.raw, y, a1o.raw, a2o.raw):
                e = blob[i * 256:(i + 1) * 256].lstrip(b"\0") or b"\0"
                h.update(len(e).to_bytes(8, "big") + e)
        h.digest()
        dt = time.perf_counter() - t0
        dec = lambda o: [bytes(reversed(o.raw[i * 256:(i + 1) * 256])) for i in range(s)]
        return dt, dec(xo), dec(a1o), dec(a2o)
    if box["group"] == "secp256k1":
        pk, y, r = b"".join(row("publickeys", 33)), b"".join(row("shares", 33)), b"".join(row("responses", 32))
        t0 = time.perf_counter()
        lib.cpu_secp_verify(box["commitments"], t, pos, pk, y, r, box["challenge"], s, threads, schedule, xo, a1o, a2o)
        h = hashlib.sha256()
        for i in range(s):
            for blob in (xo.raw, y, a1o.raw, a2o.raw):
                h.update((33).to_bytes(8, "big") + blob[i * 33:(i + 1) * 33])
        h.digest()
        dt = time.perf_counter() - t0
        dec = lambda o: [o.raw[i * 33:(i + 1) * 33] for i in range(s)]
        return dt, dec(xo), dec(a1o), dec(a2o)
    raise ValueError("no CPU baseline for " + box["group"])


def spread_sample(n, s):
    return sorted({min(n - 1, (k * n) // s + (n // (2 * s))) for k in range(s)})


def reference_arm(args, n_total, t, config, cores):
    """--impl reference: the reference's CPU schedule on all host cores; never loads the GPU library."""
    sample = spread_sample(n_total, min(cores, n_total))
    box = reference_box(args.group, n_total, t, sample, args.seed, cores)
    _, _, a1, a2 = cpu_reference_step(box, sample, cores, schedule=1)   # correctness gate on the cheap schedule
    if a1 != box["expect_a1"] or a2 != box["expect_a2"]:
        raise SystemExit("CPU restatement: a1 != g^w or a2 != y^w on the synthetic box -- refusing to report")
    for _ in range(args.warmup):
        cpu_reference_step(box, sample[: max(1, len(sample) // 4)], cores)
    times = [cpu_reference_step(box, sample, cores)[0] for _ in range(args.steps)]
    per = statistics.mean(times)
    val = len(sample) / per
    return {"impl": "reference", "metric": METRICS[args.group], "value": val, "unit": "shares/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[args.group], "data": "synthetic", "config": config,
            "cpu_baseline": {"value": val, "unit": "shares/s", "cores": cores, "per_core": val / cores, "kind": "port",
                             "sample": f"{len(sample)} participants per step at positions spread over "
                                       f"1..{n_total}, full t={t}, reference schedule (t+4 exponentiations per "
                                       "share, participant.rs:423-447) + framed SHA-256 of their rows, on " +
                                       CPU_PROXY[args.group] + "; box synthesised with OpenSSL/Python, GPU library "
                                       "not loaded"},
            "e2e": {"value": val, "unit": "shares/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ----------------------------------------------------------------- GPU arm ----
class Runner:
    """One synthetic box on one group context (with or without a communicator); times resident steps and
    full calls."""

    def __init__(self, group, box, torch, dist, rank, world):
        self.g, self.box, self.torch, self.dist, self.rank, self.world = group, box, torch, dist, rank, world
        self.lib, self.h = group.ctx.lib, group.ctx.h
        pin = lambda b: torch.frombuffer(bytearray(b), dtype=torch.uint8).pin_memory()
        self.host = {k: pin(box[k]) for k in ("commitments", "publickeys", "shares", "responses", "challenge")}
        self.ok = ctypes.c_int(0)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        self.modp = box["group"] == "modp"
        self.check = True
        self.outputs = None     # see keep_outputs()

    def P(self, key):
        return ctypes.cast(self.host[key].data_ptr(), ctypes.POINTER(ctypes.c_uint8))

    def stage(self):
        b = self.box
        self.g.ctx.check(self.lib.mpvss_verify_distribution_stage(
            self.h, b["n"], b["t"], self.P("commitments"), None, self.P("publickeys"), self.P("shares"),
            self.P("responses"), self.P("challenge")))

    def run(self, x_out=None, digest=None, a1_out=None, a2_out=None):
        self.g.ctx.check(self.lib.mpvss_verify_distribution_run(self.h, ctypes.byref(self.ok), x_out, a1_out, a2_out,
                                                                digest))
        return self.ok.value, self.g.ctx.last_kernel_ms, self.g.ctx.last_phase_ms(2 if self.modp else 0)

    def keep_outputs(self):
        """make the last timed resident step receive every output of the call: the digest, and X_i / a1 / a2 on
        one GPU (the library returns no rows through a communicator)"""
        from mpvss_rs_b200.lib import buf
        rows = self.box["n"] * self.box["eb"]
        self.outputs = {k: (buf(size=rows) if self.world == 1 else None) for k in ("x", "a1", "a2")}
        self.outputs["digest"] = buf(size=32)

    def run_keep(self):
        from mpvss_rs_b200.lib import ptr
        o = self.outputs
        r = self.run(ptr(o["x"]), ptr(o["digest"]), ptr(o["a1"]), ptr(o["a2"]))
        o["verdict"] = r[0]
        return r

    def full(self):
        b = self.box
        self.g.ctx.check(self.lib.mpvss_verify_distribution(
            self.h, b["n"], b["t"], self.P("commitments"), None, self.P("publickeys"), self.P("shares"),
            self.P("responses"), self.P("challenge"), ctypes.byref(self.ok), None, None, None, None))
        return self.ok.value

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def maxr(self, x):
        if self.dist is None:
            return x
        tns = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(tns, op=self.dist.ReduceOp.MAX)
        return float(tns.item())

    def timed(self, fn, steps, warmup, last=None):
        """warmup + steps calls of fn (the final one `last` when given); returns the timed steps"""
        out = []
        for i in range(warmup + steps):
            self.flush.zero_()
            self.barrier()
            t0 = time.perf_counter()
            r = last() if last is not None and i == warmup + steps - 1 else fn()
            self.barrier()
            dt = self.maxr(time.perf_counter() - t0)
            if i >= warmup:
                out.append((dt, r))
        return out

    def measure(self, steps, warmup):
        """resident steps, then full calls; returns a dict of means (max over ranks per step)"""
        self.stage()
        res = self.timed(self.run, steps, warmup, self.run_keep if self.outputs is not None else None)
        assert not self.check or all(r[1][0] == 1 for r in res), "synthetic box did not verify"
        launches = self.g.ctx.last_kernel_launches * steps * self.world
        sq, ml = self.g.ctx.last_horner_products()
        e2e = self.timed(self.full, steps, warmup)
        assert not self.check or all(r[1] == 1 for r in e2e)
        return {"ms": statistics.mean(r[0] for r in res) * 1e3,
                "kernel_ms": statistics.mean(self.maxr(r[1][1]) for r in res),
                "horner_ms": statistics.mean(self.maxr(r[1][2]) for r in res),
                "e2e_ms": statistics.mean(r[0] for r in e2e) * 1e3, "launches": launches, "sqr": sq, "mul": ml}


def dump_outputs(path, runner, seed):
    """--dump-outputs: what the last timed resident step returned, one .npy per output.  verdict.npy (float64,
    1 = the box verifies); digest.npy (float32, the 32 bytes of the transcript's SHA-256); on one GPU x.npy,
    a1.npy and a2.npy (float32, [rows, element bytes], each row a participant's element in the ABI's boundary
    encoding, one byte per entry) and participant_index.npy (float64, the 0-based participant of each row).  When
    all rows would exceed DUMP_BYTES, the rows are a sample of participants drawn with the box's seed."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    o, eb = runner.outputs, runner.box["eb"]
    save = lambda name, a: np.save(os.path.join(path, name + ".npy"), a)
    save("verdict", np.array([o["verdict"]], dtype=np.float64))
    save("digest", np.frombuffer(bytes(o["digest"]), dtype=np.uint8).astype(np.float32))
    if o["x"] is None:
        return
    n = len(o["x"]) // eb
    fit = (DUMP_BYTES - (1 << 20)) // (3 * 4 * eb + 8)
    idx = np.arange(n) if n <= fit else np.sort(np.random.default_rng(seed).choice(n, fit, replace=False))
    save("participant_index", idx.astype(np.float64))
    for k in ("x", "a1", "a2"):
        save(k, np.frombuffer(bytes(o[k]), dtype=np.uint8).reshape(n, eb)[idx].astype(np.float32))


# dram__bytes_read.sum + dram__bytes_write.sum of the dominant launch at n = 4096, t = 2731 on one GPU, from the
# ncu --set full captures summarised under profiles/ (horner_r02_ncu.txt, ec_horner_*_r02_ncu.txt)
# (values of the final round-2 captures; DRAM traffic of these launches moves by a few hundred KB from run to run)
NCU_TRAFFIC = {"modp": 1161472 + 0, "secp256k1": 307712 + 2316544, "ristretto255": 259584 + 26141696}


def modp_roofline(m, n_local, imad_lo, imad_wide, peak_src, traffic=None):
    hm = m["sqr"] * SQR_MACS + m["mul"] * MUL_MACS
    achieved = 2.0 * hm / (m["horner_ms"] * 1e-3) / 1e12        # TIMAD/s, 1 MAC = 2 IMAD issues (SURVEY 8d)
    total = hm + dleq_macs(n_local)
    step = 2.0 * total / (m["kernel_ms"] * 1e-3) / 1e12
    return {
        "bound": "imad", "kernel": "modp::horner_kernel (X_i multi-exponentiation, addition chains)",
        "achieved": achieved, "peak": imad_lo, "unit": "TIMAD/s", "frac": achieved / imad_lo if imad_lo else None,
        "peak_source": peak_src + "; 32-bit IMAD issue rate, 1 MAC (32x32->64) = 2 IMAD",
        "achieved_tmac_per_s": achieved / 2, "wide_mac_peak_tmac_per_s": imad_wide,
        "frac_of_wide_mac_peak": (achieved / 2) / imad_wide if imad_wide else None,
        "algorithmic_macs_per_launch": hm, "modsqr_per_launch": m["sqr"], "modmul_per_launch": m["mul"],
        "kernel_ms": m["horner_ms"], "share_of_step_macs": hm / total, "traffic": traffic,
        "traffic_note": "dram bytes read+written by the Horner launch, ncu --set full (profiles/)",
        "note": "kernel_ms = CUDA events around the Horner launch on the library stream (max over ranks); "
                "algorithmic MACs = products the executed addition chains contain (library counter, rank 0's "
                "participants), squarings at 6240 and multiplications at 8256 MACs; padding products excluded",
        "whole_step": {"achieved": step, "frac": step / imad_lo if imad_lo else None, "algorithmic_macs": total,
                       "kernel_ms": m["kernel_ms"],
                       "what": "all kernels of the step (Horner + both DLEQ launches; g^r from the fixed-base table)"}}


def ec_roofline(m, group_name, imad_lo, imad_wide, peak_src, traffic=None):
    macs = m["sqr"] * EC_SQR_MACS[group_name] + m["mul"] * EC_MUL_MACS[group_name]
    achieved = 2.0 * macs / (m["horner_ms"] * 1e-3) / 1e12
    return {"bound": "imad", "kernel": f"ec::horner_kernel<{group_name}> (chunked X_i Horner incl. chunk scaling)",
            "achieved": achieved, "peak": imad_lo, "unit": "TIMAD/s", "frac": achieved / imad_lo if imad_lo else None,
            "peak_source": peak_src, "frac_of_wide_mac_peak": (achieved / 2) / imad_wide if imad_wide else None,
            "algorithmic_macs_per_launch": macs, "field_sqr_per_launch": m["sqr"], "field_mul_per_launch": m["mul"],
            "kernel_ms": m["horner_ms"], "traffic": traffic,
            "traffic_note": "dram bytes read+written by the Horner launch, ncu --set full (profiles/)",
            "note": "field products executed by the Horner launches (library counter) x 72 / 44 MACs "
                    "(8x8 limb product or 36 distinct squaring products + 8 for the special-form fold)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # long spellings too: under torchrun, `--n` / `--t` collide with abbreviations of its own options
    ap.add_argument("--n", "--participants-per-gpu", dest="n", type=int, default=4096, help="participants per GPU")
    ap.add_argument("--t", "--threshold", dest="t", type=int, default=0, help="threshold (default ceil(2n/3))")
    ap.add_argument("--tpi", type=int, default=0, help="override lanes per 2048-bit value")
    ap.add_argument("--seed", type=int, default=SEED)
    ap.add_argument("--group", default="modp", choices=["modp", "secp256k1", "ristretto255"])
    ap.add_argument("--ec-threads", type=int, default=0)
    ap.add_argument("--overlap", type=int, default=-1, help="override modp_overlap (0, 2 or 3)")
    ap.add_argument("--wpc", type=int, default=0, help="override warps per CTA of the MODP Horner launch (1..4)")
    ap.add_argument("--chunks", type=int, default=0, help="override chunks per position of the MODP Horner launch")
    ap.add_argument("--subset", type=int, default=0, help="kernel experiments: verify only the first M participants of "
                    "the box (the verdict is then false by construction and not asserted; not a reportable number)")
    ap.add_argument("--device-hash", action="store_true", help="experiment: whole-box transcript hashed by one device "
                    "thread (device_hash tunable) instead of the host's SHA-NI")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--c5", action="store_true", help="also time BASELINE config 5 (n=65536 t=43691) [default at 8 GPUs]")
    ap.add_argument("--no-c5", action="store_true", help="skip config 5 at 8 GPUs (short re-runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    n = args.n
    t = args.t or -(-2 * n // 3)
    n_total = n * world
    cores = os.cpu_count() or 1
    config = {"workload": f"{args.group} verify_distribution_shares n={n} per GPU (box of {n_total}), t={t}",
              "group": args.group, "n_per_gpu": n, "n_total": n_total, "t": t,
              "x_schedule": "Horner in the exponent; acc^i by power-tree addition chains (DESIGN.md section 2)",
              "residency": "value: box resident in HBM, staging excluded; e2e: host buffers, staging included",
              "l2": "flushed between timed steps (256 MiB write)",
              "sharding": f"participants round-robin over {world} rank(s) inside the library, one ncclAllGather of "
                          "the framed transcript rows per step, every rank hashes"}

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs dumps the GPU path (--impl ours)")
        if rank == 0:
            print(json.dumps(reference_arm(args, n_total, t, config, cores)))
        return 0

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: mpvss_rs_b200 has no CPU path")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import mpvss_rs_b200 as m
    from mpvss_rs_b200.lib import buf, ptr

    def make_group(name, joined):
        g = m.Group(name, device=local)
        if args.tpi and name == "modp":
            g.ctx.set_int("modp_tpi", args.tpi)
        if args.ec_threads and name != "modp":
            g.ctx.set_int("ec_threads", args.ec_threads)
        if args.overlap >= 0 and name == "modp":
            g.ctx.set_int("modp_overlap", args.overlap)
        if args.wpc and name == "modp":
            g.ctx.set_int("modp_wpc", args.wpc)
        if args.chunks and name == "modp":
            g.ctx.set_int("modp_chunks", args.chunks)
        if args.device_hash:
            g.ctx.set_int("device_hash", 1)
        if joined and world > 1:
            g.join(rank, world, dist)           # NCCL communicator inside the library
        return g

    group = make_group(args.group, True)
    eb = group.codec.eb
    box = build_box(group, n_total, t, args.seed)
    if args.subset:      # kernel experiment: the first M participants only (transcript no longer matches)
        box = dict(box, n=args.subset)
        runner = Runner(group, box, torch, dist, rank, world)
        runner.check = False
        if args.dump_outputs:
            runner.keep_outputs()
        m_ = runner.measure(args.steps, args.warmup)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, runner, args.seed)
        if rank == 0:
            print(json.dumps({"experiment": f"first {args.subset} participants of a box of {n_total}, t={t}", "ms": m_["ms"],
                              "kernel_ms": m_["kernel_ms"], "horner_ms": m_["horner_ms"], "chunks": args.chunks}))
        return 0
    runner = Runner(group, box, torch, dist, rank, world)

    # correctness gates before timing: the box verifies; the verifier's X equals the dealer's g^P(i); at N>1 the
    # sharded transcript digest equals the single-GPU digest of the same box
    runner.stage()
    dig = buf(size=32)
    if world == 1:
        x_chk = buf(size=n * eb)
        okv, _, _ = runner.run(ptr(x_chk), ptr(dig))
        if okv != 1:
            raise SystemExit("verification of the synthetic box failed -- refusing to report a number")
        if bytes(x_chk) != box["x_dealer"]:
            raise SystemExit("verifier X_i differs from dealer X_i -- refusing to report a number")
    else:
        okv, _, _ = runner.run(None, ptr(dig))
        if okv != 1:
            raise SystemExit("sharded verification of the synthetic box failed -- refusing to report a number")
        if rank == 0 and n_total <= 16384:
            solo = make_group(args.group, False)
            r1 = Runner(solo, box, torch, None, 0, 1)
            r1.stage()
            d1 = buf(size=32)
            ok1, _, _ = r1.run(None, ptr(d1))
            if ok1 != 1 or bytes(d1) != bytes(dig):
                raise SystemExit("sharded transcript digest != single-GPU digest -- refusing to report a number")
            config["digest_check"] = "sharded transcript digest == single-GPU digest of the same box (rank 0)"
            solo.ctx.close()
        runner.barrier()

    imad_lo, imad_wide, peak_src = measure_imad_peak() if rank == 0 else (0, 0, "")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if args.dump_outputs:
        runner.keep_outputs()
    meas = runner.measure(args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, runner, args.seed)

    also = {}
    if world > 1 and not args.no_also:
        # strong scaling: the metric's box (n = 4096 in total) split over the N GPUs
        sg = make_group(args.group, True)
        sbox = build_box(sg, n, t, args.seed)
        sm = Runner(sg, sbox, torch, dist, rank, world).measure(args.steps, args.warmup)
        also["strong"] = {"scaling": "strong", "n_total": n, "t": t, "value": n / (sm["ms"] * 1e-3), "unit": "shares/s",
                          "ms_per_step": sm["ms"], "kernel_ms_per_step": sm["kernel_ms"],
                          "e2e": {"value": n / (sm["e2e_ms"] * 1e-3), "unit": "shares/s"},
                          "note": "one box of n participants in total, sharded over all ranks"}
        sg.ctx.close()
    if (args.c5 or world == 8) and not args.no_c5 and args.group == "modp" and not args.no_also:
        # BASELINE config 5: ModpGroup n = 65536, t = 43691, distribute + verify sharded over the ranks
        cg = make_group("modp", True)
        t0 = time.perf_counter()
        cbox = build_box(cg, 65536, 43691, args.seed)
        dist_s = runner.maxr(time.perf_counter() - t0)
        cm = Runner(cg, cbox, torch, dist, rank, world).measure(2, 1)
        c5 = {"workload": "modp n=65536 t=43691 (BASELINE config 5)", "n_gpus": world, "steps": 2, "warmup": 1,
              "value": 65536 / (cm["ms"] * 1e-3), "unit": "shares/s", "ms_per_step": cm["ms"],
              "kernel_ms_per_step": cm["kernel_ms"], "e2e": {"value": 65536 / (cm["e2e_ms"] * 1e-3), "unit": "shares/s"},
              "distribute_wall_s": dist_s,
              "distribute_note": "synthetic keys + mpvss_distribute (sharded dealer) incl. Python marshalling"}
        if rank == 0:
            c5["roofline"] = modp_roofline(cm, 65536 // world, imad_lo, imad_wide, peak_src)
        also["c5"] = c5
        cg.ctx.close()
    if rank != 0:
        dist.destroy_process_group()
        return 0

    value = n_total / (meas["ms"] * 1e-3)
    sb = group.codec.sb
    n_loc = n_total // world
    h2d = world * (t * eb + sb) + n_total * (2 * eb + sb)
    d2h = world * n_total * 4 * (8 + eb)
    line = {
        "metric": METRICS[args.group], "value": value, "unit": "shares/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": meas["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE[args.group], "data": "synthetic", "config": config,
        "timing": "per step: cuda-synchronize + barrier bracketed wall clock (kernels + all-gather + chunked D2H "
                  "overlapped with the host SHA-256), box resident in HBM, max over ranks; kernel_ms / roofline "
                  "from CUDA events on the library's stream",
        "kernel_ms_per_step": meas["kernel_ms"], "host_tail_ms": meas["ms"] - meas["kernel_ms"],
        "gpu_launches": meas["launches"],
        "clocks": clocks,
        "e2e": {"value": n_total / (meas["e2e_ms"] * 1e-3), "unit": "shares/s", "ms_per_step": meas["e2e_ms"],
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "call": "mpvss_verify_distribution (pinned host buffers in, verdict out; collective at N>1); the "
                        "addition-chain plan of positions 1..n is cached in the context, every box input is copied "
                        "each step"},
    }
    traffic = NCU_TRAFFIC[args.group] if (world == 1 and n == 4096 and t == 2731) else None
    if args.group == "modp":
        line["roofline"] = modp_roofline(meas, n_loc, imad_lo, imad_wide, peak_src, traffic)
    else:
        line["roofline"] = ec_roofline(meas, args.group, imad_lo, imad_wide, peak_src, traffic)
        line["phase_ms"] = {"x_horner": meas["horner_ms"], "dleq": meas["kernel_ms"] - meas["horner_ms"]}
    if not args.no_cpu_baseline and world == 1 and args.group in CPU_PROXY:
        sample = spread_sample(n_total, min(cores, n_total))
        dt, xs, _, _ = cpu_reference_step(box, sample, cores)
        for i, x in zip(sample, xs):       # the CPU restatement and the GPU agree on X_i
            assert x == box["x_dealer"][i * eb:(i + 1) * eb], "CPU baseline X_i != GPU X_i"
        dt_h = cpu_reference_step(box, sample, cores, schedule=1)[0]
        line["cpu_baseline"] = {
            "value": len(sample) / dt, "unit": "shares/s", "cores": cores, "per_core": len(sample) / dt / cores,
            "kind": "port",
            "sample": f"{len(sample)} participants (positions spread over 1..{n_total}), full t={t}, reference "
                      "schedule (t+4 full exponentiations per share) + framed SHA-256 of their rows, on " +
                      CPU_PROXY[args.group] + ", one participant per thread",
            "same_algorithm_value": len(sample) / dt_h,
            "same_algorithm_note": "CPU running the GPU's Horner schedule (baseline B, BASELINE.md section 3)"}
    if world == 1 and not args.no_also:
        also["phases"] = other_phases(group, box, args.seed)
    if args.group == "modp" and world == 1 and not args.no_also:
        # the metric names MODP + secp256k1: the same step for Secp256k1Group, reported alongside
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--group", "secp256k1", "--steps",
                                  str(args.steps), "--warmup", str(args.warmup), "--n", str(n), "--t", str(t)] +
                                 (["--no-cpu-baseline"] if args.no_cpu_baseline else []),
                                 capture_output=True, text=True, timeout=900)
            sec = json.loads(out.stdout.strip().splitlines()[-1])
            also["secp256k1"] = {k: sec.get(k) for k in ("metric", "value", "unit", "ms_per_step", "kernel_ms_per_step",
                                                        "e2e", "roofline", "cpu_baseline", "phase_ms", "gpu_launches")}
            also["secp256k1"]["phases"] = (sec.get("also") or {}).get("phases")
        except Exception as ex:  # the primary line stands on its own
            also["secp256k1"] = {"error": str(ex)[:200]}
    if also:
        line["also"] = also
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
