"""Host-side mirror of the reference's `Participant<G>` / `DistributionSharesBox<G>` /
`ShareBox<G>` API (src/participant.rs, src/sharebox.rs) on top of the C ABI.

Same names, argument meaning and error behaviour as the reference so that parity
tests read like the reference's own tests; every group operation goes through
libmpvss_b200.so (CUDA).  The only additions are the randomness-injection
arguments (`coeffs`, `witnesses`, `private_key`) -- the reference draws those from
`thread_rng` internally (polynomial.rs:34-47, participant.rs:223, 139-146) -- and
the batch forms `distribute_secrets` / `extract_secret_shares` / `verify_shares` /
`verify_distributions` / `reconstruct_secrets`.

Value representation at this level: MODP elements and all scalars are Python
ints (the reference uses BigInt); secp256k1 / ristretto255 elements are their
canonical encodings (33 / 32 bytes), which is also what keys the reference's
HashMaps (sharebox.rs:75-86).
"""
from __future__ import annotations

import ctypes
import secrets
from dataclasses import dataclass, field

from . import lib as _lib
from .lib import Context, buf, ptr

RFC3526_2048 = int(
    "ffffffffffffffffc90fdaa22168c234c4c6628b80dc1cd129024e088a67cc74020bbea63b139b22514a08798e3404dd"
    "ef9519b3cd3a431b302b0a6df25f14374fe1356d6d51c245e485b576625e7ec6f44c42e9a637ed6b0bff5cb6f406b7ed"
    "ee386bfb5a899fa5ae9f24117c4b1fe649286651ece45b3dc2007cb8a163bf0598da48361c55d39a69163fa8fd24cf5f"
    "83655d23dca3ad961c62f356208552bb9ed529077096966d670c354e4abc9804f1746c08ca18217c32905e462e36ce3b"
    "e39e772c180e86039b2783a2ec07a28fb5c55df06f4c52c9de2bcbf6955817183995497cea956ae515d2261898fa0510"
    "15728e5a8aacaa68ffffffffffffffff", 16)
SECP_N = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
ED_L = 2**252 + 27742317777372353535851937790883648493


class _Codec:
    """Fixed-width boundary encodings (include/mpvss_b200.h) per group."""

    def __init__(self, name):
        self.name = name
        if name == "modp":
            self.eb, self.sb = 256, 256
            self.order = RFC3526_2048 - 1          # modp.rs:101-103
            self.key_bound = RFC3526_2048          # modp.rs:165-168
        elif name == "secp256k1":
            self.eb, self.sb = 33, 32
            self.order = self.key_bound = SECP_N
        elif name == "ristretto255":
            self.eb, self.sb = 32, 32
            self.order = self.key_bound = ED_L
        else:
            raise ValueError(name)

    def enc_elem(self, e):
        return int(e).to_bytes(256, "little") if self.name == "modp" else bytes(e)

    def dec_elem(self, b):
        return int.from_bytes(b, "little") if self.name == "modp" else bytes(b)

    def enc_scalar(self, s):
        if self.name == "modp":
            return int(s).to_bytes(256, "little")
        if self.name == "secp256k1":
            return (int(s) % SECP_N).to_bytes(32, "big")
        return (int(s) % ED_L).to_bytes(32, "little")

    def dec_scalar(self, b):
        return int.from_bytes(b, "big" if self.name == "secp256k1" else "little")

    def key(self, e):
        """Group::element_to_bytes -- the HashMap key (modp.rs:150-152: minimal big-endian)."""
        if self.name == "modp":
            e = int(e)
            return e.to_bytes(max(1, (e.bit_length() + 7) // 8), "big")
        return bytes(e)

    def enc_elems(self, es):
        return b"".join(self.enc_elem(e) for e in es)

    def enc_scalars(self, ss):
        return b"".join(self.enc_scalar(s) for s in ss)

    def dec_elems(self, b, n):
        b = bytes(b)
        return [self.dec_elem(b[i * self.eb:(i + 1) * self.eb]) for i in range(n)]

    def dec_scalars(self, b, n):
        b = bytes(b)
        return [self.dec_scalar(b[i * self.sb:(i + 1) * self.sb]) for i in range(n)]


@dataclass
class DistributionSharesBox:
    """sharebox.rs:75-86."""
    commitments: list = field(default_factory=list)
    positions: dict = field(default_factory=dict)
    shares: dict = field(default_factory=dict)
    publickeys: list = field(default_factory=list)
    challenge: int = 0
    responses: dict = field(default_factory=dict)
    U: int = 0


@dataclass
class ShareBox:
    """sharebox.rs:22-27."""
    publickey: object = None
    share: object = None
    challenge: int = 0
    response: int = 0


class Group:
    """A group handle = one CUDA context (mirrors `ModpGroup::new()` etc. returning Arc<G>)."""

    def __init__(self, name="modp", device=0):
        self.name = name
        self.codec = _Codec(name)
        self.ctx = Context(name, device)

    # -- batch forms of `trait Group` (src/group.rs:24-124) --
    def batch_exp(self, bases, scalars):
        c, n = self.codec, len(scalars)
        shared = not isinstance(bases, (list, tuple))
        b = buf(c.enc_elem(bases) if shared else c.enc_elems(bases))
        s = buf(c.enc_scalars(scalars))
        out = buf(size=n * c.eb)
        self.ctx.check(self.ctx.lib.mpvss_batch_exp(self.ctx.h, ptr(b), 0 if shared else c.eb, ptr(s), n, ptr(out)))
        return c.dec_elems(out, n)

    def fixed_base_exp(self, scalars, generator=_lib.GEN_MAIN):
        c, n = self.codec, len(scalars)
        s = buf(c.enc_scalars(scalars))
        out = buf(size=n * c.eb)
        self.ctx.check(self.ctx.lib.mpvss_fixed_base_exp(self.ctx.h, generator, ptr(s), n, ptr(out)))
        return c.dec_elems(out, n)

    def batch_mul(self, a, b):
        c, n = self.codec, len(a)
        out = buf(size=n * c.eb)
        self.ctx.check(self.ctx.lib.mpvss_batch_mul(self.ctx.h, ptr(buf(c.enc_elems(a))), ptr(buf(c.enc_elems(b))),
                                                    n, ptr(out)))
        return c.dec_elems(out, n)

    def poly_eval_exp(self, commitments, positions):
        c, n = self.codec, len(positions)
        pos = (ctypes.c_int64 * n)(*positions)
        out = buf(size=n * c.eb)
        self.ctx.check(self.ctx.lib.mpvss_poly_eval_exp(self.ctx.h, ptr(buf(c.enc_elems(commitments))),
                                                        len(commitments), pos, n, ptr(out)))
        return c.dec_elems(out, n)

    def scalar_poly_eval(self, coeffs, positions):
        """Polynomial::get_value(i) % order for every position (polynomial.rs:50-58, participant.rs:202)."""
        c, n = self.codec, len(positions)
        out = buf(size=n * c.sb)
        self.ctx.check(self.ctx.lib.mpvss_scalar_poly_eval(self.ctx.h, ptr(buf(c.enc_scalars(coeffs))), len(coeffs),
                                                           (ctypes.c_int64 * n)(*positions), n, ptr(out)))
        return c.dec_scalars(out, n)

    def join(self, rank, world, dist=None):
        """Make this group's context one rank of a multi-GPU communicator (sharding.join): afterwards
        Participant.distribute_secret / verify_distribution_shares on it are collective calls."""
        from .sharding import join
        join(self.ctx, rank, world, dist)

    def dleq_verify_commit(self, g1, h1s, g2s, h2s, rs, cs):
        c, n = self.codec, len(rs)
        shared = not isinstance(cs, (list, tuple))
        cb = buf(c.enc_scalar(cs) if shared else c.enc_scalars(cs))
        a1, a2 = buf(size=n * c.eb), buf(size=n * c.eb)
        self.ctx.check(self.ctx.lib.mpvss_dleq_verify_commit(
            self.ctx.h, ptr(buf(c.enc_elem(g1))), ptr(buf(c.enc_elems(h1s))), ptr(buf(c.enc_elems(g2s))),
            ptr(buf(c.enc_elems(h2s))), ptr(buf(c.enc_scalars(rs))), ptr(cb), 0 if shared else c.sb, n,
            ptr(a1), ptr(a2)))
        return c.dec_elems(a1, n), c.dec_elems(a2, n)

    def dleq_prove_commit(self, g1, g2s, ws):
        c, n = self.codec, len(ws)
        a1, a2 = buf(size=n * c.eb), buf(size=n * c.eb)
        self.ctx.check(self.ctx.lib.mpvss_dleq_prove_commit(
            self.ctx.h, ptr(buf(c.enc_elem(g1))), ptr(buf(c.enc_elems(g2s))), ptr(buf(c.enc_scalars(ws))), n,
            ptr(a1), ptr(a2)))
        return c.dec_elems(a1, n), c.dec_elems(a2, n)

    def multi_exp(self, bases, scalars):
        c, n = self.codec, len(scalars)
        out = buf(size=c.eb)
        self.ctx.check(self.ctx.lib.mpvss_multi_exp(self.ctx.h, ptr(buf(c.enc_elems(bases))),
                                                    ptr(buf(c.enc_scalars(scalars))), n, ptr(out)))
        return c.dec_elem(bytes(out))

    def generate_public_key(self, private_key):
        """Group::generate_public_key (modp.rs:176-178)."""
        return self.fixed_base_exp([private_key])[0]

    def generate_private_key(self):
        """Group::generate_private_key (modp.rs:162-174 / secp256k1.rs:158-166)."""
        c = self.codec
        while True:
            k = secrets.randbelow(c.key_bound)
            if c.name == "modp":
                if k % 2 == 1 and k % ((RFC3526_2048 - 1) // 2) != 0:
                    return k
            elif k != 0:
                return k


class Participant:
    """src/participant.rs:64-147 (generic part) and the per-group entry points."""

    def __init__(self, group: Group):
        self.group = group
        self.privatekey = 0
        self.publickey = None

    def initialize(self, private_key=None):
        """participant.rs:139-146; `private_key` injects what the reference draws at random."""
        self.privatekey = self.group.generate_private_key() if private_key is None else private_key
        self.publickey = self.group.generate_public_key(self.privatekey)

    # -- distribute_secret: participant.rs:160-286 / 1094-1274 / 1573-1717 --
    def _deal_inputs(self, secret, publickeys, threshold, coeffs, witnesses):
        """the host checks and the randomness of one dealing: (secret bytes, coefficients, witnesses)"""
        g, c = self.group, self.group.codec
        n = len(publickeys)
        assert threshold <= n                                   # participant.rs:166
        if coeffs is None:                                      # Polynomial::init, polynomial.rs:34-47
            coeffs = [secrets.randbelow(c.order) for _ in range(threshold)]
        if witnesses is None:                                   # participant.rs:223
            witnesses = [g.generate_private_key() for _ in range(n)]
        assert len(coeffs) == threshold and len(witnesses) == n
        return secret.to_bytes(max(1, (secret.bit_length() + 7) // 8), "big"), coeffs, witnesses

    def _box(self, publickeys, comm, shares, chal, resp, u):
        """DistributionSharesBox from one box's output rows"""
        c = self.group.codec
        n = len(publickeys)
        box = DistributionSharesBox()
        box.commitments = c.dec_elems(comm, len(comm) // c.eb)
        ys, rs = c.dec_elems(shares, n), c.dec_scalars(resp, n)
        for i, pk in enumerate(publickeys):
            k = c.key(pk)
            box.positions[k] = i + 1
            box.shares[k] = ys[i]
            box.responses[k] = rs[i]
        box.publickeys = list(publickeys)
        box.challenge = c.dec_scalar(bytes(chal))
        box.U = int.from_bytes(bytes(u), "big")
        return box

    def distribute_secret(self, secret: int, publickeys, threshold: int, coeffs=None, witnesses=None):
        g, c = self.group, self.group.codec
        n = len(publickeys)
        sbytes, coeffs, witnesses = self._deal_inputs(secret, publickeys, threshold, coeffs, witnesses)
        comm, shares = buf(size=threshold * c.eb), buf(size=n * c.eb)
        chal, resp, u = buf(size=c.sb), buf(size=n * c.sb), buf(size=c.eb)
        g.ctx.check(g.ctx.lib.mpvss_distribute(
            g.ctx.h, n, threshold, ptr(buf(sbytes)), len(sbytes), ptr(buf(c.enc_scalars(coeffs))),
            ptr(buf(c.enc_scalars(witnesses))), ptr(buf(c.enc_elems(publickeys))), ptr(comm), ptr(shares),
            ptr(chal), ptr(resp), ptr(u), None))
        return self._box(publickeys, bytes(comm), bytes(shares), bytes(chal), bytes(resp), bytes(u))

    def distribute_secrets(self, jobs) -> list:
        """Batch form of distribute_secret: one DistributionSharesBox per (secret, publickeys, threshold[, coeffs[,
        witnesses]]) job, all jobs in one library call (mpvss_distribute_secrets).  A job whose box the library
        rejects (where distribute_secret would raise) is None without disturbing the others."""
        g, c = self.group, self.group.codec
        if not jobs:
            return []
        deals = []
        for job in jobs:
            secret, publickeys, threshold, coeffs, witnesses = (tuple(job) + (None, None))[:5]
            sbytes, coeffs, witnesses = self._deal_inputs(secret, publickeys, threshold, coeffs, witnesses)
            if len(sbytes) > c.eb:                              # what mpvss_distribute rejects for this secret
                raise _lib.MpvssError(_lib.ERR_ARG, "distribute_secrets: a secret is longer than one element")
            deals.append((sbytes.rjust(c.eb, b"\0"), list(publickeys), threshold, coeffs, witnesses))
        m = len(deals)
        ns, ts = [len(d[1]) for d in deals], [d[2] for d in deals]
        N, T = sum(ns), sum(ts)
        comm, shares, resp = buf(size=T * c.eb), buf(size=N * c.eb), buf(size=N * c.sb)
        chal, u, st = buf(size=m * c.sb), buf(size=m * c.eb), (ctypes.c_int * m)()
        g.ctx.check(g.ctx.lib.mpvss_distribute_secrets(
            g.ctx.h, m, (ctypes.c_size_t * m)(*ns), (ctypes.c_size_t * m)(*ts), ptr(buf(b"".join(d[0] for d in deals))),
            ptr(buf(b"".join(c.enc_scalars(d[3]) for d in deals))),
            ptr(buf(b"".join(c.enc_scalars(d[4]) for d in deals))),
            ptr(buf(b"".join(c.enc_elems(d[1]) for d in deals))), ptr(comm), ptr(shares), ptr(chal), ptr(resp), ptr(u),
            None, st))
        comm, shares, resp, chal, u = bytes(comm), bytes(shares), bytes(resp), bytes(chal), bytes(u)
        out, n0, t0 = [], 0, 0
        for b, (_, publickeys, threshold, _, _) in enumerate(deals):
            n = len(publickeys)
            out.append(None if st[b] != _lib.OK else self._box(
                publickeys, comm[t0 * c.eb:(t0 + threshold) * c.eb], shares[n0 * c.eb:(n0 + n) * c.eb],
                chal[b * c.sb:(b + 1) * c.sb], resp[n0 * c.sb:(n0 + n) * c.sb], u[b * c.eb:(b + 1) * c.eb]))
            n0, t0 = n0 + n, t0 + threshold
        return out

    # -- verify_distribution_shares: participant.rs:399-455 / 1384-1442 / 1827-1885 --
    def _flatten(self, box):
        c = self.group.codec
        pos, ys, rs = [], [], []
        for pk in box.publickeys:
            k = c.key(pk)
            p, r, y = box.positions.get(k), box.responses.get(k), box.shares.get(k)
            if p is None or r is None or y is None:             # participant.rs:415-420
                return None
            pos.append(p)
            ys.append(y)
            rs.append(r)
        return pos, ys, rs

    def verify_distribution_shares(self, box, trace=None) -> bool:
        g, c = self.group, self.group.codec
        flat = self._flatten(box)
        if flat is None:
            return False
        pos, ys, rs = flat
        n, t = len(pos), len(box.commitments)
        ok = ctypes.c_int(0)
        want = trace is not None and g.ctx.comm_size <= 1   # per-share values are not gathered across ranks
        x, a1, a2 = (buf(size=n * c.eb) if want else None for _ in range(3))
        dig = buf(size=32)
        g.ctx.check(g.ctx.lib.mpvss_verify_distribution(
            g.ctx.h, n, t, ptr(buf(c.enc_elems(box.commitments))), (ctypes.c_int64 * n)(*pos),
            ptr(buf(c.enc_elems(box.publickeys))), ptr(buf(c.enc_elems(ys))), ptr(buf(c.enc_scalars(rs))),
            ptr(buf(c.enc_scalar(box.challenge))), ctypes.byref(ok), ptr(x), ptr(a1), ptr(a2), ptr(dig)))
        if want:
            trace.update(X=c.dec_elems(x, n), a1=c.dec_elems(a1, n), a2=c.dec_elems(a2, n))
        if trace is not None:
            trace["digest"] = bytes(dig)
        return bool(ok.value)

    def verify_distributions(self, boxes, traces=None) -> list:
        """Batch form of verify_distribution_shares: one verdict per box, all boxes in one library call
        (mpvss_verify_distributions).  traces[b]["digest"] receives box b's transcript digest."""
        g, c = self.group, self.group.codec
        res = [False] * len(boxes)
        live, flats = [], []
        for b, box in enumerate(boxes):
            flat = self._flatten(box)
            if flat is not None:                                # participant.rs:415-420
                live.append(b)
                flats.append(flat)
        if not live:
            return res
        m = len(live)
        ns = [len(f[0]) for f in flats]
        ts = [len(boxes[b].commitments) for b in live]
        pos = [p for f in flats for p in f[0]]
        ok, dig = (ctypes.c_int * m)(), buf(size=32 * m)
        g.ctx.check(g.ctx.lib.mpvss_verify_distributions(
            g.ctx.h, m, (ctypes.c_size_t * m)(*ns), (ctypes.c_size_t * m)(*ts),
            ptr(buf(b"".join(c.enc_elems(boxes[b].commitments) for b in live))), (ctypes.c_int64 * len(pos))(*pos),
            ptr(buf(b"".join(c.enc_elems(boxes[b].publickeys) for b in live))),
            ptr(buf(b"".join(c.enc_elems(f[1]) for f in flats))), ptr(buf(b"".join(c.enc_scalars(f[2]) for f in flats))),
            ptr(buf(b"".join(c.enc_scalar(boxes[b].challenge) for b in live))), ok, ptr(dig)))
        for j, b in enumerate(live):
            res[b] = bool(ok[j])
            if traces is not None:
                traces[b]["digest"] = bytes(dig)[32 * j:32 * j + 32]
        return res

    # -- extract_secret_share: participant.rs:294-353 / 1282-1338 / 1725-1781 --
    def extract_secret_shares(self, box, private_keys, ws):
        """Batch form: one ShareBox (or None) per (private_key, w)."""
        g, c = self.group, self.group.codec
        n = len(private_keys)
        pks = g.fixed_base_exp(private_keys)                    # participant.rs:306
        ys, live = [], []
        for i, pk in enumerate(pks):
            y = box.shares.get(c.key(pk))                       # participant.rs:310
            if y is not None:
                live.append(i)
                ys.append(y)
        out = [None] * n
        if not live:
            return out
        m = len(live)
        pko, so, co, ro = buf(size=m * c.eb), buf(size=m * c.eb), buf(size=m * c.sb), buf(size=m * c.sb)
        st = (ctypes.c_int * m)()
        g.ctx.check(g.ctx.lib.mpvss_extract_shares(
            g.ctx.h, m, ptr(buf(c.enc_scalars([private_keys[i] for i in live]))),
            ptr(buf(c.enc_scalars([ws[i] for i in live]))), ptr(buf(c.enc_elems(ys))), ptr(pko), ptr(so), ptr(co),
            ptr(ro), st))
        pk2, ss, cs, rs = c.dec_elems(pko, m), c.dec_elems(so, m), c.dec_scalars(co, m), c.dec_scalars(ro, m)
        for j, i in enumerate(live):
            if st[j] == _lib.OK:                                # participant.rs:314 -> None
                out[i] = ShareBox(pk2[j], ss[j], cs[j], rs[j])
        return out

    def extract_secret_share(self, box, private_key, w):
        return self.extract_secret_shares(box, [private_key], [w])[0]

    # -- verify_share: participant.rs:361-386 / 1346-1371 / 1789-1814 --
    def verify_shares(self, shareboxes, box, publickeys):
        g, c = self.group, self.group.codec
        n = len(shareboxes)
        res = [False] * n
        live, ys = [], []
        for i, pk in enumerate(publickeys):
            y = box.shares.get(c.key(pk))
            if y is not None:                                   # participant.rs:371-375
                live.append(i)
                ys.append(y)
        if not live:
            return res
        m = len(live)
        ok = (ctypes.c_int * m)()
        g.ctx.check(g.ctx.lib.mpvss_verify_shares(
            g.ctx.h, m, ptr(buf(c.enc_elems([publickeys[i] for i in live]))),
            ptr(buf(c.enc_elems([shareboxes[i].share for i in live]))), ptr(buf(c.enc_elems(ys))),
            ptr(buf(c.enc_scalars([shareboxes[i].challenge for i in live]))),
            ptr(buf(c.enc_scalars([shareboxes[i].response for i in live]))), ok))
        for j, i in enumerate(live):
            res[i] = bool(ok[j])
        return res

    def verify_share(self, sharebox, box, publickey) -> bool:
        return self.verify_shares([sharebox], box, [publickey])[0]

    # -- reconstruct: participant.rs:462-519 / 1452-1513 / 1895-1950 --
    def _shares_by_position(self, share_boxes, box):
        """(positions in ascending order, their shares), or None where reconstruct returns None"""
        c = self.group.codec
        if len(share_boxes) < len(box.commitments):             # participant.rs:469
            return None
        shares = {}
        for sb in share_boxes:                                  # participant.rs:476-482
            p = box.positions.get(c.key(sb.publickey))
            if p is None:
                return None
            shares[p] = sb.share
        pos = sorted(shares)
        return pos, [shares[p] for p in pos]

    def reconstruct(self, share_boxes, box, trace=None):
        g, c = self.group, self.group.codec
        flat = self._shares_by_position(share_boxes, box)
        if flat is None:
            return None
        pos, ss = flat
        k = len(pos)
        sec, gs = buf(size=c.eb), buf(size=c.eb)
        g.ctx.check(g.ctx.lib.mpvss_reconstruct(
            g.ctx.h, k, (ctypes.c_int64 * k)(*pos), ptr(buf(c.enc_elems(ss))),
            ptr(buf(box.U.to_bytes(c.eb, "big"))), ptr(sec), ptr(gs)))
        if trace is not None:
            trace["G_s"] = c.dec_elem(bytes(gs))
        return int.from_bytes(bytes(sec), "big")

    def reconstruct_secrets(self, jobs, traces=None) -> list:
        """Batch form of reconstruct: one secret (or None) per (share_boxes, box) job, all jobs in one library call
        (mpvss_reconstruct_secrets).  A job for which reconstruct returns None, or whose box the library rejects
        (where reconstruct would raise), is None without disturbing the others.  traces[j]["G_s"] receives G^s."""
        g, c = self.group, self.group.codec
        res = [None] * len(jobs)
        live, flats = [], []
        for j, (share_boxes, box) in enumerate(jobs):
            flat = self._shares_by_position(share_boxes, box)
            if flat is not None:
                live.append(j)
                flats.append(flat)
        if not live:
            return res
        m = len(live)
        pos = [p for f in flats for p in f[0]]
        sec, gs, st = buf(size=m * c.eb), buf(size=m * c.eb), (ctypes.c_int * m)()
        g.ctx.check(g.ctx.lib.mpvss_reconstruct_secrets(
            g.ctx.h, m, (ctypes.c_size_t * m)(*[len(f[0]) for f in flats]), (ctypes.c_int64 * len(pos))(*pos),
            ptr(buf(b"".join(c.enc_elems(f[1]) for f in flats))),
            ptr(buf(b"".join(jobs[j][1].U.to_bytes(c.eb, "big") for j in live))), ptr(sec), ptr(gs), st))
        for i, j in enumerate(live):
            if st[i] != _lib.OK:
                continue
            res[j] = int.from_bytes(bytes(sec)[i * c.eb:(i + 1) * c.eb], "big")
            if traces is not None:
                traces[j]["G_s"] = c.dec_elem(bytes(gs)[i * c.eb:(i + 1) * c.eb])
        return res


def string_to_secret(message: str) -> int:
    """lib.rs:49-52."""
    return int.from_bytes(message.encode(), "big")


def string_from_secret(secret: int) -> str:
    """lib.rs:54-57."""
    return secret.to_bytes((secret.bit_length() + 7) // 8, "big").decode()
