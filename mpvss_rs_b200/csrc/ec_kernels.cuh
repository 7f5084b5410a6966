// Kernel bodies for the elliptic-curve groups (Secp256k1Group, Ristretto255Group), one
// instance per thread, templated on a curve policy (secp.cuh: SecpCurve, rist.cuh:
// RistCurve).  `tid` is the global thread index; bodies return immediately for tid >= n (no
// warp-collective operations are used).
//
// Reference call sites replaced (paths under /root/reference/src; secp256k1 / ristretto255):
//   exp2_body    : group.exp / DLEQ commitments  secp256k1.rs:91-100, ristretto255.rs:161-170,
//                  dleq.rs:37-39, 66-84, participant.rs:1143,1187,1202-1203,1300,1316-1317,1544 /
//                  1608,1645,1660-1661,1743,1759-1760,1992
//   horner_body  : X_i = sum_j (i^j) C_j  participant.rs:1174-1184, 1411-1421 / 1630-1642, 1854-1864
//   add_body     : group.mul  secp256k1.rs:102-107, ristretto255.rs:172-177
//   poly_body    : P(i) mod order  polynomial.rs:50-58 via participant.rs:1155-1157 / 1619-1621
//   lagrange_body: lambda_i  participant.rs:1518-1557 / 1955-2002
//   inv_body     : scalar inverse  secp256k1.rs:109-112, ristretto255.rs:179-187
#pragma once
#include "fp256.cuh"

namespace ec {

using fp256::Fe;
using fp256::Modulus;

MP_DEV uint32_t nibble(const uint32_t* e, int w) { return (e[w >> 3] >> ((w & 7) * 4)) & 15u; }

// table[i] = i * p for i = 0..15
template <class Cv>
MP_DEV void build_table(typename Cv::Point* tbl, const typename Cv::Point& p, const typename Cv::Consts& C) {
  tbl[0] = Cv::infinity(C);
  tbl[1] = p;
  tbl[2] = Cv::dbl(p, C);
#pragma unroll 1
  for (int i = 3; i < 16; ++i) tbl[i] = (i & 1) ? Cv::add(tbl[i - 1], p, C) : Cv::dbl(tbl[i >> 1], C);
}

// e1 * p1 [+ e2 * p2]: fixed 4-bit windows, doublings shared between the two scalars
// (scalars: 8 little-endian u32 limbs)
template <class Cv>
MP_DEV typename Cv::Point scalar_mul2(const typename Cv::Point& p1, const uint32_t* e1, const typename Cv::Point* p2,
                                      const uint32_t* e2, typename Cv::Point* tbl1, typename Cv::Point* tbl2,
                                      const typename Cv::Consts& C) {
  build_table<Cv>(tbl1, p1, C);
  if (p2) build_table<Cv>(tbl2, *p2, C);
  typename Cv::Point acc = Cv::infinity(C);
#pragma unroll 1
  for (int w = 63; w >= 0; --w) {
    if (w != 63) {
      acc = Cv::dbl(acc, C);
      acc = Cv::dbl(acc, C);
      acc = Cv::dbl(acc, C);
      acc = Cv::dbl(acc, C);
    }
    uint32_t d = nibble(e1, w);
    if (d) acc = Cv::add(acc, tbl1[d], C);
    if (p2) {
      d = nibble(e2, w);
      if (d) acc = Cv::add(acc, tbl2[d], C);
    }
  }
  return acc;
}

// The small-integer multiple [pos]acc of the Horner step is the curve policy's Cv::small_mul (fixed
// 2-bit windows, one addition call site per window so that a warp whose lanes hold different digits
// still executes a single point addition).

// ------------------------------------------------------------ e1*B1 [+ e2*B2] ----
template <class Cv>
struct Exp2Args {
  const typename Cv::Consts* C;
  const uint8_t* b1;   // compressed points, stride b1_stride bytes (0 = one shared base)
  const uint32_t* e1;  // scalars, 8 little-endian limbs each, stride e1_stride limbs
  const uint8_t* b2;   // optional second base / scalar
  const uint32_t* e2;
  uint8_t* out;        // encoded results (Cv::EB bytes each), or nullptr
  typename Cv::Point* out_jac;  // projective results, or nullptr
  uint32_t* status;    // per instance: 0 ok, 1 invalid encoding
  uint32_t n, b1_stride, e1_stride, b2_stride, e2_stride;
  const uint32_t* comb1;  // optional fixed-base table of b1 (COMB_WORDS words, CombArgs layout): e1 * b1 becomes 64
                          // mixed additions of table entries, no doublings (b1 is then not decoded)
};

// ---- fixed-base table of the generator ("comb"): T[w][d-1] = (d * 16^w) G, affine, w < 64, d = 1..15 ----
// 960 entries x 64 bytes = 60 KB: the kernels that use it stage it through shared memory once per CTA
// (north_star: "fixed-base precomputed tables staged through shared memory"), then every scalar
// multiplication by G is 64 table lookups and at most 64 mixed additions.
constexpr int COMB_ENTRIES = 64 * 15;
constexpr int COMB_WORDS = COMB_ENTRIES * 16;

template <class Cv>
MP_DEV typename Cv::Point comb_mul(const uint32_t* tbl, const uint32_t* e, const typename Cv::Consts& C) {
  typename Cv::Point acc = Cv::infinity(C);
#pragma unroll 1
  for (int w = 0; w < 64; ++w) {
    const uint32_t d = nibble(e, w);
    if (d) {
      const uint32_t* q = tbl + (size_t)(w * 15 + (d - 1)) * 16;
      typename Cv::Affine a;
      a.x = fp256::load(q);
      a.y = fp256::load(q + 8);
      a.inf = 0;
      acc = Cv::madd(acc, a, C);
    }
  }
  return acc;
}

template <class Cv>
struct CombArgs {
  const typename Cv::Consts* C;
  const uint8_t* gen;  // encoded generator
  uint32_t* tbl;       // COMB_WORDS words
};
// entry (w, d): one thread each, (d << 4w) * G by the generic ladder, then to affine
template <class Cv>
MP_DEV void comb_build_body(const CombArgs<Cv>& A, uint32_t tid) {
  if (tid >= (uint32_t)COMB_ENTRIES) return;
  using Point = typename Cv::Point;
  const typename Cv::Consts& C = *A.C;
  const uint32_t w = tid / 15, d = tid % 15 + 1;
  typename Cv::Affine g;
  Cv::decode(g, A.gen, C);
  uint32_t e[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  e[w >> 3] = d << ((w & 7) * 4);
  Point tbl[16];
  Point r = scalar_mul2<Cv>(Cv::from_aff(g, C), e, nullptr, e, tbl, tbl, C);
  typename Cv::Affine a = Cv::to_affine(r, C);
  fp256::store(A.tbl + (size_t)tid * 16, a.x);
  fp256::store(A.tbl + (size_t)tid * 16 + 8, a.y);
}

// out[i] = e[i] * G from the table (Group::exp with a generator: commitments, public keys, a1 = w * G)
template <class Cv>
struct FixedArgs {
  const typename Cv::Consts* C;
  const uint32_t* tbl;   // global copy of the table
  const uint32_t* e;     // n scalars, 8 little-endian limbs each
  uint8_t* out;          // n encodings
  uint32_t n;
};
template <class Cv>
MP_DEV void fixed_body(const FixedArgs<Cv>& A, uint32_t tid, const uint32_t* tbl) {
  if (tid >= A.n) return;
  uint32_t e[8];
  for (int i = 0; i < 8; ++i) e[i] = A.e[(size_t)tid * 8 + i];
  Cv::encode(A.out + (size_t)tid * Cv::EB, comb_mul<Cv>(tbl, e, *A.C), *A.C);
}

// `comb` = the staged table of b1 (shared memory) when A.comb1 is set, else unused
template <class Cv>
MP_DEV void exp2_body(const Exp2Args<Cv>& A, uint32_t tid, const uint32_t* comb = nullptr) {
  if (tid >= A.n) return;
  using Point = typename Cv::Point;
  const typename Cv::Consts& C = *A.C;
  typename Cv::Affine a1, a2;
  bool ok = true;
  if (!A.comb1) ok = Cv::decode(a1, A.b1 + (size_t)tid * A.b1_stride, C);
  if (A.b2) ok = Cv::decode(a2, A.b2 + (size_t)tid * A.b2_stride, C) && ok;
  if (A.status) A.status[tid] = ok ? 0u : 1u;
  Point tbl1[16], tbl2[16];
  Point p1, p2;
  if (!A.comb1) p1 = Cv::from_aff(a1, C);
  if (A.b2) p2 = Cv::from_aff(a2, C);
  uint32_t e1[8], e2[8];
  for (int i = 0; i < 8; ++i) {
    e1[i] = A.e1[(size_t)tid * A.e1_stride + i];
    e2[i] = A.b2 ? A.e2[(size_t)tid * A.e2_stride + i] : 0u;
  }
  Point r = Cv::infinity(C);
  if (ok) {
    if (A.comb1) {
      r = comb_mul<Cv>(comb, e1, C);
      if (A.b2) r = Cv::add(r, scalar_mul2<Cv>(p2, e2, nullptr, e2, tbl2, tbl2, C), C);
    } else {
      r = scalar_mul2<Cv>(p1, e1, A.b2 ? &p2 : nullptr, e2, tbl1, tbl2, C);
    }
  }
  if (A.out_jac) A.out_jac[tid] = r;
  if (A.out) Cv::encode(A.out + (size_t)tid * Cv::EB, r, C);
}

// ----------------------------------------------------------------- decode ----
template <class Cv>
struct DecodeArgs {
  const typename Cv::Consts* C;
  const uint8_t* in;   // n compressed points
  uint32_t* xy;        // n x 16 limbs: x, y in Montgomery form (identity: all zero)
  uint32_t* status;
  uint32_t n;
};
template <class Cv>
MP_DEV void decode_body(const DecodeArgs<Cv>& A, uint32_t tid) {
  if (tid >= A.n) return;
  typename Cv::Affine a;
  bool ok = Cv::decode(a, A.in + (size_t)tid * Cv::EB, *A.C);
  fp256::store(A.xy + (size_t)tid * 16, a.x);
  fp256::store(A.xy + (size_t)tid * 16 + 8, a.y);
  A.status[tid] = ok ? (a.inf ? 2u : 0u) : 1u;
}

// ----------------------------------------------------------------- Horner ----
// Instance (k, i) = tid / n, tid % n evaluates chunk k of the commitment polynomial at
// position pos[i] by Horner in the group, then scales by pos^(k*B) so that the K partial
// results of a position add up to X_i (chunking only adds parallelism; the group element is
// the same as the reference's sum of t scalar multiplications).
template <class Cv>
struct HornerArgs {
  const typename Cv::Consts* C;
  const uint32_t* cxy;     // t commitments, affine Montgomery (decode_body layout)
  const uint32_t* cstatus; // decode status per commitment (2 = identity)
  const uint32_t* pos;     // n positions
  typename Cv::Point* out; // K * n partial results, index k * n + i
  uint32_t t, n, K, B;     // K chunks of B coefficients (last one shorter)
};

MP_DEV uint32_t digits4(uint32_t p) {
  uint32_t d = 1;
  while (d < 16 && (p >> (2 * d))) ++d;
  return d;
}
template <class Cv>
MP_DEV typename Cv::Affine load_aff(const uint32_t* xy, uint32_t status) {
  typename Cv::Affine a;
  a.x = fp256::load(xy);
  a.y = fp256::load(xy + 8);
  a.inf = status == 2u;
  return a;
}

template <class Cv>
MP_DEV void horner_body(const HornerArgs<Cv>& A, uint32_t tid) {
  if (tid >= A.n * A.K) return;
  using Point = typename Cv::Point;
  const typename Cv::Consts& C = *A.C;
  const uint32_t k = tid / A.n, i = tid % A.n;
  const uint32_t lo = k * A.B, hi = (lo + A.B < A.t) ? lo + A.B : A.t;
  const uint32_t pos = A.pos[i], nd = digits4(pos);
  Point acc = Cv::from_aff(load_aff<Cv>(A.cxy + (size_t)(hi - 1) * 16, A.cstatus[hi - 1]), C);
#pragma unroll 1
  for (int j = (int)hi - 2; j >= (int)lo; --j) {
    acc = Cv::small_mul(acc, pos, nd, C);
    acc = Cv::madd(acc, load_aff<Cv>(A.cxy + (size_t)j * 16, A.cstatus[j]), C);
  }
  if (k > 0) {
    // e = pos^(k*B) mod n in the scalar field, then acc <- e * acc
    using namespace fp256;
    Fe b = fe_zero();
    b.v[0] = pos;
    b = to_mont(b, C.N);
    Fe e = mont_one(C.N);
    uint32_t ex = lo;
    bool started = false;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      if (started) e = sqr(e, C.N);
      if ((ex >> bit) & 1u) {
        e = started ? mul(e, b, C.N) : b;
        started = true;
      }
    }
    e = from_mont(e, C.N);
    acc = Cv::scalar_mul_wide(acc, e.v, C);
  }
  A.out[tid] = acc;
}

// Multi-box Horner (mpvss_verify_distributions): the positions of several boxes are concatenated, and
// position i belongs to a box whose t_b commitments start at cxy row coff[i].  Instance (k, i) evaluates
// chunk k = [k B_b, min((k+1) B_b, t_b)), B_b = ceil(t_b / K), of that box's polynomial; a chunk that lies
// past t_b (boxes with fewer than K coefficients) contributes the identity.  The body repeats horner_body
// instead of sharing a helper with it so that the single-box kernel's code stays exactly as it is.  Running the
// single-box calls through this kernel as one box was measured and not taken: at 128 registers it keeps 264
// bytes of stack against horner_kernel's 256 (secp256k1), and the secp256k1 X_i phase of the n = 4096 verify
// took 26.02-26.10 ms against 25.98-26.00 ms (NVIDIA B200, 1000 W, 3 alternating runs each).
template <class Cv>
struct HornerBoxesArgs {
  const typename Cv::Consts* C;
  const uint32_t* cxy;      // commitments of all boxes, concatenated (decode_body layout)
  const uint32_t* cstatus;  // decode status per commitment (2 = identity)
  const uint32_t* pos;      // n positions, concatenated over the boxes
  const uint32_t* coff;     // per position: first commitment of its box
  const uint32_t* ct;       // per position: commitments t_b of its box
  typename Cv::Point* out;  // K * n partial results, index k * n + i
  uint32_t n, K;
};

template <class Cv>
MP_DEV void horner_boxes_body(const HornerBoxesArgs<Cv>& A, uint32_t tid) {
  if (tid >= A.n * A.K) return;
  using Point = typename Cv::Point;
  const typename Cv::Consts& C = *A.C;
  const uint32_t k = tid / A.n, i = tid % A.n;
  const uint32_t t = A.ct[i], B = (t + A.K - 1) / A.K, lo = k * B;
  if (lo >= t) {
    A.out[tid] = Cv::infinity(C);
    return;
  }
  const uint32_t hi = (lo + B < t) ? lo + B : t;
  const uint32_t* cxy = A.cxy + (size_t)A.coff[i] * 16;
  const uint32_t* cst = A.cstatus + A.coff[i];
  const uint32_t pos = A.pos[i], nd = digits4(pos);
  Point acc = Cv::from_aff(load_aff<Cv>(cxy + (size_t)(hi - 1) * 16, cst[hi - 1]), C);
#pragma unroll 1
  for (int j = (int)hi - 2; j >= (int)lo; --j) {
    acc = Cv::small_mul(acc, pos, nd, C);
    acc = Cv::madd(acc, load_aff<Cv>(cxy + (size_t)j * 16, cst[j]), C);
  }
  if (k > 0) {
    // e = pos^(k*B) mod n in the scalar field, then acc <- e * acc
    using namespace fp256;
    Fe b = fe_zero();
    b.v[0] = pos;
    b = to_mont(b, C.N);
    Fe e = mont_one(C.N);
    bool started = false;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      if (started) e = sqr(e, C.N);
      if ((lo >> bit) & 1u) {
        e = started ? mul(e, b, C.N) : b;
        started = true;
      }
    }
    e = from_mont(e, C.N);
    acc = Cv::scalar_mul_wide(acc, e.v, C);
  }
  A.out[tid] = acc;
}

// --------------------------------------------------------- sums / encoding ----
template <class Cv>
struct SumArgs {
  const typename Cv::Consts* C;
  const typename Cv::Point* in;  // element (g, j) at in[g * g_stride + j * j_stride], j < count (clipped to total)
  typename Cv::Point* out_jac;   // groups results (or nullptr)
  uint8_t* out;                  // groups encoded results (or nullptr)
  uint32_t groups, count, g_stride, j_stride, total;
};
template <class Cv>
MP_DEV void sum_body(const SumArgs<Cv>& A, uint32_t tid) {
  if (tid >= A.groups) return;
  const typename Cv::Consts& C = *A.C;
  typename Cv::Point acc = A.in[(size_t)tid * A.g_stride];
#pragma unroll 1
  for (uint32_t j = 1; j < A.count; ++j) {
    size_t idx = (size_t)tid * A.g_stride + (size_t)j * A.j_stride;
    if (idx >= A.total) break;
    acc = Cv::add(acc, A.in[idx], C);
  }
  if (A.out_jac) A.out_jac[tid] = acc;
  if (A.out) Cv::encode(A.out + (size_t)tid * Cv::EB, acc, C);
}

// Segmented sum (mpvss_reconstruct_secrets): group g adds the seg[2g + 1] >= 1 points from row seg[2g]; the host
// plans the segments with sum_boxes_level so that none crosses a box boundary.
template <class Cv>
struct SumBoxesArgs {
  const typename Cv::Consts* C;
  const typename Cv::Point* in;
  const uint32_t* seg;           // groups x (first row, count)
  typename Cv::Point* out_jac;   // groups results (or nullptr)
  uint8_t* out;                  // groups encoded results (or nullptr)
  uint32_t groups;
};
template <class Cv>
MP_DEV void sum_boxes_body(const SumBoxesArgs<Cv>& A, uint32_t tid) {
  if (tid >= A.groups) return;
  const typename Cv::Consts& C = *A.C;
  const uint32_t first = A.seg[2 * tid], count = A.seg[2 * tid + 1];
  typename Cv::Point acc = A.in[first];
#pragma unroll 1
  for (uint32_t j = 1; j < count; ++j) acc = Cv::add(acc, A.in[first + j], C);
  if (A.out_jac) A.out_jac[tid] = acc;
  if (A.out) Cv::encode(A.out + (size_t)tid * Cv::EB, acc, C);
}

// One level of the segmented sum (host planning, shared with the tests): box b holds cnt[b] points from row
// start[b]; every 64 consecutive points of a box form one group, and the groups are numbered in box order.
// Writes the groups' (first row, count) to `seg`, moves start / cnt to the box's group results and returns the
// group count.  A level planned while every cnt is at most 64 has one group per box: group b is box b.
inline uint32_t sum_boxes_level(uint32_t* start, uint32_t* cnt, uint32_t boxes, uint32_t* seg) {
  uint32_t m = 0;
  for (uint32_t b = 0; b < boxes; ++b) {
    const uint32_t first = m;
    for (uint32_t j = 0; j < cnt[b]; j += 64) {
      seg[2 * m] = start[b] + j;
      seg[2 * m + 1] = cnt[b] - j < 64 ? cnt[b] - j : 64;
      ++m;
    }
    start[b] = first;
    cnt[b] = m - first;
  }
  return m;
}

// out[i] = a[i] + b[i]   (Group::mul)
template <class Cv>
struct AddArgs {
  const typename Cv::Consts* C;
  const uint8_t *a, *b;
  uint8_t* out;
  uint32_t* status;
  uint32_t n;
};
template <class Cv>
MP_DEV void add_body(const AddArgs<Cv>& A, uint32_t tid) {
  if (tid >= A.n) return;
  const typename Cv::Consts& C = *A.C;
  typename Cv::Affine a, b;
  bool ok = Cv::decode(a, A.a + (size_t)tid * Cv::EB, C);
  ok = Cv::decode(b, A.b + (size_t)tid * Cv::EB, C) && ok;
  A.status[tid] = ok ? 0u : 1u;
  typename Cv::Point r = Cv::madd(Cv::from_aff(a, C), b, C);
  Cv::encode(A.out + (size_t)tid * Cv::EB, r, C);
}

// ------------------------------------------------------- transcript frames ----
// Row j of the Fiat-Shamir transcript (dleq.rs:58-61, 87-99): F(X_j) F(Y_j) F(a1_j) F(a2_j) with
// F(e) = len_u64_be || encoding; the curves' encodings have fixed length eb (33 / 32), so a row is
// 4 * (8 + eb) bytes.  One thread per frame.  `bad` marks a row set whose inputs did not decode: the
// first byte of the rank's first row becomes 0xff (never part of a valid length), which every rank sees
// after the all-gather.
struct FrameArgs {
  const uint8_t *x, *y, *a1, *a2;  // n encodings each
  uint8_t* out;
  uint32_t n, eb;
};
MP_DEV void frame_body(const FrameArgs& A, uint32_t tid) {
  const uint32_t j = tid >> 2, e = tid & 3u;
  if (j >= A.n) return;
  const uint8_t* src = (e == 0 ? A.x : e == 1 ? A.y : e == 2 ? A.a1 : A.a2) + (size_t)j * A.eb;
  uint8_t* dst = A.out + ((size_t)j * 4 + e) * (8 + A.eb);
  for (int k = 0; k < 7; ++k) dst[k] = 0;
  dst[7] = (uint8_t)A.eb;
  for (uint32_t k = 0; k < A.eb; ++k) dst[8 + k] = src[k];
}

// ---------------------------------------------------------- scalar kernels ----
// p_i = P(pos_i) mod n by Horner in the scalar field (coefficients: 8 LE limbs, < n)
struct PolyArgs {
  const Modulus* N;
  const uint32_t* coeffs;  // t x 8 limbs
  const uint32_t* pos;     // n positions
  uint32_t* out;           // n x 8 limbs
  uint32_t t, n;
};
MP_DEV void poly_body(const PolyArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  using namespace fp256;
  const Modulus& N = *A.N;
  Fe x = fe_zero();
  x.v[0] = A.pos[tid];
  x = to_mont(x, N);
  Fe acc = to_mont(load(A.coeffs + (size_t)(A.t - 1) * 8), N);
#pragma unroll 1
  for (int j = (int)A.t - 2; j >= 0; --j) acc = add(mul(acc, x, N), to_mont(load(A.coeffs + (size_t)j * 8), N), N);
  store(A.out + (size_t)tid * 8, from_mont(acc, N));
}

// Several boxes at once (mpvss_distribute_secrets): the coefficients and the instances of the boxes are
// concatenated, and instance i evaluates the polynomial of its own box: t_b = bt[i] coefficients from row coff[i],
// the box's instances starting at row ioff[i].
struct PolyBoxesArgs {
  const Modulus* N;
  const uint32_t* coeffs;  // sum t_b x 8 limbs, concatenated over the boxes
  const uint32_t* pos;     // n positions, concatenated over the boxes
  const uint32_t* coff;    // per instance: first coefficient row of its box
  const uint32_t* bt;      // per instance: coefficients t_b of its box
  const uint32_t* ioff;    // per instance: first instance row of its box
  uint32_t* out;           // n x 8 limbs
  uint32_t n;
};
MP_DEV void poly_boxes_body(const PolyBoxesArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  const uint32_t off = A.ioff[tid];
  poly_body(PolyArgs{A.N, A.coeffs + (size_t)A.coff[tid] * 8, A.pos + off, A.out + (size_t)off * 8, A.bt[tid], A.n - off},
            tid - off);
}

// Lagrange coefficients at 0 for the given positions, in the scalar field, with the sign of
// the reference folded in:  lambda_i = prod_{j != i} x_j / (x_j - x_i)  (participant.rs:1518-1557
// computes |x_j - x_i| and a separate sign, then negates the point; negating the scalar gives
// the same group element).
struct LagrangeArgs {
  const Modulus* N;
  const uint32_t* pos;  // k positions
  uint32_t* out;        // k x 8 limbs
  uint32_t k;
};
// acc <- acc * f for a 256-bit plain integer and a 32-bit factor (the caller keeps the product below 2^256)
MP_DEV void mul_small(uint32_t (&acc)[8], uint32_t f) {
  uint32_t carry = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint64_t t = (uint64_t)acc[i] * f + carry;
    acc[i] = (uint32_t)t;
    carry = (uint32_t)(t >> 32);
  }
}
MP_DEV void lagrange_body(const LagrangeArgs& A, uint32_t tid) {
  if (tid >= A.k) return;
  using namespace fp256;
  const Modulus& N = *A.N;
  const uint32_t xi = A.pos[tid];
  Fe num = mont_one(N), den = mont_one(N);
  bool negative = false;
  // The factors are 32-bit numbers: eight of them are multiplied as plain integers (8 MACs each) before one
  // Montgomery product folds them into the running value -- a quarter of the field products of the
  // factor-by-factor loop, which was 5 ms of dependent products per thread at k = 2731.
  Fe na = fe_zero(), da = fe_zero();
  na.v[0] = da.v[0] = 1;
  uint32_t pending = 0;
#pragma unroll 1
  for (uint32_t j = 0; j < A.k; ++j) {
    if (j == tid) continue;
    const uint32_t xj = A.pos[j];
    if (xj < xi) negative = !negative;
    mul_small(na.v, xj);
    mul_small(da.v, xj < xi ? xi - xj : xj - xi);
    if (++pending == 8) {
      num = mul(num, to_mont(na, N), N);
      den = mul(den, to_mont(da, N), N);
      na = fe_zero();
      da = fe_zero();
      na.v[0] = da.v[0] = 1;
      pending = 0;
    }
  }
  if (pending) {
    num = mul(num, to_mont(na, N), N);
    den = mul(den, to_mont(da, N), N);
  }
  Fe lam = mul(num, inv(den, N), N);  // den = 0 (duplicate position) -> lambda = 0, as ristretto255.rs falls back
  if (negative) lam = neg(lam, N);
  store(A.out + (size_t)tid * 8, from_mont(lam, N));
}

// Several boxes at once (mpvss_reconstruct_secrets): the positions of the boxes are concatenated, position i
// belongs to the box of bk[i] positions that starts at boff[i], and its coefficient is lagrange_body's over
// that box alone.
struct LagrangeBoxesArgs {
  const Modulus* N;
  const uint32_t* pos;   // n positions, concatenated over the boxes
  const uint32_t* boff;  // per position: first position of its box
  const uint32_t* bk;    // per position: positions k_b of its box
  uint32_t* out;         // n x 8 limbs
  uint32_t n;
};
MP_DEV void lagrange_boxes_body(const LagrangeBoxesArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  const uint32_t off = A.boff[tid];
  lagrange_body(LagrangeArgs{A.N, A.pos + off, A.out + (size_t)off * 8, A.bk[tid]}, tid - off);
}

// out[i] = in[i]^-1 in the scalar field (0 -> 0, flagged in status)
struct InvArgs {
  const Modulus* N;
  const uint32_t* in;
  uint32_t* out;
  uint32_t* status;
  uint32_t n;
};
MP_DEV void inv_body(const InvArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  using namespace fp256;
  Fe x = load(A.in + (size_t)tid * 8);
  A.status[tid] = is_zero(x) ? 1u : 0u;
  store(A.out + (size_t)tid * 8, from_mont(inv(to_mont(x, *A.N), *A.N), *A.N));
}

// ------------------------------------------------- per-share DLEQ transcripts ----
// Second half of a per-share Fiat-Shamir step once shadev::row_hash_body has hashed the share's row
// (sha2_dev.cuh): reduce hash_to_scalar's integer into the scalar field and either
//   extract (sk, w given): c and r = w - sk * c  (participant.rs:1323-1333 / 1766-1776; dleq.rs:42-50), or
//   verify  (c_in given):  ok = (c == c_in)      (dleq.rs:119-126 via participant.rs:1370 / 1813).
// wide = 0: h is int_be(SHA-256(digest)) < 2^256 < 2n, one conditional subtraction (secp256k1.rs:121-131);
// wide = 1: h is the 512-bit int_le(SHA-512(digest)), reduced as lo + hi * 2^256 with Montgomery products by
// R^2 (ristretto255.rs:196-205, Scalar::from_bytes_mod_order_wide).  Scalars leave in the boundary encoding.
struct ProofArgs {
  const Modulus* N;
  const uint32_t* h;       // n x (wide ? 16 : 8) limbs
  const uint32_t *sk, *w;  // extract: n x 8 limbs each
  const uint8_t* c_in;     // verify: n x 32 bytes
  uint8_t *c_out, *r_out;  // extract: n x 32 bytes each
  uint32_t* ok;            // verify
  uint32_t n, wide, big_endian;
};
MP_DEV void scalar_bytes_out(uint8_t* o, const fp256::Fe& v, bool big_endian) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint32_t x = v.v[i];
    if (big_endian) {
      uint8_t* q = o + 4 * (7 - i);
      q[0] = (uint8_t)(x >> 24); q[1] = (uint8_t)(x >> 16); q[2] = (uint8_t)(x >> 8); q[3] = (uint8_t)x;
    } else {
      uint8_t* q = o + 4 * i;
      q[0] = (uint8_t)x; q[1] = (uint8_t)(x >> 8); q[2] = (uint8_t)(x >> 16); q[3] = (uint8_t)(x >> 24);
    }
  }
}
MP_DEV fp256::Fe scalar_bytes_in(const uint8_t* p, bool big_endian) {
  fp256::Fe v;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (big_endian) {
      const uint8_t* q = p + 4 * (7 - i);
      v.v[i] = (uint32_t)q[0] << 24 | (uint32_t)q[1] << 16 | (uint32_t)q[2] << 8 | q[3];
    } else {
      const uint8_t* q = p + 4 * i;
      v.v[i] = (uint32_t)q[3] << 24 | (uint32_t)q[2] << 16 | (uint32_t)q[1] << 8 | q[0];
    }
  }
  return v;
}
MP_DEV void proof_body(const ProofArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  using namespace fp256;
  const Modulus& N = *A.N;
  Fe c;
  if (A.wide) {
    const uint32_t* h = A.h + (size_t)tid * 16;
    const Fe r2 = load(N.r2);
    Fe lo = mul(load(h), r2, N);               // lo * R
    Fe hi = mul(mul(load(h + 8), r2, N), r2, N);  // hi * R * R = (hi * 2^256) * R
    c = from_mont(add(lo, hi, N), N);
  } else {
    c = cond_sub(load(A.h + (size_t)tid * 8), 0, N);
  }
  const bool be = A.big_endian != 0;
  if (A.c_in) {
    A.ok[tid] = eq(c, scalar_bytes_in(A.c_in + (size_t)tid * 32, be)) ? 1u : 0u;
  } else {
    Fe sk = load(A.sk + (size_t)tid * 8), w = load(A.w + (size_t)tid * 8);
    Fe r = sub(w, mul(sk, to_mont(c, N), N), N);  // mont(sk, c R) = sk c
    scalar_bytes_out(A.c_out + (size_t)tid * 32, c, be);
    scalar_bytes_out(A.r_out + (size_t)tid * 32, r, be);
  }
}

}  // namespace ec
