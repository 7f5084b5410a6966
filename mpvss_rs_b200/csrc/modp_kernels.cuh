// Kernel bodies for the ModpGroup hot path.  Each body is written against simt.h so
// that the CUDA build (modp.cu) and the lane-per-thread emulator (tests/emu) run
// the same source.  A body is executed by whole warps; `wg` is the global warp
// index and `wsm` the warp's private slice of dynamic shared memory.  No block
// barrier is used anywhere (warps are independent), only warp shuffles/barriers.
//
// Reference call sites replaced (paths under /root/reference/src):
//   horner_body  : X_i = prod_j C_j^(i^j)  participant.rs:207-215, 423-434; mpvss.rs:114-123
//   exp2_body    : group.exp / DLEQ commitments  modp.rs:122-128, dleq.rs:37-39, 66-84,
//                  participant.rs:219, 236-237, 316, 331-332, 553
//   mul_body     : group.mul  modp.rs:130-132
#pragma once
#include "modp_arith.cuh"
#include "modp_sqr.cuh"

namespace modp {

// Layout of the constant block (device global memory, u32 limbs):
//   [0,64) q   [64,128) 2^2048-q   [128,192) R mod q (Montgomery one)
//   [192,256) R^2 mod q   [256] -q^-1 mod 2^32   [260,324) (q+1)/2
// Per-group shared buffers are strided by their size plus GPAD words, so that the 32/TPI groups of a warp
// start 8 banks apart: the LDS.64 that fetches the next two digits of b (every group reads the same word
// index of its own buffer) then touches 2 x 4 distinct banks instead of one bank pair four times
// (round-1 ncu: 4.2e9 shared-memory bank conflicts per Horner launch with a stride of 256 words).
constexpr int GPAD = 8;
enum { C_Q = 0, C_NQ = 64, C_ONE = 128, C_R2 = 192, C_NP = 256, C_QH = 260, C_WORDS = 324 };

template <int TPI>
MP_DEV void load_mod(Mod<Cfg<TPI>::L>& M, const uint32_t* consts, const Lane& ln) {
  load_slice<TPI>(M.q, consts + C_Q, ln);
  load_slice<TPI>(M.nq, consts + C_NQ, ln);
  M.np = consts[C_NP];
  M.qh = consts + C_QH;
}

// copy 64 limbs global -> this warp's shared buffer (lane l moves limbs 2l, 2l+1)
MP_DEV void warp_copy64(uint32_t* dst, const uint32_t* src) {
  uint32_t l = simt::lane_id();
  simt::syncwarp();  // earlier readers of dst are done
  dst[2 * l] = src[2 * l];
  dst[2 * l + 1] = src[2 * l + 1];
}

// Shared-memory scratch and per-lane plan of the split squaring (modp_sqr.cuh); empty unless the
// build selects it (MPVSS_MODP_SPLIT_SQR, TPI = 8 only).
#ifdef MPVSS_MODP_SPLIT_SQR
template <int TPI>
constexpr int sqr_scratch_words = TPI == 8 ? SQS_WORDS : 0;
#else
template <int TPI>
constexpr int sqr_scratch_words = 0;
#endif
struct SqrCtx {
  uint32_t* scratch;
  SqPlan pl;
};
template <int TPI>
MP_DEV SqrCtx make_sqr_ctx(uint32_t* scratch, const Lane& ln) {
  SqrCtx c;
  c.scratch = scratch;
  if (sqr_scratch_words<TPI> != 0) {
    c.pl = make_sq_plan(ln.k);
    scratch[SQS_ZERO + ln.k] = 0;
  }
  return c;
}

template <int TPI>
MP_DEV void sqr_plain(uint32_t (&acc)[Cfg<TPI>::L], uint32_t* sq, const Mod<Cfg<TPI>::L>& M, const Lane& ln) {
  stage_shared<TPI>(sq, acc, ln);
  simt::syncwarp();
  mont_mul<TPI>(acc, acc, sq, M, ln);
}

template <int TPI>
MP_DEV void sqr_inplace(uint32_t (&acc)[Cfg<TPI>::L], uint32_t* sq, const SqrCtx& sc, const Mod<Cfg<TPI>::L>& M,
                        const Lane& ln) {
  stage_shared<TPI>(sq, acc, ln);
  simt::syncwarp();
  // Three squarings exist: through mont_mul (1696 instructions per product at TPI = 8, 1024 wide MACs),
  // mont_sqr (symmetric rows in the fused loop: 832 MACs, 2304 instructions) and the split squaring of
  // modp_sqr.cuh (804 MACs, ~1940 instructions).  At n = 4096 (1.74 warps per scheduler) the launch
  // is latency-bound per warp and the instruction count decides: Horner 256 / 263 / 288 ms
  // (DESIGN.md section 5).  The dedicated ones are compile-time options for large batches.
  if constexpr (sqr_scratch_words<TPI> != 0) {
    mont_sqr_split(acc, acc, sq, sc.scratch, sc.pl, M, ln);
  } else {
#ifdef MPVSS_MODP_DEDICATED_SQR
    mont_sqr<TPI>(acc, acc, sq, M, ln);
#else
    mont_mul<TPI>(acc, acc, sq, M, ln);
#endif
  }
}

// Leave Montgomery form (multiply by 1), reduce below q, store 64 limbs.
template <int TPI>
MP_DEV void finish_store(uint32_t (&acc)[Cfg<TPI>::L], uint32_t* sq, uint32_t* dst64, bool live,
                         const Mod<Cfg<TPI>::L>& M, const Lane& ln) {
  constexpr int L = Cfg<TPI>::L;
  uint32_t one[L];
#pragma unroll
  for (int i = 0; i < L; ++i) one[i] = 0;
  if (ln.k == 0) one[0] = 1;
  stage_shared<TPI>(sq, one, ln);
  simt::syncwarp();
  mont_mul<TPI>(acc, acc, sq, M, ln);
  canonical<TPI>(acc, M, ln);
  if (live) stage<TPI>(dst64, acc, ln);
}

// ---------------------------------------------------------------- Horner ----
// X_i = (...((C_{t-1})^i * C_{t-2})^i ...)^i * C_0 : t-1 steps of "raise to the small integer i and
// multiply by C_j".  acc^i follows a short addition chain per position (modp_chain.h: power tree, 13.4
// products for a 12-bit i instead of the 16 of fixed 2-bit windows); the host lowers it to a list of ops
//     if (save) slot[save-1] <- acc;  if (a) acc <- slot[a-1];  acc <- acc * B(b)
// (bits 0-3 b, 4-7 a, 8-11 save; B(6) = Montgomery one = padding, B(7) = C_j closes the step: both are
// kept as per-group copies behind the chain slots, so that the operand address is ONE expression of the
// op field -- a select between two buffers cost 18 register moves per 10 digits in the product loop).
// Every lane group of a warp runs its own chain: the op fields only select shared-memory addresses, the
// instruction stream is the same for all groups, so only the LENGTH of the op list has to agree inside
// a warp (positions are sorted by it, shorter lists padded with products by one).
struct HornerArgs {
  const uint32_t* consts;  // constant block
  const uint32_t* cm;      // t commitments, Montgomery form, 64 limbs each
  const uint16_t* ops;     // n x HC_OPS ops (one Horner step of each instance)
  const uint32_t* slot;    // n output slots (nullptr: instance i writes slot i; 0xffffffff: padding)
  const uint32_t* nops;    // ops per step, per CTA (all instances of a CTA share it; the launcher passes
                           // nops[blockIdx.x], which keeps the schedule provably block-uniform so that
                           // ptxas needs no WARPSYNC around the shuffles); nullptr: `nops_all` everywhere
  uint32_t* out;           // results, canonical, 64 limbs each, indexed by slot
  uint32_t t, n, nops_all;
  uint32_t warps_per_cta;  // launch shape (0 = 1); nops is indexed by CTA
  // Chunked evaluation (few positions: the polynomial is cut into K contiguous chunks so that K times as many
  // lane groups run chains 1/K as long; the host combines X = prod_k H_k^(pos^(k B))).  Per CTA: index of the
  // chunk's top coefficient and its number of Horner steps; nullptr = the whole polynomial (t-1, t-1).
  const uint32_t* cfirst;
  const uint32_t* csteps;
};

constexpr int HC_SLOTS = 6;   // == modp_chain::SLOTS; slot 6 = Montgomery one, slot 7 = C_j
constexpr int HC_OPS = 48;    // == modp_chain::OPS_MAX
constexpr int HC_GSTRIDE = (HC_SLOTS + 2) * 64 + GPAD;

template <int TPI>
constexpr int horner_smem_words = (32 / TPI) * (HC_GSTRIDE + HC_OPS / 2);

// NP1: the modulus satisfies -q^-1 = 1 mod 2^32 (true for the RFC 3526 prime, whose low 64 bits are all
// ones), so the Montgomery digit is the low limb itself and one multiply leaves the per-digit critical path.
// CHUNKED: first / steps come from the per-CTA arrays; otherwise they are t - 1, a kernel parameter, and the
// loop control stays in uniform registers.  The shape of this loop moves the launch by a few per cent although
// it is outside the product: bounds passed in as two values and compared against each other 225.3 ms, bounds
// from the parameter 220.2 ms, per-CTA arrays with the count-down-to-zero loop on a shifted base (below)
// 217.4 ms at n = 4096, t = 2731 -- the last one is what the library launches.
template <int TPI, bool NP1 = false, bool CHUNKED = false>
MP_DEV void horner_body(const HornerArgs& A, uint32_t wg, uint32_t* wsm, uint32_t nops, uint32_t cta = 0) {
  const uint32_t first = CHUNKED ? A.cfirst[cta] : A.t - 1, steps = CHUNKED ? A.csteps[cta] : A.t - 1;
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  uint32_t inst = wg * GPW + gi;
  const bool live = inst < A.n;
  if (!live) inst = A.n - 1;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  if (NP1) M.np = 1u;
  uint32_t* gbase = wsm + gi * HC_GSTRIDE;  // this group's chain slots, then one and C_j
  uint16_t* opsm = reinterpret_cast<uint16_t*>(wsm + GPW * HC_GSTRIDE) + gi * HC_OPS;
  for (int k = ln.k; k < HC_OPS; k += TPI) opsm[k] = A.ops[(size_t)inst * HC_OPS + k];
  uint32_t acc[L];
  load_slice<TPI>(acc, A.consts + C_ONE, ln);
  stage<TPI>(gbase + HC_SLOTS * 64, acc, ln);
  load_slice<TPI>(acc, A.cm + (size_t)first * 64, ln);
  simt::syncwarp();
  // the chunk's coefficients are cmb[steps-1 .. 0]: the loop counts down to zero on a shifted base
  const uint32_t* cmb = CHUNKED ? A.cm + (size_t)(first - steps) * 64 : A.cm;
  for (int j = (int)steps - 1; j >= 0; --j) {
    {
      uint32_t cj[L];
      load_slice<TPI>(cj, cmb + (size_t)j * 64, ln);
      stage_shared<TPI>(gbase + (HC_SLOTS + 1) * 64, cj, ln);  // visible after the first op's barrier
    }
    uint32_t op = opsm[0];
#pragma unroll 1
    for (uint32_t k = 0; k < nops; ++k) {  // one code instance of the product for the whole step
      const uint32_t nxt = opsm[k + 1 < (uint32_t)HC_OPS ? k + 1 : k];
      const uint32_t sv = (op >> 8) & 15u, a = (op >> 4) & 15u, b = op & 15u;
      simt::syncwarp();  // earlier readers of the slot are done
      if (sv) stage<TPI>(gbase + (sv - 1) * 64, acc, ln);
      simt::syncwarp();
      if (a) load_slice<TPI>(acc, gbase + (a - 1) * 64, ln);
      mont_mul<TPI>(acc, acc, gbase + b * 64, M, ln);
      op = nxt;
    }
  }
  const uint32_t slot = A.slot ? A.slot[inst] : inst;
  finish_store<TPI>(acc, gbase, A.out + (size_t)(slot == 0xffffffffu ? 0 : slot) * 64, live && slot != 0xffffffffu, M,
                    ln);
}

// ------------------------------------------------- (double) exponentiation ----
struct Exp2Args {
  const uint32_t* consts;
  const uint32_t* b1;   // bases, normal form; stride b1_stride limbs (0 = one shared base)
  const uint32_t* e1;   // exponents, little-endian limbs, stride e1_stride
  const uint32_t* b2;   // optional second base (nullptr: single exponentiation)
  const uint32_t* e2;
  uint32_t* out;        // n results, canonical
  uint32_t n;
  uint32_t b1_stride, e1_stride, e1_windows;  // windows of 4 bits, counted from bit 0
  uint32_t b2_stride, e2_stride, e2_windows;
  const uint32_t* comb1;  // optional fixed-base table for b1 (CombArgs layout): b1^e1 becomes a product of
                          // ceil(e1_windows / 2) table entries, no squarings (b1 is then ignored)
};

template <int TPI>
constexpr int exp2_smem_words = 64 + (32 / TPI) * (16 * 64 + 64 + GPAD + sqr_scratch_words<TPI>);

template <int TPI>
MP_DEV void exp_window4(uint32_t (&acc)[Cfg<TPI>::L], const uint32_t* base64, const uint32_t* e, uint32_t windows,
                        uint32_t* tbl, uint32_t* sq, const SqrCtx& sc, const uint32_t* r2, const uint32_t* consts,
                        const Mod<Cfg<TPI>::L>& M, const Lane& ln) {
  constexpr int L = Cfg<TPI>::L;
  uint32_t x[L];
  // tbl[0] = one, tbl[1] = base in Montgomery form, tbl[i] = tbl[i-1] * base
  load_slice<TPI>(x, consts + C_ONE, ln);
  stage_shared<TPI>(tbl, x, ln);
  load_slice<TPI>(x, base64, ln);
  mont_mul<TPI>(x, x, r2, M, ln);
  stage_shared<TPI>(tbl + 64, x, ln);
  simt::syncwarp();
  for (int i = 2; i < 16; ++i) {
    mont_mul<TPI>(x, x, tbl + 64, M, ln);
    stage_shared<TPI>(tbl + i * 64, x, ln);
    simt::syncwarp();
  }
  uint32_t wi = windows - 1;
  uint32_t d = (e[wi >> 3] >> ((wi & 7u) * 4)) & 15u;
  load_slice<TPI>(acc, tbl + d * 64, ln);
  while (wi-- > 0) {
#pragma unroll 1
    for (int rep = 0; rep < 4; ++rep) sqr_inplace<TPI>(acc, sq, sc, M, ln);  // one code instance
    d = (e[wi >> 3] >> ((wi & 7u) * 4)) & 15u;
    mont_mul<TPI>(acc, acc, tbl + d * 64, M, ln);
  }
}

// Fixed-base exponentiation from a precomputed table: tbl[(w * 256 + d) * 64] = base^(d * 2^(8w)) in
// Montgomery form (d = 0: Montgomery one), so base^e = prod_w tbl[w][byte_w(e)].  Entries are staged
// through shared memory so that the Montgomery product reads its operand from there.
template <int TPI>
MP_DEV void exp_comb8(uint32_t (&acc)[Cfg<TPI>::L], const uint32_t* tbl, const uint32_t* e, uint32_t nbytes,
                      uint32_t* sq, const Mod<Cfg<TPI>::L>& M, const Lane& ln) {
  constexpr int L = Cfg<TPI>::L;
  uint32_t d = e[0] & 0xffu;
  load_slice<TPI>(acc, tbl + (size_t)d * 64, ln);
  for (uint32_t w = 1; w < nbytes; ++w) {
    d = (e[w >> 2] >> ((w & 3u) * 8)) & 0xffu;
    uint32_t x[L];
    load_slice<TPI>(x, tbl + ((size_t)w * 256 + d) * 64, ln);
    stage_shared<TPI>(sq, x, ln);
    simt::syncwarp();
    mont_mul<TPI>(acc, acc, sq, M, ln);
  }
}

// Table construction.  Step 1 (one lane group): tbl[w][1] = base^(2^(8w)) for w = 0..255.
struct CombArgs {
  const uint32_t* consts;
  const uint32_t* base;  // 64 limbs, normal form
  uint32_t* tbl;         // rows * 256 * 64 limbs
  uint32_t rows;         // byte positions covered (256 for full 2048-bit exponents)
};
template <int TPI>
constexpr int comb_smem_words = 64 + (32 / TPI) * (128 + GPAD);

template <int TPI>
MP_DEV void comb1_body(const CombArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* r2 = wsm;
  uint32_t* sq = wsm + 64 + gi * (128 + GPAD);
  warp_copy64(r2, A.consts + C_R2);
  simt::syncwarp();
  uint32_t b[L];
  load_slice<TPI>(b, A.base, ln);
  mont_mul<TPI>(b, b, r2, M, ln);
  for (uint32_t w = 0; w < A.rows; ++w) {
    if (wg == 0 && gi == 0) stage<TPI>(A.tbl + ((size_t)w * 256 + 1) * 64, b, ln);
    for (int k = 0; k < 8; ++k) sqr_plain<TPI>(b, sq, M, ln);
  }
}
// Step 2 (lane group w): tbl[w][0] = one, tbl[w][d] = tbl[w][d-1] * tbl[w][1].
template <int TPI>
MP_DEV void comb2_body(const CombArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  uint32_t w = wg * GPW + gi;
  const bool live = w < A.rows;
  if (!live) w = A.rows - 1;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* b1 = wsm + 64 + gi * (128 + GPAD);
  uint32_t* row = A.tbl + (size_t)w * 256 * 64;
  uint32_t x[L];
  load_slice<TPI>(x, A.consts + C_ONE, ln);
  if (live) stage<TPI>(row, x, ln);
  load_slice<TPI>(x, row + 64, ln);
  stage_shared<TPI>(b1, x, ln);
  simt::syncwarp();
  for (uint32_t d = 2; d < 256; ++d) {
    mont_mul<TPI>(x, x, b1, M, ln);
    if (live) stage<TPI>(row + (size_t)d * 64, x, ln);
  }
}

// out_i = b1_i^e1_i [* b2_i^e2_i]  (fixed 4-bit windows; the window count is a launch
// parameter, so every group of every warp runs the same schedule).
template <int TPI>
MP_DEV void exp2_body(const Exp2Args& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  uint32_t inst = wg * GPW + gi;
  const bool live = inst < A.n;
  if (!live) inst = A.n - 1;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* r2 = wsm;
  uint32_t* tbl = wsm + 64 + gi * (16 * 64 + 64 + GPAD + sqr_scratch_words<TPI>);
  uint32_t* sq = tbl + 16 * 64;
  const SqrCtx sc = make_sqr_ctx<TPI>(sq + 64, ln);
  warp_copy64(r2, A.consts + C_R2);
  simt::syncwarp();
  uint32_t acc[L];
  if (A.comb1)
    exp_comb8<TPI>(acc, A.comb1, A.e1 + (size_t)inst * A.e1_stride, (A.e1_windows + 1) / 2, sq, M, ln);
  else
    exp_window4<TPI>(acc, A.b1 + (size_t)inst * A.b1_stride, A.e1 + (size_t)inst * A.e1_stride, A.e1_windows, tbl,
                     sq, sc, r2, A.consts, M, ln);
  if (A.b2 != nullptr) {
    uint32_t acc2[L];
    exp_window4<TPI>(acc2, A.b2 + (size_t)inst * A.b2_stride, A.e2 + (size_t)inst * A.e2_stride, A.e2_windows, tbl,
                     sq, sc, r2, A.consts, M, ln);
    stage_shared<TPI>(sq, acc2, ln);
    simt::syncwarp();
    mont_mul<TPI>(acc, acc, sq, M, ln);
  }
  finish_store<TPI>(acc, sq, A.out + (size_t)inst * 64, live, M, ln);
}

// ------------------------------------------------------- transcript frames ----
// Row j of the Fiat-Shamir transcript (dleq.rs:58-61, 87-99; participant.rs:238-245, 438-447):
//   F(X_j) F(Y_j) F(a1_j) F(a2_j),  F(e) = len_u64_be || minimal big-endian bytes (modp.rs:150-152),
// each frame left-aligned in a slot of 8 + 256 bytes (zero padded), so that the host hashes the
// device's bytes as they are.  One thread per frame; zero encodes as the single byte 00.
struct FrameArgs {
  const uint32_t *x, *y, *a1, *a2;  // n canonical values each, 64 little-endian limbs
  uint8_t* out;                     // n rows of 4 * FRAME_BYTES
  uint32_t n;
};
constexpr int FRAME_BYTES = 8 + 256;

MP_DEV void frame_body(const FrameArgs& A, uint32_t tid) {
  const uint32_t j = tid >> 2, e = tid & 3u;
  if (j >= A.n) return;
  const uint32_t* src = (e == 0 ? A.x : e == 1 ? A.y : e == 2 ? A.a1 : A.a2) + (size_t)j * 64;
  uint8_t* dst = A.out + ((size_t)j * 4 + e) * FRAME_BYTES;
  int top = 63;
  while (top > 0 && src[top] == 0) --top;
  const uint32_t w = src[top];
  const uint32_t len = (uint32_t)top * 4 + ((w >> 24) ? 4u : (w >> 16) ? 3u : (w >> 8) ? 2u : 1u);
  uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);  // frames are 8-byte aligned
  d32[0] = 0;
  d32[1] = ((len & 0xffu) << 24) | ((len >> 8) << 16);  // bytes 6, 7 = big-endian length
  if (len == 256) {
#pragma unroll 8
    for (int k = 0; k < 64; ++k) {
      const uint32_t v = src[63 - k];
      d32[2 + k] = (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24);
    }
  } else {
    for (uint32_t k = 0; k < 256; ++k) {
      const uint32_t b = len - 1 - k;  // little-endian byte index; wraps above len
      dst[8 + k] = k < len ? (uint8_t)(src[b >> 2] >> ((b & 3u) * 8)) : (uint8_t)0;
    }
  }
}

// ------------------------------------------------- P(i) mod order (scalars) ----
// p_i = P(pos_i) mod order by Horner on plain integers, one position per thread, the 2048-bit
// accumulator in registers (polynomial.rs:50-58 reduced as participant.rs:202 does).  The order q-1 is
// even, so no Montgomery form: since its top limb is all ones, the part of acc*x + a_j above 2^2048
// (at most x) is folded back with delta = 2^2048 - order, twice, and one conditional subtraction at the
// end gives the canonical value.  Requires order >= 2^2048 - 2^2016 (checked by the host).
struct PolyArgs {
  const uint32_t* coeffs;  // t x 64 limbs
  const uint32_t* order;   // 64 limbs
  const uint32_t* pos;     // n positions (< 2^31)
  uint32_t* out;           // n x 64 limbs
  uint32_t t, n;
};
MP_DEV void poly_body(const PolyArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  const uint64_t x = A.pos[tid];
  uint32_t acc[64], delta[64];
  {
    uint64_t br = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      uint64_t d = (uint64_t)0 - A.order[i] - br;
      delta[i] = (uint32_t)d;
      br = (d >> 32) & 1u;
      acc[i] = 0;
    }
  }
#pragma unroll 1
  for (int j = (int)A.t - 1; j >= 0; --j) {
    const uint32_t* a = A.coeffs + (size_t)j * 64;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      c += (uint64_t)acc[i] * x + a[i];
      acc[i] = (uint32_t)c;
      c >>= 32;
    }
    // c <= x: fold c * 2^2048 = c * delta (mod order)
    uint64_t top = c, cc = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      cc += top * delta[i] + acc[i];
      acc[i] = (uint32_t)cc;
      cc >>= 32;
    }
    // at most one more wrap
    uint32_t m = 0u - (uint32_t)cc;
    uint64_t c2 = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      c2 += (uint64_t)acc[i] + (delta[i] & m);
      acc[i] = (uint32_t)c2;
      c2 >>= 32;
    }
  }
  // canonical: subtract the order once if acc >= order
  uint32_t r[64];
  uint64_t br = 0;
#pragma unroll
  for (int i = 0; i < 64; ++i) {
    uint64_t d = (uint64_t)acc[i] - A.order[i] - br;
    r[i] = (uint32_t)d;
    br = (d >> 32) & 1u;
  }
#pragma unroll
  for (int i = 0; i < 64; ++i) A.out[(size_t)tid * 64 + i] = br ? acc[i] : r[i];
}

// ------------------------------------------------- DLEQ responses (scalars) ----
// r_i = (w_i - (alpha_i * c mod order)) mod order  (dleq.rs:42-50 through modp.rs:180-192; call sites
// participant.rs:255-264, 342-347): alpha_i < order, the challenge c < 2^256, w_i < 2^2048.  One instance
// per thread on plain integers.  The order q-1 is even (no Montgomery form); its two top limbs are all
// ones, so the limbs of alpha*c above 2^2048 are folded back with delta = 2^2048 - order < 2^1984, which
// shortens the overflow by at least one limb per pass.
struct RespArgs {
  const uint32_t* order;  // 64 limbs
  const uint32_t* alpha;  // n x 64 limbs (stride alpha_stride; 0 = shared)
  const uint32_t* w;      // n x 64 limbs
  const uint32_t* c;      // challenge(s), 64 limbs each, only the low 8 are read (stride c_stride; 0 = shared)
  uint32_t* out;          // n x 64 limbs
  uint32_t n, alpha_stride, c_stride;
};
MP_DEV void resp_body(const RespArgs& A, uint32_t tid) {
  if (tid >= A.n) return;
  const uint32_t* al = A.alpha + (size_t)tid * A.alpha_stride;
  const uint32_t* cc = A.c + (size_t)tid * A.c_stride;
  uint32_t prod[72], delta[62];
  {
    uint64_t br = 0;
    for (int i = 0; i < 62; ++i) {
      uint64_t d = (uint64_t)0 - A.order[i] - br;
      delta[i] = (uint32_t)d;
      br = (d >> 32) & 1u;
    }
  }
  for (int i = 0; i < 72; ++i) prod[i] = 0;
  for (int j = 0; j < 8; ++j) {  // prod = alpha * c
    const uint64_t cj = cc[j];
    uint64_t carry = 0;
    for (int i = 0; i < 64; ++i) {
      carry += (uint64_t)al[i] * cj + prod[i + j];
      prod[i + j] = (uint32_t)carry;
      carry >>= 32;
    }
    prod[64 + j] = (uint32_t)carry;
  }
  for (int pass = 0; pass < 9; ++pass) {  // prod = lo + hi * delta until hi = 0
    uint32_t hi[8], any = 0;
    for (int j = 0; j < 8; ++j) {
      hi[j] = prod[64 + j];
      any |= hi[j];
      prod[64 + j] = 0;
    }
    if (!any) break;
    for (int j = 0; j < 8; ++j) {
      const uint64_t hj = hi[j];
      uint64_t carry = 0;
      for (int i = 0; i < 62; ++i) {
        carry += (uint64_t)delta[i] * hj + prod[i + j];
        prod[i + j] = (uint32_t)carry;
        carry >>= 32;
      }
      for (int i = 62 + j; carry && i < 72; ++i) {
        carry += prod[i];
        prod[i] = (uint32_t)carry;
        carry >>= 32;
      }
    }
  }
  // prod < 2^2048 now; bring it below the order, then r = w - prod (+ order if negative), reduced
  uint32_t r[64];
  auto sub_order = [&](uint32_t* v) {  // v -= order if v >= order
    uint32_t t[64];
    uint64_t br = 0;
    for (int i = 0; i < 64; ++i) {
      uint64_t d = (uint64_t)v[i] - A.order[i] - br;
      t[i] = (uint32_t)d;
      br = (d >> 32) & 1u;
    }
    if (!br)
      for (int i = 0; i < 64; ++i) v[i] = t[i];
  };
  sub_order(prod);
  const uint32_t* w = A.w + (size_t)tid * 64;
  uint64_t br = 0;
  for (int i = 0; i < 64; ++i) {
    uint64_t d = (uint64_t)w[i] - prod[i] - br;
    r[i] = (uint32_t)d;
    br = (d >> 32) & 1u;
  }
  if (br) {  // negative: add the order once (modp.rs:186-188)
    uint64_t c2 = 0;
    for (int i = 0; i < 64; ++i) {
      c2 += (uint64_t)r[i] + A.order[i];
      r[i] = (uint32_t)c2;
      c2 >>= 32;
    }
  } else {
    sub_order(r);  // w may exceed the order: "% order"
    sub_order(r);
  }
  for (int i = 0; i < 64; ++i) A.out[(size_t)tid * 64 + i] = r[i];
}

// ------------------------------------------------- Lagrange numerators / denominators ----
// For position x_i among k positions: num_i = prod_{j != i} x_j and den_i = prod_{j != i} |x_j - x_i|,
// both modulo the order q-1 (a multiple of the subgroup order g the coefficients live in, so the host /
// the exponentiation kernel may reduce further), and the sign of prod (x_j - x_i)
// (util.rs:47-64 + participant.rs:535-541).  One position per thread, same lazy reduction as poly_body.
// The products are cut into `parts` contiguous ranges of j and numerator / denominator run in separate threads
// (2 * parts * k threads: one thread per position did 2 k dependent 2048 x 32-bit products, 13 ms at k = 2731 on
// 86 warps); part p of position i lands in row p * k + i, the host multiplies the parts mod g with the product
// kernel and XORs the partial signs.
struct LagrangeArgs {
  const uint32_t* order;  // 64 limbs, all-ones top limb
  const uint32_t* pos;    // k positions
  uint32_t* num;          // parts x k x 64 limbs
  uint32_t* den;          // parts x k x 64 limbs
  uint32_t* negative;     // parts x k flags (partial signs)
  uint32_t k, parts;
};
MP_DEV void lagrange_product(uint32_t* out64, const LagrangeArgs& A, uint32_t tid, bool denominator, uint32_t* neg,
                             uint32_t j0, uint32_t j1) {
  const uint32_t xi = A.pos[tid];
  uint32_t acc[64], delta[64];
  {
    uint64_t br = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      uint64_t d = (uint64_t)0 - A.order[i] - br;
      delta[i] = (uint32_t)d;
      br = (d >> 32) & 1u;
      acc[i] = 0;
    }
    acc[0] = 1;
  }
  uint32_t sign = 0;
#pragma unroll 1
  for (uint32_t j = j0; j < j1; ++j) {
    if (j == tid) continue;
    const uint32_t xj = A.pos[j];
    uint64_t f = xj;
    if (denominator) {
      if (xj < xi) {
        sign ^= 1u;
        f = xi - xj;
      } else {
        f = xj - xi;
      }
    }
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      c += (uint64_t)acc[i] * f;
      acc[i] = (uint32_t)c;
      c >>= 32;
    }
    uint64_t top = c, cc = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      cc += top * delta[i] + acc[i];
      acc[i] = (uint32_t)cc;
      cc >>= 32;
    }
    uint32_t m = 0u - (uint32_t)cc;
    uint64_t c2 = 0;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
      c2 += (uint64_t)acc[i] + (delta[i] & m);
      acc[i] = (uint32_t)c2;
      c2 >>= 32;
    }
  }
  uint64_t br = 0;
  uint32_t r[64];
#pragma unroll
  for (int i = 0; i < 64; ++i) {
    uint64_t d = (uint64_t)acc[i] - A.order[i] - br;
    r[i] = (uint32_t)d;
    br = (d >> 32) & 1u;
  }
#pragma unroll
  for (int i = 0; i < 64; ++i) out64[i] = br ? acc[i] : r[i];
  if (neg) *neg = sign;
}
MP_DEV void lagrange_body(const LagrangeArgs& A, uint32_t tid) {
  const uint32_t P = A.parts ? A.parts : 1u;
  if (tid >= 2u * P * A.k) return;
  const bool denominator = tid >= P * A.k;
  const uint32_t row = denominator ? tid - P * A.k : tid, part = row / A.k, i = row % A.k;
  const uint32_t per = (A.k + P - 1) / P, j0 = part * per, j1 = j0 + per < A.k ? j0 + per : A.k;
  lagrange_product((denominator ? A.den : A.num) + (size_t)row * 64, A, i, denominator,
                   denominator ? A.negative + row : nullptr, j0 < A.k ? j0 : A.k, j1);
}

// Several boxes at once (mpvss_reconstruct_secrets): the positions of the boxes are concatenated, and position i
// belongs to the box of k_b = bk[i] positions that starts at boff[i].  Each product runs over that box only, cut
// into `parts` ranges of the box as lagrange_body cuts its k positions; part p of position i lands in row
// p * n + i.
struct LagrangeBoxesArgs {
  const uint32_t* order;  // 64 limbs, all-ones top limb
  const uint32_t* pos;    // n positions, concatenated over the boxes
  const uint32_t* boff;   // per position: first position of its box
  const uint32_t* bk;     // per position: positions k_b of its box
  uint32_t* num;          // parts x n x 64 limbs
  uint32_t* den;          // parts x n x 64 limbs
  uint32_t* negative;     // parts x n flags (partial signs)
  uint32_t n, parts;
};
MP_DEV void lagrange_boxes_body(const LagrangeBoxesArgs& A, uint32_t tid) {
  const uint32_t P = A.parts ? A.parts : 1u;
  if (tid >= 2u * P * A.n) return;
  const bool denominator = tid >= P * A.n;
  const uint32_t row = denominator ? tid - P * A.n : tid, part = row / A.n, i = row % A.n;
  const uint32_t off = A.boff[i], k = A.bk[i];
  const uint32_t per = (k + P - 1) / P, j0 = part * per, j1 = j0 + per < k ? j0 + per : k;
  const LagrangeArgs box{A.order, A.pos + off, nullptr, nullptr, nullptr, k, P};
  lagrange_product((denominator ? A.den : A.num) + (size_t)row * 64, box, i - off, denominator,
                   denominator ? A.negative + row : nullptr, j0 < k ? j0 : k, j1);
}

// --------------------------------------------- bucket multi-exponentiation ----
// prod_i S_i^(e_i) for k distinct bases and unstructured full-width exponents (the reconstruct fold,
// participant.rs:490-509, and Group-level multi_exp): Pippenger's bucket method with 8-bit windows.
//   1. the host sorts, per window w, the indices i by the byte e_i[w] (counting sort);
//   2. msm_bucket_body: one lane group per (w, d), d = 1..255: B[w][d] = prod of the bases in that bucket;
//   3. msm_window_body: one warp per window: W_w = prod_d B[w][d]^d by running products, the 255 buckets
//      cut into one segment per lane group (depth 2 * 256 / groups + ~12 instead of 510 products);
//   4. msm_fold_body: result = prod_w W_w^(2^(8w)), Horner from the top window (8 squarings + 1 product
//      per window: the 2040 sequential squarings no method can avoid for a fresh base).
// Work: windows * (k + ~600) products instead of k * (4 * windows + ...) for one exponentiation per base.
struct MsmBucketArgs {
  const uint32_t* consts;
  const uint32_t* bases;   // k values, Montgomery form
  const uint32_t* idx;     // windows * k indices, window-major, sorted by digit
  const uint32_t* start;   // windows * 257 bucket boundaries inside each window's index list
  uint32_t* buckets;       // windows * 256 values (entry d = 0 unused), Montgomery form
  uint32_t windows, k;
};
template <int TPI>
constexpr int msm_smem_words = (32 / TPI) * (2 * 64 + GPAD);

template <int TPI>
MP_DEV void msm_bucket_body(const MsmBucketArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  const uint32_t total = A.windows * 255u;
  uint32_t id = wg * GPW + gi;
  const bool live = id < total;
  if (!live) id = total - 1;
  const uint32_t w = id / 255u, d = id % 255u + 1u;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* stage_buf = wsm + gi * (2 * 64 + GPAD);
  uint32_t* one = stage_buf + 64;
  uint32_t acc[L], x[L];
  load_slice<TPI>(acc, A.consts + C_ONE, ln);
  stage_shared<TPI>(one, acc, ln);
  const uint32_t lo = A.start[w * 257u + d], hi = A.start[w * 257u + d + 1];
  uint32_t cnt = live ? hi - lo : 0u, mx = cnt;
  for (int off = 16; off >= 1; off >>= 1) {  // longest bucket of the warp: every group runs that many products
    uint32_t o = simt::shfl(mx, (int)simt::lane_id() ^ off);
    mx = o > mx ? o : mx;
  }
  simt::syncwarp();
  for (uint32_t j = 0; j < mx; ++j) {
    const bool have = j < cnt;
    if (have) load_slice<TPI>(x, A.bases + (size_t)A.idx[(size_t)w * A.k + lo + j] * 64, ln);
    simt::syncwarp();
    if (have) stage<TPI>(stage_buf, x, ln);
    simt::syncwarp();
    mont_mul<TPI>(acc, acc, have ? stage_buf : one, M, ln);
  }
  if (live) stage<TPI>(A.buckets + ((size_t)w * 256 + d) * 64, acc, ln);
}

struct MsmWindowArgs {
  const uint32_t* consts;
  const uint32_t* buckets;  // windows * 256 values (Montgomery)
  uint32_t* wprod;          // windows values (Montgomery): W_w
  uint32_t windows;
};
template <int TPI>
constexpr int msm_window_smem_words = (32 / TPI) * (4 * 64 + GPAD);

// one warp per window; lane group s owns the buckets d = s*SEG+1 .. s*SEG+SEG (SEG = 256 / groups; d = 256 does
// not exist and counts as one):  W = prod_s A_s * (R_s^SEG)^s,  A_s = prod_d B_d^(d - s*SEG),  R_s = prod_d B_d
template <int TPI>
MP_DEV void msm_window_body(const MsmWindowArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  constexpr uint32_t SEG = 256 / GPW;
  Lane ln = make_lane<TPI>();
  const uint32_t gi = simt::lane_id() / TPI;
  const uint32_t w = wg < A.windows ? wg : A.windows - 1;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* buf = wsm + gi * (4 * 64 + GPAD);  // [0] operand stage, [1] run, [2] scratch, [3] result exchange
  uint32_t run[L], acc[L], x[L];
  load_slice<TPI>(run, A.consts + C_ONE, ln);
  load_slice<TPI>(acc, A.consts + C_ONE, ln);
  simt::syncwarp();
  for (uint32_t d = SEG; d >= 1; --d) {  // running products from the top of the segment
    const uint32_t b = gi * SEG + d;
    load_slice<TPI>(x, b < 256u ? A.buckets + ((size_t)w * 256 + b) * 64 : A.consts + C_ONE, ln);
    stage_shared<TPI>(buf, x, ln);
    simt::syncwarp();
    mont_mul<TPI>(run, run, buf, M, ln);
    stage_shared<TPI>(buf + 64, run, ln);
    simt::syncwarp();
    mont_mul<TPI>(acc, acc, buf + 64, M, ln);
  }
  // run = R_s, acc = A_s.  y = R_s^SEG (log2 SEG squarings), then y^s by s - 1 products (s < groups <= 8)
  uint32_t y[L];
#pragma unroll
  for (int i = 0; i < L; ++i) y[i] = run[i];
  for (uint32_t q = SEG; q > 1; q >>= 1) sqr_plain<TPI>(y, buf, M, ln);
  stage_shared<TPI>(buf + 128, y, ln);  // y
  load_slice<TPI>(x, A.consts + C_ONE, ln);
  stage_shared<TPI>(buf + 64, x, ln);   // one
  simt::syncwarp();
  for (uint32_t e = 0; e < (uint32_t)GPW - 1; ++e)  // acc *= y while e < s, else * one (same schedule for all groups)
    mont_mul<TPI>(acc, acc, e < gi ? buf + 128 : buf + 64, M, ln);
  // product over the groups of the warp through shared memory
  stage_shared<TPI>(buf + 192, acc, ln);
  simt::syncwarp();
  load_slice<TPI>(acc, wsm + 192, ln);  // group 0's value
  for (uint32_t s = 1; s < (uint32_t)GPW; ++s) mont_mul<TPI>(acc, acc, wsm + s * (4 * 64 + GPAD) + 192, M, ln);
  if (wg < A.windows && gi == 0) stage<TPI>(A.wprod + (size_t)w * 64, acc, ln);
}

struct MsmFoldArgs {
  const uint32_t* consts;
  const uint32_t* wprod;  // windows values (Montgomery)
  uint32_t* out;          // 1 value, canonical
  uint32_t windows;
};
template <int TPI>
MP_DEV void msm_fold_body(const MsmFoldArgs& A, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  Lane ln = make_lane<TPI>();
  const uint32_t gi = simt::lane_id() / TPI;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* buf = wsm + gi * (2 * 64 + GPAD);  // every group computes the same value (one warp in all)
  uint32_t acc[L], x[L];
  load_slice<TPI>(acc, A.wprod + (size_t)(A.windows - 1) * 64, ln);
  simt::syncwarp();
  for (int w = (int)A.windows - 2; w >= 0; --w) {
#pragma unroll 1
    for (int r = 0; r < 8; ++r) sqr_plain<TPI>(acc, buf, M, ln);
    load_slice<TPI>(x, A.wprod + (size_t)w * 64, ln);
    stage_shared<TPI>(buf, x, ln);
    simt::syncwarp();
    mont_mul<TPI>(acc, acc, buf, M, ln);
  }
  finish_store<TPI>(acc, buf, A.out, gi == 0, M, ln);
}

// ------------------------------------------------------- element-wise mul ----
struct MulArgs {
  const uint32_t* consts;
  const uint32_t* a;   // n values
  const uint32_t* b;   // n values, or nullptr
  uint32_t* out;
  uint32_t n;
  uint32_t mode;       // 0: out = a*b mod q (canonical)   1: out = a*R mod q (to Montgomery form)
                       // 2: out = a*a/R mod q, a taken as is (any value below 2^2048; squaring test)
                       // 3: as 0, second product through mont_mul_il (split accumulators; test)
  uint32_t a_stride, b_stride;
};

template <int TPI>
constexpr int mul_smem_words = 64 + (32 / TPI) * (64 + GPAD);

template <int TPI>
MP_DEV void mul_body(const MulArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  uint32_t inst = wg * GPW + gi;
  const bool live = inst < A.n;
  if (!live) inst = A.n - 1;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* r2 = wsm;
  uint32_t* sq = wsm + 64 + gi * (64 + GPAD);
  warp_copy64(r2, A.consts + C_R2);
  simt::syncwarp();
  uint32_t acc[L];
  load_slice<TPI>(acc, A.a + (size_t)inst * A.a_stride, ln);
  if (A.mode == 2) {
    stage_shared<TPI>(sq, acc, ln);
    simt::syncwarp();
    mont_sqr<TPI>(acc, acc, sq, M, ln);
  } else {
    mont_mul<TPI>(acc, acc, r2, M, ln);  // a*R
  }
  if (A.mode == 0 || A.mode == 3) {
    uint32_t y[L];
    load_slice<TPI>(y, A.b + (size_t)inst * A.b_stride, ln);
    stage_shared<TPI>(sq, y, ln);
    simt::syncwarp();
    if (A.mode == 3)
      mont_mul_il<TPI>(acc, acc, sq, M, ln);  // split-accumulator product (test entry)
    else
      mont_mul<TPI>(acc, acc, sq, M, ln);  // a*R*b/R = a*b
  }
  canonical<TPI>(acc, M, ln);
  if (live) stage<TPI>(A.out + (size_t)inst * 64, acc, ln);
}

// ------------------------------------------------ gathered products (segmented tree) ----
// v[rows[3i + 2]] = v[rows[3i]] * v[rows[3i + 1]] mod q (canonical) for n host-planned row triples.  A level of
// product_tree_level writes each product over its first factor and no row is read by one triple and written by
// another, so the level runs in place.
struct MulRowsArgs {
  const uint32_t* consts;
  uint32_t* v;           // values, 64 limbs each
  const uint32_t* rows;  // n x (a, b, out)
  uint32_t n;
};

template <int TPI>
MP_DEV void mul_rows_body(const MulRowsArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int L = Cfg<TPI>::L;
  constexpr int GPW = 32 / TPI;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  uint32_t inst = wg * GPW + gi;
  const bool live = inst < A.n;
  if (!live) inst = A.n - 1;
  const uint32_t* t = A.rows + (size_t)inst * 3;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* r2 = wsm;
  uint32_t* sq = wsm + 64 + gi * (64 + GPAD);
  warp_copy64(r2, A.consts + C_R2);
  simt::syncwarp();
  uint32_t acc[L], y[L];
  load_slice<TPI>(acc, A.v + (size_t)t[0] * 64, ln);
  load_slice<TPI>(y, A.v + (size_t)t[1] * 64, ln);
  mont_mul<TPI>(acc, acc, r2, M, ln);  // a*R
  stage_shared<TPI>(sq, y, ln);
  simt::syncwarp();
  mont_mul<TPI>(acc, acc, sq, M, ln);  // a*R*b/R = a*b
  canonical<TPI>(acc, M, ln);
  if (live) stage<TPI>(A.v + (size_t)t[2] * 64, acc, ln);
}

// One level of the segmented product tree (host planning, shared with the tests): segment s holds cnt[s] values
// from row start[s].  Its first cnt / 2 rows are multiplied by the rows h = ceil(cnt / 2) further on, in place,
// and cnt becomes h; an odd middle row stays where it is.  Writes the level's (a, b, out) triples to `rows` and
// returns their number (0 once every segment is down to its product, at row start[s]).
inline uint32_t product_tree_level(const uint32_t* start, uint32_t* cnt, uint32_t segments, uint32_t* rows) {
  uint32_t m = 0;
  for (uint32_t s = 0; s < segments; ++s) {
    const uint32_t c = cnt[s], h = (c + 1) / 2;
    for (uint32_t i = 0; i < c / 2; ++i) {
      rows[3 * m] = start[s] + i;
      rows[3 * m + 1] = start[s] + i + h;
      rows[3 * m + 2] = start[s] + i;
      ++m;
    }
    cnt[s] = h;
  }
  return m;
}

// ---- split squaring, test entry (TPI = 8): out = a*a/R mod q, a taken as is ----
constexpr int sqrtest_smem_words = 64 + 4 * (64 + SQS_WORDS);
MP_DEV void sqr_split_test_body(const MulArgs& A, uint32_t wg, uint32_t* wsm) {
  constexpr int TPI = 8, L = 8, GPW = 4;
  Lane ln = make_lane<TPI>();
  const int gi = (int)simt::lane_id() / TPI;
  uint32_t inst = wg * GPW + gi;
  const bool live = inst < A.n;
  if (!live) inst = A.n - 1;
  Mod<L> M;
  load_mod<TPI>(M, A.consts, ln);
  uint32_t* sq = wsm + 64 + gi * (64 + SQS_WORDS);
  uint32_t* scratch = sq + 64;
  scratch[SQS_ZERO + ln.k] = 0;
  const SqPlan pl = make_sq_plan(ln.k);
  uint32_t acc[L];
  load_slice<TPI>(acc, A.a + (size_t)inst * A.a_stride, ln);
  for (uint32_t rep = 0; rep < (A.mode ? A.mode : 1u); ++rep) {  // mode = number of squarings in a row
    stage_shared<TPI>(sq, acc, ln);
    simt::syncwarp();
    mont_sqr_split(acc, acc, sq, scratch, pl, M, ln);
  }
  canonical<TPI>(acc, M, ln);
  if (live) stage<TPI>(A.out + (size_t)inst * 64, acc, ln);
}

}  // namespace modp
