// ModpGroup side of the C ABI: host orchestration of the CUDA kernels plus the
// CPU-resident pieces north_star keeps on the host (Fiat-Shamir SHA-256 over
// identically serialised values, scalar arithmetic mod q-1 / g).
//
// Reference semantics restated here (paths under /root/reference/src):
//   transcript framing            dleq.rs:58-61, 87-99
//   challenge = hash_to_scalar(H) participant.rs:251-252, modp.rs:142-148
//   minimal big-endian bytes      modp.rs:150-152
//   responses                     participant.rs:255-264, modp.rs:180-192
//   U mask                        participant.rs:267-272, 512-518
//   Lagrange exponents            participant.rs:526-561, util.rs:47-64
#include <algorithm>
#include <cstdlib>
#include "host_common.h"
#include "modp_chain.h"
#include "modp_launch.h"
#include "sha2.h"
#include "hash_launch.h"
#include "transcript.h"

namespace {

constexpr size_t EB = 256;  // element / scalar bytes at the boundary
constexpr size_t EW = 64;   // u32 limbs

const char* RFC3526_2048 =
    "ffffffffffffffffc90fdaa22168c234c4c6628b80dc1cd129024e088a67cc74"
    "020bbea63b139b22514a08798e3404ddef9519b3cd3a431b302b0a6df25f1437"
    "4fe1356d6d51c245e485b576625e7ec6f44c42e9a637ed6b0bff5cb6f406b7ed"
    "ee386bfb5a899fa5ae9f24117c4b1fe649286651ece45b3dc2007cb8a163bf05"
    "98da48361c55d39a69163fa8fd24cf5f83655d23dca3ad961c62f356208552bb"
    "9ed529077096966d670c354e4abc9804f1746c08ca18217c32905e462e36ce3b"
    "e39e772c180e86039b2783a2ec07a28fb5c55df06f4c52c9de2bcbf695581718"
    "3995497cea956ae515d2261898fa051015728e5a8aacaa68ffffffffffffffff";

void fill_consts(const big::Int& m, uint32_t* blk) {
  memset(blk, 0, modp::C_WORDS * 4);
  big::Int R(65, 0);
  R[64] = 1;
  big::Int nq = big::sub(R, m), one = big::mod(R, m), r2 = big::mulmod(one, one, m);
  auto put = [&](const big::Int& v, int off) {
    for (size_t i = 0; i < v.size() && i < 64; ++i) blk[off + i] = v[i];
  };
  put(m, modp::C_Q);
  put(nq, modp::C_NQ);
  put(one, modp::C_ONE);
  put(r2, modp::C_R2);
  big::Int one1(1, 1);
  put(big::shr1(big::add(m, one1)), modp::C_QH);
  uint32_t inv = 1, m0 = m[0];  // Newton: inv = m0^-1 mod 2^32
  for (int i = 0; i < 5; ++i) inv *= 2u - m0 * inv;
  blk[modp::C_NP] = 0u - inv;
}

// minimal-length big-endian bytes of a 256-byte little-endian value (modp.rs:150-152)
size_t min_be(const uint8_t* le, uint8_t* out) {
  size_t len = EB;
  while (len > 1 && le[len - 1] == 0) --len;
  for (size_t i = 0; i < len; ++i) out[i] = le[len - 1 - i];
  return len;
}
// U mask of G^s (256-byte LE): int_be(SHA-256(minimal BE bytes)) mod q  (participant.rs:269-272, 512-518)
big::Int u_mask(const mpvss_ctx* ctx, const uint8_t* gs) {
  uint8_t tmp[EB], hs[32];
  sha2::sha256(tmp, min_be(gs, tmp), hs);
  return big::mod(big::from_be(hs, 32), ctx->q);
}
// U = secret XOR (int(SHA-256(bytes(G^s))) mod q) as element-size big-endian bytes; `secret` is a big-endian
// integer of len bytes (participant.rs:267-272)
void mask_secret(const mpvss_ctx* ctx, const uint8_t* secret, size_t len, const uint8_t* gs, uint8_t* u_out) {
  big::to_be(big::bxor(big::from_be(secret, len), u_mask(ctx, gs)), u_out, EB);
}
// the order q-1 as EW little-endian limbs (the scalar kernels' modulus)
std::vector<uint32_t> order_limbs(const mpvss_ctx* ctx) {
  std::vector<uint32_t> order(EW, 0);
  for (size_t i = 0; i < ctx->qm1.size(); ++i) order[i] = ctx->qm1[i];
  return order;
}
void framed_update(sha2::Sha256& h, const uint8_t* le) {  // dleq.rs:58-61
  uint8_t tmp[EB], len8[8] = {0};
  size_t len = min_be(le, tmp);
  len8[6] = (uint8_t)(len >> 8);
  len8[7] = (uint8_t)len;
  h.update(len8, 8);
  h.update(tmp, len);
}
// challenge = int_be(SHA-256(digest)) mod g, as a 256-byte LE scalar (modp.rs:142-148)
void challenge_from_digest(const mpvss_ctx* ctx, const uint8_t digest[32], uint8_t out[EB]) {
  uint8_t h2[32];
  sha2::sha256(digest, 32, h2);
  big::Int c = big::mod(big::from_be(h2, 32), ctx->g);
  big::to_le(c, out, EB);
}
uint32_t windows_for(const uint8_t* scalars, size_t stride, size_t n) {
  size_t top = 0;  // highest non-zero byte index + 1 over all scalars
  for (size_t i = 0; i < n; ++i) {
    const uint8_t* s = scalars + i * stride;
    size_t len = EB;
    while (len > top && s[len - 1] == 0) --len;
    if (len > top) top = len;
    if (top == EB) break;
  }
  uint32_t w = (uint32_t)(top * 2);
  return w ? w : 1;
}

// device-pointer exponentiation:  out = b1^e1 [* b2^e2]
int dev_exp2(mpvss_ctx* ctx, const uint32_t* consts, const uint32_t* b1, uint32_t b1s, const uint32_t* e1,
             uint32_t e1s, uint32_t e1w, const uint32_t* b2, uint32_t b2s, const uint32_t* e2, uint32_t e2s,
             uint32_t e2w, size_t n, uint32_t* out, cudaStream_t stream = nullptr, const uint32_t* comb1 = nullptr) {
  modp::Exp2Args A{consts, b1, e1, b2, e2, out, (uint32_t)n, b1s, e1s, e1w, b2s, e2s, e2w, comb1};
  if (ctx->exp2_filler_ctas)
    MPVSS_CUDA(ctx, modp::launch_exp2_filler(ctx->modp_tpi, A, ctx->exp2_filler_ctas, stream ? stream : ctx->stream));
  else
    MPVSS_CUDA(ctx, modp::launch_exp2(ctx->modp_tpi, A, stream ? stream : ctx->stream));
  timing_launch(ctx);
  return MPVSS_OK;
}
int dev_mul(mpvss_ctx* ctx, const uint32_t* consts, const uint32_t* a, uint32_t as, const uint32_t* b, uint32_t bs,
            uint32_t mode, size_t n, uint32_t* out) {
  modp::MulArgs A{consts, a, b, out, (uint32_t)n, mode, as, bs};
  MPVSS_CUDA(ctx, modp::launch_mul(ctx->modp_tpi, A, ctx->stream));
  timing_launch(ctx);
  return MPVSS_OK;
}

// fixed-base table of generator `which` (0: G = 2, 1: g = 4), built on first use; nullptr when disabled
int comb_table(mpvss_ctx* ctx, int which, const uint32_t** out) {
  *out = nullptr;
  if (!ctx->modp_comb) return MPVSS_OK;
  DevBuf& t = ctx->comb[which];
  if (!t.p) {
    MPVSS_CUDA(ctx, t.ensure((size_t)256 * 256 * EB));
    modp::CombArgs A{ctx->consts_q.as<uint32_t>(), ctx->gens.as<uint32_t>() + which * 64, t.as<uint32_t>(), 256};
    MPVSS_CUDA(ctx, modp::launch_comb_build(ctx->modp_tpi, A, ctx->stream));
    MPVSS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  *out = t.as<uint32_t>();
  return MPVSS_OK;
}

}  // namespace

namespace modp_api {

int init(mpvss_ctx* ctx) {
  ctx->q = from_hex(RFC3526_2048);
  ctx->qm1 = big::sub(ctx->q, big::from_u64(1));
  ctx->g = big::shr1(ctx->qm1);
  std::vector<uint32_t> blk(modp::C_WORDS);
  fill_consts(ctx->q, blk.data());
  ctx->modp_np1 = blk[modp::C_NP] == 1u;
  MPVSS_TRY(h2d(ctx, ctx->consts_q, blk.data(), blk.size() * 4));
  fill_consts(ctx->g, blk.data());
  MPVSS_TRY(h2d(ctx, ctx->consts_g, blk.data(), blk.size() * 4));
  std::vector<uint32_t> gens(192, 0);
  gens[0] = 2;    // Group::generator()           modp.rs:64
  gens[64] = 4;   // Group::subgroup_generator()  modp.rs:65-66
  gens[128] = 1;  // the scalar / element 1
  MPVSS_TRY(h2d(ctx, ctx->gens, gens.data(), gens.size() * 4));
  return sync(ctx);
}

int batch_exp(mpvss_ctx* ctx, const uint8_t* bases, size_t base_stride, const uint8_t* scalars, size_t n,
              uint8_t* out) {
  MPVSS_TRY(check_args(ctx, bases && scalars && out && n > 0 && (base_stride == 0 || base_stride == EB),
                       "batch_exp: bad arguments"));
  DevBuf &db = ctx->buf(0), &de = ctx->buf(1), &dout = ctx->buf(2);
  MPVSS_TRY(h2d(ctx, db, bases, base_stride ? n * EB : EB));
  MPVSS_TRY(h2d(ctx, de, scalars, n * EB));
  MPVSS_CUDA(ctx, dout.ensure(n * EB));
  timing_begin(ctx);
  MPVSS_TRY(dev_exp2(ctx, ctx->consts_q.as<uint32_t>(), db.as<uint32_t>(), base_stride ? EW : 0, de.as<uint32_t>(), EW,
                     windows_for(scalars, EB, n), nullptr, 0, nullptr, 0, 0, n, dout.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  MPVSS_TRY(d2h(ctx, out, dout, n * EB));
  return sync(ctx);
}

int fixed_base_exp(mpvss_ctx* ctx, int generator, const uint8_t* scalars, size_t n, uint8_t* out) {
  MPVSS_TRY(check_args(ctx, scalars && out && n > 0 && (generator == MPVSS_GEN_MAIN || generator == MPVSS_GEN_SUBGROUP),
                       "fixed_base_exp: bad arguments"));
  DevBuf &de = ctx->buf(1), &dout = ctx->buf(2);
  MPVSS_TRY(h2d(ctx, de, scalars, n * EB));
  MPVSS_CUDA(ctx, dout.ensure(n * EB));
  const uint32_t* comb;
  MPVSS_TRY(comb_table(ctx, generator ? 1 : 0, &comb));
  timing_begin(ctx);
  MPVSS_TRY(dev_exp2(ctx, ctx->consts_q.as<uint32_t>(), ctx->gens.as<uint32_t>() + (generator ? 64 : 0), 0,
                     de.as<uint32_t>(), EW, windows_for(scalars, EB, n), nullptr, 0, nullptr, 0, 0, n,
                     dout.as<uint32_t>(), nullptr, comb));
  MPVSS_TRY(timing_end(ctx));
  MPVSS_TRY(d2h(ctx, out, dout, n * EB));
  return sync(ctx);
}

int batch_mul(mpvss_ctx* ctx, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  MPVSS_TRY(check_args(ctx, a && b && out && n > 0, "batch_mul: bad arguments"));
  DevBuf &da = ctx->buf(0), &db = ctx->buf(1), &dout = ctx->buf(2);
  MPVSS_TRY(h2d(ctx, da, a, n * EB));
  MPVSS_TRY(h2d(ctx, db, b, n * EB));
  MPVSS_CUDA(ctx, dout.ensure(n * EB));
  timing_begin(ctx);
  MPVSS_TRY(dev_mul(ctx, ctx->consts_q.as<uint32_t>(), da.as<uint32_t>(), EW, db.as<uint32_t>(), EW, 0, n,
                    dout.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  MPVSS_TRY(d2h(ctx, out, dout, n * EB));
  return sync(ctx);
}

// Positions are sorted by their number of base-4 digits (longest first) and every digit class
// is padded to a whole number of CTAs, so all groups of a CTA run the same fixed-window
// schedule while one launch covers every class (a single large position no longer lengthens
// everybody's schedule, and the long chains start first).  The digit count is stored per CTA.
// With many positions per launch every scheduler holds enough warps to hide latencies, and 4 lanes per
// value (16 limbs per lane) spend the fewest instructions per MAC: measured 6.4 vs 5.7 TMAC/s at
// per launch of 32768 positions (Horner 2104 vs 2149 ms); at 16384 and below 8 lanes per value win.
static int horner_tpi(const mpvss_ctx* ctx, size_t n) {
  if (!ctx->modp_tpi_auto) return ctx->modp_tpi;
  if (n >= 32768) return 4;
  // few positions (a small box, or one box split over many GPUs): 16 lanes per value double the warps;
  // below 4 warps per SM at 8 lanes the launch is latency-bound and the extra warps pay
  if (n * 8 / 32 < (size_t)4 * (size_t)ctx->sm_count) return 16;
  return ctx->modp_tpi;
}

// warps per CTA of the Horner launch ("modp_wpc" tunable; default one warp per CTA)
static int horner_wpc(const mpvss_ctx* ctx, size_t n, int tpi) {
  if (ctx->modp_wpc) return ctx->modp_wpc;
  (void)n;
  (void)tpi;
  return 1;  // measured: 4 warps per CTA change nothing at 8 .. 16 warps per SM (tools/wpc_sweep.sh)
}

// Chunks per position.  With few positions the launch is a handful of warps per SM and every chain is
// latency-bound; cutting the polynomial into K contiguous chunks gives K times the lane groups with chains
// 1/K as long, at the price of one 2048-bit exponentiation per extra chunk for the combination
// X = prod_k H_k^(pos^(k B)) (6.5 % of a chain at t = 2731) -- free while the chip is mostly idle
// (one box split over many GPUs, small boxes).  "modp_chunks": 0 = automatic.
static uint32_t horner_chunks(const mpvss_ctx* ctx, size_t n, size_t t) {
  uint32_t K = 1;
  if (ctx->modp_chunks > 0) {
    K = (uint32_t)ctx->modp_chunks;
  } else {
    const size_t warps = (n + 3) / 4, full = (size_t)8 * (size_t)ctx->sm_count;  // two warps per scheduler
    while (K < 8 && warps * (K * 2) <= full) K *= 2;
  }
  // The combination is not free: measured (tools/chunk_sweep.sh) 9 / 13 / 26 ms for K = 2 / 4 / 8 at 1024
  // positions, against 2.3 us per sequential product of a chain.  At t = 683 every K > 1 loses
  // (35.4 -> 39.5 / 38.2 ms), at t = 2731 K = 4 wins 28 % at 1024 positions and K = 8 42 % at 512.
  if (ctx->modp_chunks <= 0 && t < 1366) K = 1;
  while (K > 1 && t / K < (ctx->modp_chunks > 0 ? 32u : 340u)) K /= 2;
  return K;
}

struct PosPlan {
  int tpi = 8;
  int wpc = 1;                  // warps per CTA of the Horner launch
  uint32_t K = 1, B = 0;        // chunks per position, coefficients per chunk
  std::vector<uint32_t> first, steps;  // per CTA: top coefficient of its chunk, Horner steps
  std::vector<uint32_t> slot;   // padded instance array: output row of the instance, 0xffffffff = padding
  std::vector<uint16_t> ops;    // HC_OPS ops per instance: one Horner step (modp_chain.h)
  std::vector<uint32_t> nops;   // ops per step, per CTA
  uint64_t sqr = 0, mul = 0;    // products per Horner step summed over the live instances (roofline accounting)
  uint32_t nops_max = 1;
};
static modp_chain::PowerTree g_tree;  // shared by all contexts; grown under g_tree_mu
static std::mutex g_tree_mu;

// One box of a plan: its positions (nullptr = 1..n), its t commitments at rows [cm_off, cm_off + t) of the
// commitment array, and its results at rows row_off + k n + i.
struct PlanBox {
  const int64_t* positions;
  size_t n, t;
  uint32_t cm_off, row_off;
};

// Positions are sorted by the length of their op list (longest first) and every length class is padded to
// a whole number of CTAs, so all lane groups of a CTA run the same number of products per step while
// one launch covers every class; shorter lists inside a class do not occur, padding instances repeat
// the last live one.  With several boxes the padding is per (box, length class), so that every CTA holds
// instances of one box and reads that box's coefficients through its (first, steps) pair.  `chunked`: one
// box, cut into K chunks by horner_chunks (the single-box plan).  A batch plan (chunked = false) is always
// unchunked, K = 1, whatever its number of boxes: the batch fills the chip, and chunking inside a batch is
// not implemented (its chunk exponents and combination would have to follow each box's rows).
static int prep_boxes(mpvss_ctx* ctx, const PlanBox* boxes, size_t nb, bool chunked, PosPlan& plan) {
  static_assert(modp_chain::SLOTS == modp::HC_SLOTS && modp_chain::OPS_MAX == modp::HC_OPS, "kernel / host op format");
  std::vector<std::vector<uint32_t>> pos(nb);
  uint32_t maxp = 1;
  size_t n_all = 0;
  for (size_t b = 0; b < nb; ++b) {
    if (positions_u32(boxes[b].positions, boxes[b].n, pos[b]) != boxes[b].n)
      return mpvss_fail(ctx, MPVSS_ERR_ARG, "position out of range [1, 2^31)");
    for (uint32_t p : pos[b]) maxp = std::max(maxp, p);
    n_all += boxes[b].n;
  }
  std::lock_guard<std::mutex> lk(g_tree_mu);
  g_tree.build(std::min<uint32_t>(maxp, modp_chain::TREE_LIMIT));
  std::vector<std::vector<uint16_t>> ops(n_all);
  std::vector<std::vector<std::vector<uint32_t>>> by(nb, std::vector<std::vector<uint32_t>>(modp_chain::OPS_MAX + 1));
  std::vector<uint32_t> sq(n_all), ml(n_all);
  for (size_t b = 0, g = 0; b < nb; ++b)
    for (size_t i = 0; i < boxes[b].n; ++i, ++g) {  // g: instance index over all boxes
      if (!modp_chain::step_ops(pos[b][i], g_tree, ops[g], &sq[g], &ml[g]))
        return mpvss_fail(ctx, MPVSS_ERR_UNSUPPORTED, "no addition chain within the kernel's slot budget");
      by[b][ops[g].size()].push_back((uint32_t)g);
    }
  const size_t t0 = boxes[0].t;
  if (chunked && nb != 1) return mpvss_fail(ctx, MPVSS_ERR_ARG, "a chunked plan covers one box");
  plan.K = chunked ? horner_chunks(ctx, n_all, t0) : 1;
  plan.B = (uint32_t)((t0 + plan.K - 1) / plan.K);
  plan.K = (uint32_t)((t0 + plan.B - 1) / plan.B);
  plan.tpi = plan.K > 1 ? ctx->modp_tpi : horner_tpi(ctx, n_all);
  plan.wpc = horner_wpc(ctx, n_all, plan.tpi);
  const size_t per_cta = (size_t)plan.wpc * (32 / plan.tpi);
  plan.slot.clear(); plan.ops.clear(); plan.nops.clear(); plan.first.clear(); plan.steps.clear();
  plan.nops_max = 1;
  plan.sqr = plan.mul = 0;
  std::vector<uint32_t> base(nb, 0);  // instance index of each box's first position
  for (size_t b = 1; b < nb; ++b) base[b] = base[b - 1] + (uint32_t)boxes[b - 1].n;
  for (uint32_t k = 0; k < plan.K; ++k) {  // chunk k: coefficients [k B, min((k+1) B, t)), results in rows k n + i
    for (uint32_t len = modp_chain::OPS_MAX; len >= 1; --len) {
      for (size_t b = 0; b < nb; ++b) {
        const std::vector<uint32_t>& cls = by[b][len];
        if (cls.empty()) continue;
        const PlanBox& bx = boxes[b];
        const uint32_t lo = plan.K > 1 ? k * plan.B : 0, hi = (uint32_t)std::min<size_t>(bx.t, (size_t)lo + (plan.K > 1 ? plan.B : bx.t));
        plan.nops_max = std::max(plan.nops_max, len);
        auto emit = [&](uint32_t g, uint32_t slot) {
          plan.slot.push_back(slot);
          size_t at = plan.ops.size();
          plan.ops.resize(at + modp_chain::OPS_MAX, (uint16_t)modp_chain::B_ONE);
          std::copy(ops[g].begin(), ops[g].end(), plan.ops.begin() + at);
        };
        for (uint32_t g : cls) {
          emit(g, bx.row_off + k * (uint32_t)bx.n + (g - base[b]));
          plan.sqr += (uint64_t)sq[g] * (hi - lo - 1);
          plan.mul += (uint64_t)ml[g] * (hi - lo - 1);
        }
        while (plan.slot.size() % per_cta) emit(cls.back(), 0xffffffffu);
        const size_t ctas = plan.slot.size() / per_cta;
        plan.nops.resize(ctas, len);
        plan.first.resize(ctas, bx.cm_off + hi - 1);
        plan.steps.resize(ctas, hi - lo - 1);
      }
    }
  }
  return MPVSS_OK;
}
static int prep_positions(mpvss_ctx* ctx, const int64_t* positions, size_t n, size_t t, PosPlan& plan) {
  const PlanBox box{positions, n, t, 0, 0};
  return prep_boxes(ctx, &box, 1, true, plan);
}

// e_i = pos_i^E mod (q-1) for the chunk combination: q-1 = 2g, so by CRT e_i is the representative of
// pos_i^E mod g (device modexp with the constants of modulus g) that has the parity of pos_i (E >= 1).
static int dev_chunk_exponents(mpvss_ctx* ctx, const int64_t* positions, size_t n, uint32_t E, uint32_t* e_out_dev) {
  std::vector<uint8_t> base(n * EB, 0), bexp(EB, 0), e(n * EB);
  for (size_t i = 0; i < n; ++i) {
    uint32_t p = (uint32_t)(positions ? positions[i] : (int64_t)i + 1);
    memcpy(base.data() + i * EB, &p, 4);
  }
  memcpy(bexp.data(), &E, 4);
  DevBuf &db = ctx->buf(20), &dx = ctx->buf(21);
  MPVSS_TRY(h2d(ctx, db, base.data(), n * EB));
  MPVSS_TRY(h2d(ctx, dx, bexp.data(), EB));
  MPVSS_TRY(dev_exp2(ctx, ctx->consts_g.as<uint32_t>(), db.as<uint32_t>(), EW, dx.as<uint32_t>(), 0,
                     windows_for(bexp.data(), EB, 1), nullptr, 0, nullptr, 0, 0, n, e_out_dev));
  MPVSS_CUDA(ctx, cudaMemcpyAsync(e.data(), e_out_dev, n * EB, cudaMemcpyDeviceToHost, ctx->stream));
  MPVSS_TRY(sync(ctx));
  for (size_t i = 0; i < n; ++i) {
    if ((e[i * EB] & 1u) != (base[i * EB] & 1u)) {
      big::Int v = big::add(big::from_le(e.data() + i * EB, EB), ctx->g);
      big::to_le(v, e.data() + i * EB, EB);
    }
  }
  MPVSS_CUDA(ctx, cudaMemcpyAsync(e_out_dev, e.data(), n * EB, cudaMemcpyHostToDevice, ctx->stream));
  return sync(ctx);
}
// all chunk exponents of a plan: rows (k-1) n + i = pos_i^(k B) mod (q-1), k = 1 .. K-1
static int plan_chunk_exponents(mpvss_ctx* ctx, const int64_t* positions, size_t n, const PosPlan& plan, DevBuf& e) {
  if (plan.K <= 1) return MPVSS_OK;
  MPVSS_CUDA(ctx, e.ensure((size_t)(plan.K - 1) * n * EB));
  for (uint32_t k = 1; k < plan.K; ++k)
    MPVSS_TRY(dev_chunk_exponents(ctx, positions, n, k * plan.B, e.as<uint32_t>() + (size_t)(k - 1) * n * EW));
  return MPVSS_OK;
}

// Device side of a plan: everything the Horner launch and the chunk combination read.
struct PlanDev {
  const uint16_t* ops;
  const uint32_t *slot, *nops, *first, *steps;
  const uint32_t* e;  // chunk exponents (K > 1)
  size_t n_padded;
  uint32_t K;
  int tpi, wpc;
  bool boxes = false;  // a multi-box plan: only the per-CTA (first, steps) bounds describe it
};
// commitments (device, normal form) -> X (device): Montgomery conversion, Horner over every chunk, and for
// K > 1 the combination X = H_0 * prod_{k >= 1} H_k^(pos^(k B)) (one exponentiation launch + K-1 products)
static int dev_horner(mpvss_ctx* ctx, const PlanDev& P, const uint32_t* comm, DevBuf& cm, size_t t, size_t n, DevBuf& hbuf,
                      DevBuf& tbuf, uint32_t* x) {
  const uint32_t* Kq = ctx->consts_q.as<uint32_t>();
  MPVSS_CUDA(ctx, cm.ensure(t * EB));
  MPVSS_TRY(dev_mul(ctx, Kq, comm, EW, nullptr, 0, 1, t, cm.as<uint32_t>()));
  uint32_t* h = x;
  if (P.K > 1) {
    MPVSS_CUDA(ctx, hbuf.ensure((size_t)P.K * n * EB));
    MPVSS_CUDA(ctx, tbuf.ensure((size_t)(P.K - 1) * n * EB));
    h = hbuf.as<uint32_t>();
  }
  // Two instantiations of the launch exist: per-CTA (first, steps) arrays, and loop bounds taken from the kernel
  // parameter t (K = 1 only).  Measured at n = 4096, t = 2731 on the same box, alternating: arrays 217.4 ms,
  // parameter bounds 220.2 ms (the code of round 2's first half), so the arrays are used always;
  // MPVSS_HORNER_UNIFORM=1 selects the other one for comparison runs.
  static const bool uniform = getenv("MPVSS_HORNER_UNIFORM") != nullptr;
  const bool arrays = P.K > 1 || P.boxes || !uniform;
  modp::HornerArgs A{Kq, cm.as<uint32_t>(), P.ops, P.slot, P.nops, h, (uint32_t)t, (uint32_t)P.n_padded, 0,
                     (uint32_t)P.wpc, arrays ? P.first : nullptr, arrays ? P.steps : nullptr};
  MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_h0, ctx->stream));
  MPVSS_CUDA(ctx, modp::launch_horner(P.tpi, A, ctx->modp_np1, ctx->stream));
  MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_h1, ctx->stream));
  timing_launch(ctx);
  if (P.K > 1) {
    uint32_t* T = tbuf.as<uint32_t>();
    MPVSS_TRY(dev_exp2(ctx, Kq, h + n * EW, EW, P.e, EW, 512, nullptr, 0, nullptr, 0, 0, (size_t)(P.K - 1) * n, T));
    MPVSS_TRY(dev_mul(ctx, Kq, h, EW, T, EW, 0, n, x));
    for (uint32_t k = 2; k < P.K; ++k) MPVSS_TRY(dev_mul(ctx, Kq, x, EW, T + (size_t)(k - 1) * n * EW, EW, 0, n, x));
  }
  return MPVSS_OK;
}

int poly_eval_exp(mpvss_ctx* ctx, const uint8_t* commitments, size_t t, const int64_t* positions, size_t n,
                  uint8_t* out) {
  MPVSS_TRY(check_args(ctx, commitments && out && n > 0 && t > 0, "poly_eval_exp: bad arguments"));
  PosPlan plan;
  MPVSS_TRY(prep_positions(ctx, positions, n, t, plan));
  DevBuf &dc = ctx->buf(0), &dops = ctx->buf(1), &dout = ctx->buf(2), &dcm = ctx->buf(3), &dsl = ctx->buf(4),
         &dno = ctx->buf(5), &dfi = ctx->buf(6), &dstp = ctx->buf(7), &de = ctx->buf(8);
  const size_t np = plan.slot.size();
  MPVSS_TRY(h2d(ctx, dc, commitments, t * EB));
  MPVSS_TRY(h2d(ctx, dops, plan.ops.data(), plan.ops.size() * 2));
  MPVSS_TRY(h2d(ctx, dsl, plan.slot.data(), np * 4));
  MPVSS_TRY(h2d(ctx, dno, plan.nops.data(), plan.nops.size() * 4));
  MPVSS_TRY(h2d(ctx, dfi, plan.first.data(), plan.first.size() * 4));
  MPVSS_TRY(h2d(ctx, dstp, plan.steps.data(), plan.steps.size() * 4));
  MPVSS_CUDA(ctx, dout.ensure(n * EB));
  MPVSS_TRY(plan_chunk_exponents(ctx, positions, n, plan, de));
  PlanDev P{dops.as<uint16_t>(), dsl.as<uint32_t>(), dno.as<uint32_t>(), dfi.as<uint32_t>(), dstp.as<uint32_t>(),
            de.as<uint32_t>(), np, plan.K, plan.tpi, plan.wpc};
  timing_begin(ctx);
  MPVSS_TRY(dev_horner(ctx, P, dc.as<uint32_t>(), dcm, t, n, ctx->buf(9), ctx->buf(10), dout.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  ctx->horner_sqr = plan.sqr;
  ctx->horner_mul = plan.mul;
  MPVSS_TRY(d2h(ctx, out, dout, n * EB));
  return sync(ctx);
}

int dleq_verify_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* h1, const uint8_t* g2, const uint8_t* h2,
                       const uint8_t* r, const uint8_t* c, size_t c_stride, size_t n, uint8_t* a1, uint8_t* a2) {
  // a1 == a2 == nullptr (internal callers): the results stay on the device in buf(6) / buf(7)
  MPVSS_TRY(check_args(ctx, g1 && h1 && g2 && h2 && r && c && (!a1 == !a2) && n > 0 && (c_stride == 0 || c_stride == EB),
                       "dleq_verify_commit: bad arguments"));
  DevBuf &dg1 = ctx->buf(0), &dh1 = ctx->buf(1), &dg2 = ctx->buf(2), &dh2 = ctx->buf(3), &dr = ctx->buf(4),
         &dc = ctx->buf(5), &da1 = ctx->buf(6), &da2 = ctx->buf(7);
  MPVSS_TRY(h2d(ctx, dg1, g1, EB));
  MPVSS_TRY(h2d(ctx, dh1, h1, n * EB));
  MPVSS_TRY(h2d(ctx, dg2, g2, n * EB));
  MPVSS_TRY(h2d(ctx, dh2, h2, n * EB));
  MPVSS_TRY(h2d(ctx, dr, r, n * EB));
  MPVSS_TRY(h2d(ctx, dc, c, c_stride ? n * EB : EB));
  MPVSS_CUDA(ctx, da1.ensure(n * EB));
  MPVSS_CUDA(ctx, da2.ensure(n * EB));
  uint32_t rw = windows_for(r, EB, n), cw = windows_for(c, EB, c_stride ? n : 1), cs = c_stride ? EW : 0;
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  const uint32_t* comb = nullptr;  // g1 is usually one of the two generators: use its table
  {
    bool rest_zero = true;
    for (size_t i = 1; i < EB; ++i) rest_zero = rest_zero && g1[i] == 0;
    if (rest_zero && (g1[0] == 2 || g1[0] == 4)) MPVSS_TRY(comb_table(ctx, g1[0] == 4 ? 1 : 0, &comb));
  }
  timing_begin(ctx);
  MPVSS_TRY(dev_exp2(ctx, K, dg1.as<uint32_t>(), 0, dr.as<uint32_t>(), EW, rw, dh1.as<uint32_t>(), EW,
                     dc.as<uint32_t>(), cs, cw, n, da1.as<uint32_t>(), nullptr, comb));
  MPVSS_TRY(dev_exp2(ctx, K, dg2.as<uint32_t>(), EW, dr.as<uint32_t>(), EW, rw, dh2.as<uint32_t>(), EW,
                     dc.as<uint32_t>(), cs, cw, n, da2.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  if (a1) MPVSS_TRY(d2h(ctx, a1, da1, n * EB));
  if (a2) MPVSS_TRY(d2h(ctx, a2, da2, n * EB));
  return sync(ctx);
}

int dleq_prove_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* g2, const uint8_t* w, size_t n, uint8_t* a1,
                      uint8_t* a2) {
  MPVSS_TRY(check_args(ctx, g1 && g2 && w && a1 && a2 && n > 0, "dleq_prove_commit: bad arguments"));
  DevBuf &dg1 = ctx->buf(0), &dg2 = ctx->buf(2), &dw = ctx->buf(4), &da1 = ctx->buf(6), &da2 = ctx->buf(7);
  MPVSS_TRY(h2d(ctx, dg1, g1, EB));
  MPVSS_TRY(h2d(ctx, dg2, g2, n * EB));
  MPVSS_TRY(h2d(ctx, dw, w, n * EB));
  MPVSS_CUDA(ctx, da1.ensure(n * EB));
  MPVSS_CUDA(ctx, da2.ensure(n * EB));
  uint32_t ww = windows_for(w, EB, n);
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  timing_begin(ctx);
  MPVSS_TRY(dev_exp2(ctx, K, dg1.as<uint32_t>(), 0, dw.as<uint32_t>(), EW, ww, nullptr, 0, nullptr, 0, 0, n,
                     da1.as<uint32_t>()));
  MPVSS_TRY(dev_exp2(ctx, K, dg2.as<uint32_t>(), EW, dw.as<uint32_t>(), EW, ww, nullptr, 0, nullptr, 0, 0, n,
                     da2.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  MPVSS_TRY(d2h(ctx, a1, da1, n * EB));
  MPVSS_TRY(d2h(ctx, a2, da2, n * EB));
  return sync(ctx);
}

// Bucket method (Pippenger, 8-bit windows) for prod_i bases[i]^scalars[i], all on the device: counting sort of
// every window's exponent bytes, bucket products, per-window products, final fold (modp::launch_msm).
// `db` holds the bases in normal form, `de` the exponents; the result lands in dout[0].
static int multi_exp_buckets(mpvss_ctx* ctx, DevBuf& db, DevBuf& de, uint32_t windows, size_t n, DevBuf& dout) {
  DevBuf &dm = ctx->buf(15), &didx = ctx->buf(16), &dst = ctx->buf(17), &dbk = ctx->buf(18), &dwp = ctx->buf(19);
  MPVSS_CUDA(ctx, didx.ensure((size_t)windows * n * 4));
  MPVSS_CUDA(ctx, dst.ensure((size_t)windows * 257 * 4));
  MPVSS_CUDA(ctx, dm.ensure(n * EB));
  MPVSS_CUDA(ctx, dbk.ensure((size_t)windows * 256 * EB));
  MPVSS_CUDA(ctx, dwp.ensure((size_t)windows * EB));
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  MPVSS_TRY(dev_mul(ctx, K, db.as<uint32_t>(), EW, nullptr, 0, 1, n, dm.as<uint32_t>()));  // to Montgomery form
  modp::MsmBucketArgs B{K, dm.as<uint32_t>(), didx.as<uint32_t>(), dst.as<uint32_t>(), dbk.as<uint32_t>(), windows,
                        (uint32_t)n};
  MPVSS_CUDA(ctx, modp::launch_msm(B, de.as<uint32_t>(), didx.as<uint32_t>(), dst.as<uint32_t>(), dwp.as<uint32_t>(),
                                   dout.as<uint32_t>(), ctx->stream));
  timing_launch(ctx, 4);
  return MPVSS_OK;
}

// The segmented product tree that folds box j's cnt[j] rows from start[j] into row start[j]: every level planned
// on the host and uploaded to dplan at once, before the caller opens its timing bracket.  level_end[l] is the
// number of (a, b, out) triples of levels 0..l.
static int plan_product_tree(mpvss_ctx* ctx, const uint32_t* start, const uint32_t* cnt, size_t L, DevBuf& dplan,
                             std::vector<uint32_t>& level_end) {
  std::vector<uint32_t> rows(3 * ((size_t)start[L - 1] + cnt[L - 1])), c(cnt, cnt + L);
  level_end.clear();
  for (size_t m = 0, total = 0;
       (m = modp::product_tree_level(start, c.data(), (uint32_t)L, rows.data() + 3 * total)) > 0;) {
    total += m;
    level_end.push_back((uint32_t)total);
  }
  if (!level_end.empty()) MPVSS_TRY(h2d(ctx, dplan, rows.data(), (size_t)level_end.back() * 3 * 4));
  return MPVSS_OK;
}

// prod_r db[r]^de[r] per box: one exponentiation launch over rows [0, n) into dpow, then one gather-multiply launch
// per level of the tree plan_product_tree uploaded to dplan.  `windows` as dev_exp2 takes it.
static int multi_exp_direct(mpvss_ctx* ctx, const DevBuf& db, const DevBuf& de, uint32_t windows, size_t n,
                            const std::vector<uint32_t>& level_end, DevBuf& dpow, const DevBuf& dplan) {
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  MPVSS_TRY(dev_exp2(ctx, K, db.as<uint32_t>(), EW, de.as<uint32_t>(), EW, windows, nullptr, 0, nullptr, 0, 0, n,
                     dpow.as<uint32_t>()));
  for (size_t l = 0; l < level_end.size(); ++l) {
    const uint32_t lo = l ? level_end[l - 1] : 0;
    modp::MulRowsArgs MA{K, dpow.as<uint32_t>(), dplan.as<uint32_t>() + 3 * lo, level_end[l] - lo};
    MPVSS_CUDA(ctx, modp::launch_mul_rows(ctx->modp_tpi, MA, ctx->stream));
    timing_launch(ctx);
  }
  return MPVSS_OK;
}

int multi_exp(mpvss_ctx* ctx, const uint8_t* bases, const uint8_t* scalars, size_t n, uint8_t* out) {
  MPVSS_TRY(check_args(ctx, bases && scalars && out && n > 0, "multi_exp: bad arguments"));
  DevBuf &db = ctx->buf(0), &de = ctx->buf(1), &dout = ctx->buf(2);
  MPVSS_TRY(h2d(ctx, db, bases, n * EB));
  MPVSS_CUDA(ctx, dout.ensure(n * EB));
  // One exponentiation per base + product tree is ~2560 products deep whatever n is; the bucket method does
  // 8x less work but is nearly as deep (the 2040 sequential squarings of its final fold, which no method
  // avoids for fresh bases), so it wins by 1.4x at k = 2731 and by 5x at k = 43691 where the direct form
  // runs in several waves ("modp_msm": 0 never, 1 always, 2 = from msm_threshold bases on).
  const bool buckets = ctx->modp_msm == 1 || (ctx->modp_msm == 2 && n >= (size_t)ctx->msm_threshold);
  MPVSS_TRY(h2d(ctx, de, scalars, n * EB));
  const uint32_t start = 0, cnt = (uint32_t)n;
  DevBuf& dplan = ctx->buf(4);
  std::vector<uint32_t> level_end;
  if (!buckets) MPVSS_TRY(plan_product_tree(ctx, &start, &cnt, 1, dplan, level_end));
  timing_begin(ctx);
  if (buckets)
    MPVSS_TRY(multi_exp_buckets(ctx, db, de, (windows_for(scalars, EB, n) + 1) / 2, n, dout));
  else
    MPVSS_TRY(multi_exp_direct(ctx, db, de, windows_for(scalars, EB, n), n, level_end, dout, dplan));
  MPVSS_TRY(timing_end(ctx));
  MPVSS_TRY(d2h(ctx, out, dout, EB));
  return sync(ctx);
}

// P(i) mod (q-1) for the given positions (polynomial.rs:50-58 reduced as participant.rs:202 does)
int scalar_poly_eval(mpvss_ctx* ctx, const uint8_t* coeffs, size_t t, const int64_t* positions, size_t n, uint8_t* out) {
  MPVSS_TRY(check_args(ctx, coeffs && out && n > 0 && t > 0, "scalar_poly_eval: bad arguments"));
  const std::vector<uint32_t> order = order_limbs(ctx);
  std::vector<uint32_t> pos;
  if (positions_u32(positions, n, pos) != n) return mpvss_fail(ctx, MPVSS_ERR_ARG, "position out of range [1, 2^31)");
  // the kernel wants coefficients below 2^2048 and reduces lazily; bring them below the order first
  std::vector<uint8_t> co(t * EB);
  for (size_t j = 0; j < t; ++j) big::to_le(big::mod(big::from_le(coeffs + j * EB, EB), ctx->qm1), co.data() + j * EB, EB);
  DevBuf &dco = ctx->buf(0), &dp = ctx->buf(1), &dord = ctx->buf(11), &dpos = ctx->buf(12);
  MPVSS_TRY(h2d(ctx, dco, co.data(), t * EB));
  MPVSS_TRY(h2d(ctx, dord, order.data(), EB));
  MPVSS_TRY(h2d(ctx, dpos, pos.data(), n * 4));
  MPVSS_CUDA(ctx, dp.ensure(n * EB));
  timing_begin(ctx);
  modp::PolyArgs PA{dco.as<uint32_t>(), dord.as<uint32_t>(), dpos.as<uint32_t>(), dp.as<uint32_t>(), (uint32_t)t,
                    (uint32_t)n};
  MPVSS_CUDA(ctx, modp::launch_poly(PA, ctx->stream));
  timing_launch(ctx);
  MPVSS_TRY(timing_end(ctx));
  MPVSS_TRY(d2h(ctx, out, dp, n * EB));
  MPVSS_CUDA(ctx, cudaMemsetAsync(dco.p, 0, dco.cap, ctx->stream));  // coefficients are secret
  return sync(ctx);
}

// Optional input validation ("validate" tunable; SURVEY 8f-3): the reference's bytes_to_element accepts any
// integer (modp.rs:154-156).  Elements must satisfy 0 < x < q and lie in the subgroup of order g the
// protocol works in: x^g = 1 (one exponentiation each, with the kernels of modulus q).  bad[i] = 1 for
// each of the `count` device-resident elements that fails (the others are left as they are).
static int validate_elements(mpvss_ctx* ctx, const uint32_t* dev, size_t count, uint8_t* bad) {
  std::vector<uint8_t> gexp(EB), res(count * EB), in(count * EB);
  big::to_le(ctx->g, gexp.data(), EB);
  DevBuf &de = ctx->buf(20), &dout = ctx->buf(21);
  MPVSS_TRY(h2d(ctx, de, gexp.data(), EB));
  MPVSS_CUDA(ctx, dout.ensure(count * EB));
  MPVSS_TRY(dev_exp2(ctx, ctx->consts_q.as<uint32_t>(), dev, EW, de.as<uint32_t>(), 0, 512, nullptr, 0, nullptr, 0, 0,
                     count, dout.as<uint32_t>()));
  MPVSS_TRY(d2h(ctx, res.data(), dout, count * EB));
  MPVSS_CUDA(ctx, cudaMemcpyAsync(in.data(), dev, count * EB, cudaMemcpyDeviceToHost, ctx->stream));
  MPVSS_TRY(sync(ctx));
  for (size_t i = 0; i < count; ++i) {
    big::Int x = big::from_le(in.data() + i * EB, EB);
    bool one = res[i * EB] == 1;
    for (size_t k = 1; k < EB && one; ++k) one = res[i * EB + k] == 0;
    if (big::is_zero(x) || big::cmp(x, ctx->q) >= 0 || !one) bad[i] = 1;
  }
  return MPVSS_OK;
}

// ------------------------------------------------------------------- verify ----
static const transcript::Geom GEOM{EB, true};

int verify_stage(mpvss_ctx* ctx, size_t n_total, size_t t, const uint8_t* commitments, const int64_t* positions,
                 const uint8_t* publickeys, const uint8_t* shares, const uint8_t* responses, const uint8_t* challenge) {
  ctx->v_n_total = 0;
  MPVSS_TRY(check_args(ctx, n_total > 0 && t > 0 && commitments && publickeys && shares && responses && challenge,
                       "verify_distribution: bad arguments"));
  std::vector<uint32_t> pos_all;
  if (positions_u32(positions, n_total, pos_all) != n_total)  // box content, checked alike by every rank: verifies as false
    return mpvss_fail(ctx, MPVSS_ERR_ENCODING, "verify_distribution: position out of range [1, 2^31)");
  // this rank's participants: rank, rank + N, ... (every rank gets the same mix of short and long chains)
  const size_t n = transcript::local_count(n_total, ctx->nranks, ctx->rank);
  std::vector<int64_t> pos(n);
  for (size_t j = 0; j < n; ++j) pos[j] = pos_all[(size_t)ctx->rank + j * (size_t)ctx->nranks];
  // The plan depends on the positions and t only: a context that verifies boxes of the same shape again (the
  // usual case: positions 1..n) keeps the plan and its device copy from the previous call.
  PosPlan plan;
  const uint32_t want_k = n ? horner_chunks(ctx, n, t) : 1;
  const bool replan = n && !(ctx->v_plan_pos == pos && ctx->v_plan_t == t && ctx->v_plan_kreq == want_k &&
                             ctx->v_plan_tpi == (want_k > 1 ? ctx->modp_tpi : horner_tpi(ctx, n)) &&
                             ctx->v_plan_wpc == horner_wpc(ctx, n, ctx->v_plan_tpi));
  if (replan) {
    ctx->v_plan_pos.clear();
    MPVSS_TRY(prep_positions(ctx, pos.data(), n, t, plan));
    ctx->v_np = plan.slot.size();
    ctx->v_nops_max = plan.nops_max;
    ctx->v_tpi = plan.tpi;
    ctx->v_wpc = plan.wpc;
    ctx->v_k = plan.K;
    ctx->v_plan_sqr = plan.sqr;
    ctx->v_plan_mul = plan.mul;
  }
  ctx->horner_sqr = ctx->v_plan_sqr;
  ctx->horner_mul = ctx->v_plan_mul;
  std::vector<uint8_t> tpk, ty, tr;
  const uint8_t* pk = slice_rows(ctx, publickeys, n_total, EB, tpk);
  const uint8_t* y = slice_rows(ctx, shares, n_total, EB, ty);
  const uint8_t* r = slice_rows(ctx, responses, n_total, EB, tr);
  MPVSS_TRY(h2d(ctx, ctx->v_comm, commitments, t * EB));
  MPVSS_TRY(h2d(ctx, ctx->v_c, challenge, EB));
  if (replan) {
    MPVSS_TRY(h2d(ctx, ctx->v_ops, plan.ops.data(), plan.ops.size() * 2));
    MPVSS_TRY(h2d(ctx, ctx->v_slot, plan.slot.data(), ctx->v_np * 4));
    MPVSS_TRY(h2d(ctx, ctx->v_nd, plan.nops.data(), plan.nops.size() * 4));
    MPVSS_TRY(h2d(ctx, ctx->v_first, plan.first.data(), plan.first.size() * 4));
    MPVSS_TRY(h2d(ctx, ctx->v_steps, plan.steps.data(), plan.steps.size() * 4));
    MPVSS_TRY(plan_chunk_exponents(ctx, pos.data(), n, plan, ctx->v_e));
    MPVSS_TRY(sync(ctx));  // the cache key is set once the copies are done
    ctx->v_plan_pos = pos;
    ctx->v_plan_t = t;
    ctx->v_plan_kreq = want_k;
    ctx->v_plan_tpi = plan.tpi;
    ctx->v_plan_wpc = plan.wpc;
  }
  if (n) {
    MPVSS_TRY(h2d(ctx, ctx->v_pk, pk, n * EB));
    MPVSS_TRY(h2d(ctx, ctx->v_y, y, n * EB));
    MPVSS_TRY(h2d(ctx, ctx->v_r, r, n * EB));
    MPVSS_CUDA(ctx, ctx->v_x.ensure(n * EB));
    MPVSS_CUDA(ctx, ctx->v_a1.ensure(n * EB));
    MPVSS_CUDA(ctx, ctx->v_a2.ensure(n * EB));
  }
  const size_t rpr = transcript::rows_per_rank(n_total, ctx->nranks);
  MPVSS_CUDA(ctx, ctx->v_frames.ensure(rpr * GEOM.row()));
  MPVSS_CUDA(ctx, cudaMemsetAsync(ctx->v_frames.p, 0, rpr * GEOM.row(), ctx->stream));
  if (ctx->nranks > 1) MPVSS_CUDA(ctx, ctx->v_gather.ensure((size_t)ctx->nranks * rpr * GEOM.row()));
  MPVSS_TRY(comb_table(ctx, 1, &ctx->v_comb));
  ctx->v_rwin = n ? windows_for(r, EB, n) : 1;
  ctx->v_cwin = windows_for(challenge, EB, 1);
  ctx->v_challenge.assign(challenge, challenge + EB);
  ctx->v_n = n;
  ctx->v_t = t;
  MPVSS_TRY(sync(ctx));  // the host buffers may be released by the caller after return
  ctx->v_n_total = n_total;
  return MPVSS_OK;
}

// Where a2 = y^r * Y^c (n instances, independent of X) runs beside an X_i launch of np padded instances at tpi
// lanes per value whose longest chain takes `horner` products ("modp_overlap"; verify_kernels gives the
// measurements): 0 before it on the main stream, 2 regular launch / 3 persistent one-warp CTAs on a side
// stream after it.
// Mode 3 only pays when the persistent CTAs finish inside the Horner launch: rounds of one
// exponentiation per SM (about 5 products per 4-bit window) against the t-1 Horner steps of
// nops products; measured break-even near 0.6 (tools/overlap_sweep.sh).  Otherwise a2 goes first.
static int a2_placement(const mpvss_ctx* ctx, size_t n, double horner, size_t np, int tpi, uint32_t rwin, uint32_t cwin) {
  int overlap = ctx->modp_overlap;
  if (overlap == 3) {
    const size_t groups_per_warp = 32 / (size_t)ctx->modp_tpi;
    const size_t nwarps = (n + groups_per_warp - 1) / groups_per_warp;
    const size_t rounds = (nwarps + (size_t)ctx->sm_count - 1) / (size_t)ctx->sm_count;
    const double filler = (double)rounds * (5.0 * (rwin + cwin) + 30.0);
    if (filler > 0.6 * horner) overlap = 0;
    // ... and only when the Horner launch leaves a hole: W one-warp CTAs fill the 4 schedulers of every SM
    // evenly when W is a multiple of 4 * SMs; the filler warp then becomes a third warp on one scheduler per SM
    // and slows its two Horner warps for the whole launch (n = 4736 = 8 warps per SM: 308 instead of 261 ms)
    const size_t slots = (size_t)4 * (size_t)ctx->sm_count;
    const size_t hw = np / (32 / (size_t)tpi);
    const size_t holes = (slots - hw % slots) % slots;
    if (holes < (size_t)ctx->sm_count) overlap = 0;
    // Small boxes: when both launches together stay below three warps per scheduler the chip has room for a2
    // as a regular launch beside the X_i launch (measured, tools/small_box_overlap_sweep.sh: n = 1024, t = 683 36.5 -> 28.5 ms;
    // n = 2048, t = 1366 72.9 -> 71.0 ms; at n = 4096 the same mode slows the X_i warps: 265.6 against 256.5 ms)
    if (overlap == 0 && hw + nwarps <= (size_t)12 * (size_t)ctx->sm_count) overlap = 2;
  }
  return overlap;
}

// Device buffers of one verification pass over t commitments and n instances.
struct VerifyBufs {
  DevBuf &comm, &pk, &y, &r, &c;  // inputs: commitments, public keys, shares, responses, challenge(s)
  DevBuf &cm, &h, &t2;            // dev_horner's working buffers
  DevBuf &x, &a1, &a2, &frames;   // outputs: X, a1, a2, framed rows
};

// One DLEQ pass of the verify calls: X (Horner), a1 = g^r * X^c, a2 = y^r * Y^c, then the framed rows.  `cs` is the
// challenge stride in limbs (0: one challenge for all instances), `horner` the products of the longest Horner chain
// (a2_placement).  ev_mid marks the end of the X phase.  bad gets t + 2 n flags, set by validate_elements for the
// commitments, public keys and shares when the "validate" tunable is on.
static int verify_pass(mpvss_ctx* ctx, const PlanDev& P, const VerifyBufs& B, size_t t, size_t n, uint32_t cs,
                       uint32_t rwin, uint32_t cwin, double horner, const uint32_t* comb, std::vector<uint8_t>& bad) {
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  uint32_t* X = B.x.as<uint32_t>();
  // a2 = y^r * Y^c does not depend on X.  The Horner launch puts 7 one-warp CTAs on the 4 schedulers
  // of an SM, i.e. one warp slot per SM stays empty for the whole launch.  modp_overlap = 3 (default)
  // issues a2 on a side stream right AFTER the Horner launch as persistent one-warp CTAs, one per SM:
  // they take exactly that slot and a2 disappears from the step (measured: step 270.8 -> 256.5 ms,
  // Horner launch itself 245 -> 246 ms).  2: regular a2 launch on the side stream (265.6 ms, slows
  // the Horner warps); 0: a2 first on the main stream.  Issuing it first on a side stream lets it
  // claim SMs and unbalances the placement of the long-running Horner CTAs (40 % slower): no mode 1.
  MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
  auto launch_a2 = [&](cudaStream_t s) {
    return dev_exp2(ctx, K, B.pk.as<uint32_t>(), EW, B.r.as<uint32_t>(), EW, rwin, B.y.as<uint32_t>(), EW,
                    B.c.as<uint32_t>(), cs, cwin, n, B.a2.as<uint32_t>(), s);
  };
  const int overlap = a2_placement(ctx, n, horner, P.n_padded, P.tpi, rwin, cwin);
  const bool side = overlap == 2 || overlap == 3;
  if (!side) MPVSS_TRY(launch_a2(ctx->stream));
  // X_i from the commitments (participant.rs:423-434)
  MPVSS_TRY(dev_horner(ctx, P, B.comm.as<uint32_t>(), B.cm, t, n, B.h, B.t2, X));
  if (side) {
    MPVSS_CUDA(ctx, cudaStreamWaitEvent(ctx->aux[0], ctx->ev_fork, 0));
    // 3: persistent one-warp CTAs, one per SM, into the warp slot the Horner CTAs leave empty
    if (overlap == 3) ctx->exp2_filler_ctas = (size_t)ctx->sm_count;
    int rc = launch_a2(ctx->aux[0]);
    ctx->exp2_filler_ctas = 0;
    MPVSS_TRY(rc);
    MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_join[0], ctx->aux[0]));
  }
  MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_mid, ctx->stream));
  // a1 = g^r * X^c  (g^r from the fixed-base table)
  MPVSS_TRY(dev_exp2(ctx, K, ctx->gens.as<uint32_t>() + 64, 0, B.r.as<uint32_t>(), EW, rwin, X, EW,
                     B.c.as<uint32_t>(), cs, cwin, n, B.a1.as<uint32_t>(), nullptr, comb));
  if (side) MPVSS_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0));
  // transcript rows F(X) F(Y) F(a1) F(a2) in local order (dleq.rs:87-99)
  modp::FrameArgs FA{X, B.y.as<uint32_t>(), B.a1.as<uint32_t>(), B.a2.as<uint32_t>(), B.frames.as<uint8_t>(),
                     (uint32_t)n};
  MPVSS_CUDA(ctx, modp::launch_frames(FA, ctx->stream));
  timing_launch(ctx);
  bad.assign(t + 2 * n, 0);
  if (ctx->validate) {
    MPVSS_TRY(validate_elements(ctx, B.comm.as<uint32_t>(), t, bad.data()));
    MPVSS_TRY(validate_elements(ctx, B.pk.as<uint32_t>(), n, bad.data() + t));
    MPVSS_TRY(validate_elements(ctx, B.y.as<uint32_t>(), n, bad.data() + t + n));
  }
  return MPVSS_OK;
}

// kernels of the staged verification
static int verify_kernels(mpvss_ctx* ctx) {
  const size_t n = ctx->v_n, t = ctx->v_t;
  timing_begin(ctx);
  if (n == 0) {  // more ranks than participants: this rank only takes part in the all-gather
    MPVSS_TRY(timing_end(ctx));
    ctx->phase_ms[0] = ctx->phase_ms[1] = ctx->phase_ms[2] = 0.f;
    return MPVSS_OK;
  }
  PlanDev P{ctx->v_ops.as<uint16_t>(), ctx->v_slot.as<uint32_t>(), ctx->v_nd.as<uint32_t>(), ctx->v_first.as<uint32_t>(),
            ctx->v_steps.as<uint32_t>(), ctx->v_e.as<uint32_t>(), ctx->v_np, ctx->v_k, ctx->v_tpi, ctx->v_wpc};
  const VerifyBufs B{ctx->v_comm, ctx->v_pk, ctx->v_y, ctx->v_r, ctx->v_c, ctx->v_cm, ctx->v_h, ctx->v_t2,
                     ctx->v_x, ctx->v_a1, ctx->v_a2, ctx->v_frames};
  std::vector<uint8_t> bad;
  MPVSS_TRY(verify_pass(ctx, P, B, t, n, 0, ctx->v_rwin, ctx->v_cwin,
                        (double)(t > 1 ? t - 1 : 0) / (double)ctx->v_k * (double)ctx->v_nops_max, ctx->v_comb, bad));
  // mark the rank's first row: 0xff is never part of a valid length (seen by all ranks)
  if (std::find(bad.begin(), bad.end(), 1) != bad.end()) {
    const uint8_t mark = 0xff;
    MPVSS_CUDA(ctx, cudaMemcpyAsync(ctx->v_frames.p, &mark, 1, cudaMemcpyHostToDevice, ctx->stream));
  }
  MPVSS_TRY(timing_end(ctx));
  MPVSS_CUDA(ctx, cudaEventElapsedTime(&ctx->phase_ms[0], ctx->ev0, ctx->ev_mid));  // X_i (with a2 underneath)
  MPVSS_CUDA(ctx, cudaEventElapsedTime(&ctx->phase_ms[1], ctx->ev_mid, ctx->ev1));  // remaining DLEQ work
  MPVSS_CUDA(ctx, cudaEventElapsedTime(&ctx->phase_ms[2], ctx->ev_h0, ctx->ev_h1));  // the Horner launch alone
  return MPVSS_OK;
}

int verify_run(mpvss_ctx* ctx, int* ok, uint8_t* x_out, uint8_t* a1_out, uint8_t* a2_out, uint8_t* digest_out) {
  MPVSS_TRY(check_args(ctx, ok && ctx->v_n_total > 0, "verify_distribution_run: nothing staged"));
  MPVSS_TRY(check_args(ctx, ctx->nranks <= 1 || (!x_out && !a1_out && !a2_out),
                       "verify_distribution: x/a1/a2 outputs are not available with a communicator"));
  const size_t n = ctx->v_n, n_total = ctx->v_n_total;
  MPVSS_TRY(verify_kernels(ctx));
  // one all-gather of the rows per phase (SURVEY 8e), then one hash pass in participant order
  const uint8_t* rows = ctx->v_frames.as<uint8_t>();
  if (ctx->nranks > 1) {
    MPVSS_TRY(comm_allgather(ctx, ctx->v_frames.p, ctx->v_gather.p,
                             transcript::rows_per_rank(n_total, ctx->nranks) * GEOM.row()));
    MPVSS_CUDA(ctx, ctx->v_ordered.ensure(n_total * GEOM.row()));
    MPVSS_TRY(comm_reorder_rows(ctx, ctx->v_gather.p, ctx->v_ordered.p, n_total, GEOM.row()));
    rows = ctx->v_ordered.as<uint8_t>();
  }
  uint8_t digest[32], c[EB];
  if (ctx->device_hash) {  // measured alternative: the one sequential chain on one device thread
    MPVSS_TRY(transcript::device_digest(ctx, rows, n_total, ctx->nranks, GEOM, digest));
  } else {
    sha2::Sha256 h;
    MPVSS_TRY(transcript::fetch_and_hash(ctx, rows, n_total, ctx->nranks, GEOM, h, true));
    h.finalize(digest);
  }
  challenge_from_digest(ctx, digest, c);
  *ok = memcmp(c, ctx->v_challenge.data(), EB) == 0;  // participant.rs:451-454
  for (size_t r = 0; r < std::min<size_t>((size_t)ctx->nranks, n_total); ++r)  // a rank whose slice failed validation
    if (ctx->h_frames.as<uint8_t>()[r * GEOM.row()] == 0xff) *ok = 0;               // marked its first row = participant r
  if (digest_out) memcpy(digest_out, digest, 32);
  if (x_out) MPVSS_TRY(d2h(ctx, x_out, ctx->v_x, n * EB));
  if (a1_out) MPVSS_TRY(d2h(ctx, a1_out, ctx->v_a1, n * EB));
  if (a2_out) MPVSS_TRY(d2h(ctx, a2_out, ctx->v_a2, n * EB));
  return sync(ctx);
}

// ------------------------------------------------------ verify_distributions ----
// Many boxes in one pass: one Horner launch evaluates X_i of every box (prep_boxes: each CTA reads its own
// box's coefficients), a2 and a1 run once over all instances with one challenge per instance, the frames of
// all boxes come to the host in one copy and each box's row range is hashed into its own digest.  a2 is
// placed by the single-box rule (a2_placement) on the total instance count and the longest box's chain.
// Only scratch buffers are used, so the staged single-box state and its cached plan stay valid.
int verify_batch(mpvss_ctx* ctx, size_t nb, const size_t* nv, const size_t* tv, const uint8_t* commitments,
                 const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares, const uint8_t* responses,
                 const uint8_t* challenges, int* ok_out, uint8_t* digests_out) {
  std::vector<size_t> noff(nb + 1, 0), toff(nb + 1, 0);
  for (size_t b = 0; b < nb; ++b) {
    noff[b + 1] = noff[b] + nv[b];
    toff[b + 1] = toff[b] + tv[b];
  }
  const size_t N = noff[nb], Tt = toff[nb];
  // a position out of range makes its box false; the other boxes are planned
  std::vector<uint8_t> live(nb, 1);
  std::vector<PlanBox> boxes;
  std::vector<uint32_t> pos;
  for (size_t b = 0; b < nb; ++b) {
    const int64_t* p = positions ? positions + noff[b] : nullptr;
    live[b] = positions_u32(p, nv[b], pos) == nv[b];
    if (live[b]) boxes.push_back(PlanBox{p, nv[b], tv[b], (uint32_t)toff[b], (uint32_t)noff[b]});
  }
  std::vector<uint8_t> cexp(N * EB);  // the box's challenge for every instance
  for (size_t b = 0; b < nb; ++b)
    for (size_t i = noff[b]; i < noff[b + 1]; ++i) memcpy(cexp.data() + i * EB, challenges + b * EB, EB);
  const uint32_t rwin = windows_for(responses, EB, N), cwin = windows_for(challenges, EB, nb);
  DevBuf &dcomm = ctx->buf(0), &dcm = ctx->buf(1), &dpk = ctx->buf(2), &dy = ctx->buf(3), &dr = ctx->buf(4),
         &dc = ctx->buf(5), &dx = ctx->buf(6), &da1 = ctx->buf(7), &da2 = ctx->buf(8), &dfr = ctx->buf(9),
         &dops = ctx->buf(10), &dsl = ctx->buf(11), &dno = ctx->buf(12), &dfi = ctx->buf(13), &dstp = ctx->buf(14);
  MPVSS_TRY(h2d(ctx, dcomm, commitments, Tt * EB));
  MPVSS_TRY(h2d(ctx, dpk, publickeys, N * EB));
  MPVSS_TRY(h2d(ctx, dy, shares, N * EB));
  MPVSS_TRY(h2d(ctx, dr, responses, N * EB));
  MPVSS_TRY(h2d(ctx, dc, cexp.data(), N * EB));
  for (DevBuf* b : {&dx, &da1, &da2}) MPVSS_CUDA(ctx, b->ensure(N * EB));
  MPVSS_CUDA(ctx, dfr.ensure(N * GEOM.row()));
  if (boxes.size() < nb) MPVSS_CUDA(ctx, cudaMemsetAsync(dx.p, 0, N * EB, ctx->stream));  // rows no plan writes
  PosPlan plan;
  if (!boxes.empty()) {
    MPVSS_TRY(prep_boxes(ctx, boxes.data(), boxes.size(), false, plan));
    MPVSS_TRY(h2d(ctx, dops, plan.ops.data(), plan.ops.size() * 2));
    MPVSS_TRY(h2d(ctx, dsl, plan.slot.data(), plan.slot.size() * 4));
    MPVSS_TRY(h2d(ctx, dno, plan.nops.data(), plan.nops.size() * 4));
    MPVSS_TRY(h2d(ctx, dfi, plan.first.data(), plan.first.size() * 4));
    MPVSS_TRY(h2d(ctx, dstp, plan.steps.data(), plan.steps.size() * 4));
  }
  const uint32_t* comb;
  MPVSS_TRY(comb_table(ctx, 1, &comb));
  std::vector<uint8_t> bad(Tt + 2 * N, 0);  // validate: per commitment, public key and share
  timing_begin(ctx);
  if (!boxes.empty()) {
    size_t tmax = 1;
    for (const PlanBox& bx : boxes) tmax = std::max(tmax, bx.t);
    // rows of boxes left out of the plan stay unwritten
    PlanDev P{dops.as<uint16_t>(), dsl.as<uint32_t>(), dno.as<uint32_t>(), dfi.as<uint32_t>(), dstp.as<uint32_t>(),
              nullptr, plan.slot.size(), plan.K, plan.tpi, plan.wpc, true};
    const VerifyBufs B{dcomm, dpk, dy, dr, dc, dcm, ctx->buf(15), ctx->buf(16), dx, da1, da2, dfr};
    MPVSS_TRY(verify_pass(ctx, P, B, Tt, N, EW, rwin, cwin, (double)(tmax - 1) * (double)plan.nops_max, comb, bad));
  }
  MPVSS_TRY(timing_end(ctx));
  ctx->horner_sqr = plan.sqr;
  ctx->horner_mul = plan.mul;
  PinBuf& host = ctx->pin(0);
  MPVSS_CUDA(ctx, host.ensure(N * GEOM.row()));
  uint8_t* rows = host.as<uint8_t>();
  MPVSS_TRY(d2h(ctx, rows, dfr, N * GEOM.row()));
  MPVSS_TRY(sync(ctx));
  for (size_t b = 0; b < nb; ++b) {
    for (size_t j = toff[b]; j < toff[b + 1] && live[b]; ++j) live[b] = !bad[j];
    for (size_t i = noff[b]; i < noff[b + 1] && live[b]; ++i) live[b] = !bad[Tt + i] && !bad[Tt + N + i];
    uint8_t digest[32] = {0}, c[EB];
    ok_out[b] = 0;
    if (live[b]) {
      sha2::Sha256 h;
      transcript::hash_ordered(h, rows, noff[b], noff[b + 1], GEOM);
      h.finalize(digest);
      challenge_from_digest(ctx, digest, c);
      ok_out[b] = memcmp(c, challenges + b * EB, EB) == 0;  // participant.rs:451-454
    }
    if (digests_out) memcpy(digests_out + 32 * b, digest, 32);
  }
  return MPVSS_OK;
}

// --------------------------------------------------------------- distribute ----
// Device buffers of one dealing launch sequence: coefficients, secret exponents s = a_0 mod (q-1), witnesses and
// public keys in; P(i), C, G^s, X, Y, a1, a2 and the framed transcript rows out; the two fixed-base tables.
struct DealBufs {
  const uint32_t *co, *s, *w, *pk;
  uint32_t *p, *C, *Gs, *X, *Y, *A1, *A2;
  uint8_t* frames;
  const uint32_t *combG, *combg;
};
// The dealer's launches: C over t coefficients, G^s over ns secret exponents, then, for n instances, P(i) mod (q-1)
// (`poly` enqueues that one launch), X, Y, a1, a2 and the frames.  Secret exponents (coefficients, P(i), witnesses)
// always run the full window count: the schedule must not depend on their size.
template <class Poly>
static int deal_kernels(mpvss_ctx* ctx, const DealBufs& B, size_t t, size_t ns, size_t n, Poly poly) {
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  const uint32_t* G = ctx->gens.as<uint32_t>();
  const uint32_t FW = 512;
  // C_j = g^a_j (participant.rs:189-193); every rank computes all t of them (replicated, fixed-base table)
  MPVSS_TRY(dev_exp2(ctx, K, G + 64, 0, B.co, EW, FW, nullptr, 0, nullptr, 0, 0, t, B.C, nullptr, B.combg));
  // G^s (participant.rs:268)
  MPVSS_TRY(dev_exp2(ctx, K, G, 0, B.s, EW, FW, nullptr, 0, nullptr, 0, 0, ns, B.Gs, nullptr, B.combG));
  if (!n) return MPVSS_OK;
  // p_i = P(i) mod (q-1) (participant.rs:202), one position per thread
  MPVSS_CUDA(ctx, poly());
  timing_launch(ctx);
  // X_i = prod_j C_j^(i^j) = g^P(i): the dealer knows P, one fixed-base exponentiation
  // gives the same group element as the reference's t-term product (participant.rs:207-215)
  MPVSS_TRY(dev_exp2(ctx, K, G + 64, 0, B.p, EW, FW, nullptr, 0, nullptr, 0, 0, n, B.X, nullptr, B.combg));
  // Y_i = y_i^P(i) (participant.rs:219)
  MPVSS_TRY(dev_exp2(ctx, K, B.pk, EW, B.p, EW, FW, nullptr, 0, nullptr, 0, 0, n, B.Y));
  // a1 = g^w, a2 = y^w (participant.rs:236-237)
  MPVSS_TRY(dev_exp2(ctx, K, G + 64, 0, B.w, EW, FW, nullptr, 0, nullptr, 0, 0, n, B.A1, nullptr, B.combg));
  MPVSS_TRY(dev_exp2(ctx, K, B.pk, EW, B.w, EW, FW, nullptr, 0, nullptr, 0, 0, n, B.A2));
  modp::FrameArgs FA{B.X, B.Y, B.A1, B.A2, B.frames, (uint32_t)n};
  MPVSS_CUDA(ctx, modp::launch_frames(FA, ctx->stream));
  timing_launch(ctx);
  return MPVSS_OK;
}

int distribute(mpvss_ctx* ctx, size_t n_total, size_t t, const uint8_t* secret, size_t secret_len,
               const uint8_t* coeffs, const uint8_t* witnesses, const uint8_t* publickeys, uint8_t* commitments_out,
               uint8_t* shares_out, uint8_t* challenge_out, uint8_t* responses_out, uint8_t* u_out, uint8_t* x_out) {
  MPVSS_TRY(check_args(ctx, n_total > 0 && t > 0 && t <= n_total && secret && coeffs && witnesses && publickeys &&
                                commitments_out && shares_out && challenge_out && responses_out && u_out &&
                                secret_len <= EB,
                       "distribute: bad arguments (threshold <= n, participant.rs:166; secret at most 256 bytes)"));
  const std::vector<uint32_t> order = order_limbs(ctx);
  if (order[EW - 1] != 0xffffffffu || order[EW - 2] != 0xffffffffu)
    return mpvss_fail(ctx, MPVSS_ERR_UNSUPPORTED, "distribute: scalar kernels need an order with all-ones top limbs");
  // this rank's participants: rank, rank + N, ... (all of them without a communicator)
  const size_t n = transcript::local_count(n_total, ctx->nranks, ctx->rank);
  std::vector<uint32_t> pos(std::max<size_t>(n, 1));
  for (size_t j = 0; j < n; ++j) pos[j] = (uint32_t)((size_t)ctx->rank + j * (size_t)ctx->nranks + 1);
  std::vector<uint8_t> tw, tpk;
  const uint8_t* w = slice_rows(ctx, witnesses, n_total, EB, tw);
  const uint8_t* pk = slice_rows(ctx, publickeys, n_total, EB, tpk);
  DevBuf &dco = ctx->buf(0), &dp = ctx->buf(1), &dw = ctx->buf(2), &dpk = ctx->buf(3), &dC = ctx->buf(4),
         &dX = ctx->buf(5), &dY = ctx->buf(6), &dA1 = ctx->buf(7), &dA2 = ctx->buf(8), &dGs = ctx->buf(9),
         &ds = ctx->buf(10), &dord = ctx->buf(11), &dpos = ctx->buf(12), &dR = ctx->buf(13), &dc = ctx->buf(14);
  // s = P(0) mod (q-1) = a_0 mod (q-1)  (participant.rs:267)
  uint8_t s_le[EB];
  big::to_le(big::mod(big::from_le(coeffs, EB), ctx->qm1), s_le, EB);
  MPVSS_TRY(h2d(ctx, dco, coeffs, t * EB));
  MPVSS_TRY(h2d(ctx, dord, order.data(), EB));
  MPVSS_TRY(h2d(ctx, dpos, pos.data(), pos.size() * 4));
  MPVSS_TRY(h2d(ctx, ds, s_le, EB));
  if (n) {
    MPVSS_TRY(h2d(ctx, dw, w, n * EB));
    MPVSS_TRY(h2d(ctx, dpk, pk, n * EB));
  }
  const size_t nn = std::max<size_t>(n, 1);
  for (DevBuf* b : {&dp, &dX, &dY, &dA1, &dA2, &dR}) MPVSS_CUDA(ctx, b->ensure(nn * EB));
  MPVSS_CUDA(ctx, dC.ensure(t * EB));
  MPVSS_CUDA(ctx, dGs.ensure(EB));
  MPVSS_CUDA(ctx, dc.ensure(EB));
  const uint32_t *combG, *combg;
  MPVSS_TRY(comb_table(ctx, 0, &combG));
  MPVSS_TRY(comb_table(ctx, 1, &combg));
  const size_t rpr = transcript::rows_per_rank(n_total, ctx->nranks);
  MPVSS_CUDA(ctx, ctx->v_frames.ensure(rpr * GEOM.row()));
  MPVSS_CUDA(ctx, cudaMemsetAsync(ctx->v_frames.p, 0, rpr * GEOM.row(), ctx->stream));
  if (ctx->nranks > 1) MPVSS_CUDA(ctx, ctx->v_gather.ensure((size_t)ctx->nranks * rpr * GEOM.row()));
  timing_begin(ctx);
  const DealBufs B{dco.as<uint32_t>(), ds.as<uint32_t>(), dw.as<uint32_t>(), dpk.as<uint32_t>(), dp.as<uint32_t>(),
                   dC.as<uint32_t>(), dGs.as<uint32_t>(), dX.as<uint32_t>(), dY.as<uint32_t>(), dA1.as<uint32_t>(),
                   dA2.as<uint32_t>(), ctx->v_frames.as<uint8_t>(), combG, combg};
  modp::PolyArgs PA{dco.as<uint32_t>(), dord.as<uint32_t>(), dpos.as<uint32_t>(), dp.as<uint32_t>(), (uint32_t)t,
                    (uint32_t)n};
  MPVSS_TRY(deal_kernels(ctx, B, t, 1, n, [&] { return modp::launch_poly(PA, ctx->stream); }));
  MPVSS_TRY(timing_end(ctx));
  // transcript (participant.rs:238-252): one all-gather of the framed rows, one hash pass, on every rank
  const uint8_t* rows = ctx->v_frames.as<uint8_t>();
  if (ctx->nranks > 1) {
    MPVSS_TRY(comm_allgather(ctx, ctx->v_frames.p, ctx->v_gather.p, rpr * GEOM.row()));
    MPVSS_CUDA(ctx, ctx->v_ordered.ensure(n_total * GEOM.row()));
    MPVSS_TRY(comm_reorder_rows(ctx, ctx->v_gather.p, ctx->v_ordered.p, n_total, GEOM.row()));
    rows = ctx->v_ordered.as<uint8_t>();
  }
  sha2::Sha256 h;
  MPVSS_TRY(transcript::fetch_and_hash(ctx, rows, n_total, ctx->nranks, GEOM, h, true));
  uint8_t digest[32];
  h.finalize(digest);
  challenge_from_digest(ctx, digest, challenge_out);
  // responses r_i = (w_i - p_i * c) mod (q-1) on the device (participant.rs:255-264, modp.rs:180-192)
  MPVSS_TRY(h2d(ctx, dc, challenge_out, EB));
  if (n) {
    modp::RespArgs RA{dord.as<uint32_t>(), dp.as<uint32_t>(), dw.as<uint32_t>(), dc.as<uint32_t>(), dR.as<uint32_t>(),
                      (uint32_t)n, EW};
    MPVSS_CUDA(ctx, modp::launch_resp(RA, ctx->stream));
    ctx->last_launches += 1;
  }
  const void* dev_rows[3] = {dY.p, dR.p, dX.p};
  uint8_t* host_rows[3] = {shares_out, responses_out, x_out};
  const size_t widths[3] = {EB, EB, EB};
  MPVSS_TRY(transcript::gather_rows(ctx, dev_rows, host_rows, widths, x_out ? 3 : 2, n, n_total));
  uint8_t gs[EB];
  MPVSS_TRY(d2h(ctx, commitments_out, dC, t * EB));
  MPVSS_TRY(d2h(ctx, gs, dGs, EB));
  MPVSS_TRY(sync(ctx));
  mask_secret(ctx, secret, secret_len, gs, u_out);
  // the scratch buffers held secrets (coefficients, P(i), witnesses)
  for (DevBuf* b : {&dco, &dp, &dw, &ds}) MPVSS_CUDA(ctx, cudaMemsetAsync(b->p, 0, b->cap, ctx->stream));
  return sync(ctx);
}

// ------------------------------------------------------- distribute_secrets ----
// Many dealings in one pass: the launches of distribute run once over every box (C over all coefficients, G^s over
// the boxes' a_0, P(i) of every instance by the multi-box poly_boxes kernel, X / Y / a1 / a2 and the frames over all
// instances), the rows come to the host in one copy and each box's row range is hashed into its own challenge, and
// one response launch takes one challenge per instance.  ModpGroup rejects no box.  Only scratch buffers are used,
// so the staged single-box verify state stays valid.
int distribute_batch(mpvss_ctx* ctx, size_t nb, const size_t* nv, const size_t* tv, const uint8_t* secrets,
                     const uint8_t* coeffs, const uint8_t* witnesses, const uint8_t* publickeys,
                     uint8_t* commitments_out, uint8_t* shares_out, uint8_t* challenges_out, uint8_t* responses_out,
                     uint8_t* u_out, uint8_t* x_out, int* status_out) {
  const std::vector<uint32_t> order = order_limbs(ctx);
  if (order[EW - 1] != 0xffffffffu || order[EW - 2] != 0xffffffffu)
    return mpvss_fail(ctx, MPVSS_ERR_UNSUPPORTED,
                      "distribute_secrets: scalar kernels need an order with all-ones top limbs");
  std::vector<size_t> noff(nb + 1, 0), toff(nb + 1, 0);
  for (size_t b = 0; b < nb; ++b) {
    noff[b + 1] = noff[b] + nv[b];
    toff[b + 1] = toff[b] + tv[b];
  }
  const size_t N = noff[nb], Tt = toff[nb];
  // per instance: its position, then its box's first coefficient row, t_b and first instance row (poly_boxes_body)
  std::vector<uint32_t> idx(4 * N);
  std::vector<uint8_t> s_le(nb * EB);
  for (size_t b = 0; b < nb; ++b) {
    // s = a_0 mod (q-1)  (participant.rs:267)
    big::to_le(big::mod(big::from_le(coeffs + toff[b] * EB, EB), ctx->qm1), s_le.data() + b * EB, EB);
    for (size_t i = noff[b]; i < noff[b + 1]; ++i) {
      idx[i] = (uint32_t)(i - noff[b] + 1);
      idx[N + i] = (uint32_t)toff[b];
      idx[2 * N + i] = (uint32_t)tv[b];
      idx[3 * N + i] = (uint32_t)noff[b];
    }
  }
  DevBuf &dco = ctx->buf(0), &dp = ctx->buf(1), &dw = ctx->buf(2), &dpk = ctx->buf(3), &dC = ctx->buf(4),
         &dX = ctx->buf(5), &dY = ctx->buf(6), &dA1 = ctx->buf(7), &dA2 = ctx->buf(8), &dGs = ctx->buf(9),
         &ds = ctx->buf(10), &dord = ctx->buf(11), &didx = ctx->buf(12), &dR = ctx->buf(13), &dc = ctx->buf(14),
         &dfr = ctx->buf(15);
  MPVSS_TRY(h2d(ctx, dco, coeffs, Tt * EB));
  MPVSS_TRY(h2d(ctx, dord, order.data(), EB));
  MPVSS_TRY(h2d(ctx, didx, idx.data(), idx.size() * 4));
  MPVSS_TRY(h2d(ctx, ds, s_le.data(), nb * EB));
  MPVSS_TRY(h2d(ctx, dw, witnesses, N * EB));
  MPVSS_TRY(h2d(ctx, dpk, publickeys, N * EB));
  for (DevBuf* b : {&dp, &dX, &dY, &dA1, &dA2, &dR, &dc}) MPVSS_CUDA(ctx, b->ensure(N * EB));
  MPVSS_CUDA(ctx, dC.ensure(Tt * EB));
  MPVSS_CUDA(ctx, dGs.ensure(nb * EB));
  MPVSS_CUDA(ctx, dfr.ensure(N * GEOM.row()));
  const uint32_t *combG, *combg;
  MPVSS_TRY(comb_table(ctx, 0, &combG));
  MPVSS_TRY(comb_table(ctx, 1, &combg));
  timing_begin(ctx);
  const DealBufs B{dco.as<uint32_t>(), ds.as<uint32_t>(), dw.as<uint32_t>(), dpk.as<uint32_t>(), dp.as<uint32_t>(),
                   dC.as<uint32_t>(), dGs.as<uint32_t>(), dX.as<uint32_t>(), dY.as<uint32_t>(), dA1.as<uint32_t>(),
                   dA2.as<uint32_t>(), dfr.as<uint8_t>(), combG, combg};
  const uint32_t* di = didx.as<uint32_t>();
  modp::PolyBoxesArgs PA{dco.as<uint32_t>(), dord.as<uint32_t>(), di, di + N, di + 2 * N, di + 3 * N, dp.as<uint32_t>(),
                         (uint32_t)N};
  MPVSS_TRY(deal_kernels(ctx, B, Tt, nb, N, [&] { return modp::launch_poly_boxes(PA, ctx->stream); }));
  MPVSS_TRY(timing_end(ctx));
  PinBuf& host = ctx->pin(0);
  MPVSS_CUDA(ctx, host.ensure(N * GEOM.row()));
  uint8_t* rows = host.as<uint8_t>();
  MPVSS_TRY(d2h(ctx, rows, dfr, N * GEOM.row()));
  MPVSS_TRY(sync(ctx));
  // transcript per box (participant.rs:238-252), its challenge repeated for every instance of the box
  std::vector<uint8_t> cexp(N * EB);
  for (size_t b = 0; b < nb; ++b) {
    sha2::Sha256 h;
    transcript::hash_ordered(h, rows, noff[b], noff[b + 1], GEOM);
    uint8_t digest[32];
    h.finalize(digest);
    challenge_from_digest(ctx, digest, challenges_out + b * EB);
    for (size_t i = noff[b]; i < noff[b + 1]; ++i) memcpy(cexp.data() + i * EB, challenges_out + b * EB, EB);
  }
  // responses r_i = (w_i - p_i * c_b) mod (q-1) on the device (participant.rs:255-264, modp.rs:180-192)
  MPVSS_TRY(h2d(ctx, dc, cexp.data(), N * EB));
  modp::RespArgs RA{dord.as<uint32_t>(), dp.as<uint32_t>(), dw.as<uint32_t>(), dc.as<uint32_t>(), dR.as<uint32_t>(),
                    (uint32_t)N, EW, EW};
  MPVSS_CUDA(ctx, modp::launch_resp(RA, ctx->stream));
  ctx->last_launches += 1;
  std::vector<uint8_t> gs(nb * EB);
  MPVSS_TRY(d2h(ctx, shares_out, dY, N * EB));
  MPVSS_TRY(d2h(ctx, responses_out, dR, N * EB));
  if (x_out) MPVSS_TRY(d2h(ctx, x_out, dX, N * EB));
  MPVSS_TRY(d2h(ctx, commitments_out, dC, Tt * EB));
  MPVSS_TRY(d2h(ctx, gs.data(), dGs, nb * EB));
  MPVSS_TRY(sync(ctx));
  for (size_t b = 0; b < nb; ++b) {
    mask_secret(ctx, secrets + b * EB, EB, gs.data() + b * EB, u_out + b * EB);
    status_out[b] = MPVSS_OK;
  }
  // the scratch buffers held secrets (coefficients, P(i), witnesses)
  for (DevBuf* b : {&dco, &dp, &dw, &ds}) MPVSS_CUDA(ctx, cudaMemsetAsync(b->p, 0, b->cap, ctx->stream));
  return sync(ctx);
}

// ------------------------------------------------------------------ extract ----
// out[i] = v[i]^-1 mod g for n device values, none of them 0 mod g (Montgomery's trick as a tree): products of
// pairs (m, m + h) level by level on the device, ONE inversion of the root on the host (big::modinv_odd), and the
// tree walked back down with two products per node.  3 n products and 36 small launches instead of n
// exponentiations by g - 2, each 2560 products deep (6 - 8 ms at n = 2731 for a launch that is one warp per
// scheduler and therefore latency-bound).  v and out may not overlap.
static int dev_batch_inverse_g(mpvss_ctx* ctx, const uint32_t* v, size_t n, uint32_t* out) {
  const uint32_t* Kg = ctx->consts_g.as<uint32_t>();
  size_t N = 1, L = 0;
  while (N < n) N *= 2, ++L;
  DevBuf &tree = ctx->buf(21), &ia = ctx->buf(22), &ib = ctx->buf(23);
  MPVSS_CUDA(ctx, tree.ensure(2 * N * EB));
  MPVSS_CUDA(ctx, ia.ensure(N * EB));
  MPVSS_CUDA(ctx, ib.ensure(N * EB));
  uint32_t* T = tree.as<uint32_t>();
  MPVSS_CUDA(ctx, cudaMemcpyAsync(T, v, n * EB, cudaMemcpyDeviceToDevice, ctx->stream));
  if (N > n) {  // pad with ones
    std::vector<uint32_t> ones((N - n) * EW, 0);
    for (size_t i = 0; i < N - n; ++i) ones[i * EW] = 1;
    MPVSS_CUDA(ctx, cudaMemcpyAsync(T + n * EW, ones.data(), (N - n) * EB, cudaMemcpyHostToDevice, ctx->stream));
    MPVSS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `ones` is pageable and goes out of scope
  }
  std::vector<size_t> off(L + 1, 0);
  for (size_t l = 1; l <= L; ++l) off[l] = off[l - 1] + (N >> (l - 1));
  for (size_t l = 1; l <= L; ++l) {
    const size_t h = N >> l;
    MPVSS_TRY(dev_mul(ctx, Kg, T + off[l - 1] * EW, EW, T + (off[l - 1] + h) * EW, EW, 0, h, T + off[l] * EW));
  }
  uint8_t root[EB];
  MPVSS_CUDA(ctx, cudaMemcpyAsync(root, T + off[L] * EW, EB, cudaMemcpyDeviceToHost, ctx->stream));
  MPVSS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  big::Int inv;
  if (!big::modinv_odd(big::from_le(root, EB), ctx->g, &inv))
    return mpvss_fail(ctx, MPVSS_ERR_ARG, "batch inversion: an element is 0 modulo the subgroup order");
  big::to_le(inv, root, EB);
  uint32_t *cur = ia.as<uint32_t>(), *nxt = ib.as<uint32_t>();
  MPVSS_CUDA(ctx, cudaMemcpyAsync(cur, root, EB, cudaMemcpyHostToDevice, ctx->stream));
  MPVSS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  memset(root, 0, EB);  // a function of secret values when the batch holds private keys
  std::fill(inv.begin(), inv.end(), 0u);
  for (size_t l = L; l >= 1; --l) {  // inverse of a child = inverse of the parent * the sibling
    const size_t h = N >> l;
    MPVSS_TRY(dev_mul(ctx, Kg, cur, EW, T + (off[l - 1] + h) * EW, EW, 0, h, nxt));
    MPVSS_TRY(dev_mul(ctx, Kg, cur, EW, T + off[l - 1] * EW, EW, 0, h, nxt + h * EW));
    std::swap(cur, nxt);
  }
  MPVSS_CUDA(ctx, cudaMemcpyAsync(out, cur, n * EB, cudaMemcpyDeviceToDevice, ctx->stream));
  return MPVSS_OK;
}

// Per-share Fiat-Shamir transcripts on the device (SURVEY 8 f1): frame (h1, h2, a1, a2) per share, one SHA-256
// chain per thread, and hash_to_scalar's second SHA-256 (modp.rs:142-148; 256 < 2047 bits, so no reduction):
// challenges as `stride`-limb little-endian scalars (64 = boundary scalars, 8 = just the hash).  The launches are
// added to the kernel time of the call.
static int share_challenges(mpvss_ctx* ctx, const uint32_t* h1, const uint32_t* h2, const uint32_t* a1, const uint32_t* a2,
                            size_t n, uint32_t* c_out, uint32_t stride) {
  DevBuf& drows = ctx->buf(14);
  MPVSS_CUDA(ctx, drows.ensure(n * 4 * modp::FRAME_BYTES));
  const float ms0 = ctx->last_ms;
  const int l0 = ctx->last_launches;
  timing_begin(ctx);
  modp::FrameArgs FA{h1, h2, a1, a2, drows.as<uint8_t>(), (uint32_t)n};
  MPVSS_CUDA(ctx, modp::launch_frames(FA, ctx->stream));
  shadev::RowHashArgs HA{drows.as<uint8_t>(), 4u * modp::FRAME_BYTES, (uint32_t)modp::FRAME_BYTES, c_out, stride, nullptr,
                         (uint32_t)n, 0u};
  MPVSS_CUDA(ctx, shadev::launch_row_hash(HA, ctx->stream));
  timing_launch(ctx, 2);
  MPVSS_TRY(timing_end(ctx));
  ctx->last_ms += ms0;
  ctx->last_launches += l0;
  return MPVSS_OK;
}

int extract_shares(mpvss_ctx* ctx, size_t n, const uint8_t* private_keys, const uint8_t* witnesses,
                   const uint8_t* enc_shares, uint8_t* publickeys_out, uint8_t* shares_out, uint8_t* challenges_out,
                   uint8_t* responses_out, int* status_out) {
  MPVSS_TRY(check_args(ctx, n > 0 && private_keys && witnesses && enc_shares && publickeys_out && shares_out &&
                                challenges_out && responses_out,
                       "extract_shares: bad arguments"));
  const uint32_t* K = ctx->consts_q.as<uint32_t>();
  const uint32_t* Kg = ctx->consts_g.as<uint32_t>();
  const uint32_t* G = ctx->gens.as<uint32_t>();
  // sk^-1 mod (q-1), q-1 = 2g (util.rs:33-41 via participant.rs:314): by CRT it is the odd
  // representative of sk^(g-2) mod g; it exists iff sk is odd and not a multiple of g.
  std::vector<uint8_t> skg(n * EB);
  std::vector<int> st(n, MPVSS_OK);
  for (size_t i = 0; i < n; ++i) {
    big::Int sk = big::mod(big::from_le(private_keys + i * EB, EB), ctx->qm1);
    big::Int r = big::mod(sk, ctx->g);
    if (!big::is_odd(sk) || big::is_zero(r)) {
      st[i] = MPVSS_ERR_NOT_INVERTIBLE;
      r = big::from_u64(1);  // keeps the batch inversion below defined; this instance's outputs are not used
    }
    big::to_le(r, skg.data() + i * EB, EB);
  }
  DevBuf &dsk = ctx->buf(0), &dskg = ctx->buf(1), &dinv = ctx->buf(3), &dw = ctx->buf(4),
         &dY = ctx->buf(5), &dpk = ctx->buf(6), &dS = ctx->buf(7), &dA1 = ctx->buf(8), &dA2 = ctx->buf(9);
  MPVSS_TRY(h2d(ctx, dsk, private_keys, n * EB));
  MPVSS_TRY(h2d(ctx, dskg, skg.data(), n * EB));
  MPVSS_TRY(h2d(ctx, dw, witnesses, n * EB));
  MPVSS_TRY(h2d(ctx, dY, enc_shares, n * EB));
  for (DevBuf* b : {&dinv, &dpk, &dS, &dA1, &dA2}) MPVSS_CUDA(ctx, b->ensure(n * EB));
  timing_begin(ctx);
  MPVSS_TRY(dev_batch_inverse_g(ctx, dskg.as<uint32_t>(), n, dinv.as<uint32_t>()));  // one inversion for all n
  MPVSS_TRY(timing_end(ctx));
  std::vector<uint8_t> inv(n * EB);
  MPVSS_TRY(d2h(ctx, inv.data(), dinv, n * EB));
  MPVSS_TRY(sync(ctx));
  for (size_t i = 0; i < n; ++i) {
    big::Int x = big::from_le(inv.data() + i * EB, EB);
    if (!big::is_odd(x)) x = big::add(x, ctx->g);
    big::to_le(x, inv.data() + i * EB, EB);
  }
  MPVSS_TRY(h2d(ctx, dinv, inv.data(), n * EB));
  const uint32_t skw = 512, ww = 512;  // secret exponents: full window count, whatever their size
  const uint32_t* combG;
  MPVSS_TRY(comb_table(ctx, 0, &combG));
  float ms0 = ctx->last_ms;
  int l0 = ctx->last_launches;
  timing_begin(ctx);
  // pk = G^sk (participant.rs:306), S = Y^(1/sk) (:316), a1 = G^w, a2 = S^w (:331-332)
  MPVSS_TRY(dev_exp2(ctx, K, G, 0, dsk.as<uint32_t>(), EW, skw, nullptr, 0, nullptr, 0, 0, n, dpk.as<uint32_t>(),
                     nullptr, combG));
  MPVSS_TRY(dev_exp2(ctx, K, dY.as<uint32_t>(), EW, dinv.as<uint32_t>(), EW, 512, nullptr, 0, nullptr, 0, 0, n,
                     dS.as<uint32_t>()));
  MPVSS_TRY(dev_exp2(ctx, K, G, 0, dw.as<uint32_t>(), EW, ww, nullptr, 0, nullptr, 0, 0, n, dA1.as<uint32_t>(),
                     nullptr, combG));
  MPVSS_TRY(dev_exp2(ctx, K, dS.as<uint32_t>(), EW, dw.as<uint32_t>(), EW, ww, nullptr, 0, nullptr, 0, 0, n,
                     dA2.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  ctx->last_ms += ms0;
  ctx->last_launches += l0;
  {
    // challenge per share from the transcript (pk, Y, a1, a2) (participant.rs:330-340) and the response
    // r = w - sk*c mod (q-1) (dleq.rs:42-50 with modp.rs:180-192), both on the device: a1 / a2 stay there
    const std::vector<uint32_t> order = order_limbs(ctx);
    DevBuf &dord = ctx->buf(11), &dch = ctx->buf(12), &dR = ctx->buf(13);
    MPVSS_TRY(h2d(ctx, dord, order.data(), EB));
    MPVSS_CUDA(ctx, dch.ensure(n * EB));
    MPVSS_CUDA(ctx, dR.ensure(n * EB));
    MPVSS_TRY(share_challenges(ctx, dpk.as<uint32_t>(), dY.as<uint32_t>(), dA1.as<uint32_t>(), dA2.as<uint32_t>(), n,
                               dch.as<uint32_t>(), EW));
    modp::RespArgs RA{dord.as<uint32_t>(), dsk.as<uint32_t>(), dw.as<uint32_t>(), dch.as<uint32_t>(), dR.as<uint32_t>(),
                      (uint32_t)n, EW, EW};
    MPVSS_CUDA(ctx, modp::launch_resp(RA, ctx->stream));
    ctx->last_launches += 1;
    MPVSS_TRY(d2h(ctx, publickeys_out, dpk, n * EB));
    MPVSS_TRY(d2h(ctx, shares_out, dS, n * EB));
    MPVSS_TRY(d2h(ctx, challenges_out, dch, n * EB));
    MPVSS_TRY(d2h(ctx, responses_out, dR, n * EB));
    // the scratch buffers held secrets (private keys, inverses, witnesses)
    for (DevBuf* b : {&dsk, &dskg, &dinv, &dw}) MPVSS_CUDA(ctx, cudaMemsetAsync(b->p, 0, b->cap, ctx->stream));
    MPVSS_TRY(sync(ctx));
  }
  if (status_out) memcpy(status_out, st.data(), n * sizeof(int));
  return MPVSS_OK;
}

// ------------------------------------------------------------- verify_share ----
int verify_shares(mpvss_ctx* ctx, size_t n, const uint8_t* publickeys, const uint8_t* shares,
                  const uint8_t* enc_shares, const uint8_t* challenges, const uint8_t* responses, int* ok_out) {
  MPVSS_TRY(check_args(ctx, n > 0 && publickeys && shares && enc_shares && challenges && responses && ok_out,
                       "verify_shares: bad arguments"));
  std::vector<uint8_t> gen(EB, 0);
  gen[0] = 2;  // DLEQ(G, pk, S, Y)  participant.rs:378-385
  // a1 / a2 stay on the device (nullptr outputs): buf(1) = pk, buf(3) = Y, buf(6) = a1, buf(7) = a2 afterwards
  MPVSS_TRY(dleq_verify_commit(ctx, gen.data(), publickeys, shares, enc_shares, responses, challenges, EB, n, nullptr,
                               nullptr));
  // dleq.rs:275-302: per share, the transcript (h1, h2, a1, a2) = (pk, Y, a1, a2) hashed on the device; the
  // 256-bit challenges come back (32 bytes per share) and are compared here
  DevBuf& dch = ctx->buf(12);
  MPVSS_CUDA(ctx, dch.ensure(n * 32));
  MPVSS_TRY(share_challenges(ctx, ctx->buf(1).as<uint32_t>(), ctx->buf(3).as<uint32_t>(), ctx->buf(6).as<uint32_t>(),
                             ctx->buf(7).as<uint32_t>(), n, dch.as<uint32_t>(), 8));
  std::vector<uint8_t> c(n * 32);
  MPVSS_TRY(d2h(ctx, c.data(), dch, n * 32));
  MPVSS_TRY(sync(ctx));
  for (size_t i = 0; i < n; ++i) {
    const uint8_t* given = challenges + i * EB;
    bool same = memcmp(c.data() + i * 32, given, 32) == 0;
    for (size_t k = 32; k < EB && same; ++k) same = given[k] == 0;
    ok_out[i] = same;
  }
  return MPVSS_OK;
}

// -------------------------------------------------------------- reconstruct ----
// The steps after a Lagrange launch that left `parts` partial products of n numerators / denominators mod g and
// their sign flags in dnum / dden / dneg: the part products, den^-1 by one batch inversion, lambda = num * den^-1
// into dlam (which may be dnum), the end of the timing bracket the Lagrange launch opened, then lam on the host
// with the sign folded into the exponent: S^(-lambda) = S^((q-1) - lambda).
static int lagrange_lambdas(mpvss_ctx* ctx, DevBuf& dnum, DevBuf& dden, DevBuf& dneg, DevBuf& dinv, DevBuf& dlam,
                            size_t n, size_t parts, std::vector<uint8_t>& lam) {
  const uint32_t* Kg = ctx->consts_g.as<uint32_t>();
  for (size_t half = parts / 2; half >= 1; half /= 2)  // rows [0, half n) *= rows [half n, 2 half n), mod g
    for (DevBuf* b : {&dnum, &dden})
      MPVSS_TRY(dev_mul(ctx, Kg, b->as<uint32_t>(), EW, b->as<uint32_t>() + half * n * EW, EW, 0, half * n,
                        b->as<uint32_t>()));
  // den^-1 mod g: the denominators are products of non-zero integers below 2^31 < g, so none is 0 mod g
  MPVSS_TRY(dev_batch_inverse_g(ctx, dden.as<uint32_t>(), n, dinv.as<uint32_t>()));
  MPVSS_TRY(dev_mul(ctx, Kg, dnum.as<uint32_t>(), EW, dinv.as<uint32_t>(), EW, 0, n, dlam.as<uint32_t>()));
  MPVSS_TRY(timing_end(ctx));
  lam.resize(n * EB);
  std::vector<uint32_t> negf(parts * n);
  MPVSS_TRY(d2h(ctx, lam.data(), dlam, n * EB));
  MPVSS_TRY(d2h(ctx, negf.data(), dneg, parts * n * 4));
  MPVSS_TRY(sync(ctx));
  for (size_t i = 0; i < n; ++i) {
    for (size_t p = 1; p < parts; ++p) negf[i] ^= negf[p * n + i];
    if (!negf[i]) continue;
    big::Int l = big::from_le(lam.data() + i * EB, EB);
    if (!big::is_zero(l)) big::to_le(big::sub(ctx->qm1, l), lam.data() + i * EB, EB);
  }
  return MPVSS_OK;
}

// Many reconstruct calls in one (mpvss_reconstruct_secrets; mpvss_reconstruct is a batch of one box).  The live
// boxes' positions and shares are concatenated, the boxes that take the direct method first.  One box-aware
// Lagrange launch, the part products, ONE batch inversion mod g over every box's denominators, and the signs
// folded on the host: lambda_i = prod_{j != i} j / (j - i) mod g, S^(-lambda) = S^((q-1) - lambda)
// (participant.rs:535-558, element_inverse modp.rs:138-140).  Then multi_exp_direct over every direct box's
// shares, and the bucket method box after box for the others.
int reconstruct_batch(mpvss_ctx* ctx, size_t nb, const size_t* kv, const int64_t* positions, const uint8_t* shares,
                      const uint8_t* u, uint8_t* secrets_out, uint8_t* gs_out, int* status_out) {
  memset(secrets_out, 0, nb * EB);
  if (gs_out) memset(gs_out, 0, nb * EB);
  ctx->last_ms = 0.f;
  ctx->last_launches = 0;
  std::vector<size_t> live;  // boxes whose positions are in range and distinct
  std::vector<uint32_t> sorted;
  for (size_t b = 0, off = 0; b < nb; off += kv[b], ++b) {
    bool ok = positions_u32(positions + off, kv[b], sorted) == kv[b];
    if (ok) {
      std::sort(sorted.begin(), sorted.end());
      ok = std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end();
    }
    status_out[b] = ok ? MPVSS_OK : MPVSS_ERR_ARG;
    if (ok) live.push_back(b);
  }
  if (live.empty()) return MPVSS_OK;
  // a lone box chooses as multi_exp does; in a batch a box joins the direct launch below msm_batch_threshold
  const size_t threshold = live.size() == 1 ? (size_t)ctx->msm_threshold : mpvss_ctx::msm_batch_threshold;
  auto buckets = [&](size_t b) { return ctx->modp_msm == 1 || (ctx->modp_msm == 2 && kv[b] >= threshold); };
  std::stable_partition(live.begin(), live.end(), [&](size_t b) { return !buckets(b); });
  LiveBoxes B = pack_live_boxes(nb, kv, positions, shares, EB, live);
  const size_t L = live.size(), n = B.n;
  const std::vector<uint32_t> &start = B.start, &cnt = B.cnt;
  size_t L_direct = 0, kmax = 0;  // boxes of the direct launch
  for (size_t j = 0; j < L; ++j) {
    kmax = std::max<size_t>(kmax, cnt[j]);
    if (!buckets(live[j])) L_direct = j + 1;
  }
  // multi_exp_buckets holds buf(15..19) and dev_batch_inverse_g buf(21..23)
  DevBuf &dshares = ctx->buf(0), &dexp = ctx->buf(1), &dpow = ctx->buf(2), &dplan = ctx->buf(4), &didx = ctx->buf(10),
         &dord = ctx->buf(11), &dnum = ctx->buf(12), &dden = ctx->buf(13), &dneg = ctx->buf(14), &dinv = ctx->buf(20);
  const std::vector<uint32_t> order = order_limbs(ctx);
  MPVSS_TRY(h2d(ctx, didx, B.idx.data(), 3 * n * 4));
  MPVSS_TRY(h2d(ctx, dord, order.data(), EB));
  MPVSS_TRY(h2d(ctx, dshares, B.rows(shares), n * EB));
  // the k-term products are cut into `parts` ranges (more, shorter threads), multiplied together mod g afterwards
  const size_t parts = kmax >= 64 ? 8 : 1;
  for (DevBuf* b : {&dnum, &dden}) MPVSS_CUDA(ctx, b->ensure(parts * n * EB));
  MPVSS_CUDA(ctx, dinv.ensure(n * EB));
  MPVSS_CUDA(ctx, dneg.ensure(parts * n * 4));
  MPVSS_CUDA(ctx, dpow.ensure(n * EB));
  const uint32_t* di = didx.as<uint32_t>();
  modp::LagrangeBoxesArgs LA{dord.as<uint32_t>(), di, di + n, di + 2 * n, dnum.as<uint32_t>(), dden.as<uint32_t>(),
                             dneg.as<uint32_t>(), (uint32_t)n, (uint32_t)parts};
  timing_begin(ctx);
  MPVSS_CUDA(ctx, modp::launch_lagrange_boxes(LA, ctx->stream));
  timing_launch(ctx);
  std::vector<uint8_t> lam;
  MPVSS_TRY(lagrange_lambdas(ctx, dnum, dden, dneg, dinv, dnum, n, parts, lam));  // lambda in place of num
  const float ms_lambda = ctx->last_ms;
  const int launches_lambda = ctx->last_launches;
  MPVSS_TRY(h2d(ctx, dexp, lam.data(), n * EB));
  const size_t n_direct = L_direct ? (size_t)start[L_direct - 1] + cnt[L_direct - 1] : 0;  // rows of the direct boxes
  std::vector<uint32_t> level_end;
  if (L_direct) MPVSS_TRY(plan_product_tree(ctx, start.data(), cnt.data(), L_direct, dplan, level_end));
  timing_begin(ctx);
  if (L_direct)
    MPVSS_TRY(multi_exp_direct(ctx, dshares, dexp, windows_for(lam.data(), EB, n_direct), n_direct, level_end, dpow,
                               dplan));
  for (size_t j = L_direct; j < L; ++j) {
    DevBuf vb, ve, vo;  // views of box j's rows (not owned)
    vb.p = dshares.as<uint32_t>() + (size_t)start[j] * EW;
    ve.p = dexp.as<uint32_t>() + (size_t)start[j] * EW;
    vo.p = dpow.as<uint32_t>() + (size_t)start[j] * EW;
    const uint32_t windows = (windows_for(lam.data() + (size_t)start[j] * EB, EB, cnt[j]) + 1) / 2;
    MPVSS_TRY(multi_exp_buckets(ctx, vb, ve, windows, cnt[j], vo));
  }
  MPVSS_TRY(timing_end(ctx));
  ctx->last_ms += ms_lambda;
  ctx->last_launches += launches_lambda;
  // each box's result is its first row; the rows up to the last box's hold them all (one row for one box)
  std::vector<uint8_t> host(((size_t)start[L - 1] + 1) * EB);
  MPVSS_TRY(d2h(ctx, host.data(), dpow, host.size()));
  MPVSS_TRY(sync(ctx));
  for (size_t j = 0; j < L; ++j) {
    const size_t b = live[j];
    const uint8_t* gs = host.data() + (size_t)start[j] * EB;
    big::to_be(big::bxor(u_mask(ctx, gs), big::from_be(u + b * EB, EB)), secrets_out + b * EB, EB);
    if (gs_out) memcpy(gs_out + b * EB, gs, EB);
  }
  return MPVSS_OK;
}

}  // namespace modp_api

const GroupOps modp_ops = [] {
  GroupOps o{};
  o.init = modp_api::init;
  o.batch_exp = modp_api::batch_exp;
  o.fixed_base_exp = modp_api::fixed_base_exp;
  o.batch_mul = modp_api::batch_mul;
  o.poly_eval_exp = modp_api::poly_eval_exp;
  o.dleq_verify_commit = modp_api::dleq_verify_commit;
  o.dleq_prove_commit = modp_api::dleq_prove_commit;
  o.multi_exp = modp_api::multi_exp;
  o.verify_stage = modp_api::verify_stage;
  o.verify_run = modp_api::verify_run;
  o.verify_batch = modp_api::verify_batch;
  o.scalar_poly_eval = modp_api::scalar_poly_eval;
  o.distribute = modp_api::distribute;
  o.distribute_batch = modp_api::distribute_batch;
  o.extract_shares = modp_api::extract_shares;
  o.verify_shares = modp_api::verify_shares;
  o.reconstruct_batch = modp_api::reconstruct_batch;
  return o;
}();
