// Secp256k1Group / Ristretto255Group side of the C ABI: host orchestration of the
// elliptic-curve kernels plus the CPU-resident pieces (Fiat-Shamir SHA-256 transcript,
// hash_to_scalar, responses, U mask).  One template, two trait structs.
//
// Reference semantics restated here (paths under /root/reference/src; secp / ristretto):
//   transcript framing            dleq.rs:58-61, 87-99
//   hash_to_scalar                secp256k1.rs:121-131 (SHA-256, BE, mod n) /
//                                 ristretto255.rs:196-205 (SHA-512, LE, wide reduction mod l)
//   responses r = w - alpha*c     participant.rs:1221-1231 / 1679-1688
//   U mask                        participant.rs:1234-1260 / 1691-1703, unmask :1495-1512 / 1938-1949
//   Lagrange sign handling        participant.rs:1518-1557 / 1955-2002
#include "ctx.h"
#include "ec_launch.h"
#include "hash_launch.h"
#include "sha2.h"
#include "transcript.h"

namespace {

constexpr size_t SB = 32;  // scalar bytes at the boundary

big::Int hex_int(const char* s) {
  size_t n = strlen(s);
  std::vector<uint8_t> be((n + 1) / 2, 0);
  for (size_t i = 0; i < n; ++i) {
    char c = s[n - 1 - i];
    uint8_t v = c <= '9' ? c - '0' : (c | 32) - 'a' + 10;
    be[be.size() - 1 - i / 2] |= v << (4 * (i % 2));
  }
  return big::from_be(be.data(), be.size());
}
void put8(uint32_t* dst, const big::Int& v) {
  for (int i = 0; i < 8; ++i) dst[i] = i < (int)v.size() ? v[i] : 0;
}
void fill_modulus(fp256::Modulus& M, const big::Int& m) {
  big::Int R(9, 0);
  R[8] = 1;
  big::Int one = big::mod(R, m);
  put8(M.m, m);
  put8(M.one, one);
  put8(M.r2, big::mulmod(one, one, m));
  uint32_t inv = 1, m0 = m[0];
  for (int i = 0; i < 5; ++i) inv *= 2u - m0 * inv;
  M.np = 0u - inv;
}
// Field multiplications / squarings of the point operations as the kernels execute them (secp.cuh /
// rist.cuh); used only to count the algorithmic work of a Horner launch for the roofline figure.
struct OpCost {
  uint32_t m, s;
};
struct SecpTraits {
  using Cv = secp::SecpCurve;
  // dbl-2009-l 2M+5S; add-2007-bl 11M+5S; madd-2007-bl 7M+4S; small_mul_iso set-up (2P, 3P, two rescalings,
  // scale, final Z product) 16M+9S; the first window addition lands on the identity and is free
  static constexpr OpCost DBL{2, 5}, DBL_NOT{2, 5}, ADD{11, 5}, MADD{7, 4}, WIN_ADD{7, 4}, SMALL_FIXED{16, 9};
  static constexpr bool TOP_ADD_FREE = true;
  static constexpr size_t EB = 33;
  static constexpr bool SCALAR_BE = true;
  static big::Int order() { return hex_int("fffffffffffffffffffffffffffffffebaaedce6af48a03bbfd25e8cd0364141"); }
  static void consts(secp::Consts& C) {
    big::Int p = hex_int("fffffffffffffffffffffffffffffffffffffffffffffffffffffffefffffc2f");
    fill_modulus(C.P, p);
    fill_modulus(C.N, order());
    put8(C.b7, big::from_u64(7));  // base-field constants in plain representation (fpspecial.cuh)
    put8(C.gx, hex_int("79be667ef9dcbbac55a06295ce870b07029bfcdb2dce28d959f2815b16f81798"));
    put8(C.gy, hex_int("483ada7726a3c4655da4fbfc0e1108a8fd17b448a68554199c47d08ffb10d4b8"));
    put8(C.sqrt_e, big::shr1(big::shr1(big::add(p, big::from_u64(1)))));
  }
  static void generator(uint8_t* out) {  // secp256k1.rs:78-85 (both generators are G)
    big::Int gx = hex_int("79be667ef9dcbbac55a06295ce870b07029bfcdb2dce28d959f2815b16f81798");
    out[0] = 2;
    big::to_be(gx, out + 1, 32);
  }
  // secp256k1.rs:121-131: SHA-256, big-endian, reduced mod n
  static big::Int hash_to_scalar(const uint8_t* data, size_t len, const big::Int& n) {
    uint8_t h[32];
    sha2::sha256(data, len, h);
    return big::mod(big::from_be(h, 32), n);
  }
  // participant.rs:1244-1259: SHA-256(bytes) -> Scalar::from_repr(..).unwrap() -> mod n
  static bool mask_of(const uint8_t* elem, const big::Int& n, big::Int* out) {
    uint8_t h[32];
    sha2::sha256(elem, EB, h);
    big::Int v = big::from_be(h, 32);
    if (big::cmp(v, n) >= 0) return false;  // the reference would panic in from_repr().unwrap()
    *out = v;
    return true;
  }
};

struct RistTraits {
  using Cv = rist::RistCurve;
  // dbl-2008-hwcd 4M+4S (3M+4S without T); add-2008-hwcd-3 9M; adding an affine commitment 10M;
  // small_mul_ext set-up (2P, 3P) 13M+4S
  static constexpr OpCost DBL{4, 4}, DBL_NOT{3, 4}, ADD{9, 0}, MADD{10, 0}, WIN_ADD{9, 0}, SMALL_FIXED{13, 4};
  static constexpr bool TOP_ADD_FREE = false;
  static constexpr size_t EB = 32;
  static constexpr bool SCALAR_BE = false;
  static big::Int order() { return hex_int("1000000000000000000000000000000014def9dea2f79cd65812631a5cf5d3ed"); }
  static void consts(rist::Consts& C) {
    big::Int p = hex_int("7fffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffed");
    fill_modulus(C.P, p);
    fill_modulus(C.N, order());
    put8(C.d, hex_int("52036cee2b6ffe738cc740797779e89800700a4d4141d8ab75eb4dca135978a3"));
    put8(C.d2, hex_int("2406d9dc56dffce7198e80f2eef3d13000e0149a8283b156ebd69b9426b2f159"));
    put8(C.sqrt_m1, hex_int("2b8324804fc1df0b2b4d00993dfbd7a72f431806ad2fe478c4ee1b274a0ea0b0"));
    put8(C.invsqrt_a_minus_d, hex_int("786c8905cfaffca216c27b91fe01d8409d2f16175a4172be99c8fdaa805d40ea"));
    put8(C.bx, hex_int("216936d3cd6e53fec0a4e231fdd6dc5c692cc7609525a7b2c9562d608f25d51a"));
    put8(C.by, hex_int("6666666666666666666666666666666666666666666666666666666666666658"));
    big::Int e;
    big::divmod(big::sub(p, big::from_u64(5)), big::from_u64(8), &e, nullptr);
    put8(C.pm5d8, e);
  }
  static void generator(uint8_t* out) {  // RISTRETTO_BASEPOINT_POINT, ristretto255.rs:148-155
    big::Int g = hex_int("e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76");  // encoding, read big-endian
    big::to_be(g, out, 32);
  }
  // ristretto255.rs:196-205: SHA-512, little-endian, from_bytes_mod_order_wide
  static big::Int hash_to_scalar(const uint8_t* data, size_t len, const big::Int& l) {
    uint8_t h[64];
    sha2::sha512(data, len, h);
    return big::mod(big::from_le(h, 64), l);
  }
  // participant.rs:1696-1702: int_be(SHA-256(bytes)) mod l
  static bool mask_of(const uint8_t* elem, const big::Int& l, big::Int* out) {
    uint8_t h[32];
    sha2::sha256(elem, EB, h);
    *out = big::mod(big::from_be(h, 32), l);
    return true;
  }
};

int h2d(mpvss_ctx* ctx, DevBuf& b, const void* src, size_t bytes) {
  MPVSS_CUDA(ctx, b.ensure(bytes));
  MPVSS_CUDA(ctx, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return MPVSS_OK;
}
int d2h(mpvss_ctx* ctx, void* dst, const DevBuf& b, size_t bytes) {
  MPVSS_CUDA(ctx, cudaMemcpyAsync(dst, b.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return MPVSS_OK;
}
int sync(mpvss_ctx* ctx) {
  MPVSS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPVSS_OK;
}
int bad(mpvss_ctx* ctx, bool ok, const char* what) { return ok ? MPVSS_OK : mpvss_fail(ctx, MPVSS_ERR_ARG, what); }

template <class T>
struct Ec {
  using Cv = typename T::Cv;
  using Point = typename Cv::Point;
  static constexpr size_t EB = T::EB;

  static const typename Cv::Consts* K(mpvss_ctx* ctx) { return ctx->ec_consts.as<typename Cv::Consts>(); }
  static const fp256::Modulus* KN(mpvss_ctx* ctx) {
    return reinterpret_cast<const fp256::Modulus*>(ctx->ec_consts.as<char>() + sizeof(fp256::Modulus));
  }

  // boundary scalars -> device limb layout (8 little-endian u32 per scalar); report = false: a non-canonical
  // scalar returns MPVSS_ERR_ENCODING without recording a context error (per-box checks of a batch)
  static int scalars_in(mpvss_ctx* ctx, const uint8_t* s, size_t n, std::vector<uint32_t>& out, bool report = true) {
    out.resize(n * 8);
    uint32_t ord[8];
    put8(ord, ctx->ec_order);
    for (size_t i = 0; i < n; ++i) {
      // fast path, no allocation: canonical values (below the order) are just re-packed
      uint32_t* o = out.data() + i * 8;
      for (int k = 0; k < 8; ++k) {
        const uint8_t* q = s + i * SB + (T::SCALAR_BE ? 4 * (7 - k) : 4 * k);
        o[k] = T::SCALAR_BE ? ((uint32_t)q[0] << 24 | (uint32_t)q[1] << 16 | (uint32_t)q[2] << 8 | q[3])
                            : ((uint32_t)q[3] << 24 | (uint32_t)q[2] << 16 | (uint32_t)q[1] << 8 | q[0]);
      }
      bool below = false;
      for (int k = 7; k >= 0; --k)
        if (o[k] != ord[k]) {
          below = o[k] < ord[k];
          break;
        }
      if (below) continue;
      big::Int v = T::SCALAR_BE ? big::from_be(s + i * SB, SB) : big::from_le(s + i * SB, SB);
      if (big::cmp(v, ctx->ec_order) >= 0) {
        if (T::SCALAR_BE) {  // k256 Scalar::from_repr rejects non-canonical values
          if (!report) return MPVSS_ERR_ENCODING;
          return mpvss_fail(ctx, MPVSS_ERR_ENCODING, "scalar " + std::to_string(i) + " is not below the group order");
        }
        v = big::mod(v, ctx->ec_order);  // dalek Scalar::from_bytes_mod_order
      }
      put8(out.data() + i * 8, v);
    }
    return MPVSS_OK;
  }
  static void scalar_out(const big::Int& v, uint8_t* out) {
    if (T::SCALAR_BE) big::to_be(v, out, SB);
    else big::to_le(v, out, SB);
  }
  static big::Int scalar_big(const uint8_t* s) { return T::SCALAR_BE ? big::from_be(s, SB) : big::from_le(s, SB); }

  static int check_status(mpvss_ctx* ctx, const DevBuf& st, size_t n, const char* what) {
    std::vector<uint32_t> h(n);
    MPVSS_TRY(d2h(ctx, h.data(), st, n * 4));
    MPVSS_TRY(sync(ctx));
    for (size_t i = 0; i < n; ++i)
      if (h[i] == 1)
        return mpvss_fail(ctx, MPVSS_ERR_ENCODING, std::string(what) + ": invalid element encoding at index " +
                                                       std::to_string(i));
    return MPVSS_OK;
  }

  static int init(mpvss_ctx* ctx) {
    typename Cv::Consts C;
    memset(&C, 0, sizeof C);
    T::consts(C);
    ctx->ec_order = T::order();
    ctx->ec_gen.resize(EB);
    T::generator(ctx->ec_gen.data());
    MPVSS_TRY(h2d(ctx, ctx->ec_consts, &C, sizeof C));
    MPVSS_TRY(h2d(ctx, ctx->gens, ctx->ec_gen.data(), EB));
    // fixed-base table of the generator (both generators of the trait are this point): 960 affine multiples
    MPVSS_CUDA(ctx, ctx->ec_comb.ensure(ec::COMB_WORDS * 4));
    ec::CombArgs<Cv> CA{K(ctx), ctx->gens.as<uint8_t>(), ctx->ec_comb.as<uint32_t>()};
    MPVSS_CUDA(ctx, ec::launch_comb_build<Cv>(CA, ctx->stream));
    return sync(ctx);
  }

  // device-pointer launch helpers -----------------------------------------------------------
  static int dev_exp2(mpvss_ctx* ctx, const uint8_t* b1, uint32_t b1s, const uint32_t* e1, const uint8_t* b2,
                      uint32_t b2s, const uint32_t* e2, uint32_t e2s, size_t n, uint8_t* out, Point* out_jac,
                      uint32_t* status, cudaStream_t stream = nullptr, bool b1_is_generator = false) {
    ec::Exp2Args<Cv> A{K(ctx), b1, e1, b2, e2, out, out_jac, status, (uint32_t)n, b1s, 8, b2s, e2s,
                       b1_is_generator ? ctx->ec_comb.as<uint32_t>() : nullptr};
    MPVSS_CUDA(ctx, ec::launch_exp2<Cv>(A, stream ? stream : ctx->stream));
    timing_launch(ctx);
    return MPVSS_OK;
  }
  // out[i] = e[i] * G from the fixed-base table (staged through shared memory by the kernel)
  static int dev_fixed(mpvss_ctx* ctx, const uint32_t* e, size_t n, uint8_t* out) {
    ec::FixedArgs<Cv> A{K(ctx), ctx->ec_comb.as<uint32_t>(), e, out, (uint32_t)n};
    MPVSS_CUDA(ctx, ec::launch_fixed<Cv>(A, ctx->stream));
    timing_launch(ctx);
    return MPVSS_OK;
  }
  // sum `count` points per group down to one, encode the result(s) into out
  static int dev_sum_all(mpvss_ctx* ctx, Point* pts, size_t total, DevBuf& tmp, uint8_t* out) {
    // repeated 64-way partial sums until one point is left
    Point* cur = pts;
    MPVSS_CUDA(ctx, tmp.ensure(((total + 63) / 64) * sizeof(Point) * 2));
    Point* nxt = tmp.as<Point>();
    Point* alt = nxt + (total + 63) / 64;
    while (true) {
      size_t groups = (total + 63) / 64;
      bool last = groups == 1;
      ec::SumArgs<Cv> S{K(ctx), cur, last ? nullptr : nxt, last ? out : nullptr, (uint32_t)groups, 64, 64, 1,
                        (uint32_t)total};
      MPVSS_CUDA(ctx, ec::launch_sum<Cv>(S, ctx->stream));
      timing_launch(ctx);
      if (last) break;
      cur = nxt;
      std::swap(nxt, alt);
      total = groups;
    }
    return MPVSS_OK;
  }
  // commitments (device, encoded) + positions -> X (device, encoded)
  static int dev_horner(mpvss_ctx* ctx, const uint8_t* comm, size_t t, const uint32_t* pos, size_t n, DevBuf& cxy,
                        DevBuf& cst, DevBuf& part, uint8_t* x) {
    MPVSS_CUDA(ctx, cxy.ensure(t * 64));
    MPVSS_CUDA(ctx, cst.ensure(t * 4));
    ec::DecodeArgs<Cv> D{K(ctx), comm, cxy.as<uint32_t>(), cst.as<uint32_t>(), (uint32_t)t};
    MPVSS_CUDA(ctx, ec::launch_decode<Cv>(D, ctx->stream));
    timing_launch(ctx);
    // Enough chunks to fill the chip ONCE: the Horner kernel keeps 4 CTAs of 128 threads resident per SM, and
    // every extra chunk costs a full scalar multiplication, so the thread count is the largest multiple of
    // n that still fits one wave (148 x 4 x 128 = 75776 threads; 131072 threads, round 1, ran 1.73 waves and
    // twice the chunk scalings).  "ec_threads" overrides the target; at least 16 coefficients per chunk.
    const size_t target = ctx->ec_threads ? ctx->ec_threads : (size_t)ctx->sm_count * ec::HORNER_CTAS_PER_SM * 128;
    size_t Kc = std::max<size_t>(1, std::min<size_t>(target / std::max<size_t>(n, 1), std::max<size_t>(1, t / 16)));
    size_t B = (t + Kc - 1) / Kc;
    Kc = (t + B - 1) / B;
    MPVSS_CUDA(ctx, part.ensure(Kc * n * sizeof(Point)));
    ec::HornerArgs<Cv> H{K(ctx), cxy.as<uint32_t>(), cst.as<uint32_t>(), pos, part.as<Point>(),
                         (uint32_t)t, (uint32_t)n, (uint32_t)Kc, (uint32_t)B};
    MPVSS_CUDA(ctx, ec::launch_horner<Cv>(H, ctx->stream));
    timing_launch(ctx);
    ec::SumArgs<Cv> S{K(ctx), part.as<Point>(), nullptr, x, (uint32_t)n, (uint32_t)Kc, 1, (uint32_t)n,
                      (uint32_t)(Kc * n)};
    MPVSS_CUDA(ctx, ec::launch_sum<Cv>(S, ctx->stream));
    timing_launch(ctx);
    ctx->ec_chunks = Kc;
    return MPVSS_OK;
  }
  // field products of the Horner + chunk-scaling + chunk-sum launches for these positions (roofline accounting)
  // one position p of a polynomial of t coefficients cut into Kc non-empty chunks
  static void count_position(uint32_t p, uint64_t t, uint64_t Kc, uint64_t& M, uint64_t& S) {
    auto add = [&](OpCost c, uint64_t times) {
      M += c.m * times;
      S += c.s * times;
    };
    uint32_t nd = 1, nz = 0;
    while (nd < 16 && (p >> (2 * nd))) ++nd;
    for (uint32_t d = 0; d + 1 < nd; ++d) nz += ((p >> (2 * d)) & 3u) != 0;
    const uint64_t steps = t - Kc;                       // Horner steps of all chunks of this position
    add(T::SMALL_FIXED, steps);
    add(T::DBL_NOT, steps * (nd - 1));
    add(T::DBL, steps * (nd - 1));
    add(T::WIN_ADD, steps * (nz + (T::TOP_ADD_FREE ? 0 : 1)));
    add(T::MADD, steps);
    // chunks 1..K-1: acc <- pos^(kB) * acc, fixed 4-bit windows (7 dbl + 7 add table, 63 x 4 dbl, ~60 adds)
    add(T::DBL, (Kc - 1) * (7 + 252));
    add(T::ADD, (Kc - 1) * (7 + 60));
    add(T::ADD, Kc - 1);                                  // chunk sum
  }
  static void count_horner(mpvss_ctx* ctx, const std::vector<uint32_t>& pos, size_t t) {
    const uint64_t Kc = ctx->ec_chunks ? ctx->ec_chunks : 1;
    uint64_t M = 0, S = 0;
    for (uint32_t p : pos) count_position(p, t, Kc, M, S);
    ctx->horner_sqr = S;
    ctx->horner_mul = M;
  }

  static int positions_u32(mpvss_ctx* ctx, const int64_t* positions, size_t n, std::vector<uint32_t>& pos) {
    pos.resize(n);
    for (size_t i = 0; i < n; ++i) {
      int64_t p = positions ? positions[i] : (int64_t)i + 1;
      if (p < 1 || p > 0x7fffffff) return mpvss_fail(ctx, MPVSS_ERR_ARG, "position out of range [1, 2^31)");
      pos[i] = (uint32_t)p;
    }
    return MPVSS_OK;
  }

  // ---- batch forms of trait Group ------------------------------------------------------------
  static int batch_exp(mpvss_ctx* ctx, const uint8_t* bases, size_t base_stride, const uint8_t* scalars, size_t n,
                       uint8_t* out) {
    MPVSS_TRY(bad(ctx, bases && scalars && out && n > 0 && (base_stride == 0 || base_stride == EB),
                  "batch_exp: bad arguments"));
    std::vector<uint32_t> e;
    MPVSS_TRY(scalars_in(ctx, scalars, n, e));
    DevBuf &db = ctx->buf(0), &de = ctx->buf(1), &dout = ctx->buf(2), &dst = ctx->buf(3);
    MPVSS_TRY(h2d(ctx, db, bases, base_stride ? n * EB : EB));
    MPVSS_TRY(h2d(ctx, de, e.data(), n * 32));
    MPVSS_CUDA(ctx, dout.ensure(n * EB));
    MPVSS_CUDA(ctx, dst.ensure(n * 4));
    timing_begin(ctx);
    MPVSS_TRY(dev_exp2(ctx, db.as<uint8_t>(), (uint32_t)base_stride, de.as<uint32_t>(), nullptr, 0, nullptr, 0, n,
                       dout.as<uint8_t>(), nullptr, dst.as<uint32_t>()));
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(check_status(ctx, dst, n, "batch_exp"));
    MPVSS_TRY(d2h(ctx, out, dout, n * EB));
    return sync(ctx);
  }
  static int fixed_base_exp(mpvss_ctx* ctx, int generator, const uint8_t* scalars, size_t n, uint8_t* out) {
    MPVSS_TRY(bad(ctx, (generator == MPVSS_GEN_MAIN || generator == MPVSS_GEN_SUBGROUP) && scalars && out && n > 0,
                  "fixed_base_exp: bad arguments"));
    std::vector<uint32_t> e;
    MPVSS_TRY(scalars_in(ctx, scalars, n, e));
    DevBuf &de = ctx->buf(1), &dout = ctx->buf(2);
    MPVSS_TRY(h2d(ctx, de, e.data(), n * 32));
    MPVSS_CUDA(ctx, dout.ensure(n * EB));
    timing_begin(ctx);
    MPVSS_TRY(dev_fixed(ctx, de.as<uint32_t>(), n, dout.as<uint8_t>()));
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(d2h(ctx, out, dout, n * EB));
    MPVSS_CUDA(ctx, cudaMemsetAsync(de.p, 0, de.cap, ctx->stream));  // private keys / witnesses pass through here
    return sync(ctx);
  }
  static int batch_mul(mpvss_ctx* ctx, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
    MPVSS_TRY(bad(ctx, a && b && out && n > 0, "batch_mul: bad arguments"));
    DevBuf &da = ctx->buf(0), &db = ctx->buf(1), &dout = ctx->buf(2), &dst = ctx->buf(3);
    MPVSS_TRY(h2d(ctx, da, a, n * EB));
    MPVSS_TRY(h2d(ctx, db, b, n * EB));
    MPVSS_CUDA(ctx, dout.ensure(n * EB));
    MPVSS_CUDA(ctx, dst.ensure(n * 4));
    timing_begin(ctx);
    ec::AddArgs<Cv> A{K(ctx), da.as<uint8_t>(), db.as<uint8_t>(), dout.as<uint8_t>(), dst.as<uint32_t>(), (uint32_t)n};
    MPVSS_CUDA(ctx, ec::launch_add<Cv>(A, ctx->stream));
    timing_launch(ctx);
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(check_status(ctx, dst, n, "batch_mul"));
    MPVSS_TRY(d2h(ctx, out, dout, n * EB));
    return sync(ctx);
  }
  static int poly_eval_exp(mpvss_ctx* ctx, const uint8_t* commitments, size_t t, const int64_t* positions, size_t n,
                           uint8_t* out) {
    MPVSS_TRY(bad(ctx, commitments && out && n > 0 && t > 0, "poly_eval_exp: bad arguments"));
    std::vector<uint32_t> pos;
    MPVSS_TRY(positions_u32(ctx, positions, n, pos));
    DevBuf &dc = ctx->buf(0), &dp = ctx->buf(1), &dout = ctx->buf(2);
    MPVSS_TRY(h2d(ctx, dc, commitments, t * EB));
    MPVSS_TRY(h2d(ctx, dp, pos.data(), n * 4));
    MPVSS_CUDA(ctx, dout.ensure(n * EB));
    timing_begin(ctx);
    MPVSS_TRY(dev_horner(ctx, dc.as<uint8_t>(), t, dp.as<uint32_t>(), n, ctx->buf(3), ctx->buf(4), ctx->buf(5),
                         dout.as<uint8_t>()));
    count_horner(ctx, pos, t);
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(check_status(ctx, ctx->buf(4), t, "poly_eval_exp (commitments)"));
    MPVSS_TRY(d2h(ctx, out, dout, n * EB));
    return sync(ctx);
  }
  // `undecodable`: when given, instances whose elements or scalars do not decode are flagged there (and get
  // an arbitrary a1 / a2) instead of failing the whole call -- verify_share returns false for them
  static int dleq_verify_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* h1, const uint8_t* g2,
                                const uint8_t* h2, const uint8_t* r, const uint8_t* c, size_t c_stride, size_t n,
                                uint8_t* a1, uint8_t* a2, std::vector<uint8_t>* undecodable = nullptr) {
    MPVSS_TRY(bad(ctx, g1 && h1 && g2 && h2 && r && c && ((a1 && a2) || undecodable) && n > 0 &&
                           (c_stride == 0 || c_stride == SB),
                  "dleq_verify_commit: bad arguments"));
    std::vector<uint32_t> rl, cl;
    if (undecodable) {
      undecodable->assign(n, 0);
      rl.assign(n * 8, 0);
      cl.assign((c_stride ? n : 1) * 8, 0);
      std::vector<uint32_t> one;
      for (size_t i = 0; i < n; ++i) {  // per-instance: a non-canonical scalar only spoils its own share
        if (scalars_in(ctx, r + i * SB, 1, one) != MPVSS_OK) (*undecodable)[i] = 1;
        else memcpy(&rl[i * 8], one.data(), 32);
        if (c_stride || i == 0) {
          if (scalars_in(ctx, c + i * c_stride, 1, one) != MPVSS_OK) (*undecodable)[i] = 1;
          else memcpy(&cl[i * 8], one.data(), 32);
        }
      }
    } else {
      MPVSS_TRY(scalars_in(ctx, r, n, rl));
      MPVSS_TRY(scalars_in(ctx, c, c_stride ? n : 1, cl));
    }
    DevBuf &dg1 = ctx->buf(0), &dh1 = ctx->buf(1), &dg2 = ctx->buf(2), &dh2 = ctx->buf(3), &dr = ctx->buf(4),
           &dc = ctx->buf(5), &da1 = ctx->buf(6), &da2 = ctx->buf(7), &ds1 = ctx->buf(8), &ds2 = ctx->buf(9);
    MPVSS_TRY(h2d(ctx, dg1, g1, EB));
    MPVSS_TRY(h2d(ctx, dh1, h1, n * EB));
    MPVSS_TRY(h2d(ctx, dg2, g2, n * EB));
    MPVSS_TRY(h2d(ctx, dh2, h2, n * EB));
    MPVSS_TRY(h2d(ctx, dr, rl.data(), n * 32));
    MPVSS_TRY(h2d(ctx, dc, cl.data(), cl.size() * 4));
    for (DevBuf* b : {&da1, &da2}) MPVSS_CUDA(ctx, b->ensure(n * EB));
    for (DevBuf* b : {&ds1, &ds2}) MPVSS_CUDA(ctx, b->ensure(n * 4));
    uint32_t cs = c_stride ? 8 : 0;
    timing_begin(ctx);
    const bool gen = memcmp(g1, ctx->ec_gen.data(), EB) == 0;  // the usual case: fixed-base table
    MPVSS_TRY(dev_exp2(ctx, dg1.as<uint8_t>(), 0, dr.as<uint32_t>(), dh1.as<uint8_t>(), EB, dc.as<uint32_t>(), cs, n,
                       da1.as<uint8_t>(), nullptr, ds1.as<uint32_t>(), nullptr, gen));
    MPVSS_TRY(dev_exp2(ctx, dg2.as<uint8_t>(), EB, dr.as<uint32_t>(), dh2.as<uint8_t>(), EB, dc.as<uint32_t>(), cs, n,
                       da2.as<uint8_t>(), nullptr, ds2.as<uint32_t>()));
    MPVSS_TRY(timing_end(ctx));
    if (undecodable) {
      std::vector<uint32_t> s1(n), s2(n);
      MPVSS_TRY(d2h(ctx, s1.data(), ds1, n * 4));
      MPVSS_TRY(d2h(ctx, s2.data(), ds2, n * 4));
      MPVSS_TRY(sync(ctx));
      for (size_t i = 0; i < n; ++i)
        if (s1[i] == 1 || s2[i] == 1) (*undecodable)[i] = 1;
    } else {
      MPVSS_TRY(check_status(ctx, ds1, n, "dleq_verify_commit (g1/h1)"));
      MPVSS_TRY(check_status(ctx, ds2, n, "dleq_verify_commit (g2/h2)"));
    }
    if (a1) MPVSS_TRY(d2h(ctx, a1, da1, n * EB));  // nullptr: the caller continues on the device (verify_shares)
    if (a2) MPVSS_TRY(d2h(ctx, a2, da2, n * EB));
    return sync(ctx);
  }
  static int dleq_prove_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* g2, const uint8_t* w, size_t n,
                               uint8_t* a1, uint8_t* a2) {
    MPVSS_TRY(bad(ctx, g1 && g2 && w && a1 && a2 && n > 0, "dleq_prove_commit: bad arguments"));
    MPVSS_TRY(batch_exp(ctx, g1, 0, w, n, a1));
    float ms = ctx->last_ms;
    int l = ctx->last_launches;
    MPVSS_TRY(batch_exp(ctx, g2, EB, w, n, a2));
    ctx->last_ms += ms;
    ctx->last_launches += l;
    return MPVSS_OK;
  }
  static int multi_exp_limbs(mpvss_ctx* ctx, const uint8_t* bases, const uint32_t* scalar_limbs_dev,
                             const uint32_t* scalar_limbs_host, size_t n, uint8_t* out) {
    DevBuf &db = ctx->buf(0), &de = ctx->buf(1), &dj = ctx->buf(2), &dst = ctx->buf(3), &dout = ctx->buf(4),
           &tmp = ctx->buf(5);
    MPVSS_TRY(h2d(ctx, db, bases, n * EB));
    if (scalar_limbs_host) MPVSS_TRY(h2d(ctx, de, scalar_limbs_host, n * 32));
    const uint32_t* e = scalar_limbs_host ? de.as<uint32_t>() : scalar_limbs_dev;
    MPVSS_CUDA(ctx, dj.ensure(n * sizeof(Point)));
    MPVSS_CUDA(ctx, dst.ensure(n * 4));
    MPVSS_CUDA(ctx, dout.ensure(EB));
    timing_begin(ctx);
    MPVSS_TRY(dev_exp2(ctx, db.as<uint8_t>(), EB, e, nullptr, 0, nullptr, 0, n, nullptr, dj.as<Point>(),
                       dst.as<uint32_t>()));
    MPVSS_TRY(dev_sum_all(ctx, dj.as<Point>(), n, tmp, dout.as<uint8_t>()));
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(check_status(ctx, dst, n, "multi_exp"));
    MPVSS_TRY(d2h(ctx, out, dout, EB));
    return sync(ctx);
  }
  static int multi_exp(mpvss_ctx* ctx, const uint8_t* bases, const uint8_t* scalars, size_t n, uint8_t* out) {
    MPVSS_TRY(bad(ctx, bases && scalars && out && n > 0, "multi_exp: bad arguments"));
    std::vector<uint32_t> e;
    MPVSS_TRY(scalars_in(ctx, scalars, n, e));
    return multi_exp_limbs(ctx, bases, nullptr, e.data(), n, out);
  }

  // ---- verify_distribution_shares --------------------------------------------------------------
  static transcript::Geom geom() { return transcript::Geom{EB, false}; }
  static const uint8_t* slice_rows(const mpvss_ctx* ctx, const uint8_t* all, size_t n_total, size_t width,
                                   std::vector<uint8_t>& tmp) {
    if (ctx->nranks <= 1) return all;
    tmp.clear();
    for (size_t i = (size_t)ctx->rank; i < n_total; i += (size_t)ctx->nranks)
      tmp.insert(tmp.end(), all + i * width, all + (i + 1) * width);
    return tmp.data();
  }
  static int verify_stage(mpvss_ctx* ctx, size_t n_total, size_t t, const uint8_t* commitments,
                          const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares,
                          const uint8_t* responses, const uint8_t* challenge) {
    ctx->v_n_total = 0;
    MPVSS_TRY(bad(ctx, n_total > 0 && t > 0 && commitments && publickeys && shares && responses && challenge,
                  "verify_distribution: bad arguments"));
    // every rank checks ALL positions and scalars, so that a malformed box is rejected by all ranks alike
    std::vector<uint32_t> pos_all, rl_all, cl;
    if (positions_u32(ctx, positions, n_total, pos_all) != MPVSS_OK)   // box content: verifies as false
      return mpvss_fail(ctx, MPVSS_ERR_ENCODING, "verify_distribution: position out of range [1, 2^31)");
    MPVSS_TRY(scalars_in(ctx, responses, n_total, rl_all));
    MPVSS_TRY(scalars_in(ctx, challenge, 1, cl));
    const size_t n = transcript::local_count(n_total, ctx->nranks, ctx->rank), N = (size_t)ctx->nranks;
    std::vector<uint32_t> pos(n), rl(n * 8);
    for (size_t j = 0; j < n; ++j) {
      const size_t i = (size_t)ctx->rank + j * N;
      pos[j] = pos_all[i];
      memcpy(&rl[j * 8], &rl_all[i * 8], 32);
    }
    std::vector<uint8_t> tpk, ty;
    const uint8_t* pk = slice_rows(ctx, publickeys, n_total, EB, tpk);
    const uint8_t* y = slice_rows(ctx, shares, n_total, EB, ty);
    MPVSS_TRY(h2d(ctx, ctx->v_comm, commitments, t * EB));
    MPVSS_TRY(h2d(ctx, ctx->v_c, cl.data(), 32));
    if (n) {
      MPVSS_TRY(h2d(ctx, ctx->v_pos, pos.data(), n * 4));
      MPVSS_TRY(h2d(ctx, ctx->v_pk, pk, n * EB));
      MPVSS_TRY(h2d(ctx, ctx->v_y, y, n * EB));
      MPVSS_TRY(h2d(ctx, ctx->v_r, rl.data(), n * 32));
      for (DevBuf* b : {&ctx->v_x, &ctx->v_a1, &ctx->v_a2}) MPVSS_CUDA(ctx, b->ensure(n * EB));
      MPVSS_CUDA(ctx, ctx->v_st.ensure(2 * n * 4));  // status of the two DLEQ launches
    }
    const size_t rpr = transcript::rows_per_rank(n_total, ctx->nranks), row = geom().row();
    MPVSS_CUDA(ctx, ctx->v_frames.ensure(rpr * row));
    MPVSS_CUDA(ctx, cudaMemsetAsync(ctx->v_frames.p, 0, rpr * row, ctx->stream));
    if (ctx->nranks > 1) MPVSS_CUDA(ctx, ctx->v_gather.ensure(N * rpr * row));
    ctx->v_challenge.assign(challenge, challenge + SB);
    ctx->v_n = n;
    ctx->v_t = t;
    ctx->v_hpos = pos;
    MPVSS_TRY(sync(ctx));
    ctx->v_n_total = n_total;
    return MPVSS_OK;
  }
  // X (chunked Horner), a1 = r*g + c*X, a2 = r*y + c*Y, framed rows.  *decoded = false if an element of the
  // box is not a valid encoding (the rows are then marked instead of failing: the all-gather must still run)
  static int verify_kernels(mpvss_ctx* ctx, bool* decoded) {
    const size_t n = ctx->v_n, t = ctx->v_t;
    *decoded = true;
    timing_begin(ctx);
    if (n == 0) {
      MPVSS_TRY(timing_end(ctx));
      ctx->phase_ms[0] = ctx->phase_ms[1] = 0.f;
      return MPVSS_OK;
    }
    uint8_t* X = ctx->v_x.as<uint8_t>();
    uint32_t* st = ctx->v_st.as<uint32_t>();
    MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
    MPVSS_TRY(dev_horner(ctx, ctx->v_comm.as<uint8_t>(), t, ctx->v_pos.as<uint32_t>(), n, ctx->v_cm, ctx->v_cst,
                         ctx->buf(12), X));
    count_horner(ctx, ctx->v_hpos, t);
    // a2 = r*y + c*Y does not depend on X: a small grid (one thread per share) on a side stream, issued
    // after the Horner launches so that it only takes CTA slots they leave free
    MPVSS_CUDA(ctx, cudaStreamWaitEvent(ctx->aux[0], ctx->ev_fork, 0));
    MPVSS_TRY(dev_exp2(ctx, ctx->v_pk.as<uint8_t>(), EB, ctx->v_r.as<uint32_t>(), ctx->v_y.as<uint8_t>(), EB,
                       ctx->v_c.as<uint32_t>(), 0, n, ctx->v_a2.as<uint8_t>(), nullptr, st + n, ctx->aux[0]));
    MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_join[0], ctx->aux[0]));
    MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev_mid, ctx->stream));
    // a1 = r*g + c*X  (dleq.rs:66-84)
    MPVSS_TRY(dev_exp2(ctx, ctx->gens.as<uint8_t>(), 0, ctx->v_r.as<uint32_t>(), X, EB, ctx->v_c.as<uint32_t>(), 0, n,
                       ctx->v_a1.as<uint8_t>(), nullptr, st, nullptr, true));
    MPVSS_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0));
    ec::FrameArgs FA{X, ctx->v_y.as<uint8_t>(), ctx->v_a1.as<uint8_t>(), ctx->v_a2.as<uint8_t>(),
                     ctx->v_frames.as<uint8_t>(), (uint32_t)n, (uint32_t)EB};
    MPVSS_CUDA(ctx, ec::launch_frames(FA, ctx->stream));
    timing_launch(ctx);
    MPVSS_TRY(timing_end(ctx));
    MPVSS_CUDA(ctx, cudaEventElapsedTime(&ctx->phase_ms[0], ctx->ev0, ctx->ev_mid));
    MPVSS_CUDA(ctx, cudaEventElapsedTime(&ctx->phase_ms[1], ctx->ev_mid, ctx->ev1));
    int s1 = check_status(ctx, ctx->v_cst, t, "verify_distribution (commitments)");
    int s2 = s1 == MPVSS_OK ? check_status(ctx, ctx->v_st, 2 * n, "verify_distribution (public keys / shares)") : s1;
    if (s2 == MPVSS_ERR_ENCODING) {
      *decoded = false;
      const uint8_t mark = 0xff;
      MPVSS_CUDA(ctx, cudaMemcpyAsync(ctx->v_frames.p, &mark, 1, cudaMemcpyHostToDevice, ctx->stream));
      MPVSS_TRY(sync(ctx));
      return MPVSS_OK;
    }
    return s2;
  }
  static void framed(sha2::Sha256& h, const uint8_t* e) {  // dleq.rs:58-61
    uint8_t len8[8] = {0, 0, 0, 0, 0, 0, 0, (uint8_t)EB};
    h.update(len8, 8);
    h.update(e, EB);
  }
  static big::Int challenge_of(mpvss_ctx* ctx, sha2::Sha256& h, uint8_t* digest_out) {
    uint8_t digest[32];
    h.finalize(digest);
    if (digest_out) memcpy(digest_out, digest, 32);
    return T::hash_to_scalar(digest, 32, ctx->ec_order);  // the digest is hashed again (participant.rs:1217-1218)
  }
  static int verify_run(mpvss_ctx* ctx, int* ok, uint8_t* x_out, uint8_t* a1_out, uint8_t* a2_out,
                        uint8_t* digest_out) {
    MPVSS_TRY(bad(ctx, ok && ctx->v_n_total > 0, "verify_distribution_run: nothing staged"));
    MPVSS_TRY(bad(ctx, ctx->nranks <= 1 || (!x_out && !a1_out && !a2_out),
                  "verify_distribution: x/a1/a2 outputs are not available with a communicator"));
    const size_t n = ctx->v_n, n_total = ctx->v_n_total;
    bool decoded = true;
    MPVSS_TRY(verify_kernels(ctx, &decoded));
    const transcript::Geom g = geom();
    const size_t rpr = transcript::rows_per_rank(n_total, ctx->nranks);
    const uint8_t* rows = ctx->v_frames.as<uint8_t>();
    if (ctx->nranks > 1) {
      MPVSS_TRY(comm_allgather(ctx, ctx->v_frames.p, ctx->v_gather.p, rpr * g.row()));
      MPVSS_CUDA(ctx, ctx->v_ordered.ensure(n_total * g.row()));
      MPVSS_TRY(comm_reorder_rows(ctx, ctx->v_gather.p, ctx->v_ordered.p, n_total, g.row()));
      rows = ctx->v_ordered.as<uint8_t>();
    }
    big::Int c;
    if (ctx->device_hash) {  // measured alternative: the one sequential chain on one device thread
      uint8_t digest[32];
      MPVSS_TRY(transcript::device_digest(ctx, rows, n_total, ctx->nranks, g, digest));
      if (digest_out) memcpy(digest_out, digest, 32);
      c = T::hash_to_scalar(digest, 32, ctx->ec_order);
    } else {
      sha2::Sha256 h;
      MPVSS_TRY(transcript::fetch_and_hash(ctx, rows, n_total, ctx->nranks, g, h, true));
      c = challenge_of(ctx, h, digest_out);
    }
    *ok = big::cmp(c, scalar_big(ctx->v_challenge.data())) == 0;
    for (size_t r = 0; r < std::min<size_t>((size_t)ctx->nranks, n_total); ++r)  // a rank whose slice did not decode
      if (ctx->h_frames.as<uint8_t>()[r * g.row()] == 0xff) *ok = 0;      // marked its first row = participant r
    if (!decoded) *ok = 0;
    if (x_out) MPVSS_TRY(d2h(ctx, x_out, ctx->v_x, n * EB));
    if (a1_out) MPVSS_TRY(d2h(ctx, a1_out, ctx->v_a1, n * EB));
    if (a2_out) MPVSS_TRY(d2h(ctx, a2_out, ctx->v_a2, n * EB));
    return sync(ctx);
  }

  // ---- mpvss_verify_distributions: many boxes, one launch per kernel ---------------------------------
  // Positions and scalars are checked per box on the host; a box that fails verifies as false with a zero
  // digest and leaves the others alone.  All commitments are decoded in one launch, X_i of every box comes
  // from one multi-box Horner launch and one chunk sum, a1 / a2 take one challenge per instance, and the
  // frames of all boxes come to the host in one copy, where each box's row range is hashed on its own.
  // Uses scratch buffers only: the staged single-box state (v_*) is left as it was.
  static int verify_batch(mpvss_ctx* ctx, size_t nb, const size_t* nv, const size_t* tv, const uint8_t* commitments,
                          const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares,
                          const uint8_t* responses, const uint8_t* challenges, int* ok_out, uint8_t* digests_out) {
    std::vector<size_t> noff(nb + 1, 0), toff(nb + 1, 0);
    size_t tmax = 1;
    for (size_t b = 0; b < nb; ++b) {
      noff[b + 1] = noff[b] + nv[b];
      toff[b + 1] = toff[b] + tv[b];
      tmax = std::max(tmax, tv[b]);
    }
    const size_t N = noff[nb], Tt = toff[nb];
    std::vector<uint8_t> live(nb, 1);
    // a rejected box is only false: these checks record no context error, the call succeeds
    std::vector<uint32_t> pos(N, 1), coff(N), ct(N), rl(N * 8, 0), cl(N * 8, 0), br, bc;
    for (size_t b = 0; b < nb; ++b) {
      for (size_t i = noff[b]; positions && i < noff[b + 1] && live[b]; ++i)
        live[b] = positions[i] >= 1 && positions[i] <= 0x7fffffff;
      if (!live[b] || scalars_in(ctx, responses + noff[b] * SB, nv[b], br, false) != MPVSS_OK ||
          scalars_in(ctx, challenges + b * SB, 1, bc, false) != MPVSS_OK)
        live[b] = 0;
      for (size_t j = 0, i = noff[b]; j < nv[b]; ++j, ++i) {
        coff[i] = (uint32_t)toff[b];
        ct[i] = (uint32_t)tv[b];
        if (!live[b]) continue;
        pos[i] = positions ? (uint32_t)positions[i] : (uint32_t)(j + 1);
        memcpy(&rl[i * 8], &br[j * 8], 32);
        memcpy(&cl[i * 8], bc.data(), 32);
      }
    }
    DevBuf &dc = ctx->buf(0), &dxy = ctx->buf(1), &dcst = ctx->buf(2), &dpos = ctx->buf(3), &dcoff = ctx->buf(4),
           &dct = ctx->buf(5), &dpk = ctx->buf(6), &dy = ctx->buf(7), &dr = ctx->buf(8), &dch = ctx->buf(9),
           &dpart = ctx->buf(10), &dx = ctx->buf(11), &da1 = ctx->buf(12), &da2 = ctx->buf(13), &dst = ctx->buf(14),
           &dfr = ctx->buf(15);
    MPVSS_TRY(h2d(ctx, dc, commitments, Tt * EB));
    MPVSS_TRY(h2d(ctx, dpos, pos.data(), N * 4));
    MPVSS_TRY(h2d(ctx, dcoff, coff.data(), N * 4));
    MPVSS_TRY(h2d(ctx, dct, ct.data(), N * 4));
    MPVSS_TRY(h2d(ctx, dpk, publickeys, N * EB));
    MPVSS_TRY(h2d(ctx, dy, shares, N * EB));
    MPVSS_TRY(h2d(ctx, dr, rl.data(), N * 32));
    MPVSS_TRY(h2d(ctx, dch, cl.data(), N * 32));
    const transcript::Geom g = geom();
    const size_t row = g.row();
    for (DevBuf* b : {&dx, &da1, &da2}) MPVSS_CUDA(ctx, b->ensure(N * EB));
    MPVSS_CUDA(ctx, dxy.ensure(Tt * 64));
    MPVSS_CUDA(ctx, dcst.ensure(Tt * 4));
    MPVSS_CUDA(ctx, dst.ensure(2 * N * 4));
    MPVSS_CUDA(ctx, dfr.ensure(N * row));
    // chunks per position: the one-wave rule of dev_horner on the total position count
    const size_t target = ctx->ec_threads ? ctx->ec_threads : (size_t)ctx->sm_count * ec::HORNER_CTAS_PER_SM * 128;
    const size_t Kc = std::max<size_t>(1, std::min<size_t>(target / N, std::max<size_t>(1, tmax / 16)));
    MPVSS_CUDA(ctx, dpart.ensure(Kc * N * sizeof(Point)));
    uint32_t* st = dst.as<uint32_t>();
    timing_begin(ctx);
    ec::DecodeArgs<Cv> D{K(ctx), dc.as<uint8_t>(), dxy.as<uint32_t>(), dcst.as<uint32_t>(), (uint32_t)Tt};
    MPVSS_CUDA(ctx, ec::launch_decode<Cv>(D, ctx->stream));
    timing_launch(ctx);
    ec::HornerBoxesArgs<Cv> H{K(ctx), dxy.as<uint32_t>(), dcst.as<uint32_t>(), dpos.as<uint32_t>(), dcoff.as<uint32_t>(),
                              dct.as<uint32_t>(), dpart.as<Point>(), (uint32_t)N, (uint32_t)Kc};
    MPVSS_CUDA(ctx, ec::launch_horner_boxes<Cv>(H, ctx->stream));
    timing_launch(ctx);
    ec::SumArgs<Cv> S{K(ctx), dpart.as<Point>(), nullptr, dx.as<uint8_t>(), (uint32_t)N, (uint32_t)Kc, 1, (uint32_t)N,
                      (uint32_t)(Kc * N)};
    MPVSS_CUDA(ctx, ec::launch_sum<Cv>(S, ctx->stream));
    timing_launch(ctx);
    // a2 = r*y + c*Y, a1 = r*g + c*X  (dleq.rs:66-84), one challenge per instance
    MPVSS_TRY(dev_exp2(ctx, dpk.as<uint8_t>(), EB, dr.as<uint32_t>(), dy.as<uint8_t>(), EB, dch.as<uint32_t>(), 8, N,
                       da2.as<uint8_t>(), nullptr, st + N));
    MPVSS_TRY(dev_exp2(ctx, ctx->gens.as<uint8_t>(), 0, dr.as<uint32_t>(), dx.as<uint8_t>(), EB, dch.as<uint32_t>(), 8, N,
                       da1.as<uint8_t>(), nullptr, st, nullptr, true));
    ec::FrameArgs FA{dx.as<uint8_t>(), dy.as<uint8_t>(), da1.as<uint8_t>(), da2.as<uint8_t>(), dfr.as<uint8_t>(),
                     (uint32_t)N, (uint32_t)EB};
    MPVSS_CUDA(ctx, ec::launch_frames(FA, ctx->stream));
    timing_launch(ctx);
    MPVSS_TRY(timing_end(ctx));
    uint64_t M = 0, Sq = 0;
    for (size_t b = 0; b < nb; ++b) {
      const uint64_t B = (tv[b] + Kc - 1) / Kc, Kb = (tv[b] + B - 1) / B;
      for (size_t i = noff[b]; i < noff[b + 1]; ++i) count_position(pos[i], tv[b], Kb, M, Sq);
    }
    ctx->horner_sqr = Sq;
    ctx->horner_mul = M;
    // rows, then the decode status of the commitments and of the two DLEQ launches, in one pinned buffer
    PinBuf& host = ctx->pin(0);
    MPVSS_CUDA(ctx, host.ensure(N * row + (Tt + 2 * N) * 4));
    uint8_t* rows = host.as<uint8_t>();
    uint32_t* hcst = reinterpret_cast<uint32_t*>(rows + N * row);
    uint32_t* hst = hcst + Tt;
    MPVSS_TRY(d2h(ctx, rows, dfr, N * row));
    MPVSS_TRY(d2h(ctx, hcst, dcst, Tt * 4));
    MPVSS_TRY(d2h(ctx, hst, dst, 2 * N * 4));
    MPVSS_TRY(sync(ctx));
    for (size_t b = 0; b < nb; ++b) {
      for (size_t j = toff[b]; j < toff[b + 1] && live[b]; ++j) live[b] = hcst[j] != 1;
      for (size_t i = noff[b]; i < noff[b + 1] && live[b]; ++i) live[b] = hst[i] != 1 && hst[N + i] != 1;
      uint8_t digest[32] = {0};
      ok_out[b] = 0;
      if (live[b]) {
        sha2::Sha256 h;
        transcript::hash_ordered(h, rows, noff[b], noff[b + 1], g);
        const big::Int c = challenge_of(ctx, h, digest);
        ok_out[b] = big::cmp(c, scalar_big(challenges + b * SB)) == 0;
      }
      if (digests_out) memcpy(digests_out + 32 * b, digest, 32);
    }
    return MPVSS_OK;
  }

  static int scalar_poly_eval(mpvss_ctx* ctx, const uint8_t* coeffs, size_t t, const int64_t* positions, size_t n,
                              uint8_t* out) {
    MPVSS_TRY(bad(ctx, coeffs && out && n > 0 && t > 0, "scalar_poly_eval: bad arguments"));
    std::vector<uint32_t> co, pos, p(n * 8);
    MPVSS_TRY(scalars_in(ctx, coeffs, t, co));
    MPVSS_TRY(positions_u32(ctx, positions, n, pos));
    DevBuf &dco = ctx->buf(0), &dp = ctx->buf(1), &dpos = ctx->buf(9);
    MPVSS_TRY(h2d(ctx, dco, co.data(), t * 32));
    MPVSS_TRY(h2d(ctx, dpos, pos.data(), n * 4));
    MPVSS_CUDA(ctx, dp.ensure(n * 32));
    timing_begin(ctx);
    ec::PolyArgs PA{KN(ctx), dco.as<uint32_t>(), dpos.as<uint32_t>(), dp.as<uint32_t>(), (uint32_t)t, (uint32_t)n};
    MPVSS_CUDA(ctx, ec::launch_poly(PA, ctx->stream));
    timing_launch(ctx);
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(d2h(ctx, p.data(), dp, n * 32));
    MPVSS_TRY(sync(ctx));
    for (size_t i = 0; i < n; ++i) {
      big::Int v(p.begin() + i * 8, p.begin() + i * 8 + 8);
      big::trim(v);
      scalar_out(v, out + i * SB);
    }
    MPVSS_CUDA(ctx, cudaMemsetAsync(dco.p, 0, dco.cap, ctx->stream));  // coefficients are secret
    return sync(ctx);
  }

  // ---- distribute_secret -------------------------------------------------------------------------
  // With a communicator the call is collective: rank r deals participants r, r + N, ... (commitments are
  // computed by every rank), one all-gather carries the framed transcript rows, a second one the shares,
  // responses and X of all ranks.
  static int distribute(mpvss_ctx* ctx, size_t n_total, size_t t, const uint8_t* secret, size_t secret_len,
                        const uint8_t* coeffs, const uint8_t* witnesses, const uint8_t* publickeys,
                        uint8_t* commitments_out, uint8_t* shares_out, uint8_t* challenge_out, uint8_t* responses_out,
                        uint8_t* u_out, uint8_t* x_out) {
    MPVSS_TRY(bad(ctx, n_total > 0 && t > 0 && t <= n_total && secret && coeffs && witnesses && publickeys &&
                           commitments_out && shares_out && challenge_out && responses_out && u_out && secret_len <= EB,
                  "distribute: bad arguments (threshold <= n, participant.rs:1100; secret at most one element long)"));
    std::vector<uint32_t> co, wl_all;
    MPVSS_TRY(scalars_in(ctx, coeffs, t, co));
    MPVSS_TRY(scalars_in(ctx, witnesses, n_total, wl_all));   // every rank checks all of them alike
    const size_t n = transcript::local_count(n_total, ctx->nranks, ctx->rank), N = (size_t)ctx->nranks;
    const size_t nn = std::max<size_t>(n, 1);
    std::vector<uint32_t> pos(nn), wl(nn * 8);
    for (size_t j = 0; j < n; ++j) {
      const size_t i = (size_t)ctx->rank + j * N;
      pos[j] = (uint32_t)(i + 1);
      memcpy(&wl[j * 8], &wl_all[i * 8], 32);
    }
    std::vector<uint8_t> tpk;
    const uint8_t* pk = slice_rows(ctx, publickeys, n_total, EB, tpk);
    DevBuf &dco = ctx->buf(0), &dp = ctx->buf(1), &dw = ctx->buf(2), &dpk = ctx->buf(3), &dC = ctx->buf(4),
           &dX = ctx->buf(5), &dY = ctx->buf(6), &dA1 = ctx->buf(7), &dA2 = ctx->buf(8), &dpos = ctx->buf(9),
           &dst = ctx->buf(10), &dR = ctx->buf(13);
    MPVSS_TRY(h2d(ctx, dco, co.data(), t * 32));
    MPVSS_TRY(h2d(ctx, dw, wl.data(), nn * 32));
    if (n) MPVSS_TRY(h2d(ctx, dpk, pk, n * EB));
    MPVSS_TRY(h2d(ctx, dpos, pos.data(), nn * 4));
    MPVSS_CUDA(ctx, dp.ensure(nn * 32));
    MPVSS_CUDA(ctx, dR.ensure(nn * 32));
    MPVSS_CUDA(ctx, dC.ensure(t * EB));
    for (DevBuf* b : {&dX, &dY, &dA1, &dA2}) MPVSS_CUDA(ctx, b->ensure(nn * EB));
    MPVSS_CUDA(ctx, dst.ensure(2 * nn * 4));
    const transcript::Geom g = geom();
    const size_t rpr = transcript::rows_per_rank(n_total, ctx->nranks);
    MPVSS_CUDA(ctx, ctx->v_frames.ensure(rpr * g.row()));
    MPVSS_CUDA(ctx, cudaMemsetAsync(ctx->v_frames.p, 0, rpr * g.row(), ctx->stream));
    if (ctx->nranks > 1) MPVSS_CUDA(ctx, ctx->v_gather.ensure(N * rpr * g.row()));
    timing_begin(ctx);
    // C_j = a_j * g (participant.rs:1130-1146 / 1603-1610), fixed-base table; every rank computes all of them
    MPVSS_TRY(dev_fixed(ctx, dco.as<uint32_t>(), t, dC.as<uint8_t>()));
    if (n) {
      // p_i = P(i) mod order (participant.rs:1155-1157 / 1619-1621)
      ec::PolyArgs PA{KN(ctx), dco.as<uint32_t>(), dpos.as<uint32_t>(), dp.as<uint32_t>(), (uint32_t)t, (uint32_t)n};
      MPVSS_CUDA(ctx, ec::launch_poly(PA, ctx->stream));
      timing_launch(ctx);
      // X_i = p_i * g (dealer shortcut: same element as sum_j i^j C_j) ; Y_i = p_i * y_i ; a1 = w * g ; a2 = w * y_i
      MPVSS_TRY(dev_fixed(ctx, dp.as<uint32_t>(), n, dX.as<uint8_t>()));
      MPVSS_TRY(dev_exp2(ctx, dpk.as<uint8_t>(), EB, dp.as<uint32_t>(), nullptr, 0, nullptr, 0, n, dY.as<uint8_t>(),
                         nullptr, dst.as<uint32_t>()));
      MPVSS_TRY(dev_fixed(ctx, dw.as<uint32_t>(), n, dA1.as<uint8_t>()));
      MPVSS_TRY(dev_exp2(ctx, dpk.as<uint8_t>(), EB, dw.as<uint32_t>(), nullptr, 0, nullptr, 0, n, dA2.as<uint8_t>(),
                         nullptr, dst.as<uint32_t>() + n));
      ec::FrameArgs FA{dX.as<uint8_t>(), dY.as<uint8_t>(), dA1.as<uint8_t>(), dA2.as<uint8_t>(),
                       ctx->v_frames.as<uint8_t>(), (uint32_t)n, (uint32_t)EB};
      MPVSS_CUDA(ctx, ec::launch_frames(FA, ctx->stream));
      timing_launch(ctx);
    }
    MPVSS_TRY(timing_end(ctx));
    // an undecodable public key: mark the rows (the collectives below must still run on every rank)
    int bad_pk = n ? check_status(ctx, dst, 2 * n, "distribute (public keys)") : MPVSS_OK;
    if (bad_pk != MPVSS_OK && bad_pk != MPVSS_ERR_ENCODING) return bad_pk;
    if (bad_pk == MPVSS_ERR_ENCODING) {
      const uint8_t mark = 0xff;
      MPVSS_CUDA(ctx, cudaMemcpyAsync(ctx->v_frames.p, &mark, 1, cudaMemcpyHostToDevice, ctx->stream));
    }
    const uint8_t* rows = ctx->v_frames.as<uint8_t>();
    if (ctx->nranks > 1) {
      MPVSS_TRY(comm_allgather(ctx, ctx->v_frames.p, ctx->v_gather.p, rpr * g.row()));
      MPVSS_CUDA(ctx, ctx->v_ordered.ensure(n_total * g.row()));
      MPVSS_TRY(comm_reorder_rows(ctx, ctx->v_gather.p, ctx->v_ordered.p, n_total, g.row()));
      rows = ctx->v_ordered.as<uint8_t>();
    }
    sha2::Sha256 h;  // participant.rs:1205-1212: (X, Y, a1, a2) in publickeys order
    MPVSS_TRY(transcript::fetch_and_hash(ctx, rows, n_total, ctx->nranks, g, h, true));
    for (size_t r = 0; r < std::min<size_t>((size_t)ctx->nranks, n_total); ++r)
      if (ctx->h_frames.as<uint8_t>()[r * g.row()] == 0xff)
        return mpvss_fail(ctx, MPVSS_ERR_ENCODING, "distribute: invalid public key encoding");
    big::Int c = challenge_of(ctx, h, nullptr);
    scalar_out(c, challenge_out);
    const big::Int& ord = ctx->ec_order;
    std::vector<uint32_t> p(nn * 8);
    std::vector<uint8_t> resp(nn * SB);
    MPVSS_TRY(d2h(ctx, p.data(), dp, nn * 32));
    MPVSS_TRY(sync(ctx));
    for (size_t j = 0; j < n; ++j) {  // r = w - p*c (participant.rs:1221-1231 / 1679-1688)
      big::Int pi(p.begin() + j * 8, p.begin() + j * 8 + 8), wi(wl.begin() + j * 8, wl.begin() + j * 8 + 8);
      big::trim(pi);
      big::trim(wi);
      scalar_out(big::submod(wi, big::mulmod(pi, c, ord), ord), resp.data() + j * SB);
    }
    MPVSS_TRY(h2d(ctx, dR, resp.data(), nn * SB));
    const void* dev_rows[3] = {dY.p, dR.p, dX.p};
    uint8_t* host_rows[3] = {shares_out, responses_out, x_out};
    const size_t widths[3] = {EB, SB, EB};
    MPVSS_TRY(transcript::gather_rows(ctx, dev_rows, host_rows, widths, x_out ? 3 : 2, n, n_total));
    MPVSS_TRY(d2h(ctx, commitments_out, dC, t * EB));
    MPVSS_TRY(sync(ctx));
    // U = secret XOR mask(a_0 * G)  (participant.rs:1234-1260 / 1691-1703); C_0 is that point
    big::Int mask;
    if (!T::mask_of(commitments_out, ord, &mask))
      return mpvss_fail(ctx, MPVSS_ERR_ENCODING, "distribute: SHA-256(G^s) is not a canonical scalar");
    big::to_be(big::bxor(big::from_be(secret, secret_len), mask), u_out, EB);
    // the scratch buffers held secrets (coefficients, P(i), witnesses)
    for (DevBuf* b : {&dco, &dp, &dw}) MPVSS_CUDA(ctx, cudaMemsetAsync(b->p, 0, b->cap, ctx->stream));
    return sync(ctx);
  }

  // Per-share Fiat-Shamir step on device-resident encodings: frame the rows F(h1) F(h2) F(a1) F(a2), hash them
  // (sha2_dev.cuh) and finish in the scalar field (ec::proof_body).  Prover (sk, w given): challenge and response
  // in the boundary encoding; verifier (c_in given): ok[i] = recomputed challenge == c_in[i].  The launches are
  // added to the kernel time of the call.
  static int share_transcripts(mpvss_ctx* ctx, const uint8_t* h1, const uint8_t* h2, const uint8_t* a1, const uint8_t* a2,
                               size_t n, const uint32_t* sk, const uint32_t* w, const uint8_t* c_in, uint8_t* c_out,
                               uint8_t* r_out, uint32_t* ok) {
    const uint32_t wide = T::SCALAR_BE ? 0u : 1u;  // ristretto255: SHA-512, little-endian, 512-bit reduction
    const size_t slot = 8 + EB;
    DevBuf &drows = ctx->buf(12), &dh = ctx->buf(13);
    MPVSS_CUDA(ctx, drows.ensure(n * 4 * slot));
    MPVSS_CUDA(ctx, dh.ensure(n * (wide ? 16 : 8) * 4));
    const float ms0 = ctx->last_ms;
    const int l0 = ctx->last_launches;
    timing_begin(ctx);
    ec::FrameArgs FA{h1, h2, a1, a2, drows.as<uint8_t>(), (uint32_t)n, (uint32_t)EB};
    MPVSS_CUDA(ctx, ec::launch_frames(FA, ctx->stream));
    shadev::RowHashArgs HA{drows.as<uint8_t>(), (uint32_t)(4 * slot), (uint32_t)slot, dh.as<uint32_t>(), wide ? 16u : 8u,
                           nullptr, (uint32_t)n, wide};
    MPVSS_CUDA(ctx, shadev::launch_row_hash(HA, ctx->stream));
    ec::ProofArgs PA{KN(ctx), dh.as<uint32_t>(), sk, w, c_in, c_out, r_out, ok, (uint32_t)n, wide, T::SCALAR_BE ? 1u : 0u};
    MPVSS_CUDA(ctx, ec::launch_proof(PA, ctx->stream));
    timing_launch(ctx, 3);
    MPVSS_TRY(timing_end(ctx));
    ctx->last_ms += ms0;
    ctx->last_launches += l0;
    return MPVSS_OK;
  }

  // ---- extract_secret_share (batch) ----------------------------------------------------------------
  static int extract_shares(mpvss_ctx* ctx, size_t n, const uint8_t* private_keys, const uint8_t* witnesses,
                            const uint8_t* enc_shares, uint8_t* publickeys_out, uint8_t* shares_out,
                            uint8_t* challenges_out, uint8_t* responses_out, int* status_out) {
    MPVSS_TRY(bad(ctx, n > 0 && private_keys && witnesses && enc_shares && publickeys_out && shares_out &&
                           challenges_out && responses_out,
                  "extract_shares: bad arguments"));
    std::vector<uint32_t> sk, wl;
    MPVSS_TRY(scalars_in(ctx, private_keys, n, sk));
    MPVSS_TRY(scalars_in(ctx, witnesses, n, wl));
    DevBuf &dsk = ctx->buf(0), &dinv = ctx->buf(1), &dw = ctx->buf(2), &dY = ctx->buf(3), &dpk = ctx->buf(4),
           &dS = ctx->buf(5), &dA1 = ctx->buf(6), &dA2 = ctx->buf(7), &dst = ctx->buf(8), &dis = ctx->buf(9);
    MPVSS_TRY(h2d(ctx, dsk, sk.data(), n * 32));
    MPVSS_TRY(h2d(ctx, dw, wl.data(), n * 32));
    MPVSS_TRY(h2d(ctx, dY, enc_shares, n * EB));
    MPVSS_CUDA(ctx, dinv.ensure(n * 32));
    for (DevBuf* b : {&dpk, &dS, &dA1, &dA2}) MPVSS_CUDA(ctx, b->ensure(n * EB));
    MPVSS_CUDA(ctx, dst.ensure(2 * n * 4));
    MPVSS_CUDA(ctx, dis.ensure(n * 4));
    const uint8_t* G = ctx->gens.as<uint8_t>();
    timing_begin(ctx);
    ec::InvArgs IA{KN(ctx), dsk.as<uint32_t>(), dinv.as<uint32_t>(), dis.as<uint32_t>(), (uint32_t)n};
    MPVSS_CUDA(ctx, ec::launch_inv(IA, ctx->stream));  // 1/sk (participant.rs:1299 / 1742)
    timing_launch(ctx);
    MPVSS_TRY(dev_fixed(ctx, dsk.as<uint32_t>(), n, dpk.as<uint8_t>()));
    MPVSS_TRY(dev_exp2(ctx, dY.as<uint8_t>(), EB, dinv.as<uint32_t>(), nullptr, 0, nullptr, 0, n, dS.as<uint8_t>(),
                       nullptr, dst.as<uint32_t>()));
    MPVSS_TRY(dev_fixed(ctx, dw.as<uint32_t>(), n, dA1.as<uint8_t>()));
    MPVSS_TRY(dev_exp2(ctx, dS.as<uint8_t>(), EB, dw.as<uint32_t>(), nullptr, 0, nullptr, 0, n, dA2.as<uint8_t>(),
                       nullptr, dst.as<uint32_t>() + n));
    MPVSS_TRY(timing_end(ctx));
    MPVSS_TRY(check_status(ctx, dst, 2 * n, "extract_shares (encrypted shares)"));
    // Per-share transcript (pk, Y, a1, a2), challenge and response r = w - sk c on the device (SURVEY 8 f1):
    // n independent SHA-256 chains, one per thread; a1 / a2 never leave the GPU.
    DevBuf &dc = ctx->buf(14), &dr = ctx->buf(15);
    MPVSS_CUDA(ctx, dc.ensure(n * SB));
    MPVSS_CUDA(ctx, dr.ensure(n * SB));
    MPVSS_TRY(share_transcripts(ctx, dpk.as<uint8_t>(), dY.as<uint8_t>(), dA1.as<uint8_t>(), dA2.as<uint8_t>(), n,
                                dsk.as<uint32_t>(), dw.as<uint32_t>(), nullptr, dc.as<uint8_t>(), dr.as<uint8_t>(),
                                nullptr));
    std::vector<uint32_t> inv_st(n);
    MPVSS_TRY(d2h(ctx, publickeys_out, dpk, n * EB));
    MPVSS_TRY(d2h(ctx, shares_out, dS, n * EB));
    MPVSS_TRY(d2h(ctx, challenges_out, dc, n * SB));
    MPVSS_TRY(d2h(ctx, responses_out, dr, n * SB));
    MPVSS_TRY(d2h(ctx, inv_st.data(), dis, n * 4));
    // the scratch buffers held secrets (private keys, inverses, witnesses)
    for (DevBuf* b : {&dsk, &dinv, &dw}) MPVSS_CUDA(ctx, cudaMemsetAsync(b->p, 0, b->cap, ctx->stream));
    MPVSS_TRY(sync(ctx));
    if (status_out)
      for (size_t i = 0; i < n; ++i) status_out[i] = inv_st[i] ? MPVSS_ERR_NOT_INVERTIBLE : MPVSS_OK;
    return MPVSS_OK;
  }

  static int verify_shares(mpvss_ctx* ctx, size_t n, const uint8_t* publickeys, const uint8_t* shares,
                           const uint8_t* enc_shares, const uint8_t* challenges, const uint8_t* responses,
                           int* ok_out) {
    MPVSS_TRY(bad(ctx, n > 0 && publickeys && shares && enc_shares && challenges && responses && ok_out,
                  "verify_shares: bad arguments"));
    std::vector<uint8_t> undecodable;
    // a1 = G^r pk^c, a2 = S^r Y^c stay on the device (a1 / a2 == nullptr): buf(1) = pk, buf(3) = Y, buf(6) = a1,
    // buf(7) = a2 afterwards; the per-share transcript is hashed and compared there (SURVEY 8 f1)
    MPVSS_TRY(dleq_verify_commit(ctx, ctx->ec_gen.data(), publickeys, shares, enc_shares, responses, challenges, SB, n,
                                 nullptr, nullptr, &undecodable));
    DevBuf &dcin = ctx->buf(14), &dok = ctx->buf(15);
    MPVSS_TRY(h2d(ctx, dcin, challenges, n * SB));
    MPVSS_CUDA(ctx, dok.ensure(n * 4));
    MPVSS_TRY(share_transcripts(ctx, ctx->buf(1).as<uint8_t>(), ctx->buf(3).as<uint8_t>(), ctx->buf(6).as<uint8_t>(),
                                ctx->buf(7).as<uint8_t>(), n, nullptr, nullptr, dcin.as<uint8_t>(), nullptr, nullptr,
                                dok.as<uint32_t>()));
    std::vector<uint32_t> okv(n);
    MPVSS_TRY(d2h(ctx, okv.data(), dok, n * 4));
    MPVSS_TRY(sync(ctx));
    // a share box that does not decode is simply not valid (bytes_to_element -> None in the reference)
    for (size_t i = 0; i < n; ++i) ok_out[i] = !undecodable[i] && okv[i] == 1;
    return MPVSS_OK;
  }

  static int reconstruct(mpvss_ctx* ctx, size_t k, const int64_t* positions, const uint8_t* shares, const uint8_t* u,
                         uint8_t* secret_out, uint8_t* gs_out) {
    MPVSS_TRY(bad(ctx, k > 0 && positions && shares && u && secret_out, "reconstruct: bad arguments"));
    std::vector<uint32_t> pos;
    MPVSS_TRY(positions_u32(ctx, positions, k, pos));
    DevBuf &dpos = ctx->buf(10), &dlam = ctx->buf(11);
    MPVSS_TRY(h2d(ctx, dpos, pos.data(), k * 4));
    MPVSS_CUDA(ctx, dlam.ensure(k * 32));
    ec::LagrangeArgs LA{KN(ctx), dpos.as<uint32_t>(), dlam.as<uint32_t>(), (uint32_t)k};
    timing_begin(ctx);  // the Lagrange kernel counts towards the kernel time of the call
    MPVSS_CUDA(ctx, ec::launch_lagrange(LA, ctx->stream));
    MPVSS_TRY(timing_end(ctx));
    const float ms_lambda = ctx->last_ms;
    uint8_t gs[EB];
    MPVSS_TRY(multi_exp_limbs(ctx, shares, dlam.as<uint32_t>(), nullptr, k, gs));
    ctx->last_launches += 1;
    ctx->last_ms += ms_lambda;
    big::Int mask;
    if (!T::mask_of(gs, ctx->ec_order, &mask))
      return mpvss_fail(ctx, MPVSS_ERR_ENCODING, "reconstruct: SHA-256(G^s) is not a canonical scalar");
    big::to_be(big::bxor(mask, big::from_be(u, EB)), secret_out, EB);
    if (gs_out) memcpy(gs_out, gs, EB);
    return MPVSS_OK;
  }

  // Many reconstruct calls in one (mpvss_reconstruct_secrets): the live boxes' positions and shares are
  // concatenated; one box-aware Lagrange launch, one dev_exp2 launch over every share into projective points
  // (its per-share status gives a box's ERR_ENCODING), then segmented 64-way sums that never cross a box
  // boundary until each box has one point, which the last level encodes.
  static int reconstruct_batch(mpvss_ctx* ctx, size_t nb, const size_t* kv, const int64_t* positions,
                               const uint8_t* shares, const uint8_t* u, uint8_t* secrets_out, uint8_t* gs_out,
                               int* status_out) {
    memset(secrets_out, 0, nb * EB);
    if (gs_out) memset(gs_out, 0, nb * EB);
    ctx->last_ms = 0.f;
    ctx->last_launches = 0;
    std::vector<size_t> live, first(nb);  // boxes whose positions are in range; each box's first share
    for (size_t b = 0, off = 0; b < nb; off += kv[b], ++b) {
      first[b] = off;
      status_out[b] = MPVSS_OK;
      for (size_t i = off; i < off + kv[b]; ++i)
        if (positions[i] < 1 || positions[i] > 0x7fffffff) status_out[b] = MPVSS_ERR_ARG;
      if (status_out[b] == MPVSS_OK) live.push_back(b);
    }
    if (live.empty()) return MPVSS_OK;
    const size_t L = live.size();
    size_t n = 0;
    std::vector<uint32_t> start(L), cnt(L);
    for (size_t j = 0; j < L; ++j) {
      start[j] = (uint32_t)n;
      cnt[j] = (uint32_t)kv[live[j]];
      n += cnt[j];
    }
    std::vector<uint32_t> idx(3 * n);  // positions, then per position its box's first row, then its box's k
    std::vector<uint8_t> host(n * EB);
    for (size_t j = 0; j < L; ++j) {
      for (uint32_t i = 0; i < cnt[j]; ++i) {
        idx[start[j] + i] = (uint32_t)positions[first[live[j]] + i];
        idx[n + start[j] + i] = start[j];
        idx[2 * n + start[j] + i] = cnt[j];
      }
      memcpy(host.data() + (size_t)start[j] * EB, shares + first[live[j]] * EB, cnt[j] * EB);
    }
    // every level of the segmented sum, planned here and uploaded at once
    std::vector<uint32_t> seg, level_end;
    {
      std::vector<uint32_t> s(start), c(cnt);
      for (bool last = false; !last;) {
        last = *std::max_element(c.begin(), c.end()) <= 64;
        size_t groups = 0;
        for (uint32_t x : c) groups += (x + 63) / 64;
        const size_t lo = seg.size() / 2;
        seg.resize(2 * (lo + groups));
        ec::sum_boxes_level(s.data(), c.data(), (uint32_t)L, seg.data() + 2 * lo);
        level_end.push_back((uint32_t)(lo + groups));
      }
    }
    DevBuf &dsh = ctx->buf(0), &didx = ctx->buf(1), &dlam = ctx->buf(2), &dj = ctx->buf(3), &dst = ctx->buf(4),
           &dseg = ctx->buf(5), &dtmp = ctx->buf(6), &dout = ctx->buf(7);
    MPVSS_TRY(h2d(ctx, dsh, host.data(), n * EB));
    MPVSS_TRY(h2d(ctx, didx, idx.data(), 3 * n * 4));
    MPVSS_TRY(h2d(ctx, dseg, seg.data(), seg.size() * 4));
    const size_t g1 = level_end[0];  // the first level has the most groups
    MPVSS_CUDA(ctx, dlam.ensure(n * 32));
    MPVSS_CUDA(ctx, dj.ensure(n * sizeof(Point)));
    MPVSS_CUDA(ctx, dst.ensure(n * 4));
    MPVSS_CUDA(ctx, dtmp.ensure(2 * g1 * sizeof(Point)));
    MPVSS_CUDA(ctx, dout.ensure(L * EB));
    const uint32_t* di = didx.as<uint32_t>();
    ec::LagrangeBoxesArgs LA{KN(ctx), di, di + n, di + 2 * n, dlam.as<uint32_t>(), (uint32_t)n};
    timing_begin(ctx);
    MPVSS_CUDA(ctx, ec::launch_lagrange_boxes(LA, ctx->stream));
    timing_launch(ctx);
    MPVSS_TRY(dev_exp2(ctx, dsh.as<uint8_t>(), EB, dlam.as<uint32_t>(), nullptr, 0, nullptr, 0, n, nullptr,
                       dj.as<Point>(), dst.as<uint32_t>()));
    const Point* cur = dj.as<Point>();
    Point* nxt = dtmp.as<Point>();
    Point* alt = nxt + g1;
    for (size_t l = 0; l < level_end.size(); ++l) {
      const uint32_t lo = l ? level_end[l - 1] : 0;
      const bool last = l + 1 == level_end.size();
      ec::SumBoxesArgs<Cv> S{K(ctx), cur, dseg.as<uint32_t>() + 2 * lo, last ? nullptr : nxt,
                             last ? dout.as<uint8_t>() : nullptr, level_end[l] - lo};
      MPVSS_CUDA(ctx, ec::launch_sum_boxes<Cv>(S, ctx->stream));
      timing_launch(ctx);
      cur = nxt;
      std::swap(nxt, alt);
    }
    MPVSS_TRY(timing_end(ctx));
    std::vector<uint32_t> st(n);
    std::vector<uint8_t> gs(L * EB);
    MPVSS_TRY(d2h(ctx, st.data(), dst, n * 4));
    MPVSS_TRY(d2h(ctx, gs.data(), dout, L * EB));
    MPVSS_TRY(sync(ctx));
    for (size_t j = 0; j < L; ++j) {
      const size_t b = live[j];
      big::Int mask;
      if (std::find(st.begin() + start[j], st.begin() + start[j] + cnt[j], 1u) != st.begin() + start[j] + cnt[j] ||
          !T::mask_of(gs.data() + j * EB, ctx->ec_order, &mask)) {
        status_out[b] = MPVSS_ERR_ENCODING;
        continue;
      }
      big::to_be(big::bxor(mask, big::from_be(u + b * EB, EB)), secrets_out + b * EB, EB);
      if (gs_out) memcpy(gs_out + b * EB, gs.data() + j * EB, EB);
    }
    return MPVSS_OK;
  }
};

}  // namespace

#define EC_API_NAMESPACE(ns, Traits)                                                                                 \
  namespace ns {                                                                                                     \
  int init(mpvss_ctx* c) { return Ec<Traits>::init(c); }                                                             \
  int batch_exp(mpvss_ctx* c, const uint8_t* b, size_t bs, const uint8_t* s, size_t n, uint8_t* o) {                 \
    return Ec<Traits>::batch_exp(c, b, bs, s, n, o);                                                                 \
  }                                                                                                                  \
  int fixed_base_exp(mpvss_ctx* c, int g, const uint8_t* s, size_t n, uint8_t* o) {                                  \
    return Ec<Traits>::fixed_base_exp(c, g, s, n, o);                                                                \
  }                                                                                                                  \
  int batch_mul(mpvss_ctx* c, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* o) {                            \
    return Ec<Traits>::batch_mul(c, a, b, n, o);                                                                     \
  }                                                                                                                  \
  int poly_eval_exp(mpvss_ctx* c, const uint8_t* cm, size_t t, const int64_t* p, size_t n, uint8_t* o) {             \
    return Ec<Traits>::poly_eval_exp(c, cm, t, p, n, o);                                                             \
  }                                                                                                                  \
  int dleq_verify_commit(mpvss_ctx* c, const uint8_t* g1, const uint8_t* h1, const uint8_t* g2, const uint8_t* h2,   \
                         const uint8_t* r, const uint8_t* ch, size_t cs, size_t n, uint8_t* a1, uint8_t* a2) {       \
    return Ec<Traits>::dleq_verify_commit(c, g1, h1, g2, h2, r, ch, cs, n, a1, a2);                                  \
  }                                                                                                                  \
  int dleq_prove_commit(mpvss_ctx* c, const uint8_t* g1, const uint8_t* g2, const uint8_t* w, size_t n, uint8_t* a1, \
                        uint8_t* a2) {                                                                               \
    return Ec<Traits>::dleq_prove_commit(c, g1, g2, w, n, a1, a2);                                                   \
  }                                                                                                                  \
  int multi_exp(mpvss_ctx* c, const uint8_t* b, const uint8_t* s, size_t n, uint8_t* o) {                            \
    return Ec<Traits>::multi_exp(c, b, s, n, o);                                                                     \
  }                                                                                                                  \
  int verify_stage(mpvss_ctx* c, size_t n, size_t t, const uint8_t* cm, const int64_t* p, const uint8_t* pk,         \
                   const uint8_t* y, const uint8_t* r, const uint8_t* ch) {                                          \
    return Ec<Traits>::verify_stage(c, n, t, cm, p, pk, y, r, ch);                                                   \
  }                                                                                                                  \
  int verify_run(mpvss_ctx* c, int* ok, uint8_t* x, uint8_t* a1, uint8_t* a2, uint8_t* d) {                          \
    return Ec<Traits>::verify_run(c, ok, x, a1, a2, d);                                                              \
  }                                                                                                                  \
  int verify_batch(mpvss_ctx* c, size_t nb, const size_t* n, const size_t* t, const uint8_t* cm, const int64_t* p,   \
                   const uint8_t* pk, const uint8_t* y, const uint8_t* r, const uint8_t* ch, int* ok, uint8_t* d) {  \
    return Ec<Traits>::verify_batch(c, nb, n, t, cm, p, pk, y, r, ch, ok, d);                                        \
  }                                                                                                                  \
  int scalar_poly_eval(mpvss_ctx* c, const uint8_t* co, size_t t, const int64_t* p, size_t n, uint8_t* o) {        \
    return Ec<Traits>::scalar_poly_eval(c, co, t, p, n, o);                                                          \
  }                                                                                                                  \
  int distribute(mpvss_ctx* c, size_t n, size_t t, const uint8_t* s, size_t sl, const uint8_t* co, const uint8_t* w, \
                 const uint8_t* pk, uint8_t* cm, uint8_t* sh, uint8_t* ch, uint8_t* r, uint8_t* u, uint8_t* x) {     \
    return Ec<Traits>::distribute(c, n, t, s, sl, co, w, pk, cm, sh, ch, r, u, x);                                   \
  }                                                                                                                  \
  int extract_shares(mpvss_ctx* c, size_t n, const uint8_t* sk, const uint8_t* w, const uint8_t* y, uint8_t* pk,     \
                     uint8_t* s, uint8_t* ch, uint8_t* r, int* st) {                                                 \
    return Ec<Traits>::extract_shares(c, n, sk, w, y, pk, s, ch, r, st);                                             \
  }                                                                                                                  \
  int verify_shares(mpvss_ctx* c, size_t n, const uint8_t* pk, const uint8_t* s, const uint8_t* y,                   \
                    const uint8_t* ch, const uint8_t* r, int* ok) {                                                  \
    return Ec<Traits>::verify_shares(c, n, pk, s, y, ch, r, ok);                                                     \
  }                                                                                                                  \
  int reconstruct(mpvss_ctx* c, size_t k, const int64_t* p, const uint8_t* s, const uint8_t* u, uint8_t* o,          \
                  uint8_t* gs) {                                                                                     \
    return Ec<Traits>::reconstruct(c, k, p, s, u, o, gs);                                                            \
  }                                                                                                                  \
  int reconstruct_batch(mpvss_ctx* c, size_t nb, const size_t* k, const int64_t* p, const uint8_t* s,              \
                        const uint8_t* u, uint8_t* o, uint8_t* gs, int* st) {                                        \
    return Ec<Traits>::reconstruct_batch(c, nb, k, p, s, u, o, gs, st);                                              \
  }                                                                                                                  \
  }

EC_API_NAMESPACE(secp_api, SecpTraits)
EC_API_NAMESPACE(rist_api, RistTraits)
