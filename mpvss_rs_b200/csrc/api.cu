// extern "C" surface of libmpvss_b200.so (declared in include/mpvss_b200.h): context
// management, error reporting and dispatch to the per-group implementations.
#include "ctx.h"
#include "transcript.h"

int mpvss_fail(mpvss_ctx* ctx, int status, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return status;
}
int mpvss_cuda_fail(mpvss_ctx* ctx, cudaError_t e, const char* what) {
  if (ctx) ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
  cudaGetLastError();  // clear the sticky flag of non-fatal errors
  return MPVSS_ERR_CUDA;
}

void timing_begin(mpvss_ctx* ctx) {
  ctx->last_launches = 0;
  ctx->last_ms = 0.f;
  cudaEventRecord(ctx->ev0, ctx->stream);
  ctx->timing_open = true;
}
void timing_launch(mpvss_ctx* ctx, int n) { ctx->last_launches += n; }
int timing_end(mpvss_ctx* ctx) {
  MPVSS_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  MPVSS_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
  MPVSS_CUDA(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  ctx->timing_open = false;
  return MPVSS_OK;
}

namespace {
struct Guard {
  mpvss_ctx* c;
  explicit Guard(mpvss_ctx* ctx) : c(ctx) {
    c->mu.lock();
    cudaSetDevice(c->device);
  }
  ~Guard() { c->mu.unlock(); }
};
int unsupported(mpvss_ctx* ctx, const char* fn) {
  return mpvss_fail(ctx, MPVSS_ERR_UNSUPPORTED, std::string(fn) + ": not available for this group in this build");
}
}  // namespace

#define DISPATCH(ctx, fn, ...)                                             \
  do {                                                                     \
    if (!(ctx)) return MPVSS_ERR_ARG;                                      \
    Guard _g(ctx);                                                         \
    switch ((ctx)->group) {                                                \
      case MPVSS_GROUP_MODP: return modp_api::fn(ctx, __VA_ARGS__);        \
      case MPVSS_GROUP_SECP256K1: return secp_api::fn(ctx, __VA_ARGS__);   \
      case MPVSS_GROUP_RISTRETTO255: return rist_api::fn(ctx, __VA_ARGS__); \
      default: return unsupported(ctx, #fn);                               \
    }                                                                      \
  } while (0)

extern "C" {

int mpvss_ctx_create(int group, int device, mpvss_ctx** out) {
  if (!out) return MPVSS_ERR_ARG;
  *out = nullptr;
  if (group < MPVSS_GROUP_MODP || group > MPVSS_GROUP_RISTRETTO255) return MPVSS_ERR_ARG;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
    cudaGetLastError();
    return MPVSS_ERR_CUDA;  // no CPU fallback: the hot path exists only on the GPU
  }
  mpvss_ctx* ctx = new mpvss_ctx();
  ctx->group = group;
  ctx->device = device;
  auto bail = [&](int s) {
    mpvss_ctx_destroy(ctx);
    return s;
  };
  if (cudaSetDevice(device) != cudaSuccess) return bail(MPVSS_ERR_CUDA);
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) ctx->sm_count = sms;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MPVSS_ERR_CUDA);
  if (cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
      cudaEventCreate(&ctx->ev_mid) != cudaSuccess || cudaEventCreate(&ctx->ev_h0) != cudaSuccess ||
      cudaEventCreate(&ctx->ev_h1) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess)
    return bail(MPVSS_ERR_CUDA);
  for (int a = 0; a < 2; ++a)
    if (cudaStreamCreateWithFlags(&ctx->aux[a], cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_join[a], cudaEventDisableTiming) != cudaSuccess)
      return bail(MPVSS_ERR_CUDA);
  for (cudaEvent_t& e : ctx->ev_chunk)
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(MPVSS_ERR_CUDA);
  int s = MPVSS_OK;
  if (group == MPVSS_GROUP_MODP) s = modp_api::init(ctx);
  if (group == MPVSS_GROUP_SECP256K1) s = secp_api::init(ctx);
  if (group == MPVSS_GROUP_RISTRETTO255) s = rist_api::init(ctx);
  if (s != MPVSS_OK) return bail(s);
  *out = ctx;
  return MPVSS_OK;
}

void mpvss_ctx_destroy(mpvss_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  comm_release(ctx);
  // scratch and pinned buffers may have held secrets (private keys, witnesses, coefficients)
  for (auto& b : ctx->scratch)
    if (b.p) cudaMemset(b.p, 0, b.cap);
  for (auto& b : ctx->pinned)
    if (b.p) memset(b.p, 0, b.cap);
  modp_api::destroy(ctx);
  ctx->h_frames.release();
  for (cudaEvent_t e : ctx->ev_chunk)
    if (e) cudaEventDestroy(e);
  ctx->ec_consts.release();
  ctx->ec_comb.release();
  for (auto& b : ctx->scratch) b.release();
  for (auto& b : ctx->pinned) b.release();
  for (cudaEvent_t e : {ctx->ev0, ctx->ev1, ctx->ev_mid, ctx->ev_h0, ctx->ev_h1, ctx->ev_fork, ctx->ev_join[0], ctx->ev_join[1]})
    if (e) cudaEventDestroy(e);
  for (int a = 0; a < 2; ++a)
    if (ctx->aux[a]) cudaStreamDestroy(ctx->aux[a]);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* mpvss_last_error(const mpvss_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int mpvss_ctx_set_int(mpvss_ctx* ctx, const char* key, int value) {
  if (!ctx || !key) return MPVSS_ERR_ARG;
  Guard g(ctx);
  if (std::string(key) == "modp_tpi") {
    if (value != 4 && value != 8 && value != 16) return mpvss_fail(ctx, MPVSS_ERR_ARG, "modp_tpi must be 4, 8 or 16");
    ctx->modp_tpi = value;
    ctx->modp_tpi_auto = false;  // an explicit choice applies to every kernel
    return MPVSS_OK;
  }
  if (std::string(key) == "ec_threads") {
    if (value != 0 && value < 32) return mpvss_fail(ctx, MPVSS_ERR_ARG, "ec_threads must be 0 (auto) or >= 32");
    ctx->ec_threads = (size_t)value;
    return MPVSS_OK;
  }
  if (std::string(key) == "modp_comb") {
    ctx->modp_comb = value != 0;
    return MPVSS_OK;
  }
  if (std::string(key) == "modp_overlap") {
    ctx->modp_overlap = value;
    return MPVSS_OK;
  }
  if (std::string(key) == "modp_chunks") {
    if (value < 0 || value > 64) return mpvss_fail(ctx, MPVSS_ERR_ARG, "modp_chunks must be 0 (automatic) .. 64");
    ctx->modp_chunks = value;
    return MPVSS_OK;
  }
  if (std::string(key) == "modp_wpc") {
    if (value < 0 || value > 4) return mpvss_fail(ctx, MPVSS_ERR_ARG, "modp_wpc must be 0 (automatic) .. 4");
    ctx->modp_wpc = value;
    return MPVSS_OK;
  }
  if (std::string(key) == "modp_msm") {
    if (value < 0 || value > 2) return mpvss_fail(ctx, MPVSS_ERR_ARG, "modp_msm must be 0, 1 or 2");
    ctx->modp_msm = value;
    return MPVSS_OK;
  }
  if (std::string(key) == "msm_threshold") {
    ctx->msm_threshold = value;
    return MPVSS_OK;
  }
  if (std::string(key) == "device_hash") {
    ctx->device_hash = value != 0;
    return MPVSS_OK;
  }
  if (std::string(key) == "validate") {
    ctx->validate = value != 0;
    return MPVSS_OK;
  }
  return mpvss_fail(ctx, MPVSS_ERR_ARG, std::string("unknown tunable: ") + key);
}

size_t mpvss_element_bytes(const mpvss_ctx* ctx) {
  if (!ctx) return 0;
  return ctx->group == MPVSS_GROUP_MODP ? 256 : ctx->group == MPVSS_GROUP_SECP256K1 ? 33 : 32;
}
size_t mpvss_scalar_bytes(const mpvss_ctx* ctx) {
  if (!ctx) return 0;
  return ctx->group == MPVSS_GROUP_MODP ? 256 : 32;
}
float mpvss_last_kernel_ms(const mpvss_ctx* ctx) { return ctx ? ctx->last_ms : 0.f; }
int mpvss_last_kernel_launches(const mpvss_ctx* ctx) { return ctx ? ctx->last_launches : 0; }
uint64_t mpvss_last_horner_products(const mpvss_ctx* ctx, int which) {
  return !ctx ? 0 : which == 0 ? ctx->horner_sqr : ctx->horner_mul;
}
float mpvss_last_phase_ms(const mpvss_ctx* ctx, int phase) {
  return (ctx && phase >= 0 && phase < 4) ? ctx->phase_ms[phase] : 0.f;
}

int mpvss_batch_exp(mpvss_ctx* ctx, const uint8_t* bases, size_t base_stride, const uint8_t* scalars, size_t n,
                    uint8_t* out) {
  DISPATCH(ctx, batch_exp, bases, base_stride, scalars, n, out);
}
int mpvss_fixed_base_exp(mpvss_ctx* ctx, int generator, const uint8_t* scalars, size_t n, uint8_t* out) {
  DISPATCH(ctx, fixed_base_exp, generator, scalars, n, out);
}
int mpvss_batch_mul(mpvss_ctx* ctx, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  DISPATCH(ctx, batch_mul, a, b, n, out);
}
int mpvss_poly_eval_exp(mpvss_ctx* ctx, const uint8_t* commitments, size_t t, const int64_t* positions, size_t n,
                        uint8_t* out) {
  DISPATCH(ctx, poly_eval_exp, commitments, t, positions, n, out);
}
int mpvss_dleq_verify_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* h1, const uint8_t* g2,
                             const uint8_t* h2, const uint8_t* r, const uint8_t* c, size_t c_stride, size_t n,
                             uint8_t* a1, uint8_t* a2) {
  if (ctx && (!a1 || !a2)) {  // only internal callers may leave the results on the device
    Guard g(ctx);
    return mpvss_fail(ctx, MPVSS_ERR_ARG, "dleq_verify_commit: bad arguments");
  }
  DISPATCH(ctx, dleq_verify_commit, g1, h1, g2, h2, r, c, c_stride, n, a1, a2);
}
int mpvss_dleq_prove_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* g2, const uint8_t* w, size_t n,
                            uint8_t* a1, uint8_t* a2) {
  DISPATCH(ctx, dleq_prove_commit, g1, g2, w, n, a1, a2);
}
int mpvss_multi_exp(mpvss_ctx* ctx, const uint8_t* bases, const uint8_t* scalars, size_t n, uint8_t* out) {
  DISPATCH(ctx, multi_exp, bases, scalars, n, out);
}
int mpvss_verify_distribution_stage(mpvss_ctx* ctx, size_t n, size_t t, const uint8_t* commitments,
                                    const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares,
                                    const uint8_t* responses, const uint8_t* challenge) {
  DISPATCH(ctx, verify_stage, n, t, commitments, positions, publickeys, shares, responses, challenge);
}
int mpvss_verify_distribution_run(mpvss_ctx* ctx, int* ok, uint8_t* x_out, uint8_t* a1_out, uint8_t* a2_out,
                                  uint8_t* digest_out) {
  DISPATCH(ctx, verify_run, ok, x_out, a1_out, a2_out, digest_out);
}
// Box contents that do not decode (bad point, non-canonical scalar, position out of range) make the
// reference return false (participant.rs:415-420, bytes_to_element -> None), not fail: only caller
// or CUDA faults are reported as errors.
static int box_verdict(int status, int* ok) {
  if (status == MPVSS_ERR_ENCODING && ok) {
    *ok = 0;
    return MPVSS_OK;
  }
  return status;
}
int mpvss_verify_distribution(mpvss_ctx* ctx, size_t n, size_t t, const uint8_t* commitments,
                              const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares,
                              const uint8_t* responses, const uint8_t* challenge, int* ok, uint8_t* x_out,
                              uint8_t* a1_out, uint8_t* a2_out, uint8_t* digest_out) {
  if (!ctx || !ok) return MPVSS_ERR_ARG;
  Guard hold(ctx);  // one lock across both steps: no other thread can stage a different box in between
  int s = mpvss_verify_distribution_stage(ctx, n, t, commitments, positions, publickeys, shares, responses, challenge);
  if (s != MPVSS_OK) return box_verdict(s, ok);
  return box_verdict(mpvss_verify_distribution_run(ctx, ok, x_out, a1_out, a2_out, digest_out), ok);
}
int mpvss_verify_distributions(mpvss_ctx* ctx, size_t n_boxes, const size_t* n, const size_t* t,
                               const uint8_t* commitments, const int64_t* positions, const uint8_t* publickeys,
                               const uint8_t* shares, const uint8_t* responses, const uint8_t* challenges,
                               int* ok_out, uint8_t* digests_out) {
  if (!ctx) return MPVSS_ERR_ARG;
  Guard hold(ctx);
  if (n_boxes == 0 || !n || !t || !commitments || !publickeys || !shares || !responses || !challenges || !ok_out)
    return mpvss_fail(ctx, MPVSS_ERR_ARG, "verify_distributions: bad arguments");
  // the kernels count positions and commitments in 32 bits
  const size_t limit = 0x7fffffff;
  size_t sum_n = 0, sum_t = 0;
  for (size_t b = 0; b < n_boxes; ++b) {
    if (n[b] == 0 || t[b] == 0 || n[b] > limit - sum_n || t[b] > limit - sum_t)
      return mpvss_fail(ctx, MPVSS_ERR_ARG, "verify_distributions: box " + std::to_string(b) +
                                                " has no participants or commitments, or the boxes are too many");
    sum_n += n[b];
    sum_t += t[b];
  }
  if (ctx->nranks > 1) return mpvss_fail(ctx, MPVSS_ERR_UNSUPPORTED, "verify_distributions: not collective");
  DISPATCH(ctx, verify_batch, n_boxes, n, t, commitments, positions, publickeys, shares, responses, challenges, ok_out,
           digests_out);
}
int mpvss_scalar_poly_eval(mpvss_ctx* ctx, const uint8_t* coeffs, size_t t, const int64_t* positions, size_t n,
                           uint8_t* out) {
  DISPATCH(ctx, scalar_poly_eval, coeffs, t, positions, n, out);
}
int mpvss_transcript_digest(int group, const uint8_t* rows, size_t n_total, int nranks, uint8_t* digest_out) {
  if (!rows || !digest_out || n_total == 0 || nranks < 1 || group < MPVSS_GROUP_MODP || group > MPVSS_GROUP_RISTRETTO255)
    return MPVSS_ERR_ARG;
  const transcript::Geom g{group == MPVSS_GROUP_MODP ? (size_t)256 : group == MPVSS_GROUP_SECP256K1 ? (size_t)33 : (size_t)32,
                           group == MPVSS_GROUP_MODP};
  sha2::Sha256 h;
  transcript::hash_range(h, rows, 0, n_total, nranks, transcript::rows_per_rank(n_total, nranks), g);
  h.finalize(digest_out);
  return MPVSS_OK;
}
int mpvss_distribute(mpvss_ctx* ctx, size_t n, size_t t, const uint8_t* secret, size_t secret_len,
                     const uint8_t* coeffs, const uint8_t* witnesses, const uint8_t* publickeys,
                     uint8_t* commitments_out, uint8_t* shares_out, uint8_t* challenge_out, uint8_t* responses_out,
                     uint8_t* u_out, uint8_t* x_out) {
  DISPATCH(ctx, distribute, n, t, secret, secret_len, coeffs, witnesses, publickeys, commitments_out, shares_out,
           challenge_out, responses_out, u_out, x_out);
}
int mpvss_extract_shares(mpvss_ctx* ctx, size_t n, const uint8_t* private_keys, const uint8_t* witnesses,
                         const uint8_t* enc_shares, uint8_t* publickeys_out, uint8_t* shares_out,
                         uint8_t* challenges_out, uint8_t* responses_out, int* status_out) {
  DISPATCH(ctx, extract_shares, n, private_keys, witnesses, enc_shares, publickeys_out, shares_out, challenges_out,
           responses_out, status_out);
}
int mpvss_verify_shares(mpvss_ctx* ctx, size_t n, const uint8_t* publickeys, const uint8_t* shares,
                        const uint8_t* enc_shares, const uint8_t* challenges, const uint8_t* responses, int* ok_out) {
  DISPATCH(ctx, verify_shares, n, publickeys, shares, enc_shares, challenges, responses, ok_out);
}
int mpvss_reconstruct(mpvss_ctx* ctx, size_t k, const int64_t* positions, const uint8_t* shares, const uint8_t* u,
                      uint8_t* secret_out, uint8_t* gs_out) {
  DISPATCH(ctx, reconstruct, k, positions, shares, u, secret_out, gs_out);
}
int mpvss_reconstruct_secrets(mpvss_ctx* ctx, size_t n_boxes, const size_t* k, const int64_t* positions,
                              const uint8_t* shares, const uint8_t* u, uint8_t* secrets_out, uint8_t* gs_out,
                              int* status_out) {
  if (!ctx) return MPVSS_ERR_ARG;
  Guard hold(ctx);
  if (n_boxes == 0 || !k || !positions || !shares || !u || !secrets_out || !status_out)
    return mpvss_fail(ctx, MPVSS_ERR_ARG, "reconstruct_secrets: bad arguments");
  const size_t limit = 0x7fffffff;  // the kernels count shares in 32 bits
  size_t sum_k = 0;
  for (size_t b = 0; b < n_boxes; ++b) {
    if (k[b] == 0 || k[b] > limit - sum_k)
      return mpvss_fail(ctx, MPVSS_ERR_ARG, "reconstruct_secrets: box " + std::to_string(b) +
                                                " has no shares, or the boxes are too many");
    sum_k += k[b];
  }
  DISPATCH(ctx, reconstruct_batch, n_boxes, k, positions, shares, u, secrets_out, gs_out, status_out);
}

}  // extern "C"
