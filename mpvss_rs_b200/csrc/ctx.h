// Internal context shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <mutex>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/mpvss_b200.h"
#include "bigint.h"

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMallocHost(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

struct GroupOps;

struct mpvss_ctx {
  int group = 0;
  const GroupOps* ops = nullptr;  // the group's entry points
  int device = 0;
  int sm_count = 148;  // multiprocessors of the device (read at context creation)
  cudaStream_t stream = nullptr;
  cudaStream_t aux[2] = {nullptr, nullptr};  // side streams for concurrent launches
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_mid = nullptr, ev_h0 = nullptr, ev_h1 = nullptr, ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
  float phase_ms[4] = {0, 0, 0, 0};  // per-phase kernel time of the last fused call
  std::recursive_mutex mu;  // one lock per public call; fused calls re-enter it for their steps
  std::string err;
  float last_ms = 0.f;
  int last_launches = 0;
  bool timing_open = false;

  // ---- ModpGroup ----
  int modp_tpi = 8;
  bool modp_tpi_auto = true;  // Horner launches pick 4 lanes per value when a launch has >= 32768 positions
  int v_tpi = 8;              // lanes per value of the staged Horner plan
  int v_wpc = 1;              // warps per CTA of the staged Horner plan
  std::vector<int64_t> v_plan_pos;  // positions the cached Horner plan (v_ops / v_slot / v_nd) was made for
  int v_plan_tpi = 0, v_plan_wpc = 0;
  size_t v_plan_t = 0;
  uint32_t v_plan_kreq = 0, v_k = 1;  // requested / actual chunks per position of the staged plan
  DevBuf v_first, v_steps, v_e, v_h, v_t2;  // per-CTA chunk bounds, chunk exponents, chunk results, their powers
  int modp_chunks = 0;                // "modp_chunks": chunks per position of the MODP Horner launch (0 = automatic)
  uint64_t v_plan_sqr = 0, v_plan_mul = 0;
  int modp_wpc = 0;           // "modp_wpc": force warps per CTA of the Horner launch (0 = automatic)
  size_t exp2_filler_ctas = 0;  // non-zero: the next dev_exp2 uses the persistent one-warp 'filler' launch with this many CTAs
  int modp_overlap = 3;  // a2 = y^r Y^c (independent of X): 0 before the Horner launch on the main stream; 2 regular launch on a
                         // side stream after it; 3 (default) persistent one-warp CTAs, one per SM, on a side stream after it
  big::Int q, qm1, g;        // modulus, order q-1, subgroup order g = (q-1)/2
  DevBuf consts_q, consts_g; // modp::C_WORDS words each (Montgomery constants for q and for g)
  DevBuf gens;               // [0,64) main generator G = 2, [64,128) subgroup generator g = 4, [128,192) one
  DevBuf comb[2];            // fixed-base tables of the two generators (built on first use, 16.8 MB each)
  int modp_comb = 1;         // use them ("modp_comb")
  int modp_msm = 2;          // multi_exp / reconstruct by buckets: 0 never, 1 always, 2 from msm_threshold bases on
  int msm_threshold = 512;   // measured on B200: buckets 9.0 / 9.8 / 12.4 / 22.5 ms against 9.2 / 13.4 / 33.1 / 119.6 ms direct
                             // at k = 683 / 2731 / 10923 / 43691 (profiles/msm_r02.json)
  // reconstruct_secrets with two or more live boxes (modp_msm = 2): a box takes the bucket method from this many
  // shares on, otherwise its exponentiations join the batch's one direct launch, where it pays only its share of
  // a launch that is already full.  Measured on B200 (profiles/reconstruct_batch_r03.json, whole batch direct vs
  // every box by buckets): 4 x 2731 shares 41.0 vs 57.5 ms, 2 x 5462 43.8 vs 35.8 ms, 2 x 10923 98.5 vs 62.1 ms.
  static constexpr size_t msm_batch_threshold = 4096;
  bool device_hash = false;  // whole-box transcript as one SHA-256 chain on one device thread (measured alternative)
  bool validate = false;     // range / subgroup check of ModpGroup elements entering the verify calls
  bool modp_np1 = false;     // -q^-1 = 1 mod 2^32: Horner kernels skip the Montgomery-digit multiply
  // ---- elliptic-curve groups ----
  size_t ec_threads = 0;        // target thread count of the chunked Horner launch ("ec_threads"); 0 = one full wave
  DevBuf ec_comb;               // fixed-base table of the generator (ec::COMB_WORDS words)
  DevBuf ec_consts;             // secp::Consts / rist::Consts
  big::Int ec_order;            // group order (scalar field modulus)
  std::vector<uint8_t> ec_gen;  // encoded generator (both generators of the trait are this point)
  std::vector<DevBuf> scratch;  // call-local device buffers, reused across calls
  std::vector<PinBuf> pinned;   // call-local pinned host buffers
  // staged verify_distribution state
  size_t v_n = 0, v_t = 0;
  uint32_t v_rwin = 0, v_cwin = 0;
  size_t v_np = 0;  // padded instance count of the Horner launch
  uint32_t v_nops_max = 1;  // products per Horner step of the longest staged addition chain
  std::vector<uint8_t> v_challenge;
  std::vector<uint32_t> v_hpos;  // staged positions (elliptic-curve groups: roofline accounting)
  size_t ec_chunks = 1;          // chunks per position of the last elliptic-curve Horner launch
  const uint32_t* v_comb = nullptr;  // fixed-base table of g for a1 = g^r * X^c
  DevBuf v_slot, v_nd, v_ops, v_comm, v_cm, v_pos, v_pk, v_y, v_r, v_c, v_x, v_a1, v_a2;
  DevBuf v_st, v_cst;  // elliptic curves: decode status of the DLEQ inputs / of the commitments
  // framed transcript rows (dleq.rs:58-61, 87-99): per participant 4 x (u64 BE length || bytes), written by the
  // device in the rank's local order; v_gather holds the rows of all ranks after the all-gather
  DevBuf v_frames, v_gather, v_ordered;  // local rows, all ranks' rows as gathered, the same in participant order
  PinBuf h_frames;
  size_t v_n_total = 0;          // participants of the whole box (== v_n without a communicator)
  uint64_t horner_sqr = 0, horner_mul = 0;  // modular squarings / multiplications of the last X_i launch
  // ---- multi-GPU (one context per GPU, one process or thread per context) ----
  void* comm = nullptr;          // ncclComm_t
  int nranks = 1, rank = 0;
  cudaEvent_t ev_chunk[16] = {};

  // fixed-size pools: references handed out by buf()/pin() stay valid for the whole call
  mpvss_ctx() : scratch(24), pinned(8) {}
  DevBuf& buf(size_t i) { return scratch.at(i); }
  PinBuf& pin(size_t i) { return pinned.at(i); }
};

int mpvss_fail(mpvss_ctx* ctx, int status, const std::string& msg);
int mpvss_cuda_fail(mpvss_ctx* ctx, cudaError_t e, const char* what);

#define MPVSS_CUDA(ctx, expr)                                        \
  do {                                                               \
    cudaError_t _e = (expr);                                         \
    if (_e != cudaSuccess) return mpvss_cuda_fail(ctx, _e, #expr);   \
  } while (0)
#define MPVSS_TRY(expr)            \
  do {                             \
    int _s = (expr);               \
    if (_s != MPVSS_OK) return _s; \
  } while (0)

// kernel-time bracket (CUDA events on the library stream)
void timing_begin(mpvss_ctx* ctx);
void timing_launch(mpvss_ctx* ctx, int n = 1);
int timing_end(mpvss_ctx* ctx);

// ---- per-group implementations ----
// One group's entry points behind the C ABI (modp_api.cu, ec_api.cu); the context holds its group's table.
struct GroupOps {
  int (*init)(mpvss_ctx*);
  int (*batch_exp)(mpvss_ctx*, const uint8_t*, size_t, const uint8_t*, size_t, uint8_t*);
  int (*fixed_base_exp)(mpvss_ctx*, int, const uint8_t*, size_t, uint8_t*);
  int (*batch_mul)(mpvss_ctx*, const uint8_t*, const uint8_t*, size_t, uint8_t*);
  int (*poly_eval_exp)(mpvss_ctx*, const uint8_t*, size_t, const int64_t*, size_t, uint8_t*);
  int (*dleq_verify_commit)(mpvss_ctx*, const uint8_t*, const uint8_t*, const uint8_t*, const uint8_t*, const uint8_t*,
                            const uint8_t*, size_t, size_t, uint8_t*, uint8_t*);
  int (*dleq_prove_commit)(mpvss_ctx*, const uint8_t*, const uint8_t*, const uint8_t*, size_t, uint8_t*, uint8_t*);
  int (*multi_exp)(mpvss_ctx*, const uint8_t*, const uint8_t*, size_t, uint8_t*);
  int (*verify_stage)(mpvss_ctx*, size_t, size_t, const uint8_t*, const int64_t*, const uint8_t*, const uint8_t*,
                      const uint8_t*, const uint8_t*);
  int (*verify_run)(mpvss_ctx*, int*, uint8_t*, uint8_t*, uint8_t*, uint8_t*);
  int (*verify_batch)(mpvss_ctx*, size_t, const size_t*, const size_t*, const uint8_t*, const int64_t*, const uint8_t*,
                      const uint8_t*, const uint8_t*, const uint8_t*, int*, uint8_t*);
  int (*scalar_poly_eval)(mpvss_ctx*, const uint8_t*, size_t, const int64_t*, size_t, uint8_t*);
  int (*distribute)(mpvss_ctx*, size_t, size_t, const uint8_t*, size_t, const uint8_t*, const uint8_t*, const uint8_t*,
                    uint8_t*, uint8_t*, uint8_t*, uint8_t*, uint8_t*, uint8_t*);
  int (*distribute_batch)(mpvss_ctx*, size_t, const size_t*, const size_t*, const uint8_t*, const uint8_t*,
                          const uint8_t*, const uint8_t*, uint8_t*, uint8_t*, uint8_t*, uint8_t*, uint8_t*, uint8_t*, int*);
  int (*extract_shares)(mpvss_ctx*, size_t, const uint8_t*, const uint8_t*, const uint8_t*, uint8_t*, uint8_t*,
                        uint8_t*, uint8_t*, int*);
  int (*verify_shares)(mpvss_ctx*, size_t, const uint8_t*, const uint8_t*, const uint8_t*, const uint8_t*,
                       const uint8_t*, int*);
  int (*reconstruct_batch)(mpvss_ctx*, size_t, const size_t*, const int64_t*, const uint8_t*, const uint8_t*, uint8_t*,
                           uint8_t*, int*);
};
extern const GroupOps modp_ops, secp_ops, rist_ops;
