/* mpvss_b200 -- C ABI of the B200 (sm_100a) back-end for the batched
 * group-exponentiation hot path of AlexiaChen/mpvss-rs.
 *
 * This is the drop-in boundary: the entry points below are what the reference's
 * FFI layer (a `build.rs` + `extern "C"` block behind new batch methods of
 * `trait Group`, src/group.rs:24-124) would bind.  INTEGRATION.md shows the Rust
 * side.  Plain pointers and sizes only; the library owns all device memory and
 * streams inside the context and never keeps a host pointer past return.
 *
 * Encodings at this boundary (fixed width, structure-of-arrays, index = position-1
 * in `publickeys` order, src/participant.rs:186,198,247):
 *   ModpGroup      element / scalar : 256 bytes, little-endian integer
 *                  (reference type: num_bigint::BigInt, src/groups/modp.rs:94-95)
 *   Secp256k1Group element : 33 bytes SEC1 compressed (src/groups/secp256k1.rs:133-136)
 *                  scalar  : 32 bytes big-endian      (src/groups/secp256k1.rs:154-156)
 *   Ristretto255   element : 32 bytes RFC 9496        (src/groups/ristretto255.rs:207-210)
 *                  scalar  : 32 bytes little-endian   (src/groups/ristretto255.rs:222-225)
 *
 * Every function returns MPVSS_OK (0) or a negative status; mpvss_last_error()
 * gives the text.  Nothing panics or throws across the boundary.  A context may
 * be used from any thread, one call at a time: every entry point holds the
 * context's lock for its whole duration (the fused calls for all their steps).  The
 * two-step pair mpvss_verify_distribution_stage / _run shares staged state between
 * two calls and must be serialised by the caller as a pair.
 * There is no CPU fallback: without a CUDA device mpvss_ctx_create fails.
 *
 * Multi-GPU: one context per GPU (one process or thread each), joined by
 * mpvss_comm_init.  Participants are independent, so the fused phase calls
 * (mpvss_verify_distribution, mpvss_distribute) shard them inside the call --
 * rank r takes participants r, r + N, ... -- and exchange the results with one
 * NCCL all-gather per phase on the library's stream (SURVEY section 8e).  Such
 * calls are collective: every rank makes the same call with the same arguments
 * and every rank receives the full result.
 */
#ifndef MPVSS_B200_H
#define MPVSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mpvss_ctx mpvss_ctx;

enum mpvss_group {
  MPVSS_GROUP_MODP = 0,        /* ModpGroup::new(), RFC 3526 group 14 (src/groups/modp.rs:44-70) */
  MPVSS_GROUP_SECP256K1 = 1,   /* Secp256k1Group::new() (src/groups/secp256k1.rs:44-55) */
  MPVSS_GROUP_RISTRETTO255 = 2 /* Ristretto255Group::new() (src/groups/ristretto255.rs:51-63) */
};

enum mpvss_status {
  MPVSS_OK = 0,
  MPVSS_ERR_CUDA = -1,        /* CUDA runtime / launch failure, or no device */
  MPVSS_ERR_ARG = -2,         /* null pointer, zero count, threshold > n, ... */
  MPVSS_ERR_ENCODING = -3,    /* invalid element / scalar encoding (reference: None / false) */
  MPVSS_ERR_UNSUPPORTED = -4, /* operation not available for this group */
  MPVSS_ERR_NOT_INVERTIBLE = -5, /* scalar without inverse (reference: extract_secret_share -> None) */
  MPVSS_ERR_COMM = -6          /* NCCL missing or a collective failed */
};

enum mpvss_generator {
  MPVSS_GEN_MAIN = 0,    /* Group::generator()          (G: public keys, G^s, share proofs) */
  MPVSS_GEN_SUBGROUP = 1 /* Group::subgroup_generator() (g: commitments, distribution proofs) */
};

/* ---- context ---------------------------------------------------------------- */
int mpvss_ctx_create(int group, int device, mpvss_ctx** out);
void mpvss_ctx_destroy(mpvss_ctx* ctx);
const char* mpvss_last_error(const mpvss_ctx* ctx);
/* tunables: "modp_tpi" (lanes per 2048-bit value: 4, 8, 16); "modp_comb" (0/1: fixed-base tables for
 * the two generators); "modp_overlap" (where the X-independent a2 = y^r Y^c runs during
 * verify_distribution and verify_distributions: 0 before the X_i launch, 2 beside it on a side stream,
 * 3 (default) beside it as one persistent one-warp CTA per SM, which takes the warp slot the X_i launch leaves idle; the default falls
 * back to 0 when that slot does not exist, or to 2 for small boxes whose two launches fit the chip together);
 * "modp_chunks" (contiguous chunks per position of the X_i launch, 0 = automatic: more than one only when the
 * launch would leave most of the chip idle); "modp_wpc" (warps per CTA of that launch); "modp_msm" /
 * "msm_threshold" (bucket method for multi_exp / reconstruct); "ec_threads" (thread target of the chunked
 * elliptic-curve Horner launch); "device_hash" (0/1, default 0: hash the whole-box transcript of
 * verify_distribution as one SHA-256 chain on one device thread instead of on the host -- a measured alternative,
 * two orders of magnitude slower than the host's SHA-NI; the per-share transcripts of extract_shares /
 * verify_shares are always hashed on the device, one chain per thread); "validate" (0/1, default 0:
 * ModpGroup elements entering verify_distribution / verify_shares are checked for range 0 < x < q and
 * subgroup membership x^g = 1 -- the reference's bytes_to_element accepts anything, modp.rs:154-156;
 * a box that fails verifies as false) */
int mpvss_ctx_set_int(mpvss_ctx* ctx, const char* key, int value);
size_t mpvss_element_bytes(const mpvss_ctx* ctx);
size_t mpvss_scalar_bytes(const mpvss_ctx* ctx);
/* device time (ms, CUDA events on the library's stream) spent in kernels by the last call,
 * and the number of kernel launches it made */
float mpvss_last_kernel_ms(const mpvss_ctx* ctx);
int mpvss_last_kernel_launches(const mpvss_ctx* ctx);
/* modular squarings (which = 0) and multiplications (which = 1) executed by the last X_i launch of a
 * ModpGroup context (summed over this rank's participants): the algorithmic work behind the roofline
 * figure bench.py reports.  EC contexts: field squarings / multiplications of the last Horner launch. */
uint64_t mpvss_last_horner_products(const mpvss_ctx* ctx, int which);
/* kernel time (ms) of one phase of the last fused call.  verify_distribution: phase 0 = X_i
 * (Montgomery conversion + Horner multi-exponentiation [+ chunk combination]; a2 runs underneath on
 * a side stream), phase 1 = remaining DLEQ commitments, phase 2 = the Horner launch alone (MODP). */
float mpvss_last_phase_ms(const mpvss_ctx* ctx, int phase);

/* ---- batch forms of `trait Group` methods ------------------------------------ */
/* Group::exp (src/group.rs:58): out[i] = bases[i] ^ scalars[i].  base_stride = 0 means one
 * shared base; otherwise the element size. */
int mpvss_batch_exp(mpvss_ctx* ctx, const uint8_t* bases, size_t base_stride, const uint8_t* scalars, size_t n,
                    uint8_t* out);
/* Group::exp with Group::generator()/subgroup_generator() as the base
 * (commitments participant.rs:189-193, public keys modp.rs:176-178, a1 = g^w dleq.rs:207-209). */
int mpvss_fixed_base_exp(mpvss_ctx* ctx, int generator, const uint8_t* scalars, size_t n, uint8_t* out);
/* Group::mul (src/group.rs:66): out[i] = a[i] * b[i]. */
int mpvss_batch_mul(mpvss_ctx* ctx, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
/* X_i = prod_j C_j^(i^j)  (participant.rs:207-215, 423-434; mpvss.rs:114-123) for the given
 * 1-based positions (NULL = 1..n). */
int mpvss_poly_eval_exp(mpvss_ctx* ctx, const uint8_t* commitments, size_t t, const int64_t* positions, size_t n,
                        uint8_t* out);
/* Polynomial::get_value reduced as its callers do (polynomial.rs:50-58; participant.rs:202, 1155-1157,
 * 1619-1621): out[i] = sum_j coeffs[j] * positions[i]^j mod order, order = q-1 / n / l.
 * positions NULL = 1..n. */
int mpvss_scalar_poly_eval(mpvss_ctx* ctx, const uint8_t* coeffs, size_t t, const int64_t* positions, size_t n,
                           uint8_t* out);
/* Verifier::commitments (dleq.rs:66-84): a1[i] = g1^r[i] * h1[i]^c[i], a2[i] = g2[i]^r[i] * h2[i]^c[i].
 * g1 is one element (a generator); c_stride = 0 means one shared challenge. */
int mpvss_dleq_verify_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* h1, const uint8_t* g2,
                             const uint8_t* h2, const uint8_t* r, const uint8_t* c, size_t c_stride, size_t n,
                             uint8_t* a1, uint8_t* a2);
/* Prover::send (dleq.rs:37-39): a1[i] = g1^w[i], a2[i] = g2[i]^w[i]. */
int mpvss_dleq_prove_commit(mpvss_ctx* ctx, const uint8_t* g1, const uint8_t* g2, const uint8_t* w, size_t n,
                            uint8_t* a1, uint8_t* a2);
/* prod_i bases[i]^scalars[i]  (the reconstruct fold, participant.rs:490-509). */
int mpvss_multi_exp(mpvss_ctx* ctx, const uint8_t* bases, const uint8_t* scalars, size_t n, uint8_t* out);

/* ---- fused phases (flattened Participant<G> entry points) ----------------------- */
/* Participant::verify_distribution_shares (participant.rs:399-455 / 1384-1442 / 1827-1885,
 * mpvss.rs:90-144).  Arrays are in `publickeys` order.  *ok = 1 iff the recomputed challenge
 * equals `challenge`.  x_out / a1_out / a2_out (n elements each) and digest_out (32 bytes,
 * SHA-256 of the framed transcript) are optional. */
int mpvss_verify_distribution(mpvss_ctx* ctx, size_t n, size_t t, const uint8_t* commitments,
                              const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares,
                              const uint8_t* responses, const uint8_t* challenge, int* ok, uint8_t* x_out,
                              uint8_t* a1_out, uint8_t* a2_out, uint8_t* digest_out);
/* Two-step form for callers that keep the box resident on the device (used by bench.py to
 * time the path without the host->device copies): stage copies the inputs, run verifies.  With a
 * communicator both are collective like mpvss_verify_distribution; x/a1/a2 outputs must then be NULL. */
int mpvss_verify_distribution_stage(mpvss_ctx* ctx, size_t n, size_t t, const uint8_t* commitments,
                                    const int64_t* positions, const uint8_t* publickeys, const uint8_t* shares,
                                    const uint8_t* responses, const uint8_t* challenge);
int mpvss_verify_distribution_run(mpvss_ctx* ctx, int* ok, uint8_t* x_out, uint8_t* a1_out, uint8_t* a2_out,
                                  uint8_t* digest_out);
/* n_boxes independent Participant::verify_distribution_shares calls in one (e.g. the n boxes of one PVSS
 * round).  Box b has n[b] participants and t[b] commitments.  Every array is the concatenation, in box order,
 * of what mpvss_verify_distribution takes for one box: commitments (sum t[b] elements), positions (sum n[b];
 * NULL = 1..n[b] in every box), publickeys and shares (sum n[b] elements), responses (sum n[b] scalars),
 * challenges (n_boxes scalars).  ok_out[b] = 1 iff box b verifies.  digests_out (optional, 32 bytes per box)
 * receives the transcript digest that mpvss_verify_distribution returns for that box alone.  Box contents that
 * do not decode, fail the "validate" check, or carry a position outside [1, 2^31) make that box verify as
 * false (its digest is then zero) and leave the other boxes alone; the call still returns MPVSS_OK.  The
 * boxes' transcripts are always hashed on the host ("device_hash" does not apply).  The staged state of
 * mpvss_verify_distribution_stage is left untouched.  Not collective: on a context with a communicator it
 * returns MPVSS_ERR_UNSUPPORTED. */
int mpvss_verify_distributions(mpvss_ctx* ctx, size_t n_boxes, const size_t* n, const size_t* t,
                               const uint8_t* commitments, const int64_t* positions, const uint8_t* publickeys,
                               const uint8_t* shares, const uint8_t* responses, const uint8_t* challenges,
                               int* ok_out, uint8_t* digests_out);

/* Participant::distribute_secret (participant.rs:160-286 / 1094-1274 / 1573-1717) with the
 * randomness injected: `coeffs` (t scalars) replaces Polynomial::init (polynomial.rs:34-47),
 * `witnesses` (n scalars) replaces generate_private_key (participant.rs:223).  `secret` is a
 * big-endian integer of secret_len bytes (lib.rs:49-52).  Outputs: commitments (t elements),
 * shares Y (n), challenge (1 scalar), responses (n scalars), u_out (element-size bytes,
 * big-endian, left-padded).  x_out is optional. */
int mpvss_distribute(mpvss_ctx* ctx, size_t n, size_t t, const uint8_t* secret, size_t secret_len,
                     const uint8_t* coeffs, const uint8_t* witnesses, const uint8_t* publickeys,
                     uint8_t* commitments_out, uint8_t* shares_out, uint8_t* challenge_out, uint8_t* responses_out,
                     uint8_t* u_out, uint8_t* x_out);
/* n_boxes independent Participant::distribute_secret calls in one (e.g. the boxes of many future beacon epochs,
 * or every dealer of a round played by one harness).  Box b has n[b] participants at positions 1..n[b] and t[b]
 * coefficients.  Every array is the concatenation, in box order, of what mpvss_distribute takes or returns for
 * one box: coeffs (sum t[b] scalars), witnesses (sum n[b] scalars), publickeys (sum n[b] elements),
 * commitments_out (sum t[b] elements), shares_out (sum n[b] elements), responses_out (sum n[b] scalars), x_out
 * (optional, sum n[b] elements), challenges_out (n_boxes scalars).  secrets and u_out hold n_boxes rows of
 * element size, big-endian and left-padded (the width mpvss_reconstruct takes U and returns secrets in).  Every
 * row of box b is byte-identical to what mpvss_distribute returns for box b alone.  status_out[b] is that box's
 * status: in secp256k1 and ristretto255 MPVSS_ERR_ENCODING for an undecodable public key, and in secp256k1 also
 * for a coefficient or witness not below the group order or a SHA-256(G^s) that is not a canonical scalar;
 * ModpGroup rejects no box.  A rejected box has zero rows in every output and leaves the other boxes alone; the
 * call still returns MPVSS_OK and records no error.  Caller errors return MPVSS_ERR_ARG: no boxes, a null
 * pointer other than x_out, n[b] == 0, t[b] == 0, t[b] > n[b], or more participants or coefficients than 32-bit
 * counts hold.  Staged mpvss_verify_distribution_stage state is left untouched.  Not collective: on a context
 * with a communicator it returns MPVSS_ERR_UNSUPPORTED. */
int mpvss_distribute_secrets(mpvss_ctx* ctx, size_t n_boxes, const size_t* n, const size_t* t,
                             const uint8_t* secrets, const uint8_t* coeffs, const uint8_t* witnesses,
                             const uint8_t* publickeys, uint8_t* commitments_out, uint8_t* shares_out,
                             uint8_t* challenges_out, uint8_t* responses_out, uint8_t* u_out, uint8_t* x_out,
                             int* status_out);

/* n independent Participant::extract_secret_share calls (participant.rs:294-353 / 1282-1338 /
 * 1725-1781): private key, witness and encrypted share per participant ->
 * ShareBox{publickey, share, challenge, response}.  status_out[i] (optional) is MPVSS_OK or
 * MPVSS_ERR_NOT_INVERTIBLE. */
int mpvss_extract_shares(mpvss_ctx* ctx, size_t n, const uint8_t* private_keys, const uint8_t* witnesses,
                         const uint8_t* enc_shares, uint8_t* publickeys_out, uint8_t* shares_out,
                         uint8_t* challenges_out, uint8_t* responses_out, int* status_out);

/* n independent Participant::verify_share calls (participant.rs:361-386 / 1346-1371 / 1789-1814). */
int mpvss_verify_shares(mpvss_ctx* ctx, size_t n, const uint8_t* publickeys, const uint8_t* shares,
                        const uint8_t* enc_shares, const uint8_t* challenges, const uint8_t* responses, int* ok_out);

/* Participant::reconstruct (participant.rs:462-519 / 1452-1513 / 1895-1950): k decrypted shares at
 * the given 1-based positions and U (element-size big-endian) -> secret (element-size big-endian,
 * left-padded).  gs_out (optional) receives G^s. */
int mpvss_reconstruct(mpvss_ctx* ctx, size_t k, const int64_t* positions, const uint8_t* shares, const uint8_t* u,
                      uint8_t* secret_out, uint8_t* gs_out);
/* n_boxes independent Participant::reconstruct calls in one (e.g. every dealer's secret of one PVSS round).
 * Box b has k[b] decrypted shares.  positions (sum k[b], 1-based) and shares (sum k[b] elements) are
 * concatenated in box order, u holds n_boxes elements (element-size big-endian each, as mpvss_reconstruct takes
 * U).  secrets_out[b] (element size) and gs_out[b] (optional) are what mpvss_reconstruct returns for box b
 * alone, and status_out[b] is its status: MPVSS_ERR_ARG for a position outside [1, 2^31) or, in ModpGroup, a
 * duplicate position; MPVSS_ERR_ENCODING for a share that does not decode or a mask the group rejects.  A box
 * that fails has zero rows in secrets_out / gs_out and leaves the other boxes alone; the call still returns
 * MPVSS_OK and records no error.  Caller errors return MPVSS_ERR_ARG: no boxes, a null pointer other than
 * gs_out, an empty box, or more shares than 32-bit counts hold.  Staged mpvss_verify_distribution_stage state
 * is left untouched.  Not collective: on a context with a communicator it runs on that context's device, as
 * mpvss_reconstruct does. */
int mpvss_reconstruct_secrets(mpvss_ctx* ctx, size_t n_boxes, const size_t* k, const int64_t* positions,
                              const uint8_t* shares, const uint8_t* u, uint8_t* secrets_out, uint8_t* gs_out,
                              int* status_out);

/* ---- multi-GPU --------------------------------------------------------------------- */
/* One context per GPU.  Rank 0 obtains an id (ncclGetUniqueId), the caller distributes its
 * MPVSS_COMM_ID_BYTES bytes to the other ranks by any means, then every rank calls mpvss_comm_init
 * (ncclCommInitRank on the context's device).  Afterwards mpvss_verify_distribution[_stage/_run] and
 * mpvss_distribute on these contexts are collective calls that shard the participants round robin and
 * all-gather the transcript rows over NVLink.  libnccl.so.2 is loaded on first use. */
#define MPVSS_COMM_ID_BYTES 128
int mpvss_comm_unique_id(uint8_t* id_out, size_t id_len);
int mpvss_comm_init(mpvss_ctx* ctx, const uint8_t* id, size_t id_len, int nranks, int rank);
int mpvss_comm_destroy(mpvss_ctx* ctx);
int mpvss_comm_size(const mpvss_ctx* ctx);
int mpvss_comm_rank(const mpvss_ctx* ctx);
/* Host-only half of the sharded transcript, exposed for tests of the gather layout: SHA-256 over the
 * framed rows of n_total participants laid out [rank][ceil(n_total / nranks)][4 frames of 8 + element
 * bytes] as the all-gather delivers them, in participant order (participant i = rank i % nranks, row
 * i / nranks).  Needs no device. */
int mpvss_transcript_digest(int group, const uint8_t* gathered_rows, size_t n_total, int nranks, uint8_t* digest_out);

#ifdef __cplusplus
}
#endif
#endif /* MPVSS_B200_H */
