// Host plumbing shared by the group implementations (modp_api.cu, ec_api.cu): copies, argument checks,
// constant parsing, rank slices and the position / box layout the kernels read.
#pragma once
#include "ctx.h"

inline int h2d(mpvss_ctx* ctx, DevBuf& b, const void* src, size_t bytes) {
  MPVSS_CUDA(ctx, b.ensure(bytes));
  MPVSS_CUDA(ctx, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return MPVSS_OK;
}
inline int d2h(mpvss_ctx* ctx, void* dst, const DevBuf& b, size_t bytes) {
  MPVSS_CUDA(ctx, cudaMemcpyAsync(dst, b.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return MPVSS_OK;
}
inline int sync(mpvss_ctx* ctx) {
  MPVSS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPVSS_OK;
}

inline int check_args(mpvss_ctx* ctx, bool ok, const char* what) {
  return ok ? MPVSS_OK : mpvss_fail(ctx, MPVSS_ERR_ARG, what);
}

inline big::Int from_hex(const char* s) {
  size_t n = strlen(s);
  std::vector<uint8_t> be((n + 1) / 2, 0);
  for (size_t i = 0; i < n; ++i) {
    char c = s[n - 1 - i];
    uint8_t v = c <= '9' ? c - '0' : (c | 32) - 'a' + 10;
    be[be.size() - 1 - i / 2] |= v << (4 * (i % 2));
  }
  return big::from_be(be.data(), be.size());
}

// rows `rank, rank + nranks, ...` of a host array of n_total rows (the whole array without a communicator)
inline const uint8_t* slice_rows(const mpvss_ctx* ctx, const uint8_t* all, size_t n_total, size_t width,
                                 std::vector<uint8_t>& tmp) {
  if (ctx->nranks <= 1) return all;
  tmp.clear();
  for (size_t i = (size_t)ctx->rank; i < n_total; i += (size_t)ctx->nranks)
    tmp.insert(tmp.end(), all + i * width, all + (i + 1) * width);
  return tmp.data();
}

// Positions as the kernels take them, 32-bit (positions == nullptr: 1..n).  Returns n, or the index of the first
// position outside [1, 2^31); the caller decides what that position means for its status.
inline size_t positions_u32(const int64_t* positions, size_t n, std::vector<uint32_t>& out) {
  out.resize(n);
  for (size_t i = 0; i < n; ++i) {
    const int64_t p = positions ? positions[i] : (int64_t)i + 1;
    if (p < 1 || p > 0x7fffffff) return i;
    out[i] = (uint32_t)p;
  }
  return n;
}

// The live boxes of a reconstruct batch packed in the order of `live`: box live[j] takes rows
// [start[j], start[j] + cnt[j]) of the n rows.  idx holds the positions, then per row its box's first row, then
// its box's share count (the box-aware Lagrange kernels' layout).  rows(shares) are the rows' shares, eb bytes
// each: the caller's array itself when every box is live in its own order (always so for a single box).
struct LiveBoxes {
  size_t n = 0;
  std::vector<uint32_t> start, cnt, idx;
  std::vector<uint8_t> packed;  // the rows' shares when they are not the caller's array as it stands
  const uint8_t* rows(const uint8_t* shares) const { return packed.empty() ? shares : packed.data(); }
};
inline LiveBoxes pack_live_boxes(size_t nb, const size_t* kv, const int64_t* positions, const uint8_t* shares,
                                 size_t eb, const std::vector<size_t>& live) {
  std::vector<size_t> first(nb, 0);  // each box's first share in the caller's arrays
  for (size_t b = 1; b < nb; ++b) first[b] = first[b - 1] + kv[b - 1];
  LiveBoxes P;
  const size_t L = live.size();
  P.start.resize(L);
  P.cnt.resize(L);
  for (size_t j = 0; j < L; ++j) {
    P.start[j] = (uint32_t)P.n;
    P.cnt[j] = (uint32_t)kv[live[j]];
    P.n += P.cnt[j];
  }
  const size_t n = P.n;
  P.idx.resize(3 * n);
  bool in_place = L == nb;
  for (size_t j = 0; j < L && in_place; ++j) in_place = live[j] == j;
  if (!in_place) P.packed.resize(n * eb);
  for (size_t j = 0; j < L; ++j) {
    const size_t b = live[j];
    for (uint32_t i = 0; i < P.cnt[j]; ++i) {
      P.idx[P.start[j] + i] = (uint32_t)positions[first[b] + i];
      P.idx[n + P.start[j] + i] = P.start[j];
      P.idx[2 * n + P.start[j] + i] = P.cnt[j];
    }
    if (!in_place) memcpy(P.packed.data() + (size_t)P.start[j] * eb, shares + first[b] * eb, P.cnt[j] * eb);
  }
  return P;
}
