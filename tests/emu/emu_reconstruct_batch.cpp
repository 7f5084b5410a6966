// CPU execution of the kernel bodies of mpvss_reconstruct_secrets (tests only): the box-aware Lagrange bodies of
// both group families, the MODP segmented product tree (product_tree_level + mul_rows_body) and the elliptic-curve
// segmented sum (exp2 into projective points, then sum_boxes_level + sum_boxes_body until one point per box).
#include <thread>
#include <vector>
#include "../../mpvss_rs_b200/csrc/modp_kernels.cuh"
#include "../../mpvss_rs_b200/csrc/secp.cuh"
#include "../../mpvss_rs_b200/csrc/rist.cuh"
#include "../../mpvss_rs_b200/csrc/ec_kernels.cuh"

namespace {
template <typename F>
void run_warps(uint32_t nwarps, size_t smem_words, F body) {
  for (uint32_t w = 0; w < nwarps; ++w) {
    simt::EmuWarp warp;
    std::vector<uint32_t> smem_raw(smem_words + 4, 0);
    uint32_t* smem = smem_raw.data();
    while (reinterpret_cast<uintptr_t>(smem) & 15) ++smem;
    std::vector<std::thread> lanes;
    for (uint32_t l = 0; l < 32; ++l)
      lanes.emplace_back([&, l] {
        simt::g_lane.warp = &warp;
        simt::g_lane.lane = l;
        simt::g_cf = 0;
        body(w, smem);
      });
    for (auto& t : lanes) t.join();
  }
}

// encoded points x scalars -> projective points (exp2_body), then the segmented sum's levels; out: one encoding per box
template <class Cv>
int sum_boxes(const void* consts, const uint8_t* pts, const uint32_t* scalars, uint32_t n, const uint32_t* start,
              const uint32_t* cnt, uint32_t boxes, uint8_t* out) {
  const typename Cv::Consts* C = (const typename Cv::Consts*)consts;
  using Point = typename Cv::Point;
  std::vector<Point> cur(n);
  std::vector<uint32_t> st(n);
  ec::Exp2Args<Cv> E{C, pts, scalars, nullptr, nullptr, nullptr, cur.data(), st.data(), n, Cv::EB, 8, 0, 0, nullptr};
  for (uint32_t i = 0; i < n; ++i) ec::exp2_body<Cv>(E, i);
  for (uint32_t i = 0; i < n; ++i)
    if (st[i]) return 1;
  std::vector<uint32_t> s(start, start + boxes), c(cnt, cnt + boxes);
  for (bool last = false; !last;) {
    last = true;
    for (uint32_t x : c) last = last && x <= 64;
    std::vector<uint32_t> seg(2 * n + 2 * boxes);
    const uint32_t groups = ec::sum_boxes_level(s.data(), c.data(), boxes, seg.data());
    std::vector<Point> nxt(groups);
    ec::SumBoxesArgs<Cv> S{C, cur.data(), seg.data(), last ? nullptr : nxt.data(), last ? out : nullptr, groups};
    for (uint32_t g = 0; g < groups; ++g) ec::sum_boxes_body<Cv>(S, g);
    cur.swap(nxt);
  }
  return 0;
}
}  // namespace

extern "C" {
// num / den / negative: parts x n rows (part p of position i in row p * n + i)
int emu_modp_lagrange_boxes(const uint32_t* order, const uint32_t* pos, const uint32_t* boff, const uint32_t* bk,
                            uint32_t n, uint32_t* num, uint32_t* den, uint32_t* negative, uint32_t parts) {
  modp::LagrangeBoxesArgs A{order, pos, boff, bk, num, den, negative, n, parts};
  for (uint32_t i = 0; i < 2 * (parts ? parts : 1) * n + 3; ++i) modp::lagrange_boxes_body(A, i);
  return 0;
}
int emu_ec_lagrange_boxes(const void* modN, const uint32_t* pos, const uint32_t* boff, const uint32_t* bk, uint32_t n,
                          uint32_t* out) {
  ec::LagrangeBoxesArgs A{(const fp256::Modulus*)modN, pos, boff, bk, out, n};
  for (uint32_t i = 0; i < n + 3; ++i) ec::lagrange_boxes_body(A, i);
  return 0;
}
// v: rows of 64 limbs; segment s holds cnt[s] rows from start[s]; its product lands in row start[s].  Returns the
// number of levels.
int emu_modp_tree(const uint32_t* consts, uint32_t* v, const uint32_t* start, const uint32_t* cnt, uint32_t segments,
                  uint32_t n) {
  constexpr int T = 8;
  std::vector<uint32_t> c(cnt, cnt + segments), rows(3 * n);
  int levels = 0;
  for (uint32_t m; (m = modp::product_tree_level(start, c.data(), segments, rows.data())) > 0; ++levels) {
    modp::MulRowsArgs A{consts, v, rows.data(), m};
    run_warps((m + 32 / T - 1) / (32 / T), modp::mul_smem_words<T>,
              [&](uint32_t w, uint32_t* s) { modp::mul_rows_body<T>(A, w, s); });
  }
  return levels;
}
int emu_secp_sum_boxes(const void* c, const uint8_t* pts, const uint32_t* e, uint32_t n, const uint32_t* start,
                       const uint32_t* cnt, uint32_t boxes, uint8_t* out) {
  return sum_boxes<secp::SecpCurve>(c, pts, e, n, start, cnt, boxes, out);
}
int emu_rist_sum_boxes(const void* c, const uint8_t* pts, const uint32_t* e, uint32_t n, const uint32_t* start,
                       const uint32_t* cnt, uint32_t boxes, uint8_t* out) {
  return sum_boxes<rist::RistCurve>(c, pts, e, n, start, cnt, boxes, out);
}
}
