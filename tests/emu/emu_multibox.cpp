// CPU execution of the multi-box elliptic-curve Horner body (tests only): the commitments of several boxes
// are decoded in one pass, horner_boxes_body evaluates K chunks of every position against its own box, and
// the chunk sum adds them up -- the launch sequence of mpvss_verify_distributions, one thread at a time.
#include "../../mpvss_rs_b200/csrc/secp.cuh"
#include "../../mpvss_rs_b200/csrc/rist.cuh"
#include "../../mpvss_rs_b200/csrc/ec_kernels.cuh"
#include <vector>

namespace {
// commitments: sum t elements; pos / coff / ct: n entries (position, its box's first commitment, its box's t)
template <class Cv>
int t_boxes(const void* consts, const uint8_t* commitments, uint32_t t_all, const uint32_t* pos, const uint32_t* coff,
            const uint32_t* ct, uint32_t n, uint32_t K, uint8_t* out) {
  const typename Cv::Consts* C = (const typename Cv::Consts*)consts;
  std::vector<uint32_t> cxy((size_t)t_all * 16), cst(t_all);
  ec::DecodeArgs<Cv> D{C, commitments, cxy.data(), cst.data(), t_all};
  for (uint32_t i = 0; i < t_all; ++i) ec::decode_body<Cv>(D, i);
  for (uint32_t i = 0; i < t_all; ++i)
    if (cst[i] == 1) return 1;
  std::vector<typename Cv::Point> part((size_t)K * n);
  ec::HornerBoxesArgs<Cv> H{C, cxy.data(), cst.data(), pos, coff, ct, part.data(), n, K};
  for (uint32_t i = 0; i < K * n; ++i) ec::horner_boxes_body<Cv>(H, i);
  ec::SumArgs<Cv> S{C, part.data(), nullptr, out, n, K, 1, n, K * n};
  for (uint32_t i = 0; i < n; ++i) ec::sum_body<Cv>(S, i);
  return 0;
}
}  // namespace

extern "C" {
int emu_secp_horner_boxes(const void* c, const uint8_t* cm, uint32_t t_all, const uint32_t* pos, const uint32_t* coff,
                          const uint32_t* ct, uint32_t n, uint32_t K, uint8_t* out) {
  return t_boxes<secp::SecpCurve>(c, cm, t_all, pos, coff, ct, n, K, out);
}
int emu_rist_horner_boxes(const void* c, const uint8_t* cm, uint32_t t_all, const uint32_t* pos, const uint32_t* coff,
                          const uint32_t* ct, uint32_t n, uint32_t K, uint8_t* out) {
  return t_boxes<rist::RistCurve>(c, cm, t_all, pos, coff, ct, n, K, out);
}
}
