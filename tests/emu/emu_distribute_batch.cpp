// CPU execution of the kernel bodies of mpvss_distribute_secrets (tests only): the multi-box polynomial bodies of
// both group families, and the MODP response body with one challenge per instance.
#include "../../mpvss_rs_b200/csrc/modp_kernels.cuh"
#include "../../mpvss_rs_b200/csrc/secp.cuh"
#include "../../mpvss_rs_b200/csrc/rist.cuh"
#include "../../mpvss_rs_b200/csrc/ec_kernels.cuh"

extern "C" {
// idx: n positions, then per instance its box's first coefficient row, t_b and first instance row
int emu_modp_poly_boxes(const uint32_t* coeffs, const uint32_t* order, const uint32_t* idx, uint32_t n, uint32_t* out) {
  modp::PolyBoxesArgs A{coeffs, order, idx, idx + n, idx + 2 * n, idx + 3 * n, out, n};
  for (uint32_t i = 0; i < n + 3; ++i) modp::poly_boxes_body(A, i);
  return 0;
}
int emu_ec_poly_boxes(const void* modN, const uint32_t* coeffs, const uint32_t* idx, uint32_t n, uint32_t* out) {
  ec::PolyBoxesArgs A{(const fp256::Modulus*)modN, coeffs, idx, idx + n, idx + 2 * n, idx + 3 * n, out, n};
  for (uint32_t i = 0; i < n + 3; ++i) ec::poly_boxes_body(A, i);
  return 0;
}
// r_i = (w_i - alpha_i * c_i) mod order, challenge i at c + i * c_stride (64-limb rows)
int emu_modp_resp(const uint32_t* order, const uint32_t* alpha, const uint32_t* w, const uint32_t* c, uint32_t c_stride,
                  uint32_t n, uint32_t* out) {
  modp::RespArgs A{order, alpha, w, c, out, n, 64, c_stride};
  for (uint32_t i = 0; i < n + 3; ++i) modp::resp_body(A, i);
  return 0;
}
}
