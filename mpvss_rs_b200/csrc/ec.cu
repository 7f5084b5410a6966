// __global__ entry points for the elliptic-curve kernels, instantiated for secp256k1 and
// ristretto255 (bodies in ec_kernels.cuh).
#include "ec_launch.h"

namespace ec {

constexpr int TPB = 128;
static inline unsigned blocks(uint32_t n) { return (n + TPB - 1) / TPB; }
#define TID (blockIdx.x * TPB + threadIdx.x)

// stage the generator's fixed-base table into shared memory (whole CTA), 128-bit copies
__device__ __forceinline__ void stage_comb(uint32_t* dst, const uint32_t* src) {
  const uint4* s4 = reinterpret_cast<const uint4*>(src);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
  for (int i = threadIdx.x; i < COMB_WORDS / 4; i += blockDim.x) d4[i] = s4[i];
  __syncthreads();
}
template <class Cv> __global__ void __launch_bounds__(TPB) exp2_kernel(Exp2Args<Cv> A) { exp2_body<Cv>(A, TID); }
template <class Cv> __global__ void __launch_bounds__(TPB) exp2_comb_kernel(Exp2Args<Cv> A) {
  extern __shared__ __align__(16) uint32_t comb_sm[];
  stage_comb(comb_sm, A.comb1);
  exp2_body<Cv>(A, TID, comb_sm);
}
template <class Cv> __global__ void __launch_bounds__(TPB) fixed_kernel(FixedArgs<Cv> A) {
  extern __shared__ __align__(16) uint32_t comb_sm[];
  stage_comb(comb_sm, A.tbl);
  fixed_body<Cv>(A, TID, comb_sm);
}
template <class Cv> __global__ void __launch_bounds__(TPB) comb_build_kernel(CombArgs<Cv> A) { comb_build_body<Cv>(A, TID); }
template <class Cv> __global__ void __launch_bounds__(TPB) decode_kernel(DecodeArgs<Cv> A) { decode_body<Cv>(A, TID); }
template <class Cv> __global__ void __launch_bounds__(TPB, EC_HORNER_MIN_BLOCKS) horner_kernel(HornerArgs<Cv> A) { horner_body<Cv>(A, TID); }
template <class Cv> __global__ void __launch_bounds__(TPB, EC_HORNER_MIN_BLOCKS) horner_boxes_kernel(HornerBoxesArgs<Cv> A) {
  horner_boxes_body<Cv>(A, TID);
}
template <class Cv> __global__ void __launch_bounds__(TPB) sum_kernel(SumArgs<Cv> A) { sum_body<Cv>(A, TID); }
template <class Cv> __global__ void __launch_bounds__(TPB) sum_boxes_kernel(SumBoxesArgs<Cv> A) { sum_boxes_body<Cv>(A, TID); }
template <class Cv> __global__ void __launch_bounds__(TPB) add_kernel(AddArgs<Cv> A) { add_body<Cv>(A, TID); }
__global__ void __launch_bounds__(TPB) frame_kernel(FrameArgs A) { frame_body(A, TID); }
__global__ void __launch_bounds__(TPB) poly_kernel(PolyArgs A) { poly_body(A, TID); }
__global__ void __launch_bounds__(TPB) poly_boxes_kernel(PolyBoxesArgs A) { poly_boxes_body(A, TID); }
__global__ void __launch_bounds__(TPB) lagrange_boxes_kernel(LagrangeBoxesArgs A) { lagrange_boxes_body(A, TID); }
__global__ void __launch_bounds__(TPB) inv_kernel(InvArgs A) { inv_body(A, TID); }
__global__ void __launch_bounds__(TPB) proof_kernel(ProofArgs A) { proof_body(A, TID); }

template <class Cv> cudaError_t launch_exp2(const Exp2Args<Cv>& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  if (A.comb1) {
    cudaError_t e = cudaFuncSetAttribute(exp2_comb_kernel<Cv>, cudaFuncAttributeMaxDynamicSharedMemorySize, COMB_WORDS * 4);
    if (e != cudaSuccess) return e;
    exp2_comb_kernel<Cv><<<blocks(A.n), TPB, COMB_WORDS * 4, s>>>(A);
  } else {
    exp2_kernel<Cv><<<blocks(A.n), TPB, 0, s>>>(A);
  }
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_fixed(const FixedArgs<Cv>& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(fixed_kernel<Cv>, cudaFuncAttributeMaxDynamicSharedMemorySize, COMB_WORDS * 4);
  if (e != cudaSuccess) return e;
  fixed_kernel<Cv><<<blocks(A.n), TPB, COMB_WORDS * 4, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_comb_build(const CombArgs<Cv>& A, cudaStream_t s) {
  comb_build_kernel<Cv><<<blocks(COMB_ENTRIES), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_decode(const DecodeArgs<Cv>& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  decode_kernel<Cv><<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_horner(const HornerArgs<Cv>& A, cudaStream_t s) {
  if (A.n == 0 || A.K == 0 || A.t == 0) return cudaErrorInvalidValue;
  horner_kernel<Cv><<<blocks(A.n * A.K), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_horner_boxes(const HornerBoxesArgs<Cv>& A, cudaStream_t s) {
  if (A.n == 0 || A.K == 0) return cudaErrorInvalidValue;
  horner_boxes_kernel<Cv><<<blocks(A.n * A.K), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_sum(const SumArgs<Cv>& A, cudaStream_t s) {
  if (A.groups == 0) return cudaErrorInvalidValue;
  sum_kernel<Cv><<<blocks(A.groups), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_sum_boxes(const SumBoxesArgs<Cv>& A, cudaStream_t s) {
  if (A.groups == 0) return cudaErrorInvalidValue;
  sum_boxes_kernel<Cv><<<blocks(A.groups), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
template <class Cv> cudaError_t launch_add(const AddArgs<Cv>& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  add_kernel<Cv><<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
cudaError_t launch_frames(const FrameArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  frame_kernel<<<blocks(A.n * 4), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
cudaError_t launch_poly(const PolyArgs& A, cudaStream_t s) {
  if (A.n == 0 || A.t == 0) return cudaErrorInvalidValue;
  poly_kernel<<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
cudaError_t launch_poly_boxes(const PolyBoxesArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  poly_boxes_kernel<<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
cudaError_t launch_lagrange_boxes(const LagrangeBoxesArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  lagrange_boxes_kernel<<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}
cudaError_t launch_inv(const InvArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  inv_kernel<<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}

cudaError_t launch_proof(const ProofArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  proof_kernel<<<blocks(A.n), TPB, 0, s>>>(A);
  return cudaGetLastError();
}

#define INSTANTIATE(Cv)                                                                  \
  template cudaError_t launch_exp2<Cv>(const Exp2Args<Cv>&, cudaStream_t);               \
  template cudaError_t launch_fixed<Cv>(const FixedArgs<Cv>&, cudaStream_t);             \
  template cudaError_t launch_comb_build<Cv>(const CombArgs<Cv>&, cudaStream_t);         \
  template cudaError_t launch_decode<Cv>(const DecodeArgs<Cv>&, cudaStream_t);           \
  template cudaError_t launch_horner<Cv>(const HornerArgs<Cv>&, cudaStream_t);           \
  template cudaError_t launch_horner_boxes<Cv>(const HornerBoxesArgs<Cv>&, cudaStream_t); \
  template cudaError_t launch_sum<Cv>(const SumArgs<Cv>&, cudaStream_t);                 \
  template cudaError_t launch_sum_boxes<Cv>(const SumBoxesArgs<Cv>&, cudaStream_t);      \
  template cudaError_t launch_add<Cv>(const AddArgs<Cv>&, cudaStream_t);
INSTANTIATE(secp::SecpCurve)
INSTANTIATE(rist::RistCurve)

}  // namespace ec
