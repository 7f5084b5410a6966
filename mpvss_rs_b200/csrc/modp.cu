// __global__ entry points for the ModpGroup kernels (bodies in modp_kernels.cuh).
#include <cuda_runtime.h>
#include "modp_kernels.cuh"
#include "modp_launch.h"

namespace modp {


template <int TPI, bool NP1, bool CHUNKED>
__global__ void __launch_bounds__(HORNER_MAX_WARPS_PER_CTA * 32) horner_kernel(HornerArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t w = threadIdx.x >> 5;
  horner_body<TPI, NP1, CHUNKED>(A, blockIdx.x * (blockDim.x >> 5) + w, smem + w * horner_smem_words<TPI>,
                                 A.nops ? A.nops[blockIdx.x] : A.nops_all, blockIdx.x);
}

template <int TPI>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) exp2_kernel(Exp2Args A) {
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t w = threadIdx.x >> 5;
  exp2_body<TPI>(A, blockIdx.x * WARPS_PER_CTA + w, smem + w * exp2_smem_words<TPI>);
}

// Persistent one-warp CTAs, one per SM: the launch only takes the warp slot the Horner launch leaves
// empty on every SM (7 one-warp CTAs on 4 schedulers).  Used for the X-independent a2 exponentiation
// (modp_overlap = 3).
template <int TPI>
__global__ void __launch_bounds__(32) exp2_filler_kernel(Exp2Args A, uint32_t nwarps) {
  extern __shared__ __align__(16) uint32_t smem[];
  for (uint32_t w = blockIdx.x; w < nwarps; w += gridDim.x) {
    exp2_body<TPI>(A, w, smem);
    __syncwarp();
  }
}

template <int TPI>
__global__ void __launch_bounds__(32) comb1_kernel(CombArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  comb1_body<TPI>(A, blockIdx.x, smem);
}
template <int TPI>
__global__ void __launch_bounds__(32) comb2_kernel(CombArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  comb2_body<TPI>(A, blockIdx.x, smem);
}

template <int TPI>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) mul_kernel(MulArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t w = threadIdx.x >> 5;
  mul_body<TPI>(A, blockIdx.x * WARPS_PER_CTA + w, smem + w * mul_smem_words<TPI>);
}

__global__ void __launch_bounds__(128) frame_kernel(FrameArgs A) { frame_body(A, blockIdx.x * 128 + threadIdx.x); }
__global__ void __launch_bounds__(64) resp_kernel(RespArgs A) { resp_body(A, blockIdx.x * 64 + threadIdx.x); }
__global__ void __launch_bounds__(64) poly_kernel(PolyArgs A) { poly_body(A, blockIdx.x * 64 + threadIdx.x); }
__global__ void __launch_bounds__(64) poly_boxes_kernel(PolyBoxesArgs A) { poly_boxes_body(A, blockIdx.x * 64 + threadIdx.x); }
__global__ void __launch_bounds__(64) lagrange_boxes_kernel(LagrangeBoxesArgs A) {
  lagrange_boxes_body(A, blockIdx.x * 64 + threadIdx.x);
}

template <int TPI>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) mul_rows_kernel(MulRowsArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t w = threadIdx.x >> 5;
  mul_rows_body<TPI>(A, blockIdx.x * WARPS_PER_CTA + w, smem + w * mul_smem_words<TPI>);
}

// Counting sort of the exponent bytes for the bucket method: CTA w orders the indices 0..k-1 by byte w of
// their exponent (idx, window-major) and writes the 257 bucket boundaries (start).  The order inside a
// bucket depends on the atomics and does not matter: a bucket is a product.
__global__ void __launch_bounds__(256) msm_sort_kernel(const uint8_t* scalars, uint32_t k, uint32_t* idx, uint32_t* start) {
  __shared__ uint32_t cnt[257], cur[256];
  const uint32_t w = blockIdx.x;
  for (uint32_t d = threadIdx.x; d < 257; d += blockDim.x) cnt[d] = 0;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < k; i += blockDim.x) atomicAdd(&cnt[scalars[(size_t)i * 256 + w] + 1u], 1u);
  __syncthreads();
  if (threadIdx.x == 0)
    for (int d = 0; d < 256; ++d) cnt[d + 1] += cnt[d];
  __syncthreads();
  for (uint32_t d = threadIdx.x; d < 257; d += blockDim.x) {
    start[w * 257u + d] = cnt[d];
    if (d < 256) cur[d] = cnt[d];
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < k; i += blockDim.x)
    idx[(size_t)w * k + atomicAdd(&cur[scalars[(size_t)i * 256 + w]], 1u)] = i;
}

template <int TPI>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) msm_bucket_kernel(MsmBucketArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t w = threadIdx.x >> 5;
  msm_bucket_body<TPI>(A, blockIdx.x * WARPS_PER_CTA + w, smem + w * msm_smem_words<TPI>);
}
template <int TPI>
__global__ void __launch_bounds__(32) msm_window_kernel(MsmWindowArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  msm_window_body<TPI>(A, blockIdx.x, smem);
}
template <int TPI>
__global__ void __launch_bounds__(32) msm_fold_kernel(MsmFoldArgs A) {
  extern __shared__ __align__(16) uint32_t smem[];
  msm_fold_body<TPI>(A, smem);
}

template <int TPI>
static uint32_t ctas_for(uint32_t n) {
  uint32_t per_cta = WARPS_PER_CTA * (32 / TPI);
  return (n + per_cta - 1) / per_cta;
}

template <typename K>
static cudaError_t set_smem(K kernel, size_t bytes) {
  // Largest shared-memory carve-out for every MODP kernel: the kernels barely use L1, and the split of
  // an SM cannot change while CTAs are resident, so a small carve-out chosen for the first launch would
  // keep a second, concurrent launch (modp_overlap) from becoming resident at all.
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

#define MODP_DISPATCH(tpi, ...)                            \
  switch (tpi) {                                           \
    case 4: { constexpr int T = 4; __VA_ARGS__; break; }   \
    case 8: { constexpr int T = 8; __VA_ARGS__; break; }   \
    case 16: { constexpr int T = 16; __VA_ARGS__; break; } \
    default: return cudaErrorInvalidValue;                 \
  }

template <int TPI, bool NP1, bool CHUNKED>
static cudaError_t horner_go(const HornerArgs& A, uint32_t grid, uint32_t wpc, size_t sm, cudaStream_t s) {
  cudaError_t e = set_smem(horner_kernel<TPI, NP1, CHUNKED>, sm);
  if (e != cudaSuccess) return e;
  horner_kernel<TPI, NP1, CHUNKED><<<grid, wpc * 32, sm, s>>>(A);
  return cudaSuccess;
}
cudaError_t launch_horner(int tpi, const HornerArgs& A, bool np_is_one, cudaStream_t s) {
  if (A.n == 0 || A.t == 0 || A.warps_per_cta > (uint32_t)HORNER_MAX_WARPS_PER_CTA) return cudaErrorInvalidValue;
  MODP_DISPATCH(tpi, {
    const uint32_t wpc = A.warps_per_cta ? A.warps_per_cta : 1u;
    size_t sm = wpc * horner_smem_words<T> * 4;
    uint32_t per_cta = wpc * (32 / T);
    uint32_t grid = (A.n + per_cta - 1) / per_cta;
    const bool chunked = A.cfirst && A.csteps;
    cudaError_t e = np_is_one ? (chunked ? horner_go<T, true, true>(A, grid, wpc, sm, s) : horner_go<T, true, false>(A, grid, wpc, sm, s))
                              : (chunked ? horner_go<T, false, true>(A, grid, wpc, sm, s) : horner_go<T, false, false>(A, grid, wpc, sm, s));
    if (e != cudaSuccess) return e;
  });
  return cudaGetLastError();
}

cudaError_t launch_exp2(int tpi, const Exp2Args& A, cudaStream_t s) {
  if (A.n == 0 || A.e1_windows == 0 || (A.b2 && A.e2_windows == 0)) return cudaErrorInvalidValue;
  MODP_DISPATCH(tpi, {
    size_t sm = WARPS_PER_CTA * exp2_smem_words<T> * 4;
    cudaError_t e = set_smem(exp2_kernel<T>, sm);
    if (e != cudaSuccess) return e;
    exp2_kernel<T><<<ctas_for<T>(A.n), WARPS_PER_CTA * 32, sm, s>>>(A);
  });
  return cudaGetLastError();
}

cudaError_t launch_exp2_filler(int tpi, const Exp2Args& A, size_t ctas, cudaStream_t s) {
  if (A.n == 0 || A.e1_windows == 0 || (A.b2 && A.e2_windows == 0)) return cudaErrorInvalidValue;
  MODP_DISPATCH(tpi, {
    size_t sm = exp2_smem_words<T> * 4;
    cudaError_t e = set_smem(exp2_filler_kernel<T>, sm);
    if (e != cudaSuccess) return e;
    uint32_t per_cta = 32 / T, nwarps = (A.n + per_cta - 1) / per_cta;
    uint32_t grid = (uint32_t)ctas;  // number of persistent CTAs (one per SM)
    exp2_filler_kernel<T><<<grid < nwarps ? grid : nwarps, 32, sm, s>>>(A, nwarps);
  });
  return cudaGetLastError();
}

cudaError_t launch_frames(const FrameArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  frame_kernel<<<(A.n * 4 + 127) / 128, 128, 0, s>>>(A);
  return cudaGetLastError();
}

cudaError_t launch_resp(const RespArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  resp_kernel<<<(A.n + 63) / 64, 64, 0, s>>>(A);
  return cudaGetLastError();
}

cudaError_t launch_poly(const PolyArgs& A, cudaStream_t s) {
  if (A.n == 0 || A.t == 0) return cudaErrorInvalidValue;
  poly_kernel<<<(A.n + 63) / 64, 64, 0, s>>>(A);
  return cudaGetLastError();
}

cudaError_t launch_poly_boxes(const PolyBoxesArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  poly_boxes_kernel<<<(A.n + 63) / 64, 64, 0, s>>>(A);
  return cudaGetLastError();
}

cudaError_t launch_lagrange_boxes(const LagrangeBoxesArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  const uint32_t threads = 2u * (A.parts ? A.parts : 1u) * A.n;
  lagrange_boxes_kernel<<<(threads + 63) / 64, 64, 0, s>>>(A);
  return cudaGetLastError();
}

cudaError_t launch_comb_build(int tpi, const CombArgs& A, cudaStream_t s) {
  MODP_DISPATCH(tpi, {
    size_t sm = comb_smem_words<T> * 4;
    comb1_kernel<T><<<1, 32, sm, s>>>(A);
    comb2_kernel<T><<<(A.rows + 32 / T - 1) / (32 / T), 32, sm, s>>>(A);
  });
  return cudaGetLastError();
}

// bucket multi-exponentiation: buckets, per-window products, final fold (8 lanes per value)
cudaError_t launch_msm(const MsmBucketArgs& B, const uint32_t* scalars, uint32_t* idx, uint32_t* start,
                       uint32_t* wprod, uint32_t* out, cudaStream_t s) {
  if (B.windows == 0 || B.windows > 256 || B.k == 0) return cudaErrorInvalidValue;
  constexpr int T = 8;
  msm_sort_kernel<<<B.windows, 256, 0, s>>>(reinterpret_cast<const uint8_t*>(scalars), B.k, idx, start);
  const uint32_t groups = B.windows * 255u, per_cta = WARPS_PER_CTA * (32 / T);
  size_t sm = WARPS_PER_CTA * msm_smem_words<T> * 4;
  msm_bucket_kernel<T><<<(groups + per_cta - 1) / per_cta, WARPS_PER_CTA * 32, sm, s>>>(B);
  MsmWindowArgs W{B.consts, B.buckets, wprod, B.windows};
  msm_window_kernel<T><<<B.windows, 32, msm_window_smem_words<T> * 4, s>>>(W);
  MsmFoldArgs F{B.consts, wprod, out, B.windows};
  msm_fold_kernel<T><<<1, 32, msm_smem_words<T> * 4, s>>>(F);
  return cudaGetLastError();
}

cudaError_t launch_mul(int tpi, const MulArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  MODP_DISPATCH(tpi, {
    size_t sm = WARPS_PER_CTA * mul_smem_words<T> * 4;
    cudaError_t e = set_smem(mul_kernel<T>, sm);
    if (e != cudaSuccess) return e;
    mul_kernel<T><<<ctas_for<T>(A.n), WARPS_PER_CTA * 32, sm, s>>>(A);
  });
  return cudaGetLastError();
}

cudaError_t launch_mul_rows(int tpi, const MulRowsArgs& A, cudaStream_t s) {
  if (A.n == 0) return cudaErrorInvalidValue;
  MODP_DISPATCH(tpi, {
    size_t sm = WARPS_PER_CTA * mul_smem_words<T> * 4;
    cudaError_t e = set_smem(mul_rows_kernel<T>, sm);
    if (e != cudaSuccess) return e;
    mul_rows_kernel<T><<<ctas_for<T>(A.n), WARPS_PER_CTA * 32, sm, s>>>(A);
  });
  return cudaGetLastError();
}

}  // namespace modp
