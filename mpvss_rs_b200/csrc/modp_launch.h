// Host-side launchers for the ModpGroup kernels.
#pragma once
#include <cuda_runtime.h>
#include "modp_kernels.cuh"

namespace modp {
constexpr int WARPS_PER_CTA = 4;     // exponentiation / multiplication kernels
// Horner launches use one warp per CTA (fine-grained op-count classes; the block scheduler then leaves one warp
// slot per SM free for the a2 filler at n = 4096); up to 4 warps per CTA through the "modp_wpc" tunable, which
// measured no different at 8 .. 16 warps per SM.
constexpr int HORNER_MAX_WARPS_PER_CTA = 4;
cudaError_t launch_horner(int tpi, const HornerArgs& A, bool np_is_one, cudaStream_t s);
cudaError_t launch_exp2(int tpi, const Exp2Args& A, cudaStream_t s);
cudaError_t launch_exp2_filler(int tpi, const Exp2Args& A, size_t ctas, cudaStream_t s);
cudaError_t launch_frames(const FrameArgs& A, cudaStream_t s);
cudaError_t launch_resp(const RespArgs& A, cudaStream_t s);
cudaError_t launch_comb_build(int tpi, const CombArgs& A, cudaStream_t s);
cudaError_t launch_poly(const PolyArgs& A, cudaStream_t s);
cudaError_t launch_poly_boxes(const PolyBoxesArgs& A, cudaStream_t s);
cudaError_t launch_lagrange_boxes(const LagrangeBoxesArgs& A, cudaStream_t s);
cudaError_t launch_mul(int tpi, const MulArgs& A, cudaStream_t s);
cudaError_t launch_mul_rows(int tpi, const MulRowsArgs& A, cudaStream_t s);
cudaError_t launch_msm(const MsmBucketArgs& B, const uint32_t* scalars, uint32_t* idx, uint32_t* start, uint32_t* wprod,
                       uint32_t* out, cudaStream_t s);
}  // namespace modp
