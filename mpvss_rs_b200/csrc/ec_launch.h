// Host-side launchers for the elliptic-curve kernels (bodies in ec_kernels.cuh).
#pragma once
#include <cuda_runtime.h>
#include "secp.cuh"
#include "rist.cuh"
#include "ec_kernels.cuh"

// resident 128-thread CTAs per SM of the Horner kernel (its register budget is 65536 / (128 x this))
#ifndef EC_HORNER_MIN_BLOCKS
#define EC_HORNER_MIN_BLOCKS 4
#endif

namespace ec {
constexpr int HORNER_CTAS_PER_SM = EC_HORNER_MIN_BLOCKS;
template <class Cv> cudaError_t launch_exp2(const Exp2Args<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_fixed(const FixedArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_comb_build(const CombArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_decode(const DecodeArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_horner(const HornerArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_horner_boxes(const HornerBoxesArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_sum(const SumArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_sum_boxes(const SumBoxesArgs<Cv>& A, cudaStream_t s);
template <class Cv> cudaError_t launch_add(const AddArgs<Cv>& A, cudaStream_t s);
cudaError_t launch_frames(const FrameArgs& A, cudaStream_t s);
cudaError_t launch_poly(const PolyArgs& A, cudaStream_t s);
cudaError_t launch_lagrange(const LagrangeArgs& A, cudaStream_t s);
cudaError_t launch_lagrange_boxes(const LagrangeBoxesArgs& A, cudaStream_t s);
cudaError_t launch_inv(const InvArgs& A, cudaStream_t s);
cudaError_t launch_proof(const ProofArgs& A, cudaStream_t s);
}  // namespace ec
