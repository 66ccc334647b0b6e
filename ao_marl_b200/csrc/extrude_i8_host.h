// Host interface of the exact integer extrusion (extrude_i8.cuh), compiled in its own translation unit.
#pragma once
#include <cuda_runtime.h>
#include "extrude_i8.cuh"

// gather + digit planes of all environments, then the digit-pair GEMM (grid NT x MT); both asynchronous on `st`
cudaError_t oz_extrude_launch(const OzGatherParams& g, const OzGemmParams& m, int MT, int NT, cudaStream_t st);

// out = X . OP^T for a per-environment float32 matrix X and an operator given as digit planes (integrator != 0: the
// least-squares integrator epilogue, with one gain per environment when m.gain_env is set): row digits of X, then the
// digit-pair GEMM; both asynchronous on `st`
cudaError_t oz_product_launch(const OzSliceParams& sl, const OzGemmParams& m, int integrator, int MT, int NT, cudaStream_t st);

