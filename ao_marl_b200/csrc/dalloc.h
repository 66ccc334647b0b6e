// Zeroed device allocation of the host side.
#pragma once
#include <cuda_runtime.h>

template <typename T>
static cudaError_t dalloc(T** p, size_t count) {
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e == cudaSuccess) e = cudaMemset(*p, 0, count * sizeof(T));
  // the fill runs on the legacy stream, the buffer may be used next on a non-blocking one: finish it here
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  return e;
}
