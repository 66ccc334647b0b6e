// Device helpers shared by the round-1 sensor kernels (wfs_mma.cuh, wfs_tma.cuh) and the pupil sweep (pupil_sweep.cuh):
// shared-memory addresses, the bounded mbarrier wait, and sin / cos with a float32 argument reduction.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define WFT_WAIT_SPINS (1u << 22)

__device__ __forceinline__ uint32_t wft_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ bool wft_mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  for (uint32_t it = 0; it < WFT_WAIT_SPINS; ++it) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return true;
  }
  // an expired wait would let the warp read a stage that was never filled: raise the error word and stop the kernel
  atomicExch(err, 2);
  __threadfence_system();
  __trap();
  return false;
}

// sin / cos of a float32 argument of any magnitude met here (|x| < ~1e4): three-term Cody-Waite
// reduction by 2 pi, then the SFU approximations on [-pi, pi] (absolute error < 5e-7)
__device__ __forceinline__ void wfm_sincos(float x, float& s, float& c) {
  const float n = rintf(x * 0.15915494309189535f);
  float r = fmaf(n, -6.28125f, x);                    // 2 pi = 6.28125 + 1.9350051879882812e-3 + 3.0199159819995e-7
  r = fmaf(n, -1.9350051879882812e-3f, r);
  r = fmaf(n, -3.0199159819995e-7f, r);
  s = __sinf(r);
  c = __cosf(r);
}
