// Translation unit of the exact integer extrusion: kernels (extrude_i8.cuh), launch geometry, operator slicing.
#define OZ_DEFINE_KERNELS
#include <math.h>
#include <string.h>
#include "dispatch.h"
#include "extrude_i8_host.h"

static cudaError_t oz_attrs() {
  static bool attr_set = false;
  if (attr_set) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(oz_gemm_kernel<0, OZ_LEVELS>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_kernel<1, OZ_LEVELS_PRODUCT>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_kernel<2, OZ_LEVELS_PRODUCT>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(oz_gemm_kernel<3, OZ_LEVELS_PRODUCT>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES);
  attr_set = e == cudaSuccess;
  return e;
}

cudaError_t oz_extrude_launch(const OzGatherParams& g, const OzGemmParams& m, int MT, int NT, cudaStream_t st) {
  cudaError_t e = oz_attrs();
  if (e != cudaSuccess) return e;
  with<false, true>(g.steps != nullptr, [&](auto PE) { oz_gather_slice_kernel<PE><<<g.E, 256, (size_t)g.KB * OZ_BK * sizeof(double), st>>>(g); });
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  oz_gemm_kernel<0, OZ_LEVELS><<<dim3(NT, MT), OZ_THREADS, OZ_SMEM_BYTES, st>>>(m);
  return cudaGetLastError();
}

cudaError_t oz_product_launch(const OzSliceParams& sl, const OzGemmParams& m, int integrator, int MT, int NT, cudaStream_t st) {
  cudaError_t e = oz_attrs();
  if (e != cudaSuccess) return e;
  oz_slice_rows_kernel<<<sl.E, 256, 0, st>>>(sl);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  with<1, 2, 3>(!integrator ? 1 : m.gain_env ? 3 : 2, [&](auto EPI) {
    oz_gemm_kernel<EPI, OZ_LEVELS_PRODUCT><<<dim3(NT, MT), OZ_THREADS, OZ_SMEM_BYTES, st>>>(m);
  });
  return cudaGetLastError();
}

void oz_slice_operator(const float* AB, int rows, int ld, int K, int KB, int NT, uint8_t* planes, int* ea) {
  for (int n = 0; n < NT * OZ_BN; ++n) {
    ea[n] = 0;
    if (n >= rows) continue;
    const float* row = AB + (size_t)n * ld;
    double amax = 0.0;
    for (int k = 0; k < K; ++k) amax = fmax(amax, fabs((double)row[k]));
    const int ex = oz_exponent(amax);
    ea[n] = ex;
    const double scale = ldexp(1.0, -ex);
    const int nt = n / OZ_BN, r = n % OZ_BN;
    for (int k = 0; k < K; ++k) {
      int q[OZ_SLICES_B];
      oz_digits<OZ_SLICES_B>((double)row[k], scale, q);
      const int kb = k / OZ_BK, kk = k % OZ_BK;
      for (int s = 0; s < OZ_SLICES_B; ++s)
        planes[((size_t)(nt * KB + kb) * OZ_SLICES_B + s) * OZ_B_TILE + oz_tile_offset(r, kk)] = (uint8_t)(int8_t)q[s];
    }
  }
}
