// Translation unit of the exact integer extrusion: kernels (extrude_i8.cuh), launch geometry, operator slicing.
#define OZ_DEFINE_KERNELS
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../../include/aomarl.h"
#include "dalloc.h"
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

int oz_operator_upload(OzOperator& op, const float* host, int rows, int ld, int K, char (&err)[512]) {
  if (!oz_operator_finite(host, rows, ld, K)) {
    snprintf(err, sizeof(err), "operator table holds a NaN or an infinity");
    return AOM_ERR_INVALID;
  }
  const int KB = (K + OZ_BK - 1) / OZ_BK, NT = (rows + OZ_BN - 1) / OZ_BN;
  const size_t bytes = (size_t)NT * KB * OZ_SLICES_B * OZ_B_TILE;
  uint8_t* planes = (uint8_t*)calloc(bytes, 1);
  int* ea = (int*)calloc((size_t)NT * OZ_BN, sizeof(int));
  if (!planes || !ea) {
    free(planes); free(ea);
    snprintf(err, sizeof(err), "out of host memory");
    return AOM_ERR_INVALID;
  }
  oz_slice_operator(host, rows, ld, K, KB, NT, planes, ea);
  oz_operator_free(op);
  cudaError_t e = cudaMalloc((void**)&op.planes, bytes);
  if (e == cudaSuccess) e = cudaMalloc((void**)&op.ea, (size_t)NT * OZ_BN * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(op.planes, planes, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(op.ea, ea, (size_t)NT * OZ_BN * sizeof(int), cudaMemcpyHostToDevice);
  free(planes); free(ea);
  if (e != cudaSuccess) {
    snprintf(err, sizeof(err), "operator digit planes: %s", cudaGetErrorString(e));
    return AOM_ERR_CUDA;
  }
  op.kb = KB; op.nt = NT;
  return AOM_OK;
}

void oz_operator_free(OzOperator& op) {
  cudaFree(op.planes); cudaFree(op.ea);
  op.planes = nullptr; op.ea = nullptr;
}

cudaError_t oz_scratch_reserve(OzScratch& s, int MT, int KB, int E, cudaStream_t st) {
  const size_t need = (size_t)MT * KB * OZ_SLICES * OZ_A_TILE;
  if (need > s.bytes) {
    cudaFree(s.zs); s.zs = nullptr; s.bytes = 0;
    cudaError_t e = cudaMalloc((void**)&s.zs, need);
    if (e == cudaSuccess) e = cudaMemsetAsync(s.zs, 0, need, st);   // a default-stream memset would not order with st
    if (e != cudaSuccess) return e;
    s.bytes = need;
  }
  return s.ev ? cudaSuccess : dalloc(&s.ev, (size_t)E);
}

void oz_scratch_free(OzScratch& s) {
  cudaFree(s.zs); cudaFree(s.ev);
  s.zs = nullptr; s.ev = nullptr; s.bytes = 0;
}
