// Host interface of the tcgen05 Shack-Hartmann frame kernel (wfs_umma.cuh), compiled in its own translation unit
// (wfs_umma.cu) and linked into libaomarl.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include "wfs_umma.cuh"

struct WfsUmmaHost {
  WfsUmmaTables f;
  CUtensorMap maps[WU_MAX_LAYERS];
};

// Launches wfs_frame_umma_kernel for the frame described by p.  full: fp32-grade products in both stages.
// Returns cudaSuccess or the error of the attribute / launch call.
// ws: the warp-specialised kernel (wfs_umma_ws.cuh) on the same tables (needs full and not ne).  p.wind != null: the
// per-environment wind instantiations of either kernel.  ne: the per-environment sensor instantiations of the fused
// kernel, which read p.noise_env / p.nph_env.
cudaError_t wfs_umma_launch(const WfsParams& p, const WfsUmmaHost& h, int num_sms, bool ws, bool full, bool ne, cudaStream_t st);
