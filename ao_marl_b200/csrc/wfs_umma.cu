// Translation unit of the tcgen05 Shack-Hartmann frame kernel: instantiations per layer count + launch geometry.
#include <string.h>
#include "dispatch.h"
#include "wfs_umma_host.h"
#include "wfs_umma_ws.cuh"

template <int NL, int FULL, int WS, bool PE, bool NE>
static cudaError_t launch_t(const WfsParams& p, const WfsUmmaHost& h, int num_sms, cudaStream_t st) {
  const long long total = (long long)p.E * p.nvalid;
  // persistent CTAs over contiguous ranges of work items: two CTAs per SM, about 4 waves, at least 8 iterations each
  long long grid = (long long)num_sms * 2 * 4;
  long long ipc = (total + grid - 1) / grid;
  if (ipc < 8 * WU_WARPS) ipc = 8 * WU_WARPS;
  ipc = (ipc + WU_WARPS - 1) / WU_WARPS * WU_WARPS;
  grid = (total + ipc - 1) / ipc;
  WfsUmmaParams P;
  memset(&P, 0, sizeof(P));
  P.p = p;
  P.f = h.f;
  P.f.items_per_cta = ipc;
  for (int l = 0; l < NL; ++l) P.maps[l] = h.maps[l];
  const size_t smem = wu_smem_bytes<NL, PE>(P.f.GW);
  if constexpr (WS != 0) {
    cudaError_t e = cudaFuncSetAttribute(wfs_frame_ws_kernel<NL, FULL, PE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    wfs_frame_ws_kernel<NL, FULL, PE><<<(unsigned)grid, WS_THREADS, smem, st>>>(P);
  } else {
    cudaError_t e = cudaFuncSetAttribute(wfs_frame_umma_kernel<NL, FULL, PE, NE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    wfs_frame_umma_kernel<NL, FULL, PE, NE><<<(unsigned)grid, WU_WARPS * 32, smem, st>>>(P);
  }
  return cudaGetLastError();
}

cudaError_t wfs_umma_launch(const WfsParams& p, const WfsUmmaHost& h, int num_sms, bool ws, bool full, bool ne, cudaStream_t st) {
  cudaError_t e = cudaErrorInvalidValue;
  with<0, 1, 2, 3, 4>(p.n_layers, [&](auto NL) {
    with<false, true>(p.wind && p.n_layers > 0, [&](auto PE) {
      with<false, true>(ws, [&](auto WS) {
        with<false, true>(full, [&](auto FULL) {
          with<false, true>(ne, [&](auto NE) {
            // per-environment winds need a layer; the specialised-warp kernel exists with FULL and without NE only
            if constexpr ((NL > 0 || !PE) && (!WS || (FULL && !NE))) e = launch_t<NL, FULL, WS, PE, NE>(p, h, num_sms, st);
          });
        });
      });
    });
  });
  return e;
}
