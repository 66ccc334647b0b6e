// Translation unit of the tcgen05 Shack-Hartmann frame kernel: instantiations per layer count + launch geometry.
#include <string.h>
#include "wfs_umma_host.h"
#include "wfs_umma_ws.cuh"

template <int NL, int FULL, int WS, bool PE, bool NE = false>
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
  if (WS) {
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

cudaError_t wfs_umma_launch(const WfsParams& p, const WfsUmmaHost& h, int num_sms, int full, int ws, cudaStream_t st) {
  if (p.noise_env || p.nph_env) {     // per-environment sensor values: the fused kernel only (the library routes so)
    if (ws) return cudaErrorInvalidValue;
#define WU_GO_NE(NL, PE) return full ? launch_t<NL, 1, 0, PE, true>(p, h, num_sms, st) : launch_t<NL, 0, 0, PE, true>(p, h, num_sms, st)
    if (p.wind && p.n_layers > 0) {
      switch (p.n_layers) {
        case 1: WU_GO_NE(1, true);
        case 2: WU_GO_NE(2, true);
        case 3: WU_GO_NE(3, true);
        case 4: WU_GO_NE(4, true);
      }
      return cudaErrorInvalidValue;
    }
    switch (p.n_layers) {
      case 0: WU_GO_NE(0, false);
      case 1: WU_GO_NE(1, false);
      case 2: WU_GO_NE(2, false);
      case 3: WU_GO_NE(3, false);
      case 4: WU_GO_NE(4, false);
    }
#undef WU_GO_NE
    return cudaErrorInvalidValue;
  }
#define WU_GO(NL, PE) return ws ? launch_t<NL, 1, 1, PE>(p, h, num_sms, st) : full ? launch_t<NL, 1, 0, PE>(p, h, num_sms, st) \
                                                                                : launch_t<NL, 0, 0, PE>(p, h, num_sms, st)
  if (p.wind && p.n_layers > 0) {     // per-environment winds
    switch (p.n_layers) {
      case 1: WU_GO(1, true);
      case 2: WU_GO(2, true);
      case 3: WU_GO(3, true);
      case 4: WU_GO(4, true);
    }
    return cudaErrorInvalidValue;
  }
  switch (p.n_layers) {
    case 0: WU_GO(0, false);
    case 1: WU_GO(1, false);
    case 2: WU_GO(2, false);
    case 3: WU_GO(3, false);
    case 4: WU_GO(4, false);
  }
#undef WU_GO
  return cudaErrorInvalidValue;
}
