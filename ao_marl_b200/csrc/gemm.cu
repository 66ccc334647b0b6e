// Translation unit of the env-batched GEMMs: the tcgen05 kernel (gemm_tc.cuh), the SIMT kernels (gemm_kernels.cuh) and
// the choice between them; and the fused actor forward (actor_tc.cuh).
#include <stdarg.h>
#include <stdio.h>

#include "../../include/aomarl.h"
#include "dispatch.h"
#include "gemm_host.h"
#include "gemm_tc.cuh"
#include "actor_tc.cuh"

// Kernels launched with more dynamic shared memory than the default: f(kernel, bytes, its template arguments) for every
// instantiation.  gemm_init sets the attribute of each and gemm_launch launches from the same list.
template <class F>
static void gemm_tc_each(F&& f) {     // tcgen05 GEMM: epilogue, column tile
  each<0, 1, 2>([&](auto EPI) {
    each<GTC_BN, GTC_BN_WIDE>([&](auto BN) { f(gemm_tc_kernel<EPI, BN>, (size_t)GTC_SMEM_BYTES_T(BN), EPI, BN); });
  });
}

#define ATC_SMEM_MAX (227 * 1024)

cudaError_t gemm_init() {
  cudaError_t ae = cudaSuccess;
  gemm_tc_each([&](auto kernel, size_t smem, auto...) {
    if (ae == cudaSuccess) ae = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  each<false, true>([&](auto PE) {
    if (ae == cudaSuccess) ae = cudaFuncSetAttribute(actor_fused_kernel<PE>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATC_SMEM_MAX);
  });
  return ae;
}

bool actor_fused_fits(int actor_in, int hidden, int heads) {
  return hidden > 0 && hidden <= 2 * GTC_BN && heads > 0 && heads <= 2 * GTC_BN && ATC_SMEM_BYTES(AOM_LD(actor_in)) <= ATC_SMEM_MAX;
}

void actor_fused_launch(const ActorParams& p, int n_agents, int* err_word, cudaStream_t st) {
  const dim3 grid((p.E + GTC_BM - 1) / GTC_BM, n_agents);
  actor_fused_kernel<false><<<grid, ATC_THREADS, ATC_SMEM_BYTES(p.nkb_in * GTC_BK), st>>>(p, err_word);
}

void actor_fused_env_launch(const ActorEnvParams& p, int n_tiles, int n_agents, int* err_word, cudaStream_t st) {
  const dim3 grid(n_tiles, n_agents);
  actor_fused_kernel<true><<<grid, ATC_THREADS, ATC_SMEM_BYTES(p.nkb_in * GTC_BK), st>>>(p, err_word);
}

static int report(char (&err)[512], int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err, sizeof(err), fmt, ap);
  va_end(ap);
  return code;
}

int gemm_launch(GemmParams p, int epi, int batch, bool exact, int gemm_path, int num_sms, int* err_word, cudaStream_t st,
                char (&err)[512]) {
  const int M = p.M, N = p.N, K = p.K, ldc = p.ldc;
  const int Kp = AOM_LD(K);
  if (p.lda < Kp || p.ldb < Kp || (p.lda & 3) || (p.ldb & 3) || (ldc & 3) || ldc < N)
    return report(err, AOM_ERR_INVALID, "gemm: leading dimensions must cover K rounded to 16 (lda %d ldb %d ldc %d K %d N %d)",
                  p.lda, p.ldb, ldc, K, N);
  p.K = Kp;
  // `exact`: float32 FFMA accumulation with round-to-nearest (the recursive screen extrusion needs it: the
  // tensor core truncates its float32 accumulator, a ~1e-5 systematic shrink that an autoregression integrates)
  if (!exact && gemm_path != AOM_GEMM_SIMT) {
    // column tile: the wide one when it saves CTA waves (two CTAs per SM)
    const long long slots = 2LL * num_sms, rows = (M + GTC_BM - 1) / GTC_BM;
    auto waves = [&](int bn) { return (double)((rows * ((ldc + bn - 1) / bn) * batch + slots - 1) / slots) * bn; };
    const int bn = (!p.Bt && waves(GTC_BN_WIDE) < waves(GTC_BN)) ? GTC_BN_WIDE : GTC_BN;
    const dim3 grid((ldc + bn - 1) / bn, (unsigned)rows, batch);
    gemm_tc_each([&](auto kernel, size_t smem, int e, int b) {
      if (e == epi && b == bn) kernel<<<grid, GTC_THREADS, smem, st>>>(p, err_word);
    });
  } else if (exact && epi == 0 && batch == 1 && !p.bias && !p.relu && gemm_path != AOM_GEMM_SIMT) {
    // shaped exact kernel: column tile 8 CN with the least padding.  Only columns < N are consumed by the
    // extrusion scatter; pad columns inside the last tile are written as zeros, the rest keep their zeros.
    int best = 9, waste = 1 << 30;
    for (int cn = 9; cn >= 8; --cn) {
      const int bn = 8 * cn, w = (N + bn - 1) / bn * bn - N;
      if (w < waste) { waste = w; best = cn; }
    }
    const int bn = 8 * best;
    // two K halves per tile when the tiles alone leave the SMs at two CTAs (8 warps) each
    const int tiles = ((N + bn - 1) / bn) * ((M + GEMM_BM - 1) / GEMM_BM);
    const int ksplit = (tiles <= 2 * num_sms && K >= 512) ? 2 : 1;
    if (ksplit > 1) {
      cudaError_t e = cudaMemsetAsync(p.C, 0, (size_t)M * ldc * sizeof(float), st);
      if (e != cudaSuccess) return report(err, AOM_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    }
    dim3 grid((N + bn - 1) / bn, (M + GEMM_BM - 1) / GEMM_BM, ksplit);
    with<8, 9>(best, [&](auto CN) { gemm_tn_exact_kernel<CN><<<grid, 128, 0, st>>>(p); });
  } else {
    dim3 grid((ldc + GEMM_BN - 1) / GEMM_BN, (M + GEMM_BM - 1) / GEMM_BM, batch);
    with<0, 1, 2>(epi, [&](auto EPI) { gemm_tn_kernel<EPI><<<grid, 256, 0, st>>>(p); });
  }
  return AOM_OK;
}
