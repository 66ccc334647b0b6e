// Host interface of the env-batched GEMMs (gemm.cu): C[b][m][n] = sum_k A[b][m][k] * B[b][n][k] (+ bias) (relu), or the
// integrator epilogue, on the tcgen05 kernel (gemm_tc.cuh) or the SIMT ones (gemm_kernels.cuh).
#pragma once
#include <cuda_runtime.h>

struct GemmParams {
  const float* A; const float* B; float* C; const float* bias;
  int lda, ldb, ldc;
  int M, N, K;          // K valid columns; the launcher rounds it up to a multiple of 16 (operands are zero padded)
  long long sA, sB, sC, sBias;   // batch strides (elements)
  int relu;
  // epilogue 1 (integrator): err = -acc ; C = err ; com += gain * err
  float* com; int ldcom; float gain; int closed;
  // gemm_tc_kernel only: the B operand already split into TF32 hi / lo planes in the UMMA tile order of 128-column tiles
  // ([n tile][k block][hi, lo][128 x 16]; gtc_pretile_host), brought in by one bulk copy per stage.  Null: B is split on the fly.
  const float* Bt; long long sBt;
  // epilogue 2: the integrator of epilogue 1 with one gain per row (environment): com += gain_env[row] * err
  const float* gain_env;
};

// Sets the dynamic shared-memory size of every tcgen05 GEMM instantiation; once per context, before any launch.
cudaError_t gemm_init();

// Launches one GEMM of `batch` products with epilogue epi (0 plain, 1 integrator, 2 integrator with p.gain_env) on st.
// `exact`: float32 FFMA accumulation with round-to-nearest, else the tcgen05 kernel unless gemm_path is AOM_GEMM_SIMT,
// whose bounded waits raise the device error word err_word.  Returns AOM_OK, or an error code with its message in err;
// the caller checks the launch itself (cudaGetLastError).
int gemm_launch(GemmParams p, int epi, int batch, bool exact, int gemm_path, int num_sms, int* err_word, cudaStream_t st,
                char (&err)[512]);
