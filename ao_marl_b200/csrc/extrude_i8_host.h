// Host interface of the exact integer extrusion (extrude_i8.cuh), compiled in its own translation unit.
#pragma once
#include <cuda_runtime.h>
#include "extrude_i8.cuh"

// An operator [rows][ld] (K valid columns) as the digit planes of the integer contraction, on the device: planes and row
// scales ea of NT column tiles of KB k blocks.  Zero: not uploaded.
struct OzOperator {
  uint8_t* planes;
  int* ea;
  int kb, nt;
};

// Replaces op by the digit planes of the host operator.  A NaN or an infinity is refused before op changes.  Returns
// AOM_OK, or an error code with its message in err.
int oz_operator_upload(OzOperator& op, const float* host, int rows, int ld, int K, char (&err)[512]);
void oz_operator_free(OzOperator& op);

// Device scratch of the contraction: digit planes of the per-environment vectors and their row scales, grown on demand.
// The two streams of aom_step contract at the same time, so each keeps its own.
struct OzScratch {
  uint8_t* zs;
  int* ev;
  size_t bytes;
};

// Room for MT row tiles of KB k blocks (new room zeroed on st, the stream that uses it) and the row scales of E rows
cudaError_t oz_scratch_reserve(OzScratch& s, int MT, int KB, int E, cudaStream_t st);
void oz_scratch_free(OzScratch& s);

// gather + digit planes of all environments, then the digit-pair GEMM (grid NT x MT); both asynchronous on `st`
cudaError_t oz_extrude_launch(const OzGatherParams& g, const OzGemmParams& m, int MT, int NT, cudaStream_t st);

// out = X . OP^T for a per-environment float32 matrix X and an operator given as digit planes (integrator != 0: the
// least-squares integrator epilogue, with one gain per environment when m.gain_env is set): row digits of X, then the
// digit-pair GEMM; both asynchronous on `st`
cudaError_t oz_product_launch(const OzSliceParams& sl, const OzGemmParams& m, int integrator, int MT, int NT, cudaStream_t st);
