// Screen extrusion as an EXACT integer contraction on the tcgen05 tensor cores (Ozaki-style slicing).
//
//   new[e][j] = sum_k AB[j][k] * v[e][k] + zref[e],   v = [screen[stencil] - zref | noise * amp]        (iterkolmo.py:255-288)
//
// is an autoregression: every new column feeds the next ~N extrusions, so the rounding of its K = S + N = 1957-term
// dot products is integrated.  Measured against the float64 oracle (profiles/r02_parity_first_run.json): float32 FFMA
// accumulation leaves the 648^2 screens 1.4e-4 (max-norm) off after the 1296 extrusions of a reset, which alone pushes
// slopes / commands / rewards of the closed loop past the 1e-4 parity bar; the tensor cores' float32 accumulators round
// towards zero, a bias the recursion turns into a drift (DESIGN.md section 4).  Integer accumulation has neither problem:
//
//   * inputs exactly as the oracle forms them: v = float64(pixel) - float64(zref) and float64(noise) * float64(amp);
//   * every row of v (per environment and extrusion) and of [A | B] (per layer, once) is scaled by a power of two to
//     (-1, 1) and cut into six signed 7-bit digits, x 2^-e = q0 2^-6 + q1 2^-13 + ... + q5 2^-41 (+ < 2^-42), each an
//     int8 in [-64, 64].  41 bits below the row maximum: exact for every float32 operator element down to 2^-17 of its
//     row maximum.  (With four operator digits the truncation -- a FIXED perturbation of the recursion -- added up
//     coherently: 648^2 screens 9.5e-5 off after a reset; measured on B200 and reproduced in numpy.)
//   * digit planes are multiplied pairwise on tcgen05.mma kind::i8 (M 128 environments, N 80 outputs, K 32) with int32
//     accumulators in TMEM; pairs with the same weight 2^-(12 + 7g), g = s + t, share one accumulator; the 21 pairs with
//     g <= 5 are kept (the dropped ones are below 2^-37 of |v|max |AB|max in rms);  every partial sum is exact:
//     64 * 64 * 1984 * 6 < 2^31;
//   * the epilogue combines the six accumulators in float64, applies 2^(ev + ea - 12), adds zref and rounds to float32
//     ONCE -- the same single rounding as the oracle's float64 evaluation, so a new pixel differs from the oracle's only
//     when the exact value sits within ~2^-40 of a float32 rounding boundary.
//
// Operand planes are stored in global memory already in the UMMA canonical K-major no-swizzle tile layout (8-row x
// 16-byte core matrices), one contiguous 16 KB / 12 KB block per (tile, k block), so the loader is two cp.async.bulk
// copies per stage and needs no tensor map.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "rng.cuh"

#define OZ_SLICES 6                               // digits of the per-extrusion inputs (41 bits below the row maximum)
#define OZ_SLICES_B 6                             // digits of the operator rows (41 bits): its truncation is a FIXED perturbation
                                                  // of the recursion and adds up coherently -- with 4 digits the 648^2 screens
                                                  // were 9.5e-5 off after a reset (measured, and reproduced in numpy)
#define OZ_LEVELS 6                               // digit pairs kept: s + t <= 5
#define OZ_LEVELS_PRODUCT 5                       // controller products (no recursion behind them): s + t <= 4, 15 MMAs per k
                                                  // block (with s + t <= 3 the 40x40 closed loop moved from 1e-6 to 1e-5 .. 4e-5
                                                  // of the oracle: measured, profiles/r02_parity_levels4.json)
#define OZ_BM 128
#define OZ_BN 80
#define OZ_BK 32
#define OZ_STAGES 3
#define OZ_A_TILE (OZ_BM * OZ_BK)                 // 4096 bytes: one digit plane of 128 rows x 32 k
#define OZ_B_TILE (OZ_BN * OZ_BK)                 // 2560 bytes
#define OZ_STAGE_BYTES (OZ_SLICES * OZ_A_TILE + OZ_SLICES_B * OZ_B_TILE)      // 39936
#define OZ_SMEM_BYTES (OZ_STAGES * OZ_STAGE_BYTES + 256)
#define OZ_THREADS 192
#define OZ_WAIT_SPINS (1u << 21)

struct OzGatherParams {
  const float* screen;      // [E][N][N]
  const int* ox; const int* oy;
  const uint32_t* count;    // [E] extrusions done since reset (RNG counter)
  const uint32_t* k0; const uint32_t* k1;
  const int* stencil;       // [S]
  float* zref;              // [E]
  int* ev;                  // [E] power-of-two scale of the environment's input row
  uint8_t* Zs;              // [MT][KB][OZ_SLICES][OZ_A_TILE] digit planes, canonical tile layout
  int N, S, E, KB, layer, axis, sign;
  float amp;
  const float* amp_env;     // [E] per-environment amplitude, or null
  const int* steps;         // per-environment winds: signed counts of this axis [E] (see ExtrudeParams), or null
  int pass;
  const int* envs;          // compacted start-up: digit row k (and zref / ev [k]) belongs to environment envs[k], or null
};

struct OzGemmParams {
  const uint8_t* Zs;        // [MT][KB][OZ_SLICES][OZ_A_TILE]
  const uint8_t* ABs;       // [NT][KB][OZ_SLICES_B][OZ_B_TILE]
  const int* ev;            // [E]
  const int* ea;            // [NT * OZ_BN]
  const float* zref;        // [E]  (extrusion epilogue)
  float* out; int ldo;      // [E][ldo]
  int E, N, KB;
  float* com; int ldcom;    // integrator epilogue: com += gain * out when closed
  float gain; int closed;
  int* err;
  const float* gain_env;    // EPI 3: one gain per environment [E]
};

// digit planes of a per-environment float32 matrix X [E][ld] (K valid columns): the A operand of oz_gemm_kernel
struct OzSliceParams {
  const float* X; int ld, K, E, KB;
  uint8_t* Zs; int* ev;
};

// element (row r, k) of a [rows x 32] int8 tile: 8-row x 16-byte core matrices, 128 B between the two k halves,
// 256 B between 8-row groups
__host__ __device__ __forceinline__ uint32_t oz_tile_offset(int r, int kk) {
  return (uint32_t)((r >> 3) * 256 + (kk >> 4) * 128 + (r & 7) * 16 + (kk & 15));
}

// NS signed 7-bit digits of x * scale, |x * scale| < 1 (every step is exact in float64 for inputs of <= 48 bits)
template <int NS>
__host__ __device__ __forceinline__ void oz_digits(double x, double scale, int (&q)[NS]) {
  double t = x * scale * 64.0;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const double r = rint(t);
    q[s] = (int)r;
    t = (t - r) * 128.0;
  }
}

// the same digits of a float32 value: every step is exact in float32 (the remainders only lose leading bits)
template <int NS>
__host__ __device__ __forceinline__ void oz_digits_f32(float x, float scale, int (&q)[NS]) {
  float t = x * scale * 64.0f;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const float r = rintf(t);
    q[s] = (int)r;
    t = (t - r) * 128.0f;
  }
}

// power of two e with |x| * 2^-e in [0.5, 1) for the row maximum x (0 for an all-zero row)
__host__ __device__ __forceinline__ int oz_exponent(double amax) {
  if (!(amax > 0.0)) return 0;
  int e;
  frexp(amax, &e);           // amax = m 2^e, m in [0.5, 1)
  return e;
}

#ifdef OZ_DEFINE_KERNELS   // the kernels are defined in one translation unit only (extrude_i8.cu)
__device__ __forceinline__ void oz_logical(int r, int c, int N, int axis, int sign, int& lr, int& lc) {
  if (axis == 0) { lr = r; lc = c; } else { lr = c; lc = r; }
  if (sign < 0) {
    if (axis == 0) { lr = N - 1 - r; lc = N - 1 - c; } else { lr = N - 1 - c; lc = N - 1 - r; }
  }
}
__device__ __forceinline__ int oz_wrap(int v, int N) { return v >= N ? v - N : v; }

// grid: E blocks of 256 threads (K with p.envs: block k serves environment envs[k] and writes row k); dynamic shared
// memory: KB * 32 doubles.
// Gathers the stencil pixels (minus the reference pixel) and the scaled innovations of one environment, finds the row
// scale, cuts the row into digit planes and stores them in the tile layout the tensor core reads.
// PE: per-environment winds -- environment e takes part in pass p.pass of the axis iff p.pass < |steps[e]|, in the
// direction of steps[e]; otherwise it stores nothing (the GEMM's row of e is computed from stale digits and not scattered).
template <bool PE = false>
__global__ void __launch_bounds__(256) oz_gather_slice_kernel(OzGatherParams p) {
  extern __shared__ double oz_v[];
  __shared__ double s_red[8];
  const int row = blockIdx.x, e = p.envs ? p.envs[row] : row, N = p.N, Kp = p.KB * OZ_BK;
  int sign = p.sign;
  if (PE) {
    const int n = p.steps[e];
    if (p.pass >= (n < 0 ? -n : n)) return;
    sign = n < 0 ? -1 : 1;
  }
  const float* scr = p.screen + (size_t)e * N * N;
  const int ox = p.ox[e], oy = p.oy[e];
  int rr, rc;
  oz_logical(0, N - 1, N, p.axis, sign, rr, rc);
  const float zr = scr[(size_t)oz_wrap(rr + oy, N) * N + oz_wrap(rc + ox, N)];
  // differences and products in float64, i.e. exactly: what the oracle (and a float64 reading of iterkolmo.py:281-284) does
  double amax = 0.0;
  const uint32_t magic = 0xFFFFFFFFu / (uint32_t)N + 1u;       // idx / N = umulhi(idx, magic) for idx < N^2 <= 2^22 (N <= 2048)
  for (int k = threadIdx.x; k < p.S; k += blockDim.x) {
    const int idx = p.stencil[k];
    const int sr = (int)__umulhi((uint32_t)idx, magic), sc = idx - sr * N;
    int lr, lc;
    oz_logical(sr, sc, N, p.axis, sign, lr, lc);
    const double v = (double)scr[(size_t)oz_wrap(lr + oy, N) * N + oz_wrap(lc + ox, N)] - (double)zr;
    oz_v[k] = v;
    amax = fmax(amax, fabs(v));
  }
  const uint32_t cnt = p.count[e], k0 = p.k0[e], k1 = p.k1[e];
  const float amp = p.amp_env ? p.amp_env[e] : p.amp;
  for (int b = threadIdx.x; 4 * b < N; b += blockDim.x) {
    const aom_u4 w = aom_philox((uint32_t)b, cnt, AOM_TAG_ATMOS, (uint32_t)p.layer, k0, k1);
    float z[4];
    aom_normal_pair(w.x, w.y, z[0], z[1]);
    aom_normal_pair(w.z, w.w, z[2], z[3]);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (4 * b + i < N) {
        const double v = (double)z[i] * (double)amp;
        oz_v[p.S + 4 * b + i] = v;
        amax = fmax(amax, fabs(v));
      }
  }
  for (int k = p.S + N + threadIdx.x; k < Kp; k += blockDim.x) oz_v[k] = 0.0;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, s));
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = amax;
  __syncthreads();
  amax = s_red[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) amax = fmax(amax, s_red[i]);
  const int ex = oz_exponent(amax);
  if (threadIdx.x == 0) { p.zref[row] = zr; p.ev[row] = ex; }
  const double scale = __longlong_as_double((long long)(1023 - ex) << 52);      // 2^-ex
  const int mt = row >> 7, r = row & 127;
  // eight values per thread and pass: the 1984 values of a 648-pixel layer keep 248 of the 256 threads busy in one pass
  for (int j = threadIdx.x; j < Kp / 8; j += blockDim.x) {
    uint32_t w[OZ_SLICES][2];
#pragma unroll
    for (int s = 0; s < OZ_SLICES; ++s) w[s][0] = w[s][1] = 0u;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int q[OZ_SLICES];
      oz_digits<OZ_SLICES>(oz_v[8 * j + i], scale, q);
#pragma unroll
      for (int s = 0; s < OZ_SLICES; ++s) w[s][i >> 2] |= ((uint32_t)q[s] & 0xffu) << (8 * (i & 3));
    }
    const int kb = j >> 2;
    uint8_t* base = p.Zs + ((size_t)(mt * p.KB + kb) * OZ_SLICES) * OZ_A_TILE + oz_tile_offset(r, (j & 3) * 8);
#pragma unroll
    for (int s = 0; s < OZ_SLICES; ++s)
      *reinterpret_cast<uint2*>(base + (size_t)s * OZ_A_TILE) = make_uint2(w[s][0], w[s][1]);
  }
}

// grid: E blocks of 256 threads.  Row scale + digit planes of one environment's input vector (slopes, commands, modes).
__global__ void __launch_bounds__(256) oz_slice_rows_kernel(OzSliceParams p) {
  __shared__ float s_red[8];
  const int e = blockIdx.x, Kp = p.KB * OZ_BK;
  const float* x = p.X + (size_t)e * p.ld;
  float amax = 0.f;
  for (int k = threadIdx.x; k < p.K; k += blockDim.x) amax = fmaxf(amax, fabsf(x[k]));
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, s));
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = amax;
  __syncthreads();
  amax = s_red[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) amax = fmaxf(amax, s_red[i]);
  const int ex = oz_exponent((double)amax);
  if (threadIdx.x == 0) p.ev[e] = ex;
  const float scale = __int_as_float((127 - ex) << 23);          // 2^-ex
  const int mt = e >> 7, r = e & 127;
  for (int j = threadIdx.x; j < Kp / 16; j += blockDim.x) {
    uint32_t w[OZ_SLICES][4];
#pragma unroll
    for (int s = 0; s < OZ_SLICES; ++s)
#pragma unroll
      for (int i = 0; i < 4; ++i) w[s][i] = 0u;
    // rows are padded to a multiple of 16 floats: whole 16-float groups can be read; columns >= K count as zeros
    float v[16];
    if (16 * j + 16 <= p.ld) {
#pragma unroll
      for (int i4 = 0; i4 < 4; ++i4) {
        const float4 f = *reinterpret_cast<const float4*>(x + 16 * j + 4 * i4);
        v[4 * i4] = f.x; v[4 * i4 + 1] = f.y; v[4 * i4 + 2] = f.z; v[4 * i4 + 3] = f.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      int q[OZ_SLICES];
      oz_digits_f32<OZ_SLICES>((16 * j + i < p.K) ? v[i] : 0.f, scale, q);
#pragma unroll
      for (int s = 0; s < OZ_SLICES; ++s) w[s][i >> 2] |= ((uint32_t)q[s] & 0xffu) << (8 * (i & 3));
    }
    const int kb = j >> 1;
    uint8_t* base = p.Zs + ((size_t)(mt * p.KB + kb) * OZ_SLICES) * OZ_A_TILE + oz_tile_offset(r, (j & 1) * 16);
#pragma unroll
    for (int s = 0; s < OZ_SLICES; ++s)
      *reinterpret_cast<uint4*>(base + (size_t)s * OZ_A_TILE) = make_uint4(w[s][0], w[s][1], w[s][2], w[s][3]);
  }
}

__device__ __forceinline__ uint32_t oz_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void oz_mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  uint32_t ns = 32;
#pragma unroll 1
  for (uint32_t it = 0; it < OZ_WAIT_SPINS; ++it) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    __nanosleep(ns);
    ns = ns < 1024u ? ns * 2u : 1024u;
  }
  atomicExch(err, 4);
  __threadfence_system();
  __trap();
}

__device__ __forceinline__ uint64_t oz_desc(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(128u >> 4) << 16;                          // leading: between the two 16-byte k chunks
  d |= (uint64_t)(256u >> 4) << 32;                          // stride: between 8-row groups
  d |= 1ull << 46;
  return d;
}

// one lane of a converged warp.  With the warp index taken through a shuffle and the lane through elect.sync the compiler
// knows the issuing path is warp-uniform and keeps descriptors in uniform registers; under `lane == 0` every MMA sat in a
// per-thread waterfall loop (ELECT / R2UR / BRA.U.ANY, ~13 instructions per MMA; measured on the denoiser kernel).
__device__ __forceinline__ bool oz_elect() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(p));
  return p != 0;
}

// descriptors given as low words (start address >> 4 | LBO 128 B >> 4 << 16); high word = SBO 256 B >> 4 | version
__device__ __forceinline__ void oz_mma_i8_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %3, {%6, %6, %6, %6}, p;\n\t}"
      :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"((256u >> 4) | (1u << 14)), "r"(0u) : "memory");
}

__device__ __forceinline__ void oz_mma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}

// grid (NT, MT), 192 threads, one CTA per SM (480 of the 512 TMEM columns):
//   warp 0  lane 0: two bulk copies per stage (24 KB of environment digits, 15 KB of operator digits)
//   warp 1  TMEM allocation; lane 0 issues the 21 digit-pair MMAs of every stage
//   warps 2-5  epilogue: TMEM lane quarter warp % 4 -> 32 environments, five int32 accumulators -> float64 -> float32
// EPI 0: screen extrusion (+ zref, every column of the row written)   1: plain product (pad columns zero)
// EPI 2: least-squares integrator: out = -product, com += gain * out when the loop is closed (rtcCompass.py:527-547)
// EPI 3: the same with one gain per environment, com += gain_env[e] * out
// LEV: digit-pair levels kept (pairs with s + t < LEV).  6 (21 MMAs per k block) for the screen recursion, which
// integrates any truncation; OZ_LEVELS_PRODUCT = 5 (15 MMAs) for the one-shot controller products, where the dropped
// pairs are below 2^-35 of |x|max |W|max per term.
template <int EPI, int LEV>
__global__ void __launch_bounds__(OZ_THREADS, 1) oz_gemm_kernel(OzGemmParams p) {
  extern __shared__ __align__(1024) uint8_t oz_smem[];
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = tid & 31;
  const int nt = blockIdx.x, mt = blockIdx.y;
  uint64_t* bars = reinterpret_cast<uint64_t*>(oz_smem + OZ_STAGES * OZ_STAGE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * OZ_STAGES + 1);
  const uint32_t full0 = oz_smem_u32(bars), empty0 = oz_smem_u32(bars + OZ_STAGES);
  const uint32_t accum_bar = oz_smem_u32(bars + 2 * OZ_STAGES);

  if (tid == 0) {
    for (int s = 0; s < 2 * OZ_STAGES + 1; ++s)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(full0 + 8 * s) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(oz_smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    if (oz_elect()) {
      const uint8_t* za = p.Zs + (size_t)mt * p.KB * OZ_SLICES * OZ_A_TILE;
      const uint8_t* ab = p.ABs + (size_t)nt * p.KB * OZ_SLICES_B * OZ_B_TILE;
      for (int kb = 0; kb < p.KB; ++kb) {
        const int s = kb % OZ_STAGES;
        const uint32_t round = (uint32_t)(kb / OZ_STAGES);
        oz_mbar_wait(empty0 + 8 * s, (round & 1u) ^ 1u, p.err);
        const uint32_t dst = oz_smem_u32(oz_smem + (size_t)s * OZ_STAGE_BYTES);
        const uint32_t bar = full0 + 8 * s;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)OZ_STAGE_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst), "l"(za + (size_t)kb * OZ_SLICES * OZ_A_TILE), "r"((uint32_t)(OZ_SLICES * OZ_A_TILE)), "r"(bar) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst + OZ_SLICES * OZ_A_TILE), "l"(ab + (size_t)kb * OZ_SLICES_B * OZ_B_TILE), "r"((uint32_t)(OZ_SLICES_B * OZ_B_TILE)), "r"(bar) : "memory");
      }
    }
  } else if (warp == 1) {
    if (oz_elect()) {
      // int8 x int8 -> int32: c_format S32 (2), a / b format signed 8 bit (1), K-major operands, N 96, M 128
      const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BN >> 3) << 17) | ((uint32_t)(OZ_BM >> 4) << 24);
      uint32_t used = 0;                                      // bit g: accumulator g has been written
      for (int kb = 0; kb < p.KB; ++kb) {
        const int s = kb % OZ_STAGES;
        const uint32_t round = (uint32_t)(kb / OZ_STAGES);
        oz_mbar_wait(full0 + 8 * s, round & 1u, p.err);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a0 = ((oz_smem_u32(oz_smem) + (uint32_t)s * OZ_STAGE_BYTES) >> 4) | ((128u >> 4) << 16);
        const uint32_t b0 = a0 + (OZ_SLICES * OZ_A_TILE >> 4);
#pragma unroll
        for (int g = 0; g < LEV; ++g)
#pragma unroll
          for (int sa = 0; sa < OZ_SLICES; ++sa) {
            const int sb = g - sa;
            if (sb < 0 || sb >= OZ_SLICES_B || sa >= OZ_SLICES) continue;
            oz_mma_i8_lo(tmem_base + (uint32_t)(g * OZ_BN), a0 + sa * (OZ_A_TILE >> 4), b0 + sb * (OZ_B_TILE >> 4), idesc,
                         (used >> g) & 1u);
            used |= 1u << g;
          }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(empty0 + 8 * s) : "memory");
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(accum_bar) : "memory");
    }
  } else {
    oz_mbar_wait(accum_bar, 0u, p.err);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int q = warp & 3;                                   // TMEM lane quarter this warp may read
    const int e = mt * OZ_BM + 32 * q + lane;
    const bool live = e < p.E;
    const int ev = live ? p.ev[e] : 0;
    const double zr = (EPI == 0 && live) ? (double)p.zref[e] : 0.0;
    const float gn = (EPI == 3 && live) ? p.gain_env[e] : p.gain;     // integrator gain of this row's environment
#pragma unroll 1
    for (int cb = 0; cb < OZ_BN / 8; ++cb) {
      uint32_t v[LEV][8];
#pragma unroll
      for (int g = 0; g < LEV; ++g) {
        const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(g * OZ_BN + cb * 8);
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(v[g][0]), "=r"(v[g][1]), "=r"(v[g][2]), "=r"(v[g][3]), "=r"(v[g][4]), "=r"(v[g][5]), "=r"(v[g][6]), "=r"(v[g][7])
                     : "r"(taddr) : "memory");
      }
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (live) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int n = nt * OZ_BN + cb * 8 + j;
          // sum_g acc_g 2^(-7 g) in float64 (each accumulator < 2^26; the sum spans 61 bits, rounded at 2^-53)
          double acc = (double)(int)v[LEV - 1][j];
#pragma unroll
          for (int g = LEV - 2; g >= 0; --g) acc = fma(acc, 0.0078125, (double)(int)v[g][j]);
          const int ex = ev + p.ea[n] - 12;
          const double sc = __longlong_as_double((long long)(1023 + ex) << 52);
          if (EPI == 0) o[j] = (float)fma(acc, sc, zr);        // pad columns get zref: harmless, the scatter reads n < N
          else {
            const float r = (float)(acc * sc);
            o[j] = (n < p.N) ? (EPI >= 2 ? -r : r) : 0.f;       // pad columns stay zero
          }
        }
        const int n0 = nt * OZ_BN + cb * 8;
        float* dst = p.out + (size_t)e * p.ldo + n0;
        if (n0 + 8 <= p.ldo) {
          *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<float4*>(dst + 4) = make_float4(o[4], o[5], o[6], o[7]);
          if (EPI >= 2 && p.closed) {
            float4* cp = reinterpret_cast<float4*>(p.com + (size_t)e * p.ldcom + n0);
            float4 c0 = cp[0], c1 = cp[1];
            c0.x = fmaf(gn, o[0], c0.x); c0.y = fmaf(gn, o[1], c0.y); c0.z = fmaf(gn, o[2], c0.z); c0.w = fmaf(gn, o[3], c0.w);
            c1.x = fmaf(gn, o[4], c1.x); c1.y = fmaf(gn, o[5], c1.y); c1.z = fmaf(gn, o[6], c1.z); c1.w = fmaf(gn, o[7], c1.w);
            cp[0] = c0; cp[1] = c1;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (n0 + j < p.ldo) {
              dst[j] = o[j];
              if (EPI >= 2 && p.closed) p.com[(size_t)e * p.ldcom + n0 + j] = fmaf(gn, o[j], p.com[(size_t)e * p.ldcom + n0 + j]);
            }
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}
#endif  // OZ_DEFINE_KERNELS
