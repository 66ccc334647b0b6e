// Env-batched contractions on the 5th-generation tensor cores (tcgen05 + TMEM), float32 in / float32 out.
//
//        C[b][m][n] = sum_k A[b][m][k] * B[b][n][k]  (+ bias[b][n]) (relu)   |   integrator epilogue
//
// Same contract as gemm_tn_kernel (gemm_kernels.cuh): A = per-environment vectors [E][ld], B = shared
// operator [rows][ld], both K-major with zero-padded leading dimensions.  Serves the screen extrusion
// (A.z + B.noise, iterkolmo.py:255-288), the command-matrix reconstruction (rtcCompass.py:527-547), the
// Btt projections (rlSupervisor.py:784-818, ao_env.py:482-505) and the actors (model_rpc.py:121-158).
//
// Precision: every float32 operand is split on the fly into two TF32 numbers, hi = the leading 11
// significant bits, lo = x - hi (exact), and each product is three kind::tf32 MMAs
// (hi.hi + hi.lo + lo.hi) accumulated in float32 in TMEM: ~2^-21 relative per product, so commands,
// screens and rewards stay well inside the rel 1e-4 parity bar where a single TF32/BF16 pass does not.
//
// Structure (one 128 x 128 output tile per CTA, 288 threads, two CTAs per SM):
//   warps 0-7  loaders: coalesced 128-bit global loads of the A and B slabs (16 k-values per stage),
//              hi/lo split in registers, st.shared into the canonical K-major no-swizzle UMMA layout
//              (8-row x 16-byte core matrices), fence.proxy.async, mbarrier arrive.   Then the epilogue:
//              tcgen05.ld of their 32 TMEM lanes (two warps per lane quarter, half of the columns each), bias / relu /
//              integrator, 128-bit stores.  (Four loader warps -- the first version -- left the tensor pipe at 20-25 %.)
//   warp 8     TMEM allocation; one lane waits on the full barriers and issues the six tcgen05.mma of the
//              stage, tcgen05.commit releases the stage to the loaders and finally the accumulator.
// Every mbarrier wait is bounded: on expiry the kernel raises an error word and traps instead of hanging the
// device or publishing a wrong product.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gemm_kernels.cuh"

#define GTC_BM 128
#define GTC_BN 128
#define GTC_BK 16
#define GTC_STAGES 3
#define GTC_INFLIGHT 3                                        // slabs of global loads in flight per loader thread (register sets)
#define GTC_TILE_BYTES (GTC_BM * GTC_BK * 4)                 // 8 KB: one hi or lo slab of the A operand
#define GTC_BTILE_BYTES(BN) ((BN) * GTC_BK * 4)               // one hi or lo slab of the B operand
#define GTC_STAGE_BYTES_T(BN) (2 * GTC_TILE_BYTES + 2 * GTC_BTILE_BYTES(BN))   // A hi, A lo, B hi, B lo
#define GTC_SMEM_BYTES_T(BN) (GTC_STAGES * GTC_STAGE_BYTES_T(BN) + 128)
#define GTC_SMEM_BYTES GTC_SMEM_BYTES_T(GTC_BN)
#define GTC_BN_WIDE 144                                       // 9 x 144 = 1296: the 1283 / 1286-wide operators in one wave
#define GTC_LOADERS 8                                         // loader / epilogue warps (two per TMEM lane quarter)
#define GTC_THREADS ((GTC_LOADERS + 1) * 32)
#define GTC_WAIT_SPINS (1u << 20)

__device__ __forceinline__ uint32_t gtc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void gtc_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void gtc_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool gtc_mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: if the phase never completes the error word is raised and the kernel stops (carrying on would overwrite a
// stage the MMAs still read, or read an incomplete accumulator: silently wrong commands)
__device__ __forceinline__ bool gtc_mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  for (uint32_t it = 0; it < GTC_WAIT_SPINS; ++it)
    if (gtc_mbar_try(bar, parity)) return true;
  if (err) atomicExch(err, 1);
  __threadfence_system();
  __trap();
  return false;
}

// K-major, no swizzle: 8-row x 16-byte core matrices; LBO = 128 B between the K chunks of a row group,
// SBO = 512 B between 8-row groups (GTC_BK = 16 floats = 4 chunks per row)
__device__ __forceinline__ uint64_t gtc_desc(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(128u >> 4) << 16;
  d |= (uint64_t)(512u >> 4) << 32;
  d |= 1ull << 46;                                           // descriptor version of sm_100
  return d;
}

__device__ __forceinline__ void gtc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}

// descriptors as low words (start >> 4 | LBO 128 B >> 4 << 16); high word = SBO 512 B >> 4 | version.  Together with
// elect.sync on a shuffled warp index this keeps the issue path in uniform registers (no per-MMA waterfall loop).
__device__ __forceinline__ void gtc_mma_tf32_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, {%6, %6, %6, %6}, p;\n\t}"
      :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"((512u >> 4) | (1u << 14)), "r"(0u) : "memory");
}
__device__ __forceinline__ bool gtc_elect() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(p));
  return p != 0;
}

__device__ __forceinline__ void gtc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void gtc_split4(const float4& v, float4& hi, float4& lo) {
  hi.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
  hi.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
  hi.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
  hi.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
  lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
}

// BN: column tile (multiple of 16, 128 or GTC_BN_WIDE).  With M = 4096 rows the 1283 / 1286-wide operators give
// 11 x 32 = 352 tiles of 128 columns on 296 CTA slots -- a second wave that keeps 56 tiles' worth of SMs busy while
// the rest idle (ncu: SMs active 56 % of the launch) -- and 9 x 32 = 288 tiles of 144 columns: one wave.
template <int EPI, int BN>
__global__ void __launch_bounds__(GTC_THREADS, 2) gemm_tc_kernel(GemmParams p, int* err) {
  constexpr int STAGE_BYTES = GTC_STAGE_BYTES_T(BN);
  constexpr int B_OFF = 2 * GTC_TILE_BYTES;                    // B hi at B_OFF, B lo at B_OFF + GTC_BTILE_BYTES(BN)
  constexpr int ROWS_PER_PASS = GTC_LOADERS * 8;               // 64 rows of a slab per pass of the loaders
  constexpr int A_ITERS = GTC_BM / ROWS_PER_PASS;
  constexpr int B_ITERS = (BN + ROWS_PER_PASS - 1) / ROWS_PER_PASS;
  constexpr uint32_t TMEM_COLS = BN <= 128 ? 128u : 256u;
  extern __shared__ __align__(1024) uint8_t gtc_smem[];
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = tid & 31;
  const int bz = blockIdx.z;
  const float* __restrict__ A = p.A + (long long)bz * p.sA;
  const float* __restrict__ B = p.B + (long long)bz * p.sB;
  float* __restrict__ C = p.C + (long long)bz * p.sC;
  const int m0 = blockIdx.y * GTC_BM;
  const int n0 = blockIdx.x * BN;
  const int nkb = (p.K + GTC_BK - 1) / GTC_BK;
  // pre-tiled B (static weights, 128-column tiles only): [n tile][k block][hi, lo][BN x 16 floats]
  const bool pre = (BN == GTC_BN) && p.Bt != nullptr;
  const float* __restrict__ Bt = pre ? p.Bt + (long long)bz * p.sBt + (size_t)blockIdx.x * nkb * (2 * BN * GTC_BK) : nullptr;

  uint8_t* tiles = gtc_smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(gtc_smem + GTC_STAGES * STAGE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * GTC_STAGES + 1);
  const uint32_t full0 = gtc_smem_u32(bars), empty0 = gtc_smem_u32(bars + GTC_STAGES);
  const uint32_t accum_bar = gtc_smem_u32(bars + 2 * GTC_STAGES);

  if (tid == 0) {
    for (int s = 0; s < GTC_STAGES; ++s) {
      gtc_mbar_init(full0 + 8 * s, GTC_LOADERS + (pre ? 1 : 0));   // one arrive per loader warp (+ the bulk copy's expect_tx)
      gtc_mbar_init(empty0 + 8 * s, 1);       // tcgen05.commit
    }
    gtc_mbar_init(accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == GTC_LOADERS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(gtc_smem_u32(tmem_slot)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp < GTC_LOADERS) {
    // ===== loaders =====
    // eight consecutive lanes take the same 16-byte chunk (4 k-values) of eight consecutive rows: their st.shared.v4 fill
    // one 128-byte core matrix without bank conflicts (with chunk = tid & 3 the four chunks of a row landed 128 B apart on
    // the same banks: 75 % of the shared-memory wavefronts were replays, profiles/r01_gemmtc_E4096_metrics.csv); the
    // global loads of a warp still cover whole 64-byte row segments
    const int c = (tid >> 3) & 3;
    const int r0 = (tid >> 5) * 8 + (tid & 7);   // rows r0, r0 + 64 (eight loader warps: 64 rows per pass)
    // two slabs of global loads stay in flight (register sets 0 / 1): one slab alone left every stage waiting
    // for HBM/L2 latency longer than its three MMAs take
    float4 va[GTC_INFLIGHT][A_ITERS], vb[GTC_INFLIGHT][B_ITERS];
    auto load_regs = [&](int kb, float4 (&xa)[A_ITERS], float4 (&xb)[B_ITERS]) {
      const int k = kb * GTC_BK + c * 4;
      const bool kin = k < p.K;
#pragma unroll
      for (int i = 0; i < A_ITERS; ++i) {
        const int ra = m0 + r0 + ROWS_PER_PASS * i;
        xa[i] = (kin && ra < p.M) ? __ldg(reinterpret_cast<const float4*>(A + (long long)ra * p.lda + k))
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (!pre) {
#pragma unroll
        for (int i = 0; i < B_ITERS; ++i) {
          const int r = r0 + ROWS_PER_PASS * i, rb = n0 + r;
          xb[i] = (kin && r < BN && rb < p.N) ? __ldg(reinterpret_cast<const float4*>(B + (long long)rb * p.ldb + k))
                                              : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    auto stage_out = [&](int kb, float4 (&xa)[A_ITERS], float4 (&xb)[B_ITERS]) {
      const int s = kb % GTC_STAGES;
      const uint32_t round = (uint32_t)(kb / GTC_STAGES);
      gtc_mbar_wait(empty0 + 8 * s, (round & 1u) ^ 1u, err);
      uint8_t* st = tiles + (size_t)s * STAGE_BYTES;
#pragma unroll
      for (int i = 0; i < A_ITERS; ++i) {
        const int r = r0 + ROWS_PER_PASS * i;
        const uint32_t off = (uint32_t)((r >> 3) * 512 + c * 128 + (r & 7) * 16);
        float4 hi, lo;
        gtc_split4(xa[i], hi, lo);
        *reinterpret_cast<float4*>(st + off) = hi;
        *reinterpret_cast<float4*>(st + GTC_TILE_BYTES + off) = lo;
      }
      if (pre) {
        // the stage's B planes (hi then lo, contiguous in the pre-tiled table) by one bulk copy, off the L1 / LSU path
        if (tid == 0) {
          const uint32_t bar = full0 + 8 * s, bytes = 2u * GTC_BTILE_BYTES(BN);
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(gtc_smem_u32(st + B_OFF)), "l"(Bt + (size_t)kb * (2 * BN * GTC_BK)), "r"(bytes), "r"(bar) : "memory");
        }
      } else {
#pragma unroll
        for (int i = 0; i < B_ITERS; ++i) {
          const int r = r0 + ROWS_PER_PASS * i;
          if (r < BN) {
            const uint32_t off = (uint32_t)((r >> 3) * 512 + c * 128 + (r & 7) * 16);
            float4 hi, lo;
            gtc_split4(xb[i], hi, lo);
            *reinterpret_cast<float4*>(st + B_OFF + off) = hi;
            *reinterpret_cast<float4*>(st + B_OFF + GTC_BTILE_BYTES(BN) + off) = lo;
          }
        }
      }
      if (kb + GTC_INFLIGHT < nkb) load_regs(kb + GTC_INFLIGHT, xa, xb);   // refill this register set GTC_INFLIGHT slabs ahead
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) gtc_mbar_arrive(full0 + 8 * s);
    };
#pragma unroll
    for (int j = 0; j < GTC_INFLIGHT; ++j)
      if (j < nkb) load_regs(j, va[j], vb[j]);
    for (int kb = 0; kb < nkb; kb += GTC_INFLIGHT) {
#pragma unroll
      for (int j = 0; j < GTC_INFLIGHT; ++j)
        if (kb + j < nkb) stage_out(kb + j, va[j], vb[j]);
    }

    // ===== epilogue: TMEM lanes 32 q .. 32 q + 31 (q = warp & 3) are rows m0 + 32 q + lane; the two warps of a lane
    //       quarter take the lower / upper half of the column blocks =====
    gtc_mbar_wait(accum_bar, 0u, err);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int lq = warp & 3;
    const int row = m0 + lq * 32 + lane;
    constexpr int NCB = BN / 16, CB_SPLIT = (NCB + 1) / 2;
    const int cb_lo = (warp < 4) ? 0 : CB_SPLIT, cb_hi = (warp < 4) ? CB_SPLIT : NCB;
    const float* bias = p.bias ? p.bias + (long long)bz * p.sBias : nullptr;
#pragma unroll 1
    for (int cb = cb_lo; cb < cb_hi; ++cb) {
      uint32_t v[16];
      const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(cb * 16);
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
          "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
            "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
          : "r"(taddr)
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (row < p.M) {
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int col = n0 + cb * 16 + j4 * 4;
          if (col >= p.ldc) continue;
          float o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int cc = col + j;
            float x = (nkb > 0) ? __uint_as_float(v[j4 * 4 + j]) : 0.f;
            if (EPI == 0) {
              if (bias && cc < p.N) x += bias[cc];
              if (p.relu) x = fmaxf(x, 0.f);
            } else {
              x = -x;
            }
            o[j] = (cc < p.N) ? x : 0.f;         // pad columns stay zero
          }
          *reinterpret_cast<float4*>(C + (long long)row * p.ldc + col) = make_float4(o[0], o[1], o[2], o[3]);
          if ((EPI == 1 || EPI == 2) && p.closed) {
            const float g = (EPI == 2) ? p.gain_env[row] : p.gain;
            float4* cp = reinterpret_cast<float4*>(p.com + (long long)row * p.ldcom + col);
            float4 c4 = *cp;
            c4.x = fmaf(g, o[0], c4.x); c4.y = fmaf(g, o[1], c4.y);
            c4.z = fmaf(g, o[2], c4.z); c4.w = fmaf(g, o[3], c4.w);
            *cp = c4;
          }
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  } else if (gtc_elect()) {
    // ===== MMA issuer (one elected lane of the last warp) =====
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) |
                           ((uint32_t)(GTC_BM >> 4) << 24);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % GTC_STAGES;
      const uint32_t round = (uint32_t)(kb / GTC_STAGES);
      gtc_mbar_wait(full0 + 8 * s, round & 1u, err);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t base = ((gtc_smem_u32(tiles) + (uint32_t)s * STAGE_BYTES) >> 4) | ((128u >> 4) << 16);
#pragma unroll
      for (int k8 = 0; k8 < GTC_BK / 8; ++k8) {
        const uint32_t ko = (uint32_t)k8 * 16u;                  // two 16-byte chunks = 8 tf32 values
        const uint32_t a_hi = base + ko, a_lo = base + (GTC_TILE_BYTES >> 4) + ko;
        const uint32_t b_hi = base + (B_OFF >> 4) + ko, b_lo = base + ((B_OFF + GTC_BTILE_BYTES(BN)) >> 4) + ko;
        gtc_mma_tf32_lo(tmem_base, a_hi, b_hi, idesc, (kb | k8) ? 1u : 0u);
        gtc_mma_tf32_lo(tmem_base, a_hi, b_lo, idesc, 1u);
        gtc_mma_tf32_lo(tmem_base, a_lo, b_hi, idesc, 1u);
      }
      gtc_commit(empty0 + 8 * s);                                // stage reusable once these MMAs have read it
    }
    gtc_commit(accum_bar);                                       // accumulator complete
  }
  __syncthreads();
  if (warp == GTC_LOADERS) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

#include "gemm_tc_host.h"   // gtc_pretile_host: the pre-split, pre-tiled B operand
