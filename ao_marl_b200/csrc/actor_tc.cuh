// The batched actor forward in one tcgen05 kernel: gather of the agent's inputs from the state rows, three layers
// (relu(W1 x + b1), relu(W2 h + b2), heads) and the Gaussian-policy sampling, per 128-environment tile of one agent.
//
// The arithmetic is that of gemm_tc_kernel (gemm_tc.cuh) layer by layer: operands split into TF32 hi / lo, per k block of
// 16 and per k8 the products hi.hi, hi.lo, lo.hi into a float32 TMEM accumulator, the weights taken from the same
// pre-tiled planes (gtc_pretile_host), bias / relu / zeroed pad columns in the epilogue.  What changes is where the
// operands live: the activations never leave the SM, and no intermediate goes through HBM.
//
// TMEM (512 columns, one CTA per SM): H1 in columns 0-255, H2 in 256-511, the heads in 0-255 again once H1 has been read.
// Shared memory: ATC_STAGES stages of [A hi, A lo (128 x 16 each), B hi, B lo (up to 256 x 16 each)], then the
// barriers and the agent's input index row.  Per stage the A slab is written by the eight loader warps (layer 1: gathered
// from the state; layers 2 and 3: read from the previous layer's accumulator) and B arrives by bulk copies.
//
//   warps 0-7  loaders / epilogue: TMEM lane quarter warp & 3, the two warps of a quarter take half of each k block;
//              after the heads: bias, then sampling of the actions (actor_sample_kernel's arithmetic).
//   warp 8     TMEM allocation; one lane issues the MMAs and commits stages and accumulators.
//   warp 9     one lane issues the weight copies, running ahead of the loaders by up to ATC_STAGES stages.
// Every mbarrier wait is bounded (gtc_mbar_wait): on expiry the error word is raised and the kernel traps.
//
// PE (per-environment controllers, aom_set_controller_env): the CTA runs tile blockIdx.x of the tile list
// (ctrl_tiles_host.h): its rows are the environments tile_env[tile][0..128) (-1: padding, read as zero and not sampled),
// and the weights and biases are those of the tile's policy slot.  Row by row the arithmetic is that of the uniform form.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gemm_host.h"
#include "gemm_tc.cuh"
#include "rng.cuh"

#define ATC_STAGES 4
#define ATC_A_BYTES (2 * GTC_TILE_BYTES)                     // A hi, A lo: 16 KB
#define ATC_B_LO (2 * GTC_BTILE_BYTES(GTC_BN))               // B hi of up to 256 rows (two 128-column tiles), then B lo
#define ATC_STAGE_BYTES (ATC_A_BYTES + 2 * ATC_B_LO)         // 48 KB
#define ATC_BAR_BYTES 256
#define ATC_SMEM_BYTES(ld_in) (ATC_STAGES * ATC_STAGE_BYTES + ATC_BAR_BYTES + 4 * (ld_in))
#define ATC_MMA_WARP GTC_LOADERS
#define ATC_COPY_WARP (GTC_LOADERS + 1)
#define ATC_THREADS ((GTC_LOADERS + 2) * 32)
#define ATC_H2_COL 256u

// Weights (pre-tiled planes) and biases of layer l: those of the tile's policy slot in the per-environment form
template <bool PE>
__device__ __forceinline__ const float* atc_w(const ActorArgs<PE>& p, int slot, int l) {
  if constexpr (PE) return p.ws[slot][l]; else return p.w[l];
}
template <bool PE>
__device__ __forceinline__ const float* atc_bias(const ActorArgs<PE>& p, int slot, int l) {
  if constexpr (PE) return p.bs[slot][l]; else return p.bias[l];
}

// grid (E tiles of 128, agents), PE: (tiles of the tile list, agents)
template <bool PE>
__global__ void __launch_bounds__(ATC_THREADS, 1) actor_fused_kernel(const __grid_constant__ ActorArgs<PE> p, int* err) {
  extern __shared__ __align__(1024) uint8_t atc_smem[];
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = tid & 31;
  const int a = blockIdx.y, m0 = blockIdx.x * GTC_BM;
  const int nkb1 = p.nkb_in, nkb2 = p.nkb_h;
  const int nst = nkb1 + 2 * nkb2;                            // stages of the three layers, one ring
  int slot = 0;                                               // PE: the tile's policy slot
  if constexpr (PE) slot = __ldg(p.tile_slot + blockIdx.x);

  uint8_t* ring = atc_smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(atc_smem + ATC_STAGES * ATC_STAGE_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * ATC_STAGES + 3);
  int* idx_s = reinterpret_cast<int*>(atc_smem + ATC_STAGES * ATC_STAGE_BYTES + ATC_BAR_BYTES);
  const uint32_t full0 = gtc_smem_u32(bars), empty0 = full0 + 8 * ATC_STAGES, acc0 = empty0 + 8 * ATC_STAGES;

  // the agent's input row: -1 (no input) and k >= actor_in read as 0
  for (int k = tid; k < nkb1 * GTC_BK; k += ATC_THREADS)
    idx_s[k] = k < p.actor_in ? __ldg(p.idx + (size_t)a * p.actor_in + k) : -1;
  if (tid == 0) {
    for (int s = 0; s < ATC_STAGES; ++s) {
      gtc_mbar_init(full0 + 8 * s, GTC_LOADERS + 1);        // one arrive per loader warp + the copies' expect_tx
      gtc_mbar_init(empty0 + 8 * s, 1);                     // tcgen05.commit
    }
    for (int l = 0; l < 3; ++l) gtc_mbar_init(acc0 + 8 * l, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == ATC_MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(gtc_smem_u32(tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp < GTC_LOADERS) {
    // ===== layer 1: A = state[e][idx[k]], gathered straight into the stage (the mapping of gemm_tc_kernel's loaders:
    //       eight lanes per 16-byte chunk of eight consecutive rows, conflict-free st.shared) =====
    {
      const int c = (tid >> 3) & 3;
      const int r0 = (tid >> 5) * 8 + (tid & 7);
      int env_r[2];                                           // PE: the environments of rows r0, r0 + 64
      if constexpr (PE)
        for (int i = 0; i < 2; ++i) env_r[i] = __ldg(p.tile_env + (size_t)blockIdx.x * GTC_BM + r0 + 64 * i);
      float4 va[GTC_INFLIGHT][2];
      auto load_regs = [&](int kb, float4 (&x)[2]) {
        const int k = kb * GTC_BK + c * 4;
        const int s0 = idx_s[k], s1 = idx_s[k + 1], s2 = idx_s[k + 2], s3 = idx_s[k + 3];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          int e;
          bool in;
          if constexpr (PE) { e = env_r[i]; in = e >= 0; } else { e = m0 + r0 + 64 * i; in = e < p.E; }
          const float* srow = p.state + (size_t)e * p.ldst;
          x[i].x = (in && s0 >= 0) ? __ldg(srow + s0) : 0.f;
          x[i].y = (in && s1 >= 0) ? __ldg(srow + s1) : 0.f;
          x[i].z = (in && s2 >= 0) ? __ldg(srow + s2) : 0.f;
          x[i].w = (in && s3 >= 0) ? __ldg(srow + s3) : 0.f;
        }
      };
      auto stage_out = [&](int kb, float4 (&x)[2]) {
        const int s = kb % ATC_STAGES;
        gtc_mbar_wait(empty0 + 8 * s, ((uint32_t)(kb / ATC_STAGES) & 1u) ^ 1u, err);
        uint8_t* st = ring + (size_t)s * ATC_STAGE_BYTES;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int r = r0 + 64 * i;
          const uint32_t off = (uint32_t)((r >> 3) * 512 + c * 128 + (r & 7) * 16);
          float4 hi, lo;
          gtc_split4(x[i], hi, lo);
          *reinterpret_cast<float4*>(st + off) = hi;
          *reinterpret_cast<float4*>(st + GTC_TILE_BYTES + off) = lo;
        }
        if (kb + GTC_INFLIGHT < nkb1) load_regs(kb + GTC_INFLIGHT, x);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) gtc_mbar_arrive(full0 + 8 * s);
      };
#pragma unroll
      for (int j = 0; j < GTC_INFLIGHT; ++j)
        if (j < nkb1) load_regs(j, va[j]);
      for (int kb = 0; kb < nkb1; kb += GTC_INFLIGHT) {
#pragma unroll
        for (int j = 0; j < GTC_INFLIGHT; ++j)
          if (kb + j < nkb1) stage_out(kb + j, va[j]);
      }
    }

    // ===== layers 2 and 3: A = relu(acc + bias), pad columns zero, read from TMEM one k block at a time: row
    //       32 lq + lane, columns 8 half .. 8 half + 7 of the block (chunks 2 half, 2 half + 1) =====
    const int lq = warp & 3, half = warp >> 2;
    const int r = lq * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lq * 32) << 16);
#pragma unroll 1
    for (int l = 1; l < 3; ++l) {
      const float* __restrict__ bias = atc_bias<PE>(p, slot, l - 1) + (size_t)a * p.hidden;
      const uint32_t src = lane_addr + (l == 1 ? 0u : ATC_H2_COL);
      gtc_mbar_wait(acc0 + 8 * (l - 1), 0u, err);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
      for (int kb = 0; kb < nkb2; ++kb) {
        const int g = nkb1 + (l - 1) * nkb2 + kb, s = g % ATC_STAGES;
        const int col = kb * GTC_BK + half * 8;
        uint32_t v[8];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                     : "r"(src + (uint32_t)col)
                     : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int cc = col + j;
          float x = __uint_as_float(v[j]);
          if (cc < p.hidden) x += __ldg(bias + cc);
          x = fmaxf(x, 0.f);
          o[j] = cc < p.hidden ? x : 0.f;
        }
        gtc_mbar_wait(empty0 + 8 * s, ((uint32_t)(g / ATC_STAGES) & 1u) ^ 1u, err);
        uint8_t* st = ring + (size_t)s * ATC_STAGE_BYTES;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const uint32_t off = (uint32_t)((r >> 3) * 512 + (half * 2 + q) * 128 + (r & 7) * 16);
          float4 hi, lo;
          gtc_split4(make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]), hi, lo);
          *reinterpret_cast<float4*>(st + off) = hi;
          *reinterpret_cast<float4*>(st + GTC_TILE_BYTES + off) = lo;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // H1 read before the heads overwrite it
        __syncwarp();
        if (lane == 0) gtc_mbar_arrive(full0 + 8 * s);
      }
    }

    // ===== heads: acc + bias into a row-major scratch in the (now idle) stage ring, then one thread per environment
    //       row and Philox block samples the actions =====
    gtc_mbar_wait(acc0 + 16, 0u, err);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    float* hs = reinterpret_cast<float*>(ring);
    const int hp = p.ldh + 1;                                 // odd pitch: lanes (rows) on distinct banks
    const float* __restrict__ bias_h = atc_bias<PE>(p, slot, 2) + (size_t)a * p.heads;
    const int ncb = p.ldh / 16, cb_split = (ncb + 1) / 2;
#pragma unroll 1
    for (int cb = half ? cb_split : 0; cb < (half ? ncb : cb_split); ++cb) {
      uint32_t v[16];
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
          "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
            "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
          : "r"(lane_addr + (uint32_t)(cb * 16))
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int cc = cb * 16 + j;
        if (cc < p.heads) hs[r * hp + cc] = __uint_as_float(v[j]) + __ldg(bias_h + cc);
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.sync 1, %0;" ::"r"(GTC_LOADERS * 32) : "memory");
    const int out = p.actor_out, nb = (out + 3) >> 2;
#pragma unroll 1
    for (int t = tid; t < GTC_BM * nb; t += GTC_LOADERS * 32) {
      const int rr = t / nb, jb = t - rr * nb;
      int e;
      if constexpr (PE) {
        e = __ldg(p.tile_env + (size_t)blockIdx.x * GTC_BM + rr);
        if (e < 0) continue;
      } else {
        e = m0 + rr;
        if (e >= p.E) continue;
      }
      const uint32_t step = p.step_env ? p.step_env[e] : p.step;
      const aom_u4 w = aom_philox((uint32_t)jb, step, AOM_TAG_ACTOR, (uint32_t)a, p.k0[e], p.k1[e]);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = jb * 4 + q;
        if (j >= out) break;
        const int slot = __ldg(p.act_slot + (size_t)a * out + j);
        if (slot < 0) continue;
        const float mu = hs[rr * hp + j];
        const float ls = fminf(fmaxf(hs[rr * hp + out + j], p.log_sig_min), p.log_sig_max);
        const float eps = aom_normal_of_block(w, q);
        const float act = tanhf(mu + expf(ls) * eps) * p.act_scale + p.act_bias;
        const float mean = tanhf(mu) * p.act_scale + p.act_bias;
        p.action[(size_t)e * p.lda + slot] = p.eval_mode ? mean : act;
        p.action_mean[(size_t)e * p.lda + slot] = mean;
      }
    }
  } else if (warp == ATC_MMA_WARP) {
    if (gtc_elect()) {
      // ===== MMA issuer: one MMA over every column of the layer (N = 256 for two 128-column tiles: the operand A is read
      //       from shared memory once per k8 instead of once per tile); per accumulator the order of gemm_tc_kernel, k blocks
      //       ascending and per k8 hi.hi, hi.lo, lo.hi =====
      int g = 0;
#pragma unroll 1
      for (int l = 0; l < 3; ++l) {
        const int nkb = l == 0 ? nkb1 : nkb2, n = l == 2 ? p.ldh : GTC_BN * p.nt_hidden;
        const uint32_t d = tmem_base + (l == 1 ? ATC_H2_COL : 0u);
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(GTC_BM >> 4) << 24);
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb, ++g) {
          const int s = g % ATC_STAGES;
          gtc_mbar_wait(full0 + 8 * s, (uint32_t)(g / ATC_STAGES) & 1u, err);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t base = ((gtc_smem_u32(ring) + (uint32_t)s * ATC_STAGE_BYTES) >> 4) | ((128u >> 4) << 16);
          const uint32_t b_hi = base + (ATC_A_BYTES >> 4), b_lo = b_hi + (ATC_B_LO >> 4);
#pragma unroll
          for (int k8 = 0; k8 < GTC_BK / 8; ++k8) {
            const uint32_t ko = (uint32_t)k8 * 16u;
            const uint32_t a_hi = base + ko, a_lo = base + (GTC_TILE_BYTES >> 4) + ko;
            gtc_mma_tf32_lo(d, a_hi, b_hi + ko, idesc, (kb | k8) ? 1u : 0u);
            gtc_mma_tf32_lo(d, a_hi, b_lo + ko, idesc, 1u);
            gtc_mma_tf32_lo(d, a_lo, b_hi + ko, idesc, 1u);
          }
          gtc_commit(empty0 + 8 * s);
        }
        gtc_commit(acc0 + 8 * l);
      }
    }
  } else if (gtc_elect()) {
    // ===== weight copies: [n tile][k block][hi, lo][128 x 16] per agent.  Tile t's hi plane lands at rows 128 t of the
    //       stage's B hi operand, its lo plane at rows 128 t of B lo (8-row groups 512 B apart: one operand of up to 256
    //       rows each); a head tile narrower than 128 columns takes only its rows (the first n x 64 bytes of each plane) =====
#pragma unroll 1
    for (int g = 0; g < nst; ++g) {
      const int l = g < nkb1 ? 0 : g < nkb1 + nkb2 ? 1 : 2;
      const int kb = l == 0 ? g : l == 1 ? g - nkb1 : g - nkb1 - nkb2, nkb = l == 0 ? nkb1 : nkb2;
      const int nt = l == 2 ? p.nt_heads : p.nt_hidden, s = g % ATC_STAGES;
      const int cols = l == 2 ? p.ldh : GTC_BN * p.nt_hidden;
      gtc_mbar_wait(empty0 + 8 * s, ((uint32_t)(g / ATC_STAGES) & 1u) ^ 1u, err);
      const uint32_t bar = full0 + 8 * s;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2u * (uint32_t)cols * GTC_BK * 4u) : "memory");
      const uint32_t dst = gtc_smem_u32(ring + (size_t)s * ATC_STAGE_BYTES + ATC_A_BYTES);
      for (int t = 0; t < nt; ++t) {
        const float* src = atc_w<PE>(p, slot, l) + (size_t)a * p.w_per[l] + (size_t)(t * nkb + kb) * (2 * GTC_BN * GTC_BK);
        const uint32_t n = (uint32_t)min(GTC_BN, cols - GTC_BN * t) * GTC_BK * 4u;
        const uint32_t d = dst + (uint32_t)(t * GTC_BTILE_BYTES(GTC_BN));
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(d), "l"(src), "r"(n), "r"(bar) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(d + (uint32_t)ATC_B_LO), "l"(src + GTC_BN * GTC_BK), "r"(n), "r"(bar) : "memory");
      }
    }
  }
  __syncthreads();
  if (warp == ATC_MMA_WARP) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}
