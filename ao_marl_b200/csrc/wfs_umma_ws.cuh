// Shack-Hartmann frame, sixth generation: the tcgen05 pipeline of wfs_umma.cuh with its phases on SPECIALISED warps.
//
// The fifth-generation kernel runs the three phases of a work item (F field, C conversion of the stage-1 accumulator into
// the stage-2 operand, E epilogue) one after the other in every warp.  It is bound by latency, not by issue slots or any
// pipe (profiles/r02_wfs_umma_v5: 16 warps per SM -- the register file holds no more at 128 registers -- each issuing once
// every ~8 cycles; removing 13 % of its instructions bought 2 %).  Here a CTA has 12 warps:
//
//   warps 0-7   field warps: F phase of one subaperture each, A1 operand, arrival on a count-8 mbarrier; the last one to
//               arrive issues MMA 1 into one of TWO stage-1 accumulators (TMEM columns 0..63 / 64..127), so the field of
//               group i+1 never waits for the read-out of group i;
//   warps 8-11  transform warps: TMEM lane quarter q = warp - 8 holds rows (s, y) of subapertures 2q, 2q+1 of the stage-1
//               result -- converted to the MN-major A2 operand -- and the fx rows of subapertures q and 4 + q of the
//               stage-2 result: |.|^2, binning, centre of gravity.  The last of the four to arrive issues MMA 2.
//
// 24 warps per SM instead of 16 with the same shared memory and tensor memory, and the two halves of the work overlap
// instead of alternating.  Each role alone needs fewer registers than the fused loop did: the whole kernel fits the 80
// registers per thread that two 384-thread CTAs per SM leave (no setmaxnreg needed).  Frames with noise or a kept image
// are served by wfs_frame_umma_kernel (the host routes them).
#pragma once
#include "wfs_umma.cuh"

#define WS_THREADS 384
#define WS_MIN_BLOCKS 2                    // two CTAs per SM: 80 registers per thread

template <int NL, int FULL, bool PE = false>     // PE: per-environment winds, as in wfs_frame_umma_kernel
__global__ void __launch_bounds__(WS_THREADS, WS_MIN_BLOCKS) wfs_frame_ws_kernel(const __grid_constant__ WfsUmmaParams P) {
  const WfsParams& p = P.p;
  const WfsUmmaTables& f = P.f;
  constexpr int NLS = NL > 0 ? NL : 1;
  constexpr int AUXB = PE ? WU_AUX_BYTES_PE : WU_AUX_BYTES;
  // barrier block: [0..7] tiles of the field warps, [8], [9] MMA1 done (per accumulator buffer), [10] MMA2 done,
  //                [11] A1 written (8 field warps), [12] A2 written and Y drained (4 transform warps), [13], [14] T buffer
  //                drained (4); the TMEM slot at byte 120
  const WuSmem S = wu_smem_layout<NL, PE>();
  const int lane = wu_lane();
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int y = lane & 15, h = lane >> 4;

  const uint32_t tmem_base = wu_cta_setup(S, f, threadIdx.x, blockDim.x, warp, 15,
                                          threadIdx.x < 11 ? 1u : threadIdx.x == 11 ? (uint32_t)WU_WARPS : 4u, (uint32_t*)(S.bar + 15));

  const uint32_t mma1_bar = wu_smem_u32(S.bar + 8), mma2_bar = wu_smem_u32(S.bar + 10);
  const uint32_t a1_full = wu_smem_u32(S.bar + 11), a2_full = wu_smem_u32(S.bar + 12), t_free = wu_smem_u32(S.bar + 13);
  const uint32_t q_a1 = __shfl_sync(0xffffffffu, wu_smem_u32(S.a1) >> 4, 0), q_b1 = __shfl_sync(0xffffffffu, wu_smem_u32(S.b1) >> 4, 0);
  const uint32_t q_a2 = __shfl_sync(0xffffffffu, wu_smem_u32(S.a2) >> 4, 0), q_b2 = __shfl_sync(0xffffffffu, wu_smem_u32(S.b2) >> 4, 0);

  const long long total = (long long)p.E * p.nvalid;
  const long long base = (long long)blockIdx.x * f.items_per_cta;
  long long end = base + f.items_per_cta;
  if (end > total) end = total;
  const int n_cta = (int)(end - base);                          // > 0 by construction of the grid
  const int n_iter = (n_cta + WU_WARPS - 1) / WU_WARPS;         // groups of 8 work items

  if (warp < WU_WARPS) {
    // =============================== field warps ===============================
    unsigned char* my_tiles = S.tiles + (size_t)warp * NLS * WU_TILE_STRIDE;
    const uint32_t my_tiles_u32 = wu_smem_u32(my_tiles);
    const uint32_t my_bar_u32 = wu_smem_u32(S.bar + warp);
    unsigned char* my_aux = S.aux + (size_t)warp * 2 * AUXB;     // per parity: pm[32] | volts[32] | record
    const uint32_t my_aux_u32 = wu_smem_u32(my_aux);
    const int lane_off = y * WU_TILE_W + 8 * h;                          // floats, inside a tile
    const int amap_lane = (lane >> 2) * f.GW + (lane & 3);
    const int tt_lane = (y + p.tt_off) * p.tt_dim + 8 * h + p.tt_off;    // this lane's first pixel in the tip-tilt support
    const float* const tt_plane1 = p.tt_planes + (size_t)p.tt_dim * p.tt_dim;
    float4 tta[2], ttb[2];
    const float4 fyv = *reinterpret_cast<const float4*>(S.fyT + y * WU_NG);      // y stamp factors of this lane's row (constant)
    // phase in turns: t = phi / lambda - (x + y) / 128   (halfxy = pi (x + y) / 64, geom_init.py:690-701)
    const float kt = p.k2 * 0.15915494309189535f;
    const float hc0 = -(float)(y + 8 * h) * 0.0078125f;
    const wu_f2 hc01 = wu_pk(hc0, hc0 - 0.0078125f);

    // A1 rows of this lane: r = 16 warp + y ; chunks (re, h) (im, h) of the hi tile, the lo tile 8 KB further
    const uint32_t a1_addr = wu_smem_u32(S.a1) + (uint32_t)((2 * warp + (y >> 3)) * 512 + (y & 7) * 16 + h * 128);

    const int n_mine = (n_cta - warp + WU_WARPS - 1) / WU_WARPS;  // work items of this warp: CTA-local indices warp + 8 i
    // (e, k) of the item whose prefetch is issued next; the items in flight are kept packed (e << 16 | k)
    int e = (int)((base + warp) / p.nvalid), k = (int)((base + warp) % p.nvalid);
    int ring_e = -1;
    int rx[NLS], ry[NLS];
    uint32_t tile_phase = 0;
    uint32_t n_d = 0;                                              // tile column offsets of the item whose tiles were issued last
    bool n_seam = false;

    auto issue_tiles = [&](int pe, uint2 sb) {
      wu_issue_tiles<NL, PE>(P, my_tiles_u32, my_bar_u32, lane, pe, sb, ring_e, rx, ry, n_d, n_seam);
    };
    auto issue_aux = [&](int pe, int pk, uint2 sb, int slot, int k_after, bool has_after) {
      wu_issue_aux<NL, PE>(p, f, my_aux, my_aux_u32, S.amap, amap_lane, lane, pe, pk, sb, slot, k_after, has_after);
    };


    // ---- prologue: item 0 entirely, the record of item 1 ----
    if (n_mine > 0) {
      const uint2 sb0 = __ldg(f.sub + k);
      int k1n = k + WU_WARPS;  k1n -= (k1n >= p.nvalid) ? p.nvalid : 0;
      issue_aux(e, k, sb0, 0, k1n, n_mine > 1);
      issue_tiles(e, sb0);
    }
    uint32_t xy_cur = 0, xy_next = 0;            // (y0 << 16 | x0) of the item sampled now / next
    if (n_mine > 0) xy_cur = __ldg(f.sub + k).x;


    for (int it = 0; it < n_iter; ++it) {
      const int s = it & 1;
      const bool c_valid = it < n_mine, nx_valid = it + 1 < n_mine;
      // copies issued one iteration ago: this item's pupil word / volts (/ seam tiles), the next item's record
      asm volatile("cp.async.wait_all;" ::: "memory");
      __syncwarp();
      const uint32_t c_d = n_d;
      const bool c_seam = n_seam;

      uint32_t re_h[4], re_l[4], im_h[4], im_l[4];
      wu_f2 P[4];
      uint32_t c_pm = 0u;
      if (c_valid) {
        c_pm = *reinterpret_cast<const uint32_t*>(my_aux + s * AUXB + 4 * lane);
        const float* V = reinterpret_cast<const float*>(my_aux + s * AUXB + 128);
        // this item's mirror inputs are requested before the bookkeeping of the next item (which is full of memory-
        // clobbering copies the compiler cannot move loads across), so that their latency is covered by it
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1r = v0, v2r = v0, v3 = v0;
        float vt0 = 0.f, vt1 = 0.f;
        if (p.use_dm) {
          wu_load_tt(p, tt_plane1, tt_lane, xy_cur, tta, ttb);
          v0 = *reinterpret_cast<const float4*>(V); v1r = *reinterpret_cast<const float4*>(V + 4);
          v2r = *reinterpret_cast<const float4*>(V + 8); v3 = *reinterpret_cast<const float4*>(V + 12);
          vt0 = V[16]; vt1 = V[17];
        }
        // ---- next work item of this warp: record (fetched during the previous iteration), per-lane inputs now,
        //      tiles as soon as the current ones are sampled ----
        uint2 sb1 = make_uint2(0u, 0u);
        if (nx_valid) {
          sb1 = *reinterpret_cast<const uint2*>(my_aux + (s ^ 1) * AUXB + 256);
          sb1.x = __shfl_sync(0xffffffffu, sb1.x, 0); sb1.y = __shfl_sync(0xffffffffu, sb1.y, 0);
          k += WU_WARPS;
          if (k >= p.nvalid) { k -= p.nvalid; e += 1; }
          int k2n = k + WU_WARPS;  k2n -= (k2n >= p.nvalid) ? p.nvalid : 0;
          issue_aux(e, k, sb1, s ^ 1, k2n, it + 2 < n_mine);
          xy_next = sb1.x;
        }

        // ---- mirrors first (they need only the per-lane inputs that arrived by cp.async): the tip-tilt table loads are
        //      requested at once and consumed after the stamp arithmetic, and the tiles of the atmosphere get the whole
        //      section to land ----
        if (p.use_dm) {
          wu_mirror(v0, v1r, v2r, v3, vt0, vt1, fyv, S.fx, h, tta, ttb, P);
        } else {
        #pragma unroll
          for (int j = 0; j < 4; ++j) P[j] = 0ull;
        }

        // ---- atmosphere, on top of the mirror surface ----
        if (NL > 0) {
          WuPhase acc;
  #pragma unroll
          for (int j = 0; j < 4; ++j) acc.X[j] = P[j];
  #pragma unroll
          for (int j = 0; j < 3; ++j) acc.Y[j] = 0ull;
          acc.y0 = acc.y7 = 0.f;
          if (!c_seam) {
            wu_mbar_wait(my_bar_u32, tile_phase, f.err);
            tile_phase ^= 1u;
          }
          wu_layers<NL, PE>(my_tiles, lane_off, my_aux + s * AUXB + WU_AUX_BYTES, p, c_d, acc);
          __syncwarp();                                   // the stage is drained: re-arm it with the next item
          if (nx_valid) issue_tiles(e, sb1);
          wu_fold(acc, P);
        }

      }

      if (c_valid) {
        wu_field(P, c_pm, kt, hc01, re_h, re_l, im_h, im_l);
      }


      // A1 is free once MMA 1 of the previous group has completed
      if (it > 0) wu_mbar_wait(mma1_bar + 8u * ((it - 1) & 1), (uint32_t)(((it - 1) >> 1) & 1), f.err);
      if (c_valid) {
        wu_store_a1(a1_addr, re_h, re_l, im_h, im_l);
      }

      // ---- arrival; the last field warp issues MMA 1 of this group into accumulator buffer it & 1 ----
      if (wu_arrive(a1_full, lane, false)) {
        // the buffer was read out by the transform warps two groups ago
        if (it >= 2) wu_mbar_wait(t_free + 8u * (it & 1), (uint32_t)(((it - 2) >> 1) & 1), f.err);
        if (wu_elect_acquire(a1_full, (uint32_t)(it & 1), f.err)) {
          wu_issue_mma1(tmem_base + 64u * (uint32_t)(it & 1), q_a1, q_b1);
          wu_commit(mma1_bar + 8u * (it & 1));
        }
      }
      __syncwarp();
      xy_cur = xy_next;
    }
  } else {
    // =============================== transform warps ===============================
    const int q = warp - WU_WARPS;                                 // TMEM lane quarter
    // conversion: rows 32 q .. of the stage-1 result = subapertures 2 q + h; A2 tile q >> 1, rows m = 32 s' + fx with
    // s' = 2 (q & 1) + h, K index 16 ro + y (ro = 0: T_re columns 0..31, ro = 1: T_im columns 32..63)
    const uint32_t d1_addr = tmem_base + ((uint32_t)(32 * q) << 16);
    const uint32_t a2_addr = wu_smem_u32(S.a2) + (uint32_t)((q >> 1) * 2 * WU_A_BYTES + (4 * (2 * (q & 1) + h)) * 512 +
                                                           (y >> 3) * 128 + (y & 7) * 16);
    // epilogue: the fx rows of subaperture q (tile 0) and 4 + q (tile 1)
    const uint32_t d2_addr = tmem_base + ((uint32_t)(32 * q) << 16) + 128u;
    // (e, k) of the two subapertures of the group in the epilogue
    int ee[2], kk[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      ee[t] = (int)((base + 4 * t + q) / p.nvalid);
      kk[t] = (int)((base + 4 * t + q) % p.nvalid);
    }
    // This kernel serves frames without noise and without a kept image (the host routes the others to
    // wfs_frame_umma_kernel): the epilogue is the plain path of wu_sq_plain.
    // lane = kept fx index; fx pair lane >> 1 -> px
    const float pxf = (float)(((lane >> 1) < 8) ? 8 + (lane >> 1) : (lane >> 1) - 8);
    auto epilogue = [&](wu_f2 s0p, wu_f2 syp, int ie, int ik) {
      float a, b;
      wu_upk(s0p, a, b); float s0 = a + b;
      wu_upk(syp, a, b); float sy = a + b;
      float sx = s0 * pxf;
      wu_cog_store(p, lane, s0, sx, sy, ie, ik);
    };

    for (int j = 0; j <= n_iter; ++j) {
      const bool conv = j < n_iter, epi = j > 0;
      uint32_t tv[32];
      if (conv) {
        wu_mbar_wait(mma1_bar + 8u * (j & 1), (uint32_t)((j >> 1) & 1), f.err);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        wu_tmem_ld32(d1_addr + 64u * (uint32_t)(j & 1), tv);
      }
      // stage 2 of the previous group is complete: A2 reusable, Y(j-1) in TMEM
      if (epi) wu_mbar_wait(mma2_bar, (uint32_t)((j - 1) & 1), f.err);
      if (conv) {
#pragma unroll
        for (int ro = 0; ro < 2; ++ro) {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (ro == 1) {
            // both halves are in registers: the accumulator buffer may be overwritten (by MMA 1 of group j + 2)
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(t_free + 8u * (j & 1)) : "memory");
          }
          wu_store_a2<FULL>(a2_addr, ro * 256, tv);
          if (ro == 0) wu_tmem_ld32(d1_addr + 64u * (uint32_t)(j & 1) + 32u, tv);
        }
      }

      // ---- read-out of Y(j-1): both subapertures of this lane quarter, before MMA 2 of group j overwrites them ----
      wu_f2 s0p[2] = {0ull, 0ull}, syp[2] = {0ull, 0ull};
      if (epi) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          uint32_t yv[32];
          wu_tmem_ld32(d2_addr + 64u * t, yv);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          wu_sq_plain(yv, 8.f, s0p[t], syp[t], true);
          wu_tmem_ld32(d2_addr + 64u * t + 32u, yv);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          wu_sq_plain(yv, 0.f, s0p[t], syp[t], false);
        }
      }
      if (conv) {
        // ---- arrival (A2 written, Y drained); the last transform warp issues MMA 2 of group j ----
        if (wu_arrive(a2_full, lane, true) && wu_elect_acquire(a2_full, (uint32_t)(j & 1), f.err)) {
          wu_issue_mma2<FULL>(tmem_base + 128u, q_a2, q_b2);
          wu_commit(mma2_bar);
        }
        __syncwarp();
      }
      if (epi) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          if (8 * (j - 1) + 4 * t + q < n_cta) epilogue(s0p[t], syp[t], ee[t], kk[t]);
          kk[t] += WU_WARPS;
          if (kk[t] >= p.nvalid) { kk[t] -= p.nvalid; ee[t] += 1; }
        }
      }
    }
  }

  wu_cta_release(warp, tmem_base);
}
