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
  extern __shared__ __align__(1024) unsigned char wu_smem_raw[];
  constexpr int NLS = NL > 0 ? NL : 1;
  constexpr int AUXB = PE ? WU_AUX_BYTES_PE : WU_AUX_BYTES;
  unsigned char* s_a1 = wu_smem_raw;                                   // [hi, lo][WU_A_BYTES]
  unsigned char* s_a2 = s_a1 + 2 * WU_A_BYTES;                         // [tile][hi, lo][WU_A_BYTES]
  unsigned char* s_b1 = s_a2 + 4 * WU_A_BYTES;                         // [hi, lo][WU_B_BYTES]
  unsigned char* s_b2 = s_b1 + 2 * WU_B_BYTES;
  unsigned char* s_tiles = s_b2 + 2 * WU_B_BYTES;                      // [warp][layer][WU_TILE_STRIDE]
  // barriers: [0..7] tiles of the field warps, [8], [9] MMA1 done (per accumulator buffer), [10] MMA2 done,
  //           [11] A1 written (8 field warps), [12] A2 written and Y drained (4 transform warps), [13], [14] T buffer drained (4)
  uint64_t* s_bar = (uint64_t*)(s_tiles + (size_t)WU_WARPS * NLS * WU_TILE_STRIDE);
  uint32_t* s_cnt = (uint32_t*)(s_bar + 15) - 2;                       // [2] TMEM slot (the last 4 bytes before byte 128)
  float* s_fx = (float*)((unsigned char*)s_bar + 128);                 // [NG][16]
  float* s_fyT = s_fx + WU_NG * 16;                                    // [16][NG]
  unsigned char* s_aux = (unsigned char*)(s_fyT + 16 * WU_NG);         // [warp][parity][AUXB]
  short* s_amap = (short*)(s_aux + WU_WARPS * 2 * AUXB);

  // lane through a volatile read: the compiler otherwise re-derives it from S2R SR_TID.X at ~25 places of the loop body
  // and each of those reads stalls its warp (5 % of the stall samples in profiles/r02_wfs_umma_v5)
  int lane;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int y = lane & 15, h = lane >> 4;

  for (int i = threadIdx.x; i < 2 * WU_B_BYTES / 16; i += blockDim.x) {
    reinterpret_cast<uint4*>(s_b1)[i] = f.b1[i];
    reinterpret_cast<uint4*>(s_b2)[i] = f.b2[i];
  }
  for (int i = threadIdx.x; i < 2 * WU_NG * 16; i += blockDim.x) s_fx[i] = f.fxy[i];
  for (int i = threadIdx.x; i < f.GW * f.GW; i += blockDim.x) s_amap[i] = f.amap[i];
  // operand tiles start from zeros: rows of work items that do not exist are multiplied too
  for (int i = threadIdx.x; i < 6 * WU_A_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4*>(s_a1)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (threadIdx.x < 15)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(wu_smem_u32(s_bar + threadIdx.x)),
                 "r"(threadIdx.x < 11 ? 1u : threadIdx.x == 11 ? (uint32_t)WU_WARPS : 4u) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // B tiles / zeroed A tiles are read by the tensor core
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(wu_smem_u32(s_cnt + 2)), "r"((uint32_t)WU_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, s_cnt[2], 0);

  const uint32_t mma1_bar = wu_smem_u32(s_bar + 8), mma2_bar = wu_smem_u32(s_bar + 10);
  const uint32_t a1_full = wu_smem_u32(s_bar + 11), a2_full = wu_smem_u32(s_bar + 12), t_free = wu_smem_u32(s_bar + 13);
  const uint32_t idesc1 = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // f16 x f16 -> f32, K-major A and B
  const uint32_t idesc2 = idesc1 | (1u << 15);                                                      // A operand MN-major
  const uint32_t q_a1 = __shfl_sync(0xffffffffu, wu_smem_u32(s_a1) >> 4, 0), q_b1 = __shfl_sync(0xffffffffu, wu_smem_u32(s_b1) >> 4, 0);
  const uint32_t q_a2 = __shfl_sync(0xffffffffu, wu_smem_u32(s_a2) >> 4, 0), q_b2 = __shfl_sync(0xffffffffu, wu_smem_u32(s_b2) >> 4, 0);

  const long long total = (long long)p.E * p.nvalid;
  const long long base = (long long)blockIdx.x * f.items_per_cta;
  long long end = base + f.items_per_cta;
  if (end > total) end = total;
  const int n_cta = (int)(end - base);                          // > 0 by construction of the grid
  const int n_iter = (n_cta + WU_WARPS - 1) / WU_WARPS;         // groups of 8 work items

  if (warp < WU_WARPS) {
    // =============================== field warps ===============================
    unsigned char* my_tiles = s_tiles + (size_t)warp * NLS * WU_TILE_STRIDE;
    const uint32_t my_tiles_u32 = wu_smem_u32(my_tiles);
    const uint32_t my_bar_u32 = wu_smem_u32(s_bar + warp);
    unsigned char* my_aux = s_aux + (size_t)warp * 2 * AUXB;     // per parity: pm[32] | volts[32] | record
    const uint32_t my_aux_u32 = wu_smem_u32(my_aux);
    const int lane_off = y * WU_TILE_W + 8 * h;                          // floats, inside a tile
    const int amap_lane = (lane >> 2) * f.GW + (lane & 3);
    const int tt_lane = (y + p.tt_off) * p.tt_dim + 8 * h + p.tt_off;    // this lane's first pixel in the tip-tilt support
    const float* const tt_plane1 = p.tt_planes + (size_t)p.tt_dim * p.tt_dim;
    // The tip-tilt planes are tables (the reference's Zernike 2 / 3 are evaluated in float32 with offset centres,
    // dm_init.py:661-694 -> dm_util.py:300-380: up to 1.5 % away from a plane).  The 2 x 8 values of a lane are requested
    // at the top of the item and used after the atmosphere has been sampled (the layers are sampled one at a time so
    // that these 16 registers survive without a spill: a spill right behind the loads would wait for them).
    float4 tta[2], ttb[2];
    auto load_tta = [&](uint32_t xy) {       // first plane: requested at the top of the item
      const int to = (int)(xy >> 16) * p.tt_dim + (int)(xy & 0xffffu) + tt_lane;
      tta[0] = __ldg(reinterpret_cast<const float4*>(p.tt_planes + to));
      tta[1] = __ldg(reinterpret_cast<const float4*>(p.tt_planes + to + 4));
    };
    auto load_ttb = [&](uint32_t xy) {       // second plane: requested once the tile windows have left the registers
      const int to = (int)(xy >> 16) * p.tt_dim + (int)(xy & 0xffffu) + tt_lane;
      ttb[0] = __ldg(reinterpret_cast<const float4*>(tt_plane1 + to));
      ttb[1] = __ldg(reinterpret_cast<const float4*>(tt_plane1 + to + 4));
    };
    const float4 fyv = *reinterpret_cast<const float4*>(s_fyT + y * WU_NG);      // y stamp factors of this lane's row (constant)
    // phase in turns: t = phi / lambda - (x + y) / 128   (halfxy = pi (x + y) / 64, geom_init.py:690-701)
    const float kt = p.k2 * 0.15915494309189535f;
    const float hc0 = -(float)(y + 8 * h) * 0.0078125f;
    const wu_f2 hc01 = wu_pk(hc0, hc0 - 0.0078125f);

    // A1 rows of this lane: r = 16 warp + y ; chunks (re, h) (im, h) of the hi tile, the lo tile 8 KB further
    const uint32_t a1_addr = wu_smem_u32(s_a1) + (uint32_t)((2 * warp + (y >> 3)) * 512 + (y & 7) * 16 + h * 128);

    const int n_mine = (n_cta - warp + WU_WARPS - 1) / WU_WARPS;  // work items of this warp: CTA-local indices warp + 8 i
    // (e, k) of the item whose prefetch is issued next; the items in flight are kept packed (e << 16 | k)
    int e = (int)((base + warp) / p.nvalid), k = (int)((base + warp) % p.nvalid);
    int ring_e = -1;
    int rx[NLS], ry[NLS];
    uint32_t tile_phase = 0;
    uint32_t n_d = 0;                                              // tile column offsets of the item whose tiles were issued last
    bool n_seam = false;

    // ---- tiles of one work item (record sb): TMA boxes, or element-wise wrapped cp.async copies on the torus seam ----
    auto issue_tiles = [&](int pe, uint2 sb) {
      if (NL == 0) return;
      if (pe != ring_e) {
  #pragma unroll
        for (int l = 0; l < NL; ++l) {
          const int N = p.layer[l].N;
          int a = (PE ? __ldg(&p.wind[(size_t)l * p.E + pe].ix) : p.layer[l].ix) + p.layer[l].ox[pe];  a -= (a >= N) ? N : 0;
          int b = (PE ? __ldg(&p.wind[(size_t)l * p.E + pe].iy) : p.layer[l].iy) + p.layer[l].oy[pe];  b -= (b >= N) ? N : 0;
          rx[l] = a; ry[l] = b;
        }
        ring_e = pe;
      }
      const int x0 = (int)(sb.x & 0xffffu), y0 = (int)(sb.x >> 16);
      int tc[NLS], tr[NLS];
      bool seam = false;
      uint32_t dbits = 0;
  #pragma unroll
      for (int l = 0; l < NL; ++l) {
        const int N = p.layer[l].N;
        int c = x0 + rx[l];  c -= (c >= N) ? N : 0;
        int r = y0 + ry[l];  r -= (r >= N) ? N : 0;
        tc[l] = c & ~3; tr[l] = r;
        dbits |= (uint32_t)(c & 3) << (2 * l);
        seam |= (c + WU_TILE_H > N) | (r + WU_TILE_H > N);
      }
      n_seam = seam;
      n_d = dbits;
      if (!seam) {
        // the stage was read with plain loads: order them before the async-proxy writes of the new boxes
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (wu_elect()) {       // elect.sync: a warp-uniform issue path (no per-thread waterfall around the TMA instructions)
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(my_bar_u32), "r"(NL * WU_TILE_BYTES) : "memory");
  #pragma unroll
          for (int l = 0; l < NL; ++l)
            wu_tma_load_3d(my_tiles_u32 + l * WU_TILE_STRIDE, &P.maps[l], tc[l], tr[l], pe, my_bar_u32);
        }
      } else {
        // (rare path: keep its per-lane index arithmetic here instead of in registers that live across the whole loop)
        int ln = lane;
        asm volatile("" : "+r"(ln));
  #pragma unroll
        for (int l = 0; l < NL; ++l) {
          const int N = p.layer[l].N;
          const float* scr = p.layer[l].screen + (size_t)pe * N * N;
          const int c0 = tc[l] + (int)((dbits >> (2 * l)) & 3u), r0 = tr[l];
          const uint32_t dst0 = my_tiles_u32 + l * WU_TILE_STRIDE + ((dbits >> (2 * l)) & 3u) * 4u;
  #pragma unroll 1
          for (int i0 = 0; i0 < WU_TILE_H * WU_TILE_H; i0 += 32) {
            const int i = i0 + ln;
            if (i < WU_TILE_H * WU_TILE_H) {
              const int r = i / WU_TILE_H, c = i - r * WU_TILE_H;
              int rr = r0 + r;  rr -= (rr >= N) ? N : 0;
              int cc = c0 + c;  cc -= (cc >= N) ? N : 0;
              wu_cp_async4(dst0 + (uint32_t)(r * WU_TILE_W + c) * 4u, scr + (size_t)rr * N + cc);
            }
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      }
    };

    // ---- per-lane inputs of one work item into the parity slot: pupil word, neighbourhood volts (cp.async: no register
    //      waits for them), and the record of the item after it ----
    auto issue_aux = [&](int pe, int pk, uint2 sb, int slot, int k_after, bool has_after) {
      const uint32_t dst = my_aux_u32 + (uint32_t)slot * AUXB;
      wu_cp_async4(dst + 4u * lane, f.pmask + (size_t)pk * 32 + lane);
      if (p.use_dm && lane < 18) {
        const int idx = (lane < 16) ? (int)s_amap[(int)(sb.y & 0x7fffffffu) + amap_lane] : p.pzt_nact + lane - 16;
        if (idx >= 0) wu_cp_async4(dst + 128u + 4u * lane, p.volts + (size_t)pe * p.ldv + idx);
        else *reinterpret_cast<float*>(my_aux + slot * AUXB + 128 + 4 * lane) = 0.f;
      }
      if (has_after && lane == 0) wu_cp_async8(my_aux_u32 + (uint32_t)(slot ^ 1) * AUXB + 256u, f.sub + k_after);
      if (PE && lane < 8 * NL)      // the layer offsets of this item's environment, one word per lane
        wu_cp_async4(dst + (uint32_t)WU_AUX_BYTES + 4u * lane,
                     reinterpret_cast<const uint32_t*>(p.wind + (size_t)(lane >> 3) * p.E + pe) + (lane & 7));
      asm volatile("cp.async.commit_group;" ::: "memory");
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
          load_tta(xy_cur);
          load_ttb(xy_cur);
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
          float u[WU_NG];
          {
            wu_f2 ua = wu_mul2(wu_bc(fyv.x), wu_pk(v0.x, v0.y)), ub = wu_mul2(wu_bc(fyv.x), wu_pk(v0.z, v0.w));
            ua = wu_fma2(wu_bc(fyv.y), wu_pk(v1r.x, v1r.y), ua); ub = wu_fma2(wu_bc(fyv.y), wu_pk(v1r.z, v1r.w), ub);
            ua = wu_fma2(wu_bc(fyv.z), wu_pk(v2r.x, v2r.y), ua); ub = wu_fma2(wu_bc(fyv.z), wu_pk(v2r.z, v2r.w), ub);
            ua = wu_fma2(wu_bc(fyv.w), wu_pk(v3.x, v3.y), ua);   ub = wu_fma2(wu_bc(fyv.w), wu_pk(v3.z, v3.w), ub);
            wu_upk(ua, u[0], u[1]); wu_upk(ub, u[2], u[3]);
          }
  #pragma unroll
          for (int jx = 0; jx < WU_NG; ++jx) {
            const float4 fa = *reinterpret_cast<const float4*>(s_fx + jx * 16 + 8 * h);
            const float4 fb = *reinterpret_cast<const float4*>(s_fx + jx * 16 + 8 * h + 4);
            const wu_f2 U = wu_bc(u[jx]);
            if (jx == 0) {
              P[0] = wu_mul2(U, wu_pk(fa.x, fa.y)); P[1] = wu_mul2(U, wu_pk(fa.z, fa.w));
              P[2] = wu_mul2(U, wu_pk(fb.x, fb.y)); P[3] = wu_mul2(U, wu_pk(fb.z, fb.w));
            } else {
              P[0] = wu_fma2(U, wu_pk(fa.x, fa.y), P[0]); P[1] = wu_fma2(U, wu_pk(fa.z, fa.w), P[1]);
              P[2] = wu_fma2(U, wu_pk(fb.x, fb.y), P[2]); P[3] = wu_fma2(U, wu_pk(fb.z, fb.w), P[3]);
            }
          }
          const wu_f2 T0 = wu_bc(vt0), T1 = wu_bc(vt1);
          P[0] = wu_fma2(T0, wu_pk(tta[0].x, tta[0].y), P[0]); P[1] = wu_fma2(T0, wu_pk(tta[0].z, tta[0].w), P[1]);
          P[2] = wu_fma2(T0, wu_pk(tta[1].x, tta[1].y), P[2]); P[3] = wu_fma2(T0, wu_pk(tta[1].z, tta[1].w), P[3]);
          P[0] = wu_fma2(T1, wu_pk(ttb[0].x, ttb[0].y), P[0]); P[1] = wu_fma2(T1, wu_pk(ttb[0].z, ttb[0].w), P[1]);
          P[2] = wu_fma2(T1, wu_pk(ttb[1].x, ttb[1].y), P[2]); P[3] = wu_fma2(T1, wu_pk(ttb[1].z, ttb[1].w), P[3]);
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
  #pragma unroll
          for (int l = 0; l < NL; ++l) {
            const float* t = reinterpret_cast<const float*>(my_tiles + l * WU_TILE_STRIDE) + lane_off;
            if (PE) {
              const WindRec* wr = reinterpret_cast<const WindRec*>(my_aux + s * AUXB + WU_AUX_BYTES);
              switch ((c_d >> (2 * l)) & 3u) {
                case 0: wu_layer<0>(t, wr[l], acc); break;
                case 1: wu_layer<1>(t, wr[l], acc); break;
                case 2: wu_layer<2>(t, wr[l], acc); break;
                default: wu_layer<3>(t, wr[l], acc); break;
              }
            } else {
              switch ((c_d >> (2 * l)) & 3u) {
                case 0: wu_layer<0>(t, p.layer[l], acc); break;
                case 1: wu_layer<1>(t, p.layer[l], acc); break;
                case 2: wu_layer<2>(t, p.layer[l], acc); break;
                default: wu_layer<3>(t, p.layer[l], acc); break;
              }
            }
            asm volatile("" ::: "memory");                // one layer's window in registers at a time
          }
          __syncwarp();                                   // the stage is drained: re-arm it with the next item
          if (nx_valid) issue_tiles(e, sb1);
          // fold the right-hand taps into the pixel pairs
          float x0, x1, ya, yb;
          wu_upk(acc.X[0], x0, x1); wu_upk(acc.Y[0], ya, yb);
          P[0] = wu_pk(x0 + acc.y0, x1 + ya);
          wu_upk(acc.X[1], x0, x1); x0 += yb; wu_upk(acc.Y[1], ya, yb);
          P[1] = wu_pk(x0, x1 + ya);
          wu_upk(acc.X[2], x0, x1); x0 += yb; wu_upk(acc.Y[2], ya, yb);
          P[2] = wu_pk(x0, x1 + ya);
          wu_upk(acc.X[3], x0, x1);
          P[3] = wu_pk(x0 + yb, x1 + acc.y7);
        }

      }

      if (c_valid) {
        // ---- complex field exp(2 pi i t), t = phi / lambda - (x + y) / 128 turns; fp16 hi / lo ----
        wu_f2 RE[4], IM[4];
  #pragma unroll
        for (int c = 0; c < 4; ++c) {
          const wu_f2 t = wu_fma2(P[c], wu_bc(kt), wu_add2(hc01, wu_bc(-(float)(2 * c) * 0.0078125f)));
          float t0, t1;
          wu_upk(t, t0, t1);
          const wu_f2 ang = wu_mul2(wu_sub2(t, wu_pk(rintf(t0), rintf(t1))), wu_bc(6.283185307179586f));
          float a0, a1;
          wu_upk(ang, a0, a1);
          RE[c] = wu_pk(__cosf(a0), __cosf(a1));
          IM[c] = wu_pk(__sinf(a0), __sinf(a1));
        }
        if (c_pm != 0xffu) {
  #pragma unroll
          for (int c = 0; c < 4; ++c) {
            float r0, r1, i0, i1;
            wu_upk(RE[c], r0, r1); wu_upk(IM[c], i0, i1);
            const bool on0 = (c_pm >> (2 * c)) & 1u, on1 = (c_pm >> (2 * c + 1)) & 1u;
            RE[c] = wu_pk(on0 ? r0 : 0.f, on1 ? r1 : 0.f);
            IM[c] = wu_pk(on0 ? i0 : 0.f, on1 ? i1 : 0.f);
          }
        }
  #pragma unroll
        for (int c = 0; c < 4; ++c) {
          wu_split2(RE[c], re_h[c], re_l[c]);
          wu_split2(IM[c], im_h[c], im_l[c]);
        }
      }


      // A1 is free once MMA 1 of the previous group has completed
      if (it > 0) wu_mbar_wait(mma1_bar + 8u * ((it - 1) & 1), (uint32_t)(((it - 1) >> 1) & 1), f.err);
      if (c_valid) {
        wu_sts128(a1_addr, re_h[0], re_h[1], re_h[2], re_h[3]);
        wu_sts128(a1_addr + 256u, im_h[0], im_h[1], im_h[2], im_h[3]);
        wu_sts128(a1_addr + WU_A_BYTES, re_l[0], re_l[1], re_l[2], re_l[3]);
        wu_sts128(a1_addr + WU_A_BYTES + 256u, im_l[0], im_l[1], im_l[2], im_l[3]);
      }

      // ---- arrival; the last field warp issues MMA 1 of this group into accumulator buffer it & 1 ----
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      uint32_t pend = 0;
      if (lane == 0) {
        uint64_t st;
        asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(st) : "r"(a1_full) : "memory");
        asm volatile("mbarrier.pending_count.b64 %0, %1;" : "=r"(pend) : "l"(st));
      }
      pend = __shfl_sync(0xffffffffu, pend, 0);
      if (pend == 1u) {
        // the buffer was read out by the transform warps two groups ago
        if (it >= 2) wu_mbar_wait(t_free + 8u * (it & 1), (uint32_t)(((it - 2) >> 1) & 1), f.err);
        if (wu_elect()) {
          if (!wu_mbar_try(a1_full, (uint32_t)(it & 1))) atomicExch(f.err, 4);       // acquire; complete by construction
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          constexpr uint32_t KM = (128u >> 4) << 16, HI = (512u >> 4) | (1u << 14);     // K-major: LBO 128, SBO 512
          const uint32_t a_hi = q_a1 + KM, a_lo = a_hi + (WU_A_BYTES >> 4);
          const uint32_t b_hi = q_b1 + KM, b_lo = b_hi + (WU_B_BYTES >> 4);
          const uint32_t d = tmem_base + 64u * (uint32_t)(it & 1);
  #pragma unroll
          for (int ks = 0; ks < 2; ++ks) wu_mma_f16_lo(d, a_hi + ks * 16, b_hi + ks * 16, HI, idesc1, ks ? 1u : 0u);
  #pragma unroll
          for (int ks = 0; ks < 2; ++ks) wu_mma_f16_lo(d, a_lo + ks * 16, b_hi + ks * 16, HI, idesc1, 1u);
  #pragma unroll
          for (int ks = 0; ks < 2; ++ks) wu_mma_f16_lo(d, a_hi + ks * 16, b_lo + ks * 16, HI, idesc1, 1u);
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
    const uint32_t a2_addr = wu_smem_u32(s_a2) + (uint32_t)((q >> 1) * 2 * WU_A_BYTES + (4 * (2 * (q & 1) + h)) * 512 +
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
    // wfs_frame_umma_kernel): the centre of gravity is scale invariant and linear in |Y|^2, so the sums over the lane's 32
    // values of a half run on packed pairs straight from the accumulator: s0p = sum, syp = sum of py x value.
    auto sq_plain = [&](const uint32_t (&v)[32], float py0, wu_f2& s0p, wu_f2& syp, bool first) {
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const wu_f2 a = wu_pk(__uint_as_float(v[4 * m]), __uint_as_float(v[4 * m + 1]));
        const wu_f2 b = wu_pk(__uint_as_float(v[4 * m + 2]), __uint_as_float(v[4 * m + 3]));
        const wu_f2 t = wu_fma2(b, b, wu_mul2(a, a));
        if (first && m == 0) {
          s0p = t;
          syp = wu_mul2(t, wu_bc(py0));
        } else {
          s0p = wu_add2(s0p, t);
          syp = wu_fma2(t, wu_bc(py0 + (float)m), syp);
        }
      }
    };
    // lane = kept fx index; fx pair lane >> 1 -> px
    const float pxf = (float)(((lane >> 1) < 8) ? 8 + (lane >> 1) : (lane >> 1) - 8);
    auto epilogue = [&](wu_f2 s0p, wu_f2 syp, int ie, int ik) {
      float a, b;
      wu_upk(s0p, a, b); float s0 = a + b;
      wu_upk(syp, a, b); float sy = a + b;
      float sx = s0 * pxf;
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, sft);
        sx += __shfl_xor_sync(0xffffffffu, sx, sft);
        sy += __shfl_xor_sync(0xffffffffu, sy, sft);
      }
      if (lane == 0) {
        const float inv = __frcp_rn(s0);
        const float gx = (s0 > 0.f) ? sx * inv : p.cog_offset;
        const float gy = (s0 > 0.f) ? sy * inv : p.cog_offset;
        float* sl = p.slopes + (size_t)ie * p.lds;
        sl[ik] = (gx - p.cog_offset) * p.pixsize;
        sl[p.nvalid + ik] = (gy - p.cog_offset) * p.pixsize;
      }
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
          // ---- T -> fp16 hi / lo -> A2 (MN-major: 8 consecutive fx per 16-byte group) ----
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t hw[4], lw[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float a = __uint_as_float(tv[8 * c + 2 * i]), b = __uint_as_float(tv[8 * c + 2 * i + 1]);
              if (FULL) wu_split2(wu_pk(a, b), hw[i], lw[i]);
              else { hw[i] = wu_pack(a, b); lw[i] = 0u; }
            }
            wu_sts128(a2_addr + ro * 256 + c * 512, hw[0], hw[1], hw[2], hw[3]);
            if (FULL) wu_sts128(a2_addr + WU_A_BYTES + ro * 256 + c * 512, lw[0], lw[1], lw[2], lw[3]);
          }
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
          sq_plain(yv, 8.f, s0p[t], syp[t], true);
          wu_tmem_ld32(d2_addr + 64u * t + 32u, yv);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          sq_plain(yv, 0.f, s0p[t], syp[t], false);
        }
      }
      if (conv) {
        // ---- arrival (A2 written, Y drained); the last transform warp issues MMA 2 of group j ----
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        uint32_t pend = 0;
        if (lane == 0) {
          uint64_t st;
          asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(st) : "r"(a2_full) : "memory");
          asm volatile("mbarrier.pending_count.b64 %0, %1;" : "=r"(pend) : "l"(st));
        }
        pend = __shfl_sync(0xffffffffu, pend, 0);
        if (pend == 1u) {
          if (wu_elect()) {
            if (!wu_mbar_try(a2_full, (uint32_t)(j & 1))) atomicExch(f.err, 4);       // acquire; complete by construction
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            constexpr uint32_t KM = (128u >> 4) << 16, HI = (512u >> 4) | (1u << 14);
            const uint32_t b_hi = q_b2 + KM, b_lo = b_hi + (WU_B_BYTES >> 4);
            const uint32_t lbo = f.a2_swap ? 512u : 128u, sbo = f.a2_swap ? 128u : 512u;
            const uint32_t am = (lbo >> 4) << 16, hia = (sbo >> 4) | (1u << 14);
#pragma unroll
            for (int t = 0; t < 2; ++t) {
              const uint32_t a_hi = q_a2 + t * (2 * WU_A_BYTES >> 4) + am, a_lo = a_hi + (WU_A_BYTES >> 4);
              const uint32_t d = tmem_base + 128u + 64u * t;
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) wu_mma2(d, a_hi + ks * 16, hia, b_hi + ks * 16, HI, idesc2, ks ? 1u : 0u);
              if (FULL) {
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) wu_mma2(d, a_lo + ks * 16, hia, b_hi + ks * 16, HI, idesc2, 1u);
              }
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) wu_mma2(d, a_hi + ks * 16, hia, b_lo + ks * 16, HI, idesc2, 1u);
            }
            wu_commit(mma2_bar);
          }
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

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)WU_TMEM_COLS) : "memory");
  }
}
