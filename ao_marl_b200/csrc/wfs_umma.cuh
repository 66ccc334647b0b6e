// Shack-Hartmann frame, fifth generation: BOTH stages of the pruned 2-D DFT on the tcgen05 tensor cores.
//
// Same fused pipeline as the earlier generations (raytrace through the layers -> mirrors -> complex field -> pruned
// 64-point DFT along x, then along y, 32 kept frequencies each -> |.|^2 -> 2 x 2 binning -> flux / noise -> centre
// of gravity; WfsCompass.raytrace / compute_wfs_image / RtcCompass.do_centroids, shesha/supervisor/components/
// wfsCompass.py:334-343, sourceCompass.py:54-85, rtcCompass.py:557-563), but no warp-level mma.sync is left: the
// round-1 kernel spent 144 HMMA + ~130 fragment split / load instructions per subaperture on the legacy path and was
// bound by its instruction count (DESIGN.md section 4).  Here eight subapertures share each tensor-core tile:
//
//   one CTA = 8 warps = one group of 8 subapertures per iteration, two CTAs per SM, persistent over a contiguous
//   range of work items.  Lane (h, y) = (lane >> 4, lane & 15) of warp s owns row y, columns 8h .. 8h+7 of
//   subaperture s.
//
//   F  field      3-layer bilinear sample of TMA-staged 20 x 17 tiles + separable mirror stamp + tip-tilt -> phase in
//                 turns -> exp(2 pi i t) by SFU -> fp16 hi / lo -> four 16-byte stores into the K-major A operand
//                 A1[128 = (s, y)][32 = (re | im, x)] (UMMA canonical no-swizzle layout).
//   MMA1          D1[128][64] = A1 . B1^T, B1[64 = (re | im, fx)][32] the constant x twiddles; three fp16 products
//                 (hi.hi + lo.hi + hi.lo) = 6 tcgen05.mma (M 128, N 64, K 16) for 8 subapertures, accumulator in TMEM.
//   C  convert    warp (q, ro) reads its 32 TMEM lanes x 32 columns (T_re or T_im of two subapertures), splits to fp16
//                 hi / lo and stores 16-byte groups of 8 consecutive fx into the MN-major A operand of stage 2,
//                 A2[tile j][128 = (s', fx)][32 = (re | im, y)] -- the transposition between the two stages costs
//                 nothing: it is the choice of the MN-major descriptor.
//   MMA2          D2[j][128][64] = A2[j] . B2^T, B2[64 = (fy, re | im)][32] the y twiddles: 12 tcgen05.mma for 8
//                 subapertures.
//   E  epilogue   warp s reads the 32 fx rows x 64 columns of its own subaperture, |.|^2, binning, noise, centroid.
//
//   The three phases of one warp belong to consecutive iterations (F(i), C(i-1), E(i-2)), so every tensor-core
//   round trip has a whole field computation to complete in; every buffer is single and every wait is normally
//   already satisfied.  The MMAs are issued by lane 0 of whichever warp arrives last (a shared-memory counter), after
//   the usual generic -> async proxy fence of the writers and tcgen05 fences around the thread synchronisation.
//   Every wait is bounded; an expired wait raises the context's error word and traps.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "rng.cuh"
#include "wfs_params.cuh"
#include "wfs_lattice_host.h"

#define WU_WARPS 8
#define WU_TILE_W 20                       // box width (floats): 17 needed + up to 3 of alignment slack; rows 80 B apart
#define WU_TILE_H 17
#define WU_TILE_BYTES (WU_TILE_W * WU_TILE_H * 4)            // 1360 = bytes one box delivers
#define WU_TILE_STRIDE 1408                                  // 11 x 128
#define WU_NG WFL_NG
#define WU_MAX_LAYERS WFL_MAX_LAYERS
#define WU_A_BYTES 8192                    // 128 rows x 32 fp16
#define WU_B_BYTES 4096                    // 64 rows x 32 fp16
#define WU_TMEM_COLS 256                   // D1: 64 columns, D2: 2 x 64
#define WU_WAIT_SPINS (1u << 21)            // x ~1 us: two seconds before a wait is declared dead

struct WfsUmmaTables {
  const uint2* sub;           // [nvalid] {y0 << 16 | x0, padded-lattice index of the neighbourhood origin | fully lit << 31}
  const short* amap;          // [GW * GW] actuator index or -1 (padded by WFL_PAD cells on every side)
  const uint32_t* pmask;      // [nvalid][32] bit c = pupil(y, 8h + c) of lane (h, y)
  const uint4* b1;            // [2][WU_B_BYTES / 16] stage-1 B tiles (hi, lo), K-major canonical layout
  const uint4* b2;            // [2][WU_B_BYTES / 16] stage-2 B tiles
  const float* fxy;           // [WU_NG][16] x stamp factors, then [16][WU_NG] y stamp factors (transposed)
  int GW;
  int* err;
  long long items_per_cta;
};

struct WfsUmmaParams {
  WfsParams p;
  WfsUmmaTables f;
  CUtensorMap maps[WU_MAX_LAYERS];
};

#define WU_AUX_BYTES 288                   // per warp and parity: 32 pupil words, 32 volts, one subaperture record (+ pad)
// per-environment winds: the item's layer offsets (WindRec [WU_MAX_LAYERS], one word per lane) follow in the slot
#define WU_AUX_BYTES_PE (WU_AUX_BYTES + WU_MAX_LAYERS * 32)

template <int NL, bool PE = false>
constexpr size_t wu_smem_bytes(int gw) {
  return (size_t)2 * WU_A_BYTES + 4 * WU_A_BYTES + 4 * WU_B_BYTES + (size_t)WU_WARPS * (NL > 0 ? NL : 1) * WU_TILE_STRIDE +
         128 + 2 * WU_NG * 16 * 4 + WU_WARPS * 2 * (PE ? WU_AUX_BYTES_PE : WU_AUX_BYTES) + (((size_t)gw * gw * 2 + 15) & ~(size_t)15);
}

__device__ __forceinline__ uint32_t wu_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ bool wu_mbar_try(uint32_t bar, uint32_t parity) {
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

// Bounded wait.  The phase is normally complete already (one try); otherwise the warp sleeps in coarse steps instead
// of being woken by every unrelated mbarrier event of the CTA (round 2, first version: 375 wake-up instructions per
// subaperture).  On expiry the error word is raised and the kernel traps.
__device__ __forceinline__ void wu_mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  if (wu_mbar_try(bar, parity)) return;
  uint32_t ns = 128;
#pragma unroll 1
  for (uint32_t it = 0; it < WU_WAIT_SPINS; ++it) {
    __nanosleep(ns);
    if (wu_mbar_try(bar, parity)) return;
    ns = ns < 1024u ? ns * 2u : 1024u;
  }
  atomicExch(err, 3);
  __threadfence_system();
  __trap();
}

__device__ __forceinline__ void wu_tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// shared-memory matrix descriptor, no swizzle: 8 x 16-byte core matrices, 128 B between the two core matrices of a
// K step ("leading"), 512 B between 8-row (K-major) or 8-column (MN-major) groups ("stride")
__device__ __forceinline__ uint64_t wu_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= 1ull << 46;                                           // descriptor version of sm_100
  return d;
}

__device__ __forceinline__ void wu_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
      : "memory");
}

// the same with descriptor low words (start >> 4 | LBO >> 4 << 16) and the constant high word (SBO >> 4 | version) apart
__device__ __forceinline__ void wu_mma_f16_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, {%6, %6, %6, %6}, p;\n\t}"
      :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(hi), "r"(0u) : "memory");
}
// separate high words for A and B (the MN-major stage-2 operand has its own stride field)
__device__ __forceinline__ void wu_mma2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %6};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, {%7, %7, %7, %7}, p;\n\t}"
      :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(a_hi), "r"(b_hi), "r"(0u) : "memory");
}
__device__ __forceinline__ bool wu_elect() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ void wu_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void wu_tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void wu_sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void wu_cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void wu_cp_async8(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}

__device__ __forceinline__ uint32_t wu_pack(float lo_elem, float hi_elem) {
  __half2 h = __floats2half2_rn(lo_elem, hi_elem);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---- packed float32 pairs (Blackwell FFMA2 / FADD2 / FMUL2: one issue slot for two lanes of arithmetic; the kernel is
//      bound by its instruction stream, not by the FMA pipe) ----
typedef unsigned long long wu_f2;
__device__ __forceinline__ wu_f2 wu_pk(float lo, float hi) { wu_f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void wu_upk(wu_f2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ wu_f2 wu_fma2(wu_f2 a, wu_f2 b, wu_f2 c) { wu_f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ wu_f2 wu_mul2(wu_f2 a, wu_f2 b) { wu_f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ wu_f2 wu_add2(wu_f2 a, wu_f2 b) { wu_f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ wu_f2 wu_sub2(wu_f2 a, wu_f2 b) { wu_f2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ wu_f2 wu_bc(float v) { return wu_pk(v, v); }       // scalar broadcast (an operand modifier in SASS)

// error-free split of a pair: hi keeps the leading 11 significant bits (exact in fp16 over |v| <= 32), lo the rest
__device__ __forceinline__ void wu_split(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u);
  const float bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  hi = wu_pack(ah, bh);
  lo = wu_pack(a - ah, b - bh);
}

// the same on a packed pair (one FADD2 for the two low parts)
__device__ __forceinline__ void wu_split2(wu_f2 v, uint32_t& hi, uint32_t& lo) {
  float a, b;
  wu_upk(v, a, b);
  const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u);
  const float bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  hi = wu_pack(ah, bh);
  float la, lb;
  wu_upk(wu_sub2(v, wu_pk(ah, bh)), la, lb);
  lo = wu_pack(la, lb);
}

// Phase accumulators of a lane's 8 pixels (row y, columns 8h .. 8h+7): X[j] = pixels (2j, 2j+1); the taps one column to
// the right are register pairs shifted by one pixel, so they accumulate in their own pairing Y[j] = pixels (2j+1, 2j+2)
// plus the two end pixels as scalars, and are folded into X once after the last layer.
struct WuPhase {
  wu_f2 X[4];
  wu_f2 Y[3];
  float y0, y7;
};

// Bilinear sample of one staged tile.  The TMA box starts at the 16-byte aligned column below the tile origin (the
// start address of a box must be 16-byte aligned: profiles/dev/tma_probe.cu), so the wanted columns begin
// D = origin & 3 floats into the row; pixel c, tap b reads v[D + c + b].  The aligned register pairs (v[2k], v[2k+1])
// serve the X pairing for the taps with D + b even and the Y pairing for the others.
template <int D, class Wt>      // Wt: WfsLayer (common offset) or WindRec (the item's environment's own)
__device__ __forceinline__ void wu_layer(const float* __restrict__ t, const Wt& L, WuPhase& a) {
  float v[2][12];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const float4 q0 = *reinterpret_cast<const float4*>(t + r * WU_TILE_W);
    const float4 q1 = *reinterpret_cast<const float4*>(t + r * WU_TILE_W + 4);
    v[r][0] = q0.x; v[r][1] = q0.y; v[r][2] = q0.z; v[r][3] = q0.w;
    v[r][4] = q1.x; v[r][5] = q1.y; v[r][6] = q1.z; v[r][7] = q1.w;
    if (D == 0) {
      v[r][8] = t[r * WU_TILE_W + 8];
    } else {
      const float4 q2 = *reinterpret_cast<const float4*>(t + r * WU_TILE_W + 8);
      v[r][8] = q2.x; v[r][9] = q2.y; v[r][10] = q2.z; v[r][11] = q2.w;
    }
  }
  constexpr int d = D >> 1;
  // taps b = B_X feed the X pairing, taps b = 1 - B_X the Y pairing and the two end pixels
  constexpr int B_X = D & 1;
  const float wx0 = B_X ? L.w01 : L.w00, wx1 = B_X ? L.w11 : L.w10;       // rows 0 / 1 of the X taps
  const float wy0 = B_X ? L.w00 : L.w01, wy1 = B_X ? L.w10 : L.w11;
  const wu_f2 WX0 = wu_bc(wx0), WX1 = wu_bc(wx1), WY0 = wu_bc(wy0), WY1 = wu_bc(wy1);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int k = 2 * (d + j + B_X);
    a.X[j] = wu_fma2(WX1, wu_pk(v[1][k], v[1][k + 1]), wu_fma2(WX0, wu_pk(v[0][k], v[0][k + 1]), a.X[j]));
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int k = 2 * (d + j + 1);
    a.Y[j] = wu_fma2(WY1, wu_pk(v[1][k], v[1][k + 1]), wu_fma2(WY0, wu_pk(v[0][k], v[0][k + 1]), a.Y[j]));
  }
  // end pixels of the Y pairing: pixel 0 and pixel 7 with the tap b = 1 - B_X
  a.y0 = fmaf(wy1, v[1][D + 1 - B_X], fmaf(wy0, v[0][D + 1 - B_X], a.y0));
  a.y7 = fmaf(wy1, v[1][D + 8 - B_X], fmaf(wy0, v[0][D + 8 - B_X], a.y7));
}

// ================= pieces shared by wfs_frame_umma_kernel and wfs_frame_ws_kernel (wfs_umma_ws.cuh) =================

// Shared memory of one CTA (wu_smem_bytes).  The 128-byte barrier block is laid out by each kernel.
struct WuSmem {
  unsigned char* a1;        // [hi, lo][WU_A_BYTES]
  unsigned char* a2;        // [tile][hi, lo][WU_A_BYTES]
  unsigned char* b1;        // [hi, lo][WU_B_BYTES]
  unsigned char* b2;
  unsigned char* tiles;     // [warp][layer][WU_TILE_STRIDE]
  uint64_t* bar;            // barrier block
  float* fx;                // [NG][16]
  float* fyT;               // [16][NG]
  unsigned char* aux;       // [warp][parity][AUXB]
  short* amap;
};

template <int NL, bool PE>
__device__ __forceinline__ WuSmem wu_smem_layout() {
  extern __shared__ __align__(1024) unsigned char wu_smem_raw[];
  constexpr int NLS = NL > 0 ? NL : 1;
  constexpr int AUXB = PE ? WU_AUX_BYTES_PE : WU_AUX_BYTES;
  WuSmem S;
  S.a1 = wu_smem_raw;
  S.a2 = S.a1 + 2 * WU_A_BYTES;
  S.b1 = S.a2 + 4 * WU_A_BYTES;
  S.b2 = S.b1 + 2 * WU_B_BYTES;
  S.tiles = S.b2 + 2 * WU_B_BYTES;
  S.bar = (uint64_t*)(S.tiles + (size_t)WU_WARPS * NLS * WU_TILE_STRIDE);
  S.fx = (float*)((unsigned char*)S.bar + 128);
  S.fyT = S.fx + WU_NG * 16;
  S.aux = (unsigned char*)(S.fyT + 16 * WU_NG);
  S.amap = (short*)(S.aux + WU_WARPS * 2 * AUXB);
  return S;
}

// lane through a volatile read: the compiler otherwise re-derives it from S2R SR_TID.X at ~25 places of the loop body
// and each of those reads stalls its warp (5 % of the stall samples in profiles/r02_wfs_umma_v5)
__device__ __forceinline__ int wu_lane() {
  int lane;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
  return lane;
}

// CTA set-up: copies the constant tables, zeroes the operand tiles, initialises barriers 0 .. n_bar - 1 (count: the
// arrival count of barrier tid) and allocates the tensor memory; returns its base address, which passes through
// tmem_slot, a word of the barrier block.  tid / nthr are threadIdx.x / blockDim.x read in the kernel, where the compiler
// bounds them by its launch bounds (read here, the copy loops compile to a longer trip-count computation).
__device__ __forceinline__ uint32_t wu_cta_setup(const WuSmem& S, const WfsUmmaTables& f, uint32_t tid, uint32_t nthr, int warp,
                                                 uint32_t n_bar, uint32_t count, uint32_t* tmem_slot) {
  for (int i = tid; i < 2 * WU_B_BYTES / 16; i += nthr) {
    reinterpret_cast<uint4*>(S.b1)[i] = f.b1[i];
    reinterpret_cast<uint4*>(S.b2)[i] = f.b2[i];
  }
  for (int i = tid; i < 2 * WU_NG * 16; i += nthr) S.fx[i] = f.fxy[i];
  for (int i = tid; i < f.GW * f.GW; i += nthr) S.amap[i] = f.amap[i];
  // operand tiles start from zeros: rows of work items that do not exist are multiplied too
  for (int i = tid; i < 6 * WU_A_BYTES / 16; i += nthr) reinterpret_cast<uint4*>(S.a1)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (tid < n_bar) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(wu_smem_u32(S.bar + tid)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // B tiles / zeroed A tiles are read by the tensor core
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(wu_smem_u32(tmem_slot)), "r"((uint32_t)WU_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  return __shfl_sync(0xffffffffu, *tmem_slot, 0);
}

__device__ __forceinline__ void wu_cta_release(int warp, uint32_t tmem_base) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)WU_TMEM_COLS) : "memory");
  }
}

// ---- the F phase of a field warp: its items are the CTA-local indices warp + 8 i; the tiles and per-lane inputs of
//      the next item are in flight while the current one is sampled.  The kernels keep the per-warp state in locals
//      and pass it by reference: the order of the loads, copies and fences below is what keeps the register budget
//      (the specialised kernel fits in 80 registers) ----

// tiles of one work item (record sb): TMA boxes, or element-wise wrapped cp.async copies on the torus seam.  ring_e /
// rx / ry: the ring origins of the environment whose origins were computed last; n_d / n_seam: the tile column offsets
// and the seam flag of this item.
template <int NL, bool PE>
__device__ __forceinline__ void wu_issue_tiles(const WfsUmmaParams& P, uint32_t my_tiles_u32, uint32_t my_bar_u32, int lane, int pe,
                                               uint2 sb, int& ring_e, int (&rx)[NL > 0 ? NL : 1], int (&ry)[NL > 0 ? NL : 1],
                                               uint32_t& n_d, bool& n_seam) {
  constexpr int NLS = NL > 0 ? NL : 1;
  const WfsParams& p = P.p;
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
}

// per-lane inputs of one work item into the parity slot of my_aux (pm[32] | volts[32] | record, then with PE the layer
// offsets): pupil word, neighbourhood volts (cp.async: no register waits for them), and the record of the item after it
template <int NL, bool PE>
__device__ __forceinline__ void wu_issue_aux(const WfsParams& p, const WfsUmmaTables& f, unsigned char* my_aux, uint32_t my_aux_u32,
                                             const short* amap, int amap_lane, int lane, int pe, int pk, uint2 sb, int slot,
                                             int k_after, bool has_after) {
  constexpr int AUXB = PE ? WU_AUX_BYTES_PE : WU_AUX_BYTES;
  const uint32_t dst = my_aux_u32 + (uint32_t)slot * AUXB;
  wu_cp_async4(dst + 4u * lane, f.pmask + (size_t)pk * 32 + lane);
  if (p.use_dm && lane < 18) {
    const int idx = (lane < 16) ? (int)amap[(int)(sb.y & 0x7fffffffu) + amap_lane] : p.pzt_nact + lane - 16;
    if (idx >= 0) wu_cp_async4(dst + 128u + 4u * lane, p.volts + (size_t)pe * p.ldv + idx);
    else *reinterpret_cast<float*>(my_aux + slot * AUXB + 128 + 4 * lane) = 0.f;
  }
  if (has_after && lane == 0) wu_cp_async8(my_aux_u32 + (uint32_t)(slot ^ 1) * AUXB + 256u, f.sub + k_after);
  if (PE && lane < 8 * NL)      // the layer offsets of this item's environment, one word per lane
    wu_cp_async4(dst + (uint32_t)WU_AUX_BYTES + 4u * lane,
                 reinterpret_cast<const uint32_t*>(p.wind + (size_t)(lane >> 3) * p.E + pe) + (lane & 7));
  asm volatile("cp.async.commit_group;" ::: "memory");
}

// The tip-tilt planes are tables (the reference's Zernike 2 / 3 are evaluated in float32 with offset centres,
// dm_init.py:661-694 -> dm_util.py:300-380: up to 1.5 % away from a plane).  The 2 x 8 values of a lane are requested
// at the top of the item and used after the atmosphere has been sampled (the layers are sampled one at a time so
// that these 16 registers survive without a spill: a spill right behind the loads would wait for them).
// tt_lane: this lane's first pixel in the tip-tilt support; xy: (y0 << 16 | x0) of the item.
__device__ __forceinline__ void wu_load_tt(const WfsParams& p, const float* tt_plane1, int tt_lane, uint32_t xy, float4 (&tta)[2], float4 (&ttb)[2]) {
  const int to = (int)(xy >> 16) * p.tt_dim + (int)(xy & 0xffffu) + tt_lane;
  tta[0] = __ldg(reinterpret_cast<const float4*>(p.tt_planes + to));
  tta[1] = __ldg(reinterpret_cast<const float4*>(p.tt_planes + to + 4));
  ttb[0] = __ldg(reinterpret_cast<const float4*>(tt_plane1 + to));
  ttb[1] = __ldg(reinterpret_cast<const float4*>(tt_plane1 + to + 4));
}

// mirror surface of the lane's 8 pixels as pairs P: the separable stamp of the 4 x 4 neighbourhood volts v0..v3 (fyv:
// the y factors of the lane's row, fx: the x factors) and the tip-tilt volts vt0 / vt1 on the planes' values.  The
// tip-tilt loads were requested before the stamp arithmetic, and the tiles of the atmosphere land meanwhile.
__device__ __forceinline__ void wu_mirror(float4 v0, float4 v1r, float4 v2r, float4 v3, float vt0, float vt1, float4 fyv, const float* fx,
                                          int h, const float4 (&tta)[2], const float4 (&ttb)[2], wu_f2 (&P)[4]) {
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
    const float4 fa = *reinterpret_cast<const float4*>(fx + jx * 16 + 8 * h);
    const float4 fb = *reinterpret_cast<const float4*>(fx + jx * 16 + 8 * h + 4);
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
}

// the atmosphere on top of acc: every layer's staged tile (my_tiles + lane_off floats), with the common offsets or, with
// PE, the item's own weights (WindRec [NL] at wind_slot); c_d: the tile column offsets of the item, 2 bits per layer
template <int NL, bool PE>
__device__ __forceinline__ void wu_layers(const unsigned char* my_tiles, int lane_off, const unsigned char* wind_slot, const WfsParams& p,
                                          uint32_t c_d, WuPhase& acc) {
#pragma unroll
  for (int l = 0; l < NL; ++l) {
    const float* t = reinterpret_cast<const float*>(my_tiles + l * WU_TILE_STRIDE) + lane_off;
    if (PE) {
      const WindRec* wr = reinterpret_cast<const WindRec*>(wind_slot);
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
}

// fold the right-hand taps into the pixel pairs
__device__ __forceinline__ void wu_fold(const WuPhase& acc, wu_f2 (&P)[4]) {
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

// complex field exp(2 pi i t), t = phi / lambda - (x + y) / 128 turns (kt = k2 / 2 pi, hc01: -(x + y) / 128 of the
// lane's first pixel pair), zero outside the pupil word pm; fp16 hi / lo
__device__ __forceinline__ void wu_field(const wu_f2 (&P)[4], uint32_t pm, float kt, wu_f2 hc01, uint32_t (&re_h)[4], uint32_t (&re_l)[4],
                                         uint32_t (&im_h)[4], uint32_t (&im_l)[4]) {
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
  if (pm != 0xffu) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float r0, r1, i0, i1;
      wu_upk(RE[c], r0, r1); wu_upk(IM[c], i0, i1);
      const bool on0 = (pm >> (2 * c)) & 1u, on1 = (pm >> (2 * c + 1)) & 1u;
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
// A1 rows of the lane (a1_addr): chunks (re, h) (im, h) of the hi tile, the lo tile 8 KB further
__device__ __forceinline__ void wu_store_a1(uint32_t a1_addr, const uint32_t (&re_h)[4], const uint32_t (&re_l)[4], const uint32_t (&im_h)[4],
                                            const uint32_t (&im_l)[4]) {
  wu_sts128(a1_addr, re_h[0], re_h[1], re_h[2], re_h[3]);
  wu_sts128(a1_addr + 256u, im_h[0], im_h[1], im_h[2], im_h[3]);
  wu_sts128(a1_addr + WU_A_BYTES, re_l[0], re_l[1], re_l[2], re_l[3]);
  wu_sts128(a1_addr + WU_A_BYTES + 256u, im_l[0], im_l[1], im_l[2], im_l[3]);
}

// ---- tensor-core issue ----
// The warps of a phase arrive on a count-N mbarrier, and the elected lane of the last of them issues the MMAs.  One
// arrival per warp (release semantics, no memory barrier instruction, no atomic): the state it returns is the one before
// the arrival, and its pending count tells the last warp (== 1), which acquires the phase it has just completed
// (profiles/dev/mbar_count_probe.cu; a shared-memory counter with atom.acq_rel cost a MEMBAR.ALL.CTA and the compiler's
// warp-aggregation sequence per arrival).  The count is broadcast through a shuffle and the issuing lane chosen by
// elect.sync, so that the issue path is warp-uniform for the compiler (descriptors in uniform registers, UTCHMMA back to
// back; under `lane == 0` every MMA sat in a per-thread waterfall loop of ~13 instructions).

// the arrival of this warp's writes (generic proxy, and with tmem its tensor-memory reads); true in the last warp
__device__ __forceinline__ bool wu_arrive(uint32_t bar, int lane, bool tmem) {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (tmem) asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncwarp();
  uint32_t pend = 0;
  if (lane == 0) {
    uint64_t st;
    asm volatile("mbarrier.arrive.shared::cta.b64 %0, [%1];" : "=l"(st) : "r"(bar) : "memory");
    asm volatile("mbarrier.pending_count.b64 %0, %1;" : "=r"(pend) : "l"(st));
  }
  pend = __shfl_sync(0xffffffffu, pend, 0);
  return pend == 1u;
}
// in the last warp: true in the lane that issues, after it has acquired the completed phase
__device__ __forceinline__ bool wu_elect_acquire(uint32_t bar, uint32_t parity, int* err) {
  if (!wu_elect()) return false;
  if (!wu_mbar_try(bar, parity)) atomicExch(err, 4);       // acquire; complete by construction
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  return true;
}

constexpr uint32_t wu_idesc1 = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);  // f16 x f16 -> f32, K-major A and B
constexpr uint32_t wu_idesc2 = wu_idesc1 | (1u << 15);                                                  // A operand MN-major
constexpr uint32_t wu_km = (128u >> 4) << 16, wu_hi = (512u >> 4) | (1u << 14);     // LBO 128, SBO 512 (both majors)

// MMA 1 into TMEM column d: D1 = A1 . B1^T in three fp16 products (q_*: shared addresses >> 4)
__device__ __forceinline__ void wu_issue_mma1(uint32_t d, uint32_t q_a1, uint32_t q_b1) {
  const uint32_t a_hi = q_a1 + wu_km, a_lo = a_hi + (WU_A_BYTES >> 4);
  const uint32_t b_hi = q_b1 + wu_km, b_lo = b_hi + (WU_B_BYTES >> 4);
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) wu_mma_f16_lo(d, a_hi + ks * 16, b_hi + ks * 16, wu_hi, wu_idesc1, ks ? 1u : 0u);
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) wu_mma_f16_lo(d, a_lo + ks * 16, b_hi + ks * 16, wu_hi, wu_idesc1, 1u);
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) wu_mma_f16_lo(d, a_hi + ks * 16, b_lo + ks * 16, wu_hi, wu_idesc1, 1u);
}

// MMA 2 of both A2 tiles into TMEM columns d, d + 64
template <int FULL>
__device__ __forceinline__ void wu_issue_mma2(uint32_t d, uint32_t q_a2, uint32_t q_b2) {
  const uint32_t b_hi = q_b2 + wu_km, b_lo = b_hi + (WU_B_BYTES >> 4);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const uint32_t a_hi = q_a2 + j * (2 * WU_A_BYTES >> 4) + wu_km, a_lo = a_hi + (WU_A_BYTES >> 4);
    const uint32_t dj = d + 64u * j;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) wu_mma2(dj, a_hi + ks * 16, wu_hi, b_hi + ks * 16, wu_hi, wu_idesc2, ks ? 1u : 0u);
    if (FULL) {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) wu_mma2(dj, a_lo + ks * 16, wu_hi, b_hi + ks * 16, wu_hi, wu_idesc2, 1u);
    }
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) wu_mma2(dj, a_hi + ks * 16, wu_hi, b_lo + ks * 16, wu_hi, wu_idesc2, 1u);
  }
}

// 32 stage-1 accumulator columns -> fp16 hi / lo -> A2 (MN-major: 8 consecutive fx per 16-byte group)
template <int FULL>
__device__ __forceinline__ void wu_store_a2(uint32_t addr, uint32_t off, const uint32_t (&tv)[32]) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a = __uint_as_float(tv[8 * c + 2 * j]), b = __uint_as_float(tv[8 * c + 2 * j + 1]);
      if (FULL) wu_split2(wu_pk(a, b), hw[j], lw[j]);
      else { hw[j] = wu_pack(a, b); lw[j] = 0u; }
    }
    wu_sts128(addr + off + c * 512, hw[0], hw[1], hw[2], hw[3]);
    if (FULL) wu_sts128(addr + WU_A_BYTES + off + c * 512, lw[0], lw[1], lw[2], lw[3]);
  }
}

// ---- epilogue of one subaperture: lane = kept fx index ----
// Plain path (no noise, no image kept): the centre of gravity is scale invariant and linear in |Y|^2, so the sums over
// the lane's 32 values of a half run on packed pairs straight from the accumulator: s0p = sum, syp = sum of py x value.
__device__ __forceinline__ void wu_sq_plain(const uint32_t (&v)[32], float py0, wu_f2& s0p, wu_f2& syp, bool first) {
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
}
// centre of gravity from the lanes' partial sums and the slopes of item (ie, ik)
__device__ __forceinline__ void wu_cog_store(const WfsParams& p, int lane, float s0, float sx, float sy, int ie, int ik) {
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
}

// FULL = 1: three fp16 products in both stages (fp32-grade slopes).  0: the stage-1 result goes to stage 2 as a single
// rounded fp16 (slopes ~3e-5 relative).
// PE: per-environment winds (layer offsets from p.wind: the ring origin per environment, the weights per item through
// the aux slot)
// NE: per-environment sensor values (noise and photon count of the item's environment; whether the epilogue takes the
// plain path is decided per item -- warp-uniform, a warp's item belongs to one environment)
template <int NL, int FULL, bool PE = false, bool NE = false>
__global__ void __launch_bounds__(WU_WARPS * 32, 2) wfs_frame_umma_kernel(const __grid_constant__ WfsUmmaParams P) {
  const WfsParams& p = P.p;
  const WfsUmmaTables& f = P.f;
  constexpr int NLS = NL > 0 ? NL : 1;
  constexpr int AUXB = PE ? WU_AUX_BYTES_PE : WU_AUX_BYTES;
  // barrier block: [0..7] tiles, [8] MMA1 done, [9] MMA2 done, [10], [11] stage-1 / stage-2 arrivals of the 8 warps;
  // the TMEM slot at byte 104
  const WuSmem S = wu_smem_layout<NL, PE>();
  const int lane = wu_lane();
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int y = lane & 15, h = lane >> 4;

  const uint32_t tmem_base = wu_cta_setup(S, f, threadIdx.x, blockDim.x, warp, 12, threadIdx.x < 10 ? 1u : (uint32_t)WU_WARPS,
                                          (uint32_t*)(S.bar + 13));

  unsigned char* my_tiles = S.tiles + (size_t)warp * NLS * WU_TILE_STRIDE;
  const uint32_t my_tiles_u32 = wu_smem_u32(my_tiles);
  const uint32_t my_bar_u32 = wu_smem_u32(S.bar + warp);
  const uint32_t mma1_bar = wu_smem_u32(S.bar + 8), mma2_bar = wu_smem_u32(S.bar + 9);
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
  // conversion role: TMEM lane quarter qq = warp & 3 (rows 32 qq .. = subapertures 2 qq, 2 qq + 1), part ro = warp >> 2
  const int qq = warp & 3, ro = warp >> 2;
  const uint32_t d1_addr = tmem_base + ((uint32_t)(32 * qq) << 16) + (uint32_t)(32 * ro);
  // A2: tile qq >> 1, rows m = 32 s' + fx with s' = 2 (qq & 1) + h, K index 16 ro + y
  const uint32_t a2_addr = wu_smem_u32(S.a2) + (uint32_t)((qq >> 1) * 2 * WU_A_BYTES + (4 * (2 * (qq & 1) + h)) * 512 +
                                                         (2 * ro + (y >> 3)) * 128 + (y & 7) * 16);
  // epilogue role: own subaperture = rows 32 (warp & 3) .. of tile warp >> 2
  const uint32_t d2_addr = tmem_base + ((uint32_t)(32 * qq) << 16) + (uint32_t)(64 + 64 * ro);

  const long long total = (long long)p.E * p.nvalid;
  const long long base = (long long)blockIdx.x * f.items_per_cta;
  long long end = base + f.items_per_cta;
  if (end > total) end = total;
  const int n_cta = (int)(end - base);                          // > 0 by construction of the grid
  const int n_iter = (n_cta + WU_WARPS - 1) / WU_WARPS;         // every warp runs the same number of iterations
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

  const uint32_t q_a1 = __shfl_sync(0xffffffffu, wu_smem_u32(S.a1) >> 4, 0), q_b1 = __shfl_sync(0xffffffffu, wu_smem_u32(S.b1) >> 4, 0);
  const uint32_t q_a2 = __shfl_sync(0xffffffffu, wu_smem_u32(S.a2) >> 4, 0), q_b2 = __shfl_sync(0xffffffffu, wu_smem_u32(S.b2) >> 4, 0);
  const uint32_t arr_bar = wu_smem_u32(S.bar + 10);
  // which = 0: MMA 1 (A1 written, T drained), 1: MMA 2 (A2 written, Y drained)
  auto arrive_and_issue = [&](int which, uint32_t arr_parity) {
    if (wu_arrive(arr_bar + 8u * which, lane, true) && wu_elect_acquire(arr_bar + 8u * which, arr_parity, f.err)) {
      if (which == 0) {
        wu_issue_mma1(tmem_base, q_a1, q_b1);
        wu_commit(mma1_bar);
      } else {
        wu_issue_mma2<FULL>(tmem_base + 64u, q_a2, q_b2);
        wu_commit(mma2_bar);
      }
    }
    __syncwarp();
  };

  const bool plain = (p.noise < 0.f) && (p.bincube == nullptr);
  // q[m]: |Y|^2 of this fx row summed over the fy pair (2m, 2m+1) -> py = 8 + m (first half) or m (second half)
  auto sq_half = [&](const uint32_t (&v)[32], float (&q)[8]) {
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const float a0 = __uint_as_float(v[4 * m]), a1 = __uint_as_float(v[4 * m + 1]);
      const float a2 = __uint_as_float(v[4 * m + 2]), a3 = __uint_as_float(v[4 * m + 3]);
      q[m] = fmaf(a3, a3, fmaf(a2, a2, fmaf(a1, a1, a0 * a0)));
    }
  };
  // ---- epilogue of one subaperture: lane = kept fx index; qa / qb = the fy pairs of py 8..15 / 0..7 ----
  auto epilogue = [&](const float (&qa)[8], const float (&qb)[8], wu_f2 s0p, wu_f2 syp, int ie, int ik, bool pl) {
    const int pr = lane >> 1;                                  // fx pair: kept indices 2 pr, 2 pr + 1
    const int px = (pr < 8) ? 8 + pr : pr - 8;
    float s0 = 0.f, sx = 0.f, sy = 0.f;
    if (pl) {
      float a, b;
      wu_upk(s0p, a, b); s0 = a + b;
      wu_upk(syp, a, b); sy = a + b;
      sx = s0 * (float)px;
    } else {
      // fx half of the binning: rows 2 pr, 2 pr + 1 are lanes 2 pr, 2 pr + 1; the even lane keeps fy pairs 0..7
      // (py 8..15), the odd one 8..15 (py 0..7)
      float mine[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float give = (lane & 1) ? qa[j] : qb[j];
        const float keep = (lane & 1) ? qb[j] : qa[j];
        mine[j] = keep + __shfl_xor_sync(0xffffffffu, give, 1);
      }
      const int py0 = (lane & 1) ? 0 : 8;
      float tot = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) tot += mine[j];
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, sft);
      const float scale = nphotons_of<NE>(p, ie) * p.flux[ik] / tot;
      const float noise = noise_of<NE>(p, ie);
      const uint32_t k0 = p.k0[ie], k1 = p.k1[ie], fr = noise_frame(p, ie);
      float* cube = p.bincube ? p.bincube + ((size_t)ie * p.nvalid + ik) * 256 : nullptr;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int py = py0 + j;
        const int pidx = py * 16 + px;
        float v = mine[j] * scale;
        v = aom_pixel_noise(v, noise, (uint32_t)(ik * 256 + pidx), fr, p.wfs_index, k0, k1);
        if (cube) cube[pidx] = v;
        s0 += v;
        sx = fmaf(v, (float)px, sx);
        sy = fmaf(v, (float)py, sy);
      }
    }
    wu_cog_store(p, lane, s0, sx, sy, ie, ik);
  };

  // ---- prologue: item 0 entirely, the record of item 1 ----
  uint32_t ek0 = 0, ek1 = 0, ek2 = 0;          // (e << 16 | k) of the items in the F / C / E phases
  if (n_mine > 0) {
    const uint2 sb0 = __ldg(f.sub + k);
    ek0 = ((uint32_t)e << 16) | (uint32_t)k;
    int k1n = k + WU_WARPS;  k1n -= (k1n >= p.nvalid) ? p.nvalid : 0;
    issue_aux(e, k, sb0, 0, k1n, n_mine > 1);
    issue_tiles(e, sb0);
  }
  uint32_t xy_cur = 0, xy_next = 0;            // (y0 << 16 | x0) of the item sampled now / next
  if (n_mine > 0) xy_cur = __ldg(f.sub + k).x;

  for (int it = 0; it < n_iter + 2; ++it) {
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

    // ---- stage 1 of the previous iteration is complete: A1 reusable, T(it-1) in TMEM.  Its read-out is requested here
    //      and lands while the field below is evaluated ----
    const bool conv = it > 0 && it <= n_iter;
    uint32_t tv[32];
    if (conv) {
      wu_mbar_wait(mma1_bar, (uint32_t)((it - 1) & 1), f.err);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      wu_tmem_ld32(d1_addr, tv);
    }

    if (c_valid) {
      wu_field(P, c_pm, kt, hc01, re_h, re_l, im_h, im_l);
    }

    if (c_valid) {
      wu_store_a1(a1_addr, re_h, re_l, im_h, im_l);
    }
    if (conv) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    if (it < n_iter) arrive_and_issue(0, (uint32_t)(it & 1));             // A1(it) written and T(it-1) drained by this warp

    // stage 2 of iteration it-2 is complete: A2 reusable, Y(it-2) in TMEM
    const bool epi = it > 1;
    uint32_t yv[32];
    if (epi) {
      wu_mbar_wait(mma2_bar, (uint32_t)((it - 2) & 1), f.err);
    }
    if (conv) wu_store_a2<FULL>(a2_addr, 0u, tv);   // C(it-1): T -> fp16 hi / lo -> A2

    // ---- E(it-2) ----
    // plain path of item it-2: the batch's, or with NE its environment's (a noise-free environment of a mixed launch
    // takes exactly the path of a uniform noise-free launch)
    const bool pl = NE ? (p.bincube == nullptr && noise_of<NE>(p, (int)(ek2 >> 16)) < 0.f) : plain;
    float qa[8], qb[8];
    wu_f2 s0p = 0ull, syp = 0ull;
    if (epi) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      wu_tmem_ld32(d2_addr, yv);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (pl) wu_sq_plain(yv, 8.f, s0p, syp, true); else sq_half(yv, qa);
      wu_tmem_ld32(d2_addr + 32u, yv);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (pl) wu_sq_plain(yv, 0.f, s0p, syp, false); else sq_half(yv, qb);
    }
    if (conv) arrive_and_issue(1, (uint32_t)((it - 1) & 1));                    // A2(it-1) written and Y(it-2) drained by this warp
    if (epi && it - 2 < n_mine) epilogue(qa, qb, s0p, syp, (int)(ek2 >> 16), (int)(ek2 & 0xffffu), pl);

    xy_cur = xy_next;
    ek2 = ek1; ek1 = ek0;
    ek0 = ((uint32_t)e << 16) | (uint32_t)k;          // the item prefetched in this iteration is sampled in the next
  }

  wu_cta_release(warp, tmem_base);
}
