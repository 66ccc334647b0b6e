// Per-environment snapshots (aom_save_envs / aom_load_envs): one record per environment, a run of 16-byte-aligned
// segments.  The head (aom_env_head of aomarl.h: magic, size, configuration fingerprint, counters relative to the
// environment, wind state and resolved conditions) comes first, then one segment per row of the enumeration of the
// per-environment state (env_rows in aomarl.cu), each slot of a row padded to 16 bytes.
//
// grid (chunks + 1, n): block (c < chunks, k) moves chunk c of the segments of record k with 128-bit loads and stores
// where the context's row is 16-byte aligned (32-bit words otherwise); block (chunks, k) writes (pack) or applies
// (unpack) the head.  The command history is stored in logical order, oldest slot first: slot s of the record is
// physical slot (s + hist_head) % n_hist of the context.  Counters are stored relative to the environment's reset and
// rebased onto the context's global counters on unpack.
//
// Next to them the other per-environment bookkeeping: the restart of listed environments (aom_reset_envs), whose rows
// are those of the same enumeration, and the per-environment counters of a batch that leaves lockstep.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/aomarl.h"

// aom_reset_envs: restart listed environments while the others run on.
#define RESET_MAX_BUFS (18 + 4 * AOM_MAX_LAYERS)    // controller, state and Strehl rows + screen and ring state per layer
struct ResetEnvsParams {
  // per-environment buffers whose rows are zeroed: word (s * slot_stride + e * ld + i), s < slots, i < ld
  uint32_t* buf[RESET_MAX_BUFS];
  long long ld[RESET_MAX_BUFS], slot_stride[RESET_MAX_BUFS];
  int slots[RESET_MAX_BUFS];
  int nbuf;
  const int* envs;              // [K] environments to restart
  const uint32_t* seeds;        // [2][K] low, high words of their new seeds
  int K, E;
  uint32_t *k0, *k1;            // [E] Philox keys
  uint32_t* frame0;             // [E] noise frame of the environment's first sensor frame
  uint32_t* step_env;           // [E] actor decision counters
  int* le_n;                    // [2][E] long-exposure counts (main target, geometric target)
  int* first;                   // [E] first step pending
  uint32_t frame;
};

// grid (K, nbuf + 1): block (k, b < nbuf) zeroes the rows of buffer b of environment envs[k]; block (k, nbuf) sets its
// keys and counters.
__global__ void __launch_bounds__(256) reset_envs_kernel(const __grid_constant__ ResetEnvsParams P) {
  const int k = blockIdx.x, b = blockIdx.y, e = P.envs[k];
  if (b < P.nbuf) {
    uint32_t* base = P.buf[b] + (size_t)e * P.ld[b];
    for (int s = 0; s < P.slots[b]; ++s)
      for (long long i = threadIdx.x; i < P.ld[b]; i += blockDim.x) base[s * P.slot_stride[b] + i] = 0u;
    return;
  }
  if (threadIdx.x == 0) {
    P.k0[e] = P.seeds[k];
    P.k1[e] = P.seeds[P.K + k];
    P.frame0[e] = P.frame;
    P.step_env[e] = 0u;
    P.le_n[e] = 0;
    P.le_n[P.E + e] = 0;
    P.first[e] = 1;
  }
}

// The per-environment counters when the batch stops running in lockstep: every environment at the batch's counts.
__global__ void stagger_counters_kernel(uint32_t* frame0, uint32_t* step_env, int* le_n, int* first, int E, uint32_t step,
                                        int n_main, int n_geo) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  frame0[e] = 0u;
  step_env[e] = step;
  le_n[e] = n_main;
  le_n[E + e] = n_geo;
  first[e] = 0;
}

// ---------------------------------------------------------------------------------------------
// aom_save_envs / aom_load_envs
#define SNAP_MAX_SEGS (RESET_MAX_BUFS + 4)    // rows aom_reset_envs clears + keys and pending target sums
#define SNAP_CHUNK_WORDS 8192                 // 32 KB of a slot per block
#define SNAP_THREADS 256
#define SNAP_HEAD_BYTES ((sizeof(aom_env_head) + 15) / 16 * 16)

struct SnapSeg {
  uint32_t* buf;            // word (s * slot_stride + e * ld + i) of the context, s < slots, i < ld
  long long ld, slot_stride;
  long long off, pitch;     // byte offset of the segment in the record, bytes per slot there (ld words rounded to 16 B)
  int slots, ring;          // ring: the command history (logical slot order in the record)
  int chunk0, cps;          // first chunk of the segment, chunks per slot
};

struct SnapParams {
  SnapSeg seg[SNAP_MAX_SEGS];
  int nseg, nchunks;
  const int* envs;          // [n] environments (device)
  unsigned char* rec;       // [n][bytes] records
  long long bytes;
  int E, hist_head;
  // head: constants of this context
  uint32_t magic, rec_bytes;
  uint64_t fingerprint;
  int n_layers;
  // counters: global ones, and the per-environment arrays while environments are staggered (else null)
  uint32_t frame, step;
  int le_c[2];
  uint32_t *frame0, *step_env;
  int *le_n, *first;
  // pack: wind state and conditions [aom_condition][layer], each a per-environment array while in force, else null
  const double* wind_acc;   // [L][2][E] or null
  double acc_c[AOM_MAX_LAYERS][2];
  const float* cond_env[AOM_COND_COUNT][AOM_MAX_LAYERS];
  float cond_c[AOM_COND_COUNT][AOM_MAX_LAYERS];
};

// Layers of condition k in a context of L layers (none for the unassigned value between AOM_COND_GAIN and
// AOM_COND_DELAY), and its field of layer l in a record head
__host__ __device__ __forceinline__ int cond_layers(int k, int L) {
  return k <= AOM_COND_WIND_Y ? L : k <= AOM_COND_GAIN || k == AOM_COND_DELAY ? 1 : 0;
}

__host__ __device__ __forceinline__ float& head_cond(aom_env_head& h, int k, int l) {
  switch (k) {
    case AOM_COND_AMP: return h.amp[l];
    case AOM_COND_WIND_X: return h.wind[l][0];
    case AOM_COND_WIND_Y: return h.wind[l][1];
    case AOM_COND_NOISE: return h.noise;
    case AOM_COND_NPHOTONS: return h.nphotons;
    case AOM_COND_DELAY: return h.delay;
    default: return h.gain;
  }
}

template <bool LOAD>
__device__ __forceinline__ void snap_words(uint32_t* ctx_row, uint32_t* rec_row, long long n) {
  // the record side is always 16-byte aligned; the context side is when its row starts on 16 bytes
  long long i = 0;
  if (((uintptr_t)ctx_row & 15) == 0) {
    const long long n4 = n >> 2;
    uint4* a = reinterpret_cast<uint4*>(ctx_row);
    uint4* b = reinterpret_cast<uint4*>(rec_row);
    for (long long j = threadIdx.x; j < n4; j += blockDim.x) {
      if (LOAD) a[j] = b[j];
      else b[j] = a[j];
    }
    i = n4 << 2;
  }
  for (long long j = i + threadIdx.x; j < n; j += blockDim.x) {
    if (LOAD) ctx_row[j] = rec_row[j];
    else rec_row[j] = ctx_row[j];
  }
}

template <bool LOAD>
__device__ __forceinline__ void snap_head(const SnapParams& P, int e, aom_env_head* h) {
  if (threadIdx.x) return;
  const int E = P.E;
  if (LOAD) {
    // counters rebased onto this context: the environment's noise frame stays frame - frame0[e]
    P.frame0[e] = P.frame - h->frame;
    P.step_env[e] = h->step;
    P.le_n[e] = h->le_n[0];
    P.le_n[E + e] = h->le_n[1];
    P.first[e] = h->first;
    return;
  }
  aom_env_head r{};
  r.magic = P.magic; r.bytes = P.rec_bytes; r.fingerprint = P.fingerprint; r.n_layers = P.n_layers;
  r.frame = P.frame0 ? P.frame - P.frame0[e] : P.frame;
  r.step = P.step_env ? P.step_env[e] : P.step;
  r.le_n[0] = P.le_n ? P.le_n[e] : P.le_c[0];
  r.le_n[1] = P.le_n ? P.le_n[E + e] : P.le_c[1];
  r.first = P.first ? P.first[e] : 0;
  for (int l = 0; l < P.n_layers; ++l)
    for (int a = 0; a < 2; ++a) r.acc[l][a] = P.wind_acc ? P.wind_acc[(size_t)(2 * l + a) * E + e] : P.acc_c[l][a];
  for (int k = 0; k < AOM_COND_COUNT; ++k)
    for (int l = 0; l < cond_layers(k, P.n_layers); ++l) head_cond(r, k, l) = P.cond_env[k][l] ? P.cond_env[k][l][e] : P.cond_c[k][l];
  *h = r;
}

template <bool LOAD>
__device__ __forceinline__ void snap_move(const SnapParams& P) {
  const int k = blockIdx.y, e = P.envs[k], c = blockIdx.x;
  unsigned char* rec = P.rec + (size_t)k * P.bytes;
  if (c == P.nchunks) {
    snap_head<LOAD>(P, e, reinterpret_cast<aom_env_head*>(rec));
    return;
  }
  int s = 0;
  while (s + 1 < P.nseg && P.seg[s + 1].chunk0 <= c) ++s;
  const SnapSeg& G = P.seg[s];
  const int cc = c - G.chunk0, slot = cc / G.cps, part = cc - slot * G.cps;
  const int phys = G.ring ? (slot + P.hist_head) % G.slots : slot;
  const long long i0 = (long long)part * SNAP_CHUNK_WORDS;
  const long long n = min((long long)SNAP_CHUNK_WORDS, G.ld - i0);
  uint32_t* row = G.buf + (long long)phys * G.slot_stride + (long long)e * G.ld + i0;
  uint32_t* dst = reinterpret_cast<uint32_t*>(rec + G.off + (long long)slot * G.pitch) + i0;
  snap_words<LOAD>(row, dst, n);
}

__global__ void __launch_bounds__(SNAP_THREADS) env_pack_kernel(const __grid_constant__ SnapParams P) { snap_move<false>(P); }
__global__ void __launch_bounds__(SNAP_THREADS) env_unpack_kernel(const __grid_constant__ SnapParams P) { snap_move<true>(P); }
