// Shared device helpers for libwbk (sm_100a).  Block-wide helpers are written with
// block-stride loops + barriers so they are valid for any blockDim that is a multiple
// of 32 (and for the fibre emulator used by the CPU-only tests).
#pragma once

#ifndef WBK_EMU
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#define WBK_LAUNCH_RAW(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define WBK_DYN_SMEM(type, name)                        \
  extern __shared__ __align__(16) unsigned char wbk_dyn_smem_raw[]; \
  type* name = reinterpret_cast<type*>(wbk_dyn_smem_raw)
#endif

#include "../../include/wbk.h"

// kernel ids for the profiler (names in wbk_core.cu)
enum WbkKernelId {
  KID_SMOOTH = 0, KID_CONVOLVE, KID_NAN_BORDER, KID_MFLUX, KID_FLIP, KID_SYNTH, KID_MS_SEGMENTS, KID_CONTOUR_LINK,
  KID_CONTOUR_PACK, KID_SELECT, KID_OVERTURNING, KID_STREAMER_PREP, KID_TILE_SCAN, KID_PAIR_SCAN, KID_CASCADE,
  KID_EVENT_LIST, KID_EVENTS_RASTER, KID_RINGS_RASTER, KID_OWNER, KID_EVENTS_GATHER, KID_TRACK_OVERLAP, KID_MISC, KID_SPLIT, KID_SPLIT_RASTER, KID_TOUCH, KID_FINISH, KID_SMOOTH_MS, KID_TRACK_PAIRS, KID_TRACK_EXACT, KID_TRACK_DIST,
  KID_FLAG_COUNTS, KID_TRACK_APPEND
};
void wbk_prof_begin(int kid, void* stream);
void wbk_prof_end(int kid, void* stream);
#ifdef WBK_EMU
#define WBK_LAUNCH_RAW(kernel, grid, block, smem, stream, ...) simt::launch(kernel, dim3(grid), dim3(block), (size_t)(smem), __VA_ARGS__)
#endif
// launch with launch counting / optional event timing
#define WBK_LAUNCH(kid, kernel, grid, block, smem, stream, ...)             \
  do {                                                                      \
    wbk_prof_begin((kid), (void*)(stream));                                 \
    WBK_LAUNCH_RAW(kernel, grid, block, smem, stream, __VA_ARGS__);         \
    wbk_prof_end((kid), (void*)(stream));                                   \
  } while (0)

#define WBK_FULL 0xffffffffu
#define WBK_NONE 0xffffffffu

typedef unsigned int u32;
typedef unsigned long long u64;
typedef long long i64;

// ---------------------------------------------------------------- small utilities
__device__ __forceinline__ int wbk_tid() { return threadIdx.x; }
__device__ __forceinline__ int wbk_nthreads() { return blockDim.x; }
__device__ __forceinline__ int wbk_lane() { return threadIdx.x & 31; }
__device__ __forceinline__ int wbk_warp() { return threadIdx.x >> 5; }

__host__ __device__ __forceinline__ u32 wbk_pow2_ceil(u32 v) {
  u32 p = 1;
  while (p < v) p <<= 1;
  return p;
}
__host__ __device__ __forceinline__ int wbk_log2_ceil(u32 v) {
  int l = 0;
  while ((1u << l) < v) ++l;
  return l;
}

__device__ __forceinline__ u32 wbk_hash32(u32 x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}
__device__ __forceinline__ u32 wbk_hash64(u64 x) {
  x ^= x >> 33;
  x *= 0xff51afd7ed558ccdULL;
  x ^= x >> 33;
  x *= 0xc4ceb9fe1a85ec53ULL;
  x ^= x >> 33;
  return (u32)x;
}

// packed lattice point: x in the low 16 bits, y in the high 16 bits
__host__ __device__ __forceinline__ u32 wbk_pack_xy(int x, int y) { return (u32)(x & 0xffff) | ((u32)y << 16); }
__host__ __device__ __forceinline__ int wbk_px(u32 p) { return (int)(p & 0xffffu); }
__host__ __device__ __forceinline__ int wbk_py(u32 p) { return (int)(p >> 16); }

// ---------------------------------------------------------------- warp collectives
__device__ __forceinline__ int wbk_warp_incl_scan(int v) {
  int lane = wbk_lane();
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(WBK_FULL, v, d);
    if (lane >= d) v += t;
  }
  return v;
}
__device__ __forceinline__ int wbk_warp_sum(int v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(WBK_FULL, v, d);
  return v;
}
__device__ __forceinline__ int wbk_warp_max(int v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = max(v, __shfl_xor_sync(WBK_FULL, v, d));
  return v;
}
__device__ __forceinline__ int wbk_warp_min(int v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = min(v, __shfl_xor_sync(WBK_FULL, v, d));
  return v;
}
__device__ __forceinline__ double wbk_warp_sum_f64(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(WBK_FULL, v, d);
  return v;
}

// ---------------------------------------------------------------- block collectives
// Exclusive prefix sum over data[0..n) in place (int); returns the total to every thread.
// scratch: >= 34 ints of shared memory.  All threads of the block must call.
__device__ inline int wbk_block_excl_scan(int* data, int n, int* scratch) {
  const int tid = wbk_tid(), nt = wbk_nthreads();
  const int lane = wbk_lane(), warp = wbk_warp(), nwarps = nt >> 5;
  // each thread owns a contiguous chunk
  const int chunk = (n + nt - 1) / nt;
  const int b = min(n, tid * chunk), e = min(n, b + chunk);
  int s = 0;
  for (int i = b; i < e; ++i) s += data[i];
  int incl = wbk_warp_incl_scan(s);
  if (lane == 31) scratch[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = lane < nwarps ? scratch[lane] : 0;
    int wi = wbk_warp_incl_scan(w);
    if (lane < nwarps) scratch[lane] = wi - w;
    if (lane == 31) scratch[32] = wi;
  }
  __syncthreads();
  int run = scratch[warp] + incl - s;
  const int total = scratch[32];
  for (int i = b; i < e; ++i) {
    int v = data[i];
    data[i] = run;
    run += v;
  }
  __syncthreads();
  return total;
}

// Inclusive running maximum over data[0..n) in place.
__device__ inline void wbk_block_incl_max_scan(int* data, int n, int* scratch) {
  const int tid = wbk_tid(), nt = wbk_nthreads();
  const int lane = wbk_lane(), warp = wbk_warp(), nwarps = nt >> 5;
  const int chunk = (n + nt - 1) / nt;
  const int b = min(n, tid * chunk), e = min(n, b + chunk);
  const int NEG = -2147483647 - 1;
  int s = NEG;
  for (int i = b; i < e; ++i) s = max(s, data[i]);
  int incl = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(WBK_FULL, incl, d);
    if (lane >= d) incl = max(incl, t);
  }
  if (lane == 31) scratch[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = lane < nwarps ? scratch[lane] : NEG;
    int wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int t = __shfl_up_sync(WBK_FULL, wi, d);
      if (lane >= d) wi = max(wi, t);
    }
    // exclusive: max of previous warps
    int prev = __shfl_up_sync(WBK_FULL, wi, 1);
    if (lane == 0) prev = NEG;
    if (lane < nwarps) scratch[lane] = prev;
  }
  __syncthreads();
  int before = __shfl_up_sync(WBK_FULL, incl, 1);
  if (lane == 0) before = NEG;
  int run = max(scratch[warp], before);
  for (int i = b; i < e; ++i) {
    run = max(run, data[i]);
    data[i] = run;
  }
  __syncthreads();
}

// Block-wide double sum in a fixed (deterministic) tree order; result to every thread.
__device__ inline double wbk_block_sum_f64(double v, double* scratch /* >= 33 doubles */) {
  const int lane = wbk_lane(), warp = wbk_warp(), nwarps = wbk_nthreads() >> 5;
  v = wbk_warp_sum_f64(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  if (warp == 0) {
    double w = lane < nwarps ? scratch[lane] : 0.0;
    w = wbk_warp_sum_f64(w);
    if (lane == 0) scratch[32] = w;
  }
  __syncthreads();
  return scratch[32];
}

// In-place ascending bitonic sort of keys[0..npow2) (npow2 a power of two; pad with ~0).
// Works on shared or global memory; all threads of the block must call.
__device__ inline void wbk_block_bitonic_sort(u64* keys, u32 npow2) {
  const int tid = wbk_tid(), nt = wbk_nthreads();
  for (u32 k = 2; k <= npow2; k <<= 1) {
    for (u32 j = k >> 1; j > 0; j >>= 1) {
      for (u32 i = tid; i < npow2; i += nt) {
        u32 ixj = i ^ j;
        if (ixj > i) {
          u64 a = keys[i], b = keys[ixj];
          bool up = ((i & k) == 0);
          if ((a > b) == up) {
            keys[i] = b;
            keys[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------- open-addressing hash (u32 key -> u32 val)
// table: 2*cap u32 (keys then vals); cap power of two; keys initialised to WBK_NONE.
__device__ __forceinline__ void wbk_hash_insert32(u32* keys, u32* vals, u32 cap, u32 key, u32 val) {
  u32 h = wbk_hash32(key) & (cap - 1);
  while (true) {
    u32 prev = atomicCAS(&keys[h], (u32)WBK_NONE, key);
    if (prev == WBK_NONE || prev == key) {
      vals[h] = val;
      return;
    }
    h = (h + 1) & (cap - 1);
  }
}
__device__ __forceinline__ u32 wbk_hash_find32(const u32* keys, const u32* vals, u32 cap, u32 key) {
  u32 h = wbk_hash32(key) & (cap - 1);
  while (true) {
    u32 k = keys[h];
    if (k == key) return vals[h];
    if (k == WBK_NONE) return WBK_NONE;
    h = (h + 1) & (cap - 1);
  }
}

// u64 key -> slot index (insert-or-find); keys initialised to ~0ull.  Returns the slot.
__device__ __forceinline__ u32 wbk_hash_slot64(u64* keys, u32 cap, u64 key, bool* is_new) {
  u32 h = wbk_hash64(key) & (cap - 1);
  while (true) {
    u64 prev = atomicCAS(&keys[h], ~0ull, key);
    if (prev == ~0ull) {
      if (is_new) *is_new = true;
      return h;
    }
    if (prev == key) {
      if (is_new) *is_new = false;
      return h;
    }
    h = (h + 1) & (cap - 1);
  }
}
__device__ __forceinline__ u32 wbk_hash_lookup64(const u64* keys, u32 cap, u64 key) {
  u32 h = wbk_hash64(key) & (cap - 1);
  while (true) {
    u64 k = keys[h];
    if (k == key) return h;
    if (k == ~0ull) return WBK_NONE;
    h = (h + 1) & (cap - 1);
  }
}

// ---------------------------------------------------------------- host side error plumbing
void wbk_set_error(const char* fmt, ...);
#ifndef WBK_EMU
#define WBK_CUDA_CHECK(expr)                                                          \
  do {                                                                                \
    cudaError_t e_ = (expr);                                                          \
    if (e_ != cudaSuccess) {                                                          \
      wbk_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return WBK_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)
#else
#define WBK_CUDA_CHECK(expr) do { (void)(expr); } while (0)
#endif
#define WBK_LAUNCH_CHECK() WBK_CUDA_CHECK(cudaGetLastError())
