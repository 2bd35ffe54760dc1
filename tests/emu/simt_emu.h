// SIMT emulation shim -- TEST INFRASTRUCTURE ONLY.
//
// Lets the CUDA sources under wavebreaking_b200/csrc/ be compiled by g++ (-x c++
// -include simt_emu.h -DWBK_EMU) and executed on the host so that the integer / index
// logic of the kernels can be unit-tested in the CPU-only CI container.  Every CUDA
// thread of a CTA runs as a ucontext fiber; __syncthreads() and the warp collectives
// are rendezvous points between fibers.  CTAs run one after another.  "Device" memory
// is plain host memory.  The product package never loads a library built this way
// (wavebreaking_b200/_lib.py only loads the nvcc-built libwbk.so and refuses to run
// without a CUDA device); tests/emu builds and loads it explicitly.
#pragma once
#include <ucontext.h>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <algorithm>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __grid_constant__
#define __restrict__
#define __launch_bounds__(...)
#define __shared__ static
#define __constant__ static
#define __align__(n) __attribute__((aligned(n)))

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct uint3_ { unsigned x, y, z; };

typedef int cudaError_t;
typedef void* cudaStream_t;
#define cudaSuccess 0
enum cudaMemcpyKind { cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };

namespace simt {
struct Fiber {
  ucontext_t ctx;
  char* stack;
  uint3_ tid;
  int lin;          // linear thread id
  int state;        // 0 runnable, 1 waiting at CTA barrier, 2 waiting at warp barrier, 3 done
  unsigned long long xchg;  // shuffle / ballot exchange slot
};
extern Fiber* cur;
extern ucontext_t sched_ctx;
extern uint3_ g_blockIdx;
extern dim3 g_blockDim, g_gridDim;
extern unsigned char* g_dyn_smem;
extern std::vector<Fiber> fibers;
void yield_wait(int state);
void run_grid(void (*entry)(void*), void* args, dim3 grid, dim3 block, size_t smem);
inline int warp_base() { return (cur->lin / 32) * 32; }
inline int warp_lanes() {
  int total = (int)(g_blockDim.x * g_blockDim.y * g_blockDim.z);
  int b = warp_base();
  return std::min(32, total - b);
}
void warp_sync();
}  // namespace simt

#define threadIdx (simt::cur->tid)
#define blockIdx (simt::g_blockIdx)
#define blockDim (simt::g_blockDim)
#define gridDim (simt::g_gridDim)
#define warpSize 32

inline void __syncthreads() { simt::yield_wait(1); }
inline void __syncwarp(unsigned = 0xffffffffu) { simt::warp_sync(); }
inline void __threadfence() {}
inline void __threadfence_block() {}

template <typename T>
inline T simt_shfl_from(T v, int src_lane) {
  unsigned long long raw = 0;
  std::memcpy(&raw, &v, sizeof(T));
  simt::cur->xchg = raw;
  simt::warp_sync();
  int base = simt::warp_base();
  int n = simt::warp_lanes();
  T out = v;
  if (src_lane >= 0 && src_lane < n) {
    unsigned long long r = simt::fibers[base + src_lane].xchg;
    std::memcpy(&out, &r, sizeof(T));
  }
  simt::warp_sync();
  return out;
}
template <typename T>
inline T __shfl_sync(unsigned, T v, int src, int width = 32) {
  int lane = simt::cur->lin % 32;
  int seg = (lane / width) * width;
  return simt_shfl_from(v, seg + (src % width));
}
template <typename T>
inline T __shfl_up_sync(unsigned, T v, unsigned d, int width = 32) {
  int lane = simt::cur->lin % 32;
  int seg = (lane / width) * width;
  int src = lane - (int)d;
  return simt_shfl_from(v, src < seg ? lane : src);
}
template <typename T>
inline T __shfl_down_sync(unsigned, T v, unsigned d, int width = 32) {
  int lane = simt::cur->lin % 32;
  int seg = (lane / width) * width;
  int src = lane + (int)d;
  return simt_shfl_from(v, src >= seg + width ? lane : src);
}
template <typename T>
inline T __shfl_xor_sync(unsigned, T v, int m, int width = 32) {
  int lane = simt::cur->lin % 32;
  return simt_shfl_from(v, lane ^ m);
}
inline unsigned __ballot_sync(unsigned, int pred) {
  simt::cur->xchg = pred ? 1ull : 0ull;
  simt::warp_sync();
  int base = simt::warp_base();
  int n = simt::warp_lanes();
  unsigned out = 0;
  for (int i = 0; i < n; ++i)
    if (simt::fibers[base + i].state != 3 && simt::fibers[base + i].xchg) out |= (1u << i);
  simt::warp_sync();
  return out;
}
inline int __any_sync(unsigned m, int pred) { return __ballot_sync(m, pred) != 0; }
inline int __all_sync(unsigned m, int pred) {
  unsigned b = __ballot_sync(m, pred);
  int n = simt::warp_lanes();
  unsigned full = n == 32 ? 0xffffffffu : ((1u << n) - 1u);
  return b == full;
}
inline unsigned __activemask() { return 0xffffffffu; }
inline int __syncthreads_or(int pred) {
  static int acc;
  __syncthreads();
  if (simt::cur->lin == 0) acc = 0;
  __syncthreads();
  if (pred) acc = 1;
  __syncthreads();
  return acc;
}
inline int __syncthreads_count(int pred) {
  static int acc;
  __syncthreads();
  if (simt::cur->lin == 0) acc = 0;
  __syncthreads();
  if (pred) acc += 1;
  __syncthreads();
  return acc;
}

inline int __popc(unsigned v) { return __builtin_popcount(v); }
inline int __popcll(unsigned long long v) { return __builtin_popcountll(v); }
inline int __ffs(int v) { return __builtin_ffs(v); }
inline int __ffsll(long long v) { return __builtin_ffsll(v); }
inline int __clz(int v) { return v == 0 ? 32 : __builtin_clz((unsigned)v); }
inline int __clzll(long long v) { return v == 0 ? 64 : __builtin_clzll((unsigned long long)v); }

template <typename T> inline T atomicAdd(T* p, T v) { T o = *p; *p = o + v; return o; }
template <typename T> inline T atomicSub(T* p, T v) { T o = *p; *p = o - v; return o; }
template <typename T> inline T atomicMin(T* p, T v) { T o = *p; if (v < o) *p = v; return o; }
template <typename T> inline T atomicMax(T* p, T v) { T o = *p; if (v > o) *p = v; return o; }
template <typename T> inline T atomicOr(T* p, T v) { T o = *p; *p = o | v; return o; }
template <typename T> inline T atomicAnd(T* p, T v) { T o = *p; *p = o & v; return o; }
template <typename T> inline T atomicExch(T* p, T v) { T o = *p; *p = v; return o; }
template <typename T> inline T atomicCAS(T* p, T cmp, T v) { T o = *p; if (o == cmp) *p = v; return o; }

template <typename T> inline T __ldg(const T* p) { return *p; }
inline double __dadd_rn(double a, double b) { volatile double r = a + b; return r; }
inline double __dsub_rn(double a, double b) { volatile double r = a - b; return r; }
inline double __dmul_rn(double a, double b) { volatile double r = a * b; return r; }
inline double __ddiv_rn(double a, double b) { volatile double r = a / b; return r; }
inline float __double2float_rn(double a) { return (float)a; }
inline double __fma_rn(double a, double b, double c) { return std::fma(a, b, c); }
inline long long __double2ll_rd(double a) { return (long long)std::floor(a); }
inline int __double2int_rn(double a) { return (int)std::nearbyint(a); }
inline int __double2int_rz(double a) { return (int)a; }
inline unsigned long long __double_as_longlong(double a) { unsigned long long r; std::memcpy(&r, &a, 8); return r; }
inline double __longlong_as_double(long long a) { double r; std::memcpy(&r, &a, 8); return r; }
using std::isnan;
using std::max;
using std::min;

// ---- runtime API subset (host memory stands in for device memory)
inline cudaError_t cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t = 0) { std::memset(p, v, n); return 0; }
inline cudaError_t cudaMemset(void* p, int v, size_t n) { std::memset(p, v, n); return 0; }
inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = 0) { std::memmove(d, s, n); return 0; }
inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { std::memmove(d, s, n); return 0; }
inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
inline cudaError_t cudaDeviceSynchronize() { return 0; }
inline cudaError_t cudaGetLastError() { return 0; }
inline cudaError_t cudaPeekAtLastError() { return 0; }
inline const char* cudaGetErrorString(cudaError_t) { return "emu"; }
inline cudaError_t cudaMalloc(void** p, size_t n) { *p = std::malloc(n ? n : 1); return *p ? 0 : 2; }
inline cudaError_t cudaFree(void* p) { std::free(p); return 0; }
inline cudaError_t cudaSetDevice(int) { return 0; }
inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
struct cudaDeviceProp { int multiProcessorCount; size_t sharedMemPerBlockOptin; };
inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) { p->multiProcessorCount = 4; p->sharedMemPerBlockOptin = 227 * 1024; return 0; }
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize };
template <typename F> inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return 0; }

// ---- launch
#define WBK_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(simt::g_dyn_smem)

namespace simt {
template <typename... Args>
struct LaunchPack;
}

#include <tuple>
#include <utility>
namespace simt {
template <typename K, typename Tuple, size_t... I>
inline void call_kernel(K k, Tuple& t, std::index_sequence<I...>) { k(std::get<I>(t)...); }

template <typename K, typename... Args>
inline void launch(K kernel, dim3 grid, dim3 block, size_t smem, Args... args) {
  struct Pack { K k; std::tuple<Args...> a; } pack{kernel, std::tuple<Args...>(args...)};
  auto entry = [](void* p) {
    Pack* pk = static_cast<Pack*>(p);
    call_kernel(pk->k, pk->a, std::index_sequence_for<Args...>{});
  };
  run_grid(entry, &pack, grid, block, smem);
}
}  // namespace simt


struct double2 { double x, y; };
struct float4 { float x, y, z, w; };
struct float2 { float x, y; };
struct int2 { int x, y; };
struct int4 { int x, y, z, w; };
struct uint4 { unsigned x, y, z, w; };
#ifdef WBK_EMU_SINF_WORST
// __sinf at the worst case the CUDA programming guide documents for it (maximum absolute error 2^-21.41 on
// [-pi, pi]): the correctly rounded sine moved by that much, the sign alternating from call to call, so that the
// fp32 prefilter of the pair scan is checked against the documented bound rather than against an exact sine
inline float __sinf(float v) {
  static thread_local unsigned calls = 0;
  const double e = 3.6471e-7;  // 2^-21.41, rounded up
  return (float)((double)std::sin(v) + ((calls++ & 1u) ? e : -e));
}
#else
inline float __sinf(float v) { return std::sin(v); }
#endif
inline double2 make_double2(double x, double y) { double2 r; r.x = x; r.y = y; return r; }
inline float4 make_float4(float x, float y, float z, float w) { float4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }
inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { uint4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }
inline float __uint_as_float(unsigned v) { float f; std::memcpy(&f, &v, 4); return f; }
inline unsigned __float_as_uint(float f) { unsigned v; std::memcpy(&v, &f, 4); return v; }
