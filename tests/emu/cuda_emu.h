// A thread-per-lane emulation of ONE CUDA thread block on the host, for `-m "not gpu"` tests of kernel logic
// (test infrastructure; nothing in the product includes it).  Every CUDA thread is an OS thread; __syncthreads,
// __syncwarp and the warp collectives (ballot, match, shuffles, reduce-or - every lane of the warp calls them) are pthread barriers plus an
// exchange buffer per warp.  Blocks of a launch run in blockIdx order, `window` of them at a time, which is how
// the hardware dispatches them; a block may therefore wait for an earlier one (decoupled look-back) but never
// for a later one.
#pragma once
// b2_common.cuh compiles its device helpers (lane_id, warp_id, the warp and block scans) for the host against the
// intrinsics restated here; no helper of the product is restated in this file
#define B2_EMU_DEVICE_HELPERS 1
#define __host__
#define __device__
#define __global__
#define __shared__
#include <cuda_runtime.h>      // vector types only (uint3, uint4, dim3); no CUDA call is made
#ifndef __launch_bounds__
#define __launch_bounds__(...)
#endif
#include <pthread.h>
#include <sched.h>

#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>

struct EmuCta {
  pthread_barrier_t cta_bar;
  pthread_barrier_t warp_bar[32];
  uint32_t xchg[32][32];
  int or_word = 0;                 // __syncthreads_or
  std::vector<unsigned char> smem;
};
static thread_local EmuCta *emu_cta = nullptr;
static thread_local uint3 threadIdx, blockIdx;
static thread_local dim3 blockDim, gridDim;

inline void emu_yield() { sched_yield(); }
inline unsigned char *emu_dynamic_smem() { return emu_cta->smem.data(); }
// A kernel's static __shared__ arrays, taken in declaration order from the CTA's memory (emu_launch's smem_bytes,
// poisoned); every thread is a fresh OS thread that runs the kernel once, so all take the same offsets.
static thread_local size_t emu_shared_used = 0;
template <class T> inline T &emu_shared() {
  const size_t at = emu_shared_used;
  emu_shared_used = (at + sizeof(T) + 15) & ~(size_t)15;
  if (emu_shared_used > emu_cta->smem.size()) { fprintf(stderr, "emu_shared: %zu bytes of shared memory, launch gave %zu\n", emu_shared_used, emu_cta->smem.size()); abort(); }
  return *reinterpret_cast<T *>(emu_cta->smem.data() + at);
}

inline void __syncthreads() { pthread_barrier_wait(&emu_cta->cta_bar); }
// every thread ORs its predicate into the CTA's word between two barriers; a third keeps the word until all have
// read it, and thread 0 clears it before anyone can pass the first barrier of the next call
inline int __syncthreads_or(int p) {
  int *w = &emu_cta->or_word;
  __syncthreads();
  if (p) __atomic_fetch_or(w, 1, __ATOMIC_RELAXED);
  __syncthreads();
  const int r = __atomic_load_n(w, __ATOMIC_RELAXED);
  __syncthreads();
  if (threadIdx.x == 0) __atomic_store_n(w, 0, __ATOMIC_RELAXED);
  return r;
}
inline void __syncwarp(unsigned = 0xffffffffu) { pthread_barrier_wait(&emu_cta->warp_bar[threadIdx.x >> 5]); }
// every lane of the warp deposits a word, then reads all 32
inline void emu_exchange(uint32_t v, uint32_t out[32]) {
  EmuCta *c = emu_cta;
  const unsigned w = threadIdx.x >> 5, l = threadIdx.x & 31;
  c->xchg[w][l] = v;
  pthread_barrier_wait(&c->warp_bar[w]);
  std::memcpy(out, c->xchg[w], sizeof(uint32_t) * 32);
  pthread_barrier_wait(&c->warp_bar[w]);
}
inline uint32_t __ballot_sync(unsigned, bool p) {
  uint32_t o[32], m = 0;
  emu_exchange(p ? 1u : 0u, o);
  for (int i = 0; i < 32; i++) m |= (o[i] & 1u) << i;
  return m;
}
inline uint32_t __match_any_sync(unsigned, uint32_t v) {
  uint32_t o[32], m = 0;
  emu_exchange(v, o);
  for (int i = 0; i < 32; i++) m |= (uint32_t)(o[i] == v) << i;
  return m;
}
inline uint32_t __shfl_sync(unsigned, uint32_t v, unsigned src) { uint32_t o[32]; emu_exchange(v, o); return o[src & 31]; }
// within segments of `width` lanes: a lane whose index in its segment is below d keeps its own value
inline uint32_t __shfl_up_sync(unsigned, uint32_t v, unsigned d, int width = 32) {
  uint32_t o[32];
  emu_exchange(v, o);
  const unsigned l = threadIdx.x & 31;
  return (l & (unsigned)(width - 1)) >= d ? o[l - d] : v;
}
// 32-bit signed, 64-bit and double shuffles move every bit (two exchanges of the halves); any other argument type
// would be converted to uint32_t and silently lose bits, so it does not compile
inline int32_t __shfl_sync(unsigned m, int32_t v, unsigned src) { return (int32_t)__shfl_sync(m, (uint32_t)v, src); }
inline int32_t __shfl_up_sync(unsigned m, int32_t v, unsigned d, int width = 32) { return (int32_t)__shfl_up_sync(m, (uint32_t)v, d, width); }
inline uint64_t emu_shfl64(uint64_t v, unsigned src) { return (uint64_t)__shfl_sync(0xffffffffu, (uint32_t)v, src) | ((uint64_t)__shfl_sync(0xffffffffu, (uint32_t)(v >> 32), src) << 32); }
inline uint64_t emu_shfl_up64(uint64_t v, unsigned d, int width) { return (uint64_t)__shfl_up_sync(0xffffffffu, (uint32_t)v, d, width) | ((uint64_t)__shfl_up_sync(0xffffffffu, (uint32_t)(v >> 32), d, width) << 32); }
inline long long __shfl_sync(unsigned, long long v, unsigned src) { return (long long)emu_shfl64((uint64_t)v, src); }
inline long long __shfl_up_sync(unsigned, long long v, unsigned d, int width = 32) { return (long long)emu_shfl_up64((uint64_t)v, d, width); }
inline unsigned long long __shfl_sync(unsigned, unsigned long long v, unsigned src) { return emu_shfl64(v, src); }
inline unsigned long long __shfl_up_sync(unsigned, unsigned long long v, unsigned d, int width = 32) { return emu_shfl_up64(v, d, width); }
inline double __shfl_sync(unsigned, double v, unsigned src) { uint64_t b; std::memcpy(&b, &v, 8); b = emu_shfl64(b, src); std::memcpy(&v, &b, 8); return v; }
inline double __shfl_up_sync(unsigned, double v, unsigned d, int width = 32) { uint64_t b; std::memcpy(&b, &v, 8); b = emu_shfl_up64(b, d, width); std::memcpy(&v, &b, 8); return v; }
template <class T> T __shfl_sync(unsigned, T, unsigned) = delete;
template <class T> T __shfl_up_sync(unsigned, T, unsigned, int = 32) = delete;
inline uint32_t __shfl_xor_sync(unsigned, uint32_t v, unsigned x) { uint32_t o[32]; emu_exchange(v, o); return o[(threadIdx.x & 31) ^ x]; }
// every lane of the warp calls it; each gets the OR over the lanes of its own mask
inline uint32_t __reduce_or_sync(unsigned mask, uint32_t v) {
  uint32_t o[32], r = 0;
  emu_exchange(v, o);
  for (int i = 0; i < 32; i++) r |= ((mask >> i) & 1u) ? o[i] : 0u;
  return r;
}
inline int __popc(uint32_t x) { return __builtin_popcount(x); }
// per byte: 0xFF where the bytes of a and b are equal
inline uint32_t __vcmpeq4(uint32_t a, uint32_t b) {
  uint32_t r = 0;
  for (int k = 0; k < 32; k += 8) r |= (((a >> k) & 0xFFu) == ((b >> k) & 0xFFu) ? 0xFFu : 0u) << k;
  return r;
}
// per byte: 0xFF where the byte of a is below the byte of b (unsigned)
inline uint32_t __vcmpltu4(uint32_t a, uint32_t b) {
  uint32_t r = 0;
  for (int k = 0; k < 32; k += 8) r |= (((a >> k) & 0xFFu) < ((b >> k) & 0xFFu) ? 0xFFu : 0u) << k;
  return r;
}
// IEEE double adds, round to nearest even (the build uses -ffp-contract=off: nothing is fused)
inline double __dadd_rn(double a, double b) { return a + b; }
inline double __dsub_rn(double a, double b) { return a - b; }
inline long long __double_as_longlong(double x) { long long r; std::memcpy(&r, &x, 8); return r; }
inline double __longlong_as_double(long long x) { double r; std::memcpy(&r, &x, 8); return r; }
inline int __ffs(uint32_t x) { return __builtin_ffs((int)x); }
inline int __clz(uint32_t x) { return x ? __builtin_clz(x) : 32; }

// Runs kernel() for every thread of every block of the grid; `window` blocks are resident at a time and blocks
// start in blockIdx order.
inline void emu_launch(unsigned grid, unsigned block, size_t smem_bytes, unsigned window, const std::function<void()> &kernel) {
  std::atomic<unsigned> next{0};
  auto worker = [&]() {
    for (;;) {
      const unsigned b = next.fetch_add(1);
      if (b >= grid) return;
      EmuCta cta;
      cta.smem.assign(smem_bytes + 16, 0xCD);              // poison: the kernel must initialise what it reads
      pthread_barrier_init(&cta.cta_bar, nullptr, block);
      for (unsigned w = 0; w < (block + 31) / 32; w++) pthread_barrier_init(&cta.warp_bar[w], nullptr, std::min(32u, block - 32 * w));
      std::vector<std::thread> th;
      th.reserve(block);
      for (unsigned t = 0; t < block; t++)
        th.emplace_back([&, t]() {
          emu_cta = &cta;
          threadIdx = uint3{t, 0, 0}; blockIdx = uint3{b, 0, 0};
          blockDim = dim3(block); gridDim = dim3(grid);
          kernel();
        });
      for (auto &x : th) x.join();
      pthread_barrier_destroy(&cta.cta_bar);
      for (unsigned w = 0; w < (block + 31) / 32; w++) pthread_barrier_destroy(&cta.warp_bar[w]);
    }
  };
  // blocks start in order because `next` is taken in order; a worker that holds block b runs it to completion
  std::vector<std::thread> ws;
  for (unsigned i = 0; i < window; i++) ws.emplace_back(worker);
  for (auto &x : ws) x.join();
}

inline bool __any_sync(unsigned, bool p) { return __ballot_sync(0xffffffffu, p) != 0u; }
inline uint32_t atomicOr(uint32_t *p, uint32_t v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
inline uint32_t atomicAdd(uint32_t *p, uint32_t v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
inline uint32_t atomicMin(uint32_t *p, uint32_t v) {
  uint32_t old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v < old && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return old;
}
// loads past the L1 / fences / back-off: no reordering or caching to model for one CTA
template <class T> inline T __ldcg(const T *p) { return *p; }
inline void __threadfence() { std::atomic_thread_fence(std::memory_order_seq_cst); }
inline void __nanosleep(unsigned) { emu_yield(); }
using std::fabs;
using std::floor;
using std::max;
using std::min;
