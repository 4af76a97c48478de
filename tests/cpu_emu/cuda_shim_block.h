// TEST INFRASTRUCTURE ONLY.
// Lets g++ compile the block-level kernels of starflate_b200/csrc (pass 2 of the single-stream
// route, the parallel block chain, batch preparation, the stored-stream copy) for the host: one
// block of N warps runs as N x 32 host threads.  Every warp has its own EmuWarp (reached through a
// thread_local pointer) on which the warp primitives rendezvous, as in cuda_shim_warp.h, and
// __syncthreads is a barrier over the whole block.  __shared__ variables are `static`, so one block
// runs at a time: the blocks of a grid run one after another, forward or last block first (the
// caller chooses), so a result that depends on the order of the warps shows.  Never built into,
// loaded by, or reachable from the product library — it is not a fallback.
//
// Kept apart from cuda_shim_warp.h (its own library, libemu_block*.so): the two define EmuWarp and
// the warp primitives differently.
#pragma once
#include <barrier>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#define __device__
#define __global__
#define __host__
#define __forceinline__ inline
#define __noinline__ inline __attribute__((noinline))
#define __launch_bounds__(...)
#define __constant__ static const
#define __shared__ static
#define __align__(n) __attribute__((aligned(n)))

struct emu_dim3 { unsigned x = 0, y = 0, z = 0; };
struct uint4 { unsigned x, y, z, w; };
static inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { return uint4{x, y, z, w}; }
static thread_local emu_dim3 threadIdx, blockIdx;
static thread_local emu_dim3 blockDim, gridDim;

struct EmuWarp {
  std::barrier<> bar{32};
  uint64_t slot[32];
};
static thread_local EmuWarp* emu_warp = nullptr;
static std::barrier<>* emu_block_bar = nullptr;  // the running block's threads

template <class T> static inline T emu_exchange(T v, unsigned src)
{
  const unsigned lane = threadIdx.x & 31u;
  uint64_t raw = 0;
  std::memcpy(&raw, &v, sizeof(T));
  emu_warp->slot[lane] = raw;
  emu_warp->bar.arrive_and_wait();
  raw = emu_warp->slot[src & 31u];
  emu_warp->bar.arrive_and_wait();
  T r;
  std::memcpy(&r, &raw, sizeof(T));
  return r;
}
template <class T> static inline T __shfl_sync(unsigned, T v, int src) { return emu_exchange(v, static_cast<unsigned>(src)); }
template <class T> static inline T __shfl_down_sync(unsigned, T v, int d)
{
  const unsigned lane = threadIdx.x & 31u;
  const unsigned src = lane + static_cast<unsigned>(d);
  return emu_exchange(v, src > 31u ? lane : src);
}
static inline unsigned __ballot_sync(unsigned, int p)
{
  const unsigned lane = threadIdx.x & 31u;
  emu_warp->slot[lane] = p ? 1u : 0u;
  emu_warp->bar.arrive_and_wait();
  unsigned m = 0;
  for (unsigned i = 0; i < 32; ++i) m |= static_cast<unsigned>(emu_warp->slot[i]) << i;
  emu_warp->bar.arrive_and_wait();
  return m;
}
static inline unsigned __reduce_max_sync(unsigned, unsigned v)
{
  const unsigned lane = threadIdx.x & 31u;
  emu_warp->slot[lane] = v;
  emu_warp->bar.arrive_and_wait();
  unsigned m = 0;
  for (unsigned i = 0; i < 32; ++i) m = emu_warp->slot[i] > m ? static_cast<unsigned>(emu_warp->slot[i]) : m;
  emu_warp->bar.arrive_and_wait();
  return m;
}
static inline int __any_sync(unsigned mask, int p) { return __ballot_sync(mask, p) != 0; }
static inline int __all_sync(unsigned mask, int p) { return __ballot_sync(mask, p) == 0xffffffffu; }
static inline void __syncwarp() { emu_warp->bar.arrive_and_wait(); }
static inline void __syncthreads() { emu_block_bar->arrive_and_wait(); }
static inline unsigned __brev(unsigned v)
{
  v = ((v >> 1) & 0x55555555u) | ((v & 0x55555555u) << 1);
  v = ((v >> 2) & 0x33333333u) | ((v & 0x33333333u) << 2);
  v = ((v >> 4) & 0x0F0F0F0Fu) | ((v & 0x0F0F0F0Fu) << 4);
  v = ((v >> 8) & 0x00FF00FFu) | ((v & 0x00FF00FFu) << 8);
  return (v >> 16) | (v << 16);
}
static inline unsigned min(unsigned a, unsigned b) { return a < b ? a : b; }
static inline int __ffs(int v) { return __builtin_ffs(v); }
static inline int __clz(int v) { return v == 0 ? 32 : __builtin_clz(static_cast<unsigned>(v)); }
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned s)
{
  return static_cast<unsigned>(((static_cast<uint64_t>(hi) << 32) | lo) >> (s & 31u));
}
static inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
static inline unsigned atomicOr(unsigned* p, unsigned v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
static inline unsigned atomicAdd(unsigned* p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v)
{
  return __atomic_fetch_add(p, v, __ATOMIC_RELAXED);
}
static inline unsigned atomicCAS(unsigned* p, unsigned expect, unsigned v)
{
  __atomic_compare_exchange_n(p, &expect, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED);
  return expect;
}
static inline unsigned long long atomicMin(unsigned long long* p, unsigned long long v)
{
  unsigned long long old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v < old && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return old;
}

// One launch of `kernel` (a callable taking no arguments) as `grid` blocks of `threads` threads
// (a multiple of 32): the blocks one after another, block 0 first or (reverse) last.
template <class K> static void emu_launch(unsigned grid, unsigned threads, bool reverse, const K& kernel)
{
  for (unsigned i = 0; i < grid; ++i) {
    const unsigned b = reverse ? grid - 1u - i : i;
    std::barrier<> bar(static_cast<std::ptrdiff_t>(threads));
    std::vector<EmuWarp> warps(threads / 32u);
    emu_block_bar = &bar;
    std::vector<std::thread> th;
    th.reserve(threads);
    for (unsigned t = 0; t < threads; ++t)
      th.emplace_back([&, t] {
        threadIdx.x = t;
        blockIdx.x = b;
        blockDim.x = threads;
        gridDim.x = grid;
        emu_warp = &warps[t / 32u];
        kernel();
      });
    for (auto& x : th) x.join();
    emu_block_bar = nullptr;
  }
}
