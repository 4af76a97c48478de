// Pass 2 of the batched raw-DEFLATE decoder for sm_100a: LZ77 back-references, ONE WARP PER
// STREAM, 128-byte chunks, one aligned 32-bit word (4 output bytes) per lane.
//
// Replaces the copy half of the reference's decompress_length_distance and copy_from_before
// (src/decompress.cpp:157-187,388-398): pass 1 (huff_lanes.cuh) has already placed literals and
// stored payload at their final positions and left, for every match, a 3-byte descriptor at
// the match start plus a bit in the match-head bitmap; this pass turns each descriptor into the
// bytes the reference would have copied.  All range/room checks were made in pass 1.
//
// Per 128-byte chunk [P, P+128) of a stream's output (128-byte aligned addresses):
//   1. every lane loads its word and the 4 bitmap bits of its bytes; lanes with a match head
//      assemble the descriptor from their word and the next lane's (lane 31: the next chunk's
//      first word, which is prefetched) and publish their LAST head as one packed 30-bit value;
//   2. the match a lane's first byte may lie in is the last head of the nearest lower lane that
//      has one (ballot + FLO + one shuffle), else the match carried in from earlier chunks;
//      the lane then walks its 4 bytes, switching to its own heads as it passes them;
//   3. a covered byte's source is  start - distance + (k mod distance)  — the forward-
//      overlapping copy of copy_from_before() is periodic with period `distance` — which always
//      lies BEFORE the match start;
//   4. resolution rounds: with F the first byte of the chunk that is still unresolved, every
//      unresolved byte whose source lies below F is gathered from memory (below P: written by
//      earlier chunks; in [P, F): literals of pass 1 or bytes stored by an earlier round, made
//      visible by __syncwarp), the words are stored, F advances.  The first unresolved match
//      always resolves completely (its sources precede its start), text-like data needs 2-3
//      rounds per chunk, a chunk without near references one.
// Streams are pulled from a global counter.
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#endif

namespace sfb {

struct ResolveArgs {
  uint8_t* dst_base;           // 128-byte aligned
  uint64_t dst_delta;          // added to every dst_off (the caller's dst_base - this dst_base)
  const uint64_t* dst_off;
  const uint64_t* written;
  const uint32_t* match_bits;  // bit k <-> dst_base[k]
  uint64_t n;                          // streams of this launch: idx_base .. idx_base + n - 1,
  uint64_t idx_base;                   // or todo_list[0 .. n) when a list is given
  const uint32_t* todo_list;
  unsigned long long* stream_counter;  // zeroed before launch
};

// ---------------------------------------------------------------------------------------------
// Batch preparation: order the streams by the type of their first block (dynamic, fixed, other,
// stored) so that the 32 streams a pass-1 warp decodes together do the same kind of work — in a
// mixed batch (BASELINE config 3) a third of the lanes would otherwise sit out the token loop
// because their stream was a stored block, and the dynamic ones, which take longest, start
// first.  Two small kernels: count per type, then scatter (block-wise reserved ranges).
struct PrepArgs {
  const uint8_t* src_base;
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint64_t n;
  unsigned long long* type_count;   // [4] zeroed before launch, in the order of lz_type_rank()
  unsigned long long* type_cursor;  // [4] zeroed before launch
  uint32_t* order;                  // out: n stream indices
};

// rank of a stream in the processing order, from the BTYPE bits of its first byte
__device__ __forceinline__ uint32_t lz_type_rank(const PrepArgs& a, uint64_t i)
{
  if (a.src_len[i] == 0) return 2u;
  const uint32_t btype = (a.src_base[a.src_off[i]] >> 1) & 3u;
  return btype == 2u ? 0u : btype == 1u ? 1u : btype == 3u ? 2u : 3u;  // dynamic, fixed, invalid, stored
}

constexpr int PREP_THREADS = 256;

#if !defined(SFB_CPU_EMU) || defined(SFB_EMU_BLOCK)  // (block-level kernels: tests/cpu_emu/emu_block.cpp)

__global__ void __launch_bounds__(PREP_THREADS) prep_count_kernel(const PrepArgs a)
{
  __shared__ unsigned int cnt[4];
  if (threadIdx.x < 4) cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * PREP_THREADS + threadIdx.x;
  if (i < a.n) atomicAdd(&cnt[lz_type_rank(a, i)], 1u);
  __syncthreads();
  if (threadIdx.x < 4 && cnt[threadIdx.x]) atomicAdd(&a.type_count[threadIdx.x], static_cast<unsigned long long>(cnt[threadIdx.x]));
}

__global__ void __launch_bounds__(PREP_THREADS) prep_scatter_kernel(const PrepArgs a)
{
  __shared__ unsigned int cnt[4];
  __shared__ unsigned long long base[4];
  if (threadIdx.x < 4) cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * PREP_THREADS + threadIdx.x;
  uint32_t t = 0, r = 0;
  if (i < a.n) {
    t = lz_type_rank(a, i);
    r = atomicAdd(&cnt[t], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    unsigned long long start = 0;
    for (unsigned k = 0; k < threadIdx.x; ++k) start += a.type_count[k];
    base[threadIdx.x] = start + (cnt[threadIdx.x] ? atomicAdd(&a.type_cursor[threadIdx.x], static_cast<unsigned long long>(cnt[threadIdx.x])) : 0ull);
  }
  __syncthreads();
  if (i < a.n) a.order[base[t] + r] = static_cast<uint32_t>(i);
}
#endif  // SFB_CPU_EMU

constexpr int LZ_THREADS = 256;

// byte permute (PRMT): result byte i = byte sel.nibble[i] of the 8 bytes b:a
__device__ __forceinline__ uint32_t lz_prmt(uint32_t a, uint32_t b, uint32_t sel)
{
#ifdef SFB_CPU_EMU
  const uint64_t v = (static_cast<uint64_t>(b) << 32) | a;
  uint32_t r = 0;
  for (int i = 0; i < 4; ++i) r |= static_cast<uint32_t>((v >> (8 * ((sel >> (4 * i)) & 7u))) & 0xffu) << (8 * i);
  return r;
#else
  return __byte_perm(a, b, sel);
#endif
}
// bits [s, s+32) of hi:lo, 0 <= s < 32
__device__ __forceinline__ uint32_t lz_funnel(uint32_t lo, uint32_t hi, uint32_t s)
{
#ifdef SFB_CPU_EMU
  return static_cast<uint32_t>(((static_cast<uint64_t>(hi) << 32) | lo) >> (s & 31u));
#else
  return __funnelshift_r(lo, hi, s);
#endif
}

// k mod d for d <= k < 4096 (only overlapping matches get here, so d <= 257): multiply by a
// 20-bit reciprocal.  inv = trunc(2^20 / d) + 2 with the quotient from a fast float division
// (absolute error < 1) lies in (2^20/d, 2^20/d + 3), which makes floor(k * inv / 2^20) exact
// for k < 2^20 / (3 d)  (checked exhaustively for d < 300, k < 700 in the design notes).
__device__ __forceinline__ uint32_t lz_mod_small(uint32_t k, uint32_t d)
{
#ifdef SFB_CPU_EMU
  const uint32_t inv = static_cast<uint32_t>(1048576.0f / static_cast<float>(d)) + 2u;
#else
  const uint32_t inv = static_cast<uint32_t>(__fdividef(1048576.0f, static_cast<float>(d))) + 2u;
#endif
  return k - ((k * inv) >> 20) * d;
}

// (launched with 6 CTAs = 48 warps per SM: measured best on C2 — with 64 the streams in flight push
//  each other out of the L2, and squeezing the code under 40 registers costs more than it gains)
__global__ void __launch_bounds__(LZ_THREADS, 5) lz_resolve_kernel(const ResolveArgs a)
{
  constexpr unsigned FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t lt_mask = (1u << lane) - 1u;             // lanes below this one
  const int next_lane = static_cast<int>((lane + 1u) & 31u);
  const uint32_t bit_sh = 4u * (lane & 7u);               // my 4 bits inside my bitmap word
  for (;;) {
    unsigned long long si = 0;
    if (lane == 0) si = atomicAdd(a.stream_counter, 1ull);
    si = __shfl_sync(FULL, si, 0);
    if (si >= a.n) break;
    si = a.todo_list ? a.todo_list[si] : a.idx_base + si;
    const uint64_t off = a.dst_off[si] + a.dst_delta;
    const uint64_t wr = a.written[si];
    if (wr == 0) continue;
    // virtual positions: byte v of the view sits at base[v]; the stream occupies [q, end)
    uint8_t* const base = a.dst_base + (off & ~127ull);
    const uint32_t q = static_cast<uint32_t>(off & 127u);
    const uint32_t end = q + static_cast<uint32_t>(wr);
    // this lane's word and bitmap word of the current chunk, and of the two after it
    const uint32_t* pw = reinterpret_cast<const uint32_t*>(base) + lane;
    const uint32_t* pm = a.match_bits + ((off & ~127ull) >> 5) + (lane >> 3);
    // a word is read iff one of its bytes belongs to the stream (never a word wholly outside)
    auto load_w = [&](uint32_t P) -> uint32_t {
      const uint32_t wp = P + 4u * lane;
      return (wp + 4u > q && wp < end) ? pw[P >> 2] : 0u;
    };
    auto load_m = [&](uint32_t P) -> uint32_t { return P < end ? pm[P >> 5] : 0u; };
    uint32_t cw = load_w(0), ncw = load_w(128), mw = load_m(0), nmw = load_m(128);
    // the most recent match seen so far: [c_o, c_end) at distance c_d (none yet: empty range)
    uint32_t c_o = 0, c_end = 0, c_d = 1;
    for (uint32_t P = 0; P < end; P += 128) {
      const uint32_t nncw = load_w(P + 256), nnmw = load_m(P + 256);
      const uint32_t wp = P + 4u * lane;
      // valid bytes of my word
      uint32_t vm = 15u;
      const bool interior = P >= q && P + 128u <= end;  // (warp-uniform)
      if (!interior) {  // first / last chunk of the stream
        const uint32_t lo = q > wp ? (q - wp < 4u ? q - wp : 4u) : 0u;
        const uint32_t hi = end > wp ? (end - wp < 4u ? end - wp : 4u) : 0u;
        vm = hi > lo ? ((1u << hi) - 1u) & ~((1u << lo) - 1u) : 0u;
      }
      const uint32_t hb4 = (mw >> bit_sh) & vm;  // match heads among my bytes
      // the word after mine (lane 31: first word of the next chunk)
      const uint32_t t = __shfl_sync(FULL, cw, next_lane);
      const uint32_t u = __shfl_sync(FULL, ncw, 0);
      const uint32_t nx = lane == 31u ? u : t;
      // my last head, packed: position in chunk (7 bits) | descriptor (23 bits)
      const uint32_t hl = 31u - static_cast<uint32_t>(__clz(static_cast<int>(hb4 | 1u)));
      const uint32_t own_pack = (4u * lane + hl) | ((lz_funnel(cw, nx, 8u * hl) & 0xffffffu) << 7);
      const uint32_t hm = __ballot_sync(FULL, hb4 != 0);
      // the match my first byte may lie in
      const uint32_t below = hm & lt_mask;
      const uint32_t sl = 31u - static_cast<uint32_t>(__clz(static_cast<int>(below | 1u)));
      const uint32_t in_pack = __shfl_sync(FULL, own_pack, static_cast<int>(sl));
      uint32_t t_o = c_o, t_end = c_end, t_d = c_d;
      if (below) {
        t_o = P + (in_pack & 127u);
        t_end = t_o + ((in_pack >> 7) & 255u) + 3u;
        t_d = (in_pack >> 15) + 1u;
      }
      if (hm) {  // warp-uniform: the last head of this chunk is carried into the next ones
        const uint32_t top = 31u - static_cast<uint32_t>(__clz(static_cast<int>(hm)));
        const uint32_t pk = __shfl_sync(FULL, own_pack, static_cast<int>(top));
        c_o = P + (pk & 127u);
        c_end = c_o + ((pk >> 7) & 255u) + 3u;
        c_d = (pk >> 15) + 1u;
      }
      // ---- chunks that lie wholly inside one long match (no head, interior of the stream):
      //      every source is below the match start, hence below P and final; no per-byte
      //      bookkeeping is needed -----------------------------------------------------------
      if (interior && hm == 0 && c_end >= P + 128u && c_o < P && (c_d == 1u || c_d >= 4u)) {  // (warp-uniform)
        uint32_t v;
        if (c_d == 1u) {  // a run: all bytes equal the one before the match
          v = base[c_o - 1u] * 0x01010101u;
        } else {
          // byte 0 of my word is k bytes into the match: its source is start - d + (k mod d),
          // and so on round the period for the other three
          const uint32_t k = wp - c_o;
          const uint32_t m = k >= c_d ? lz_mod_small(k, c_d) : k;
          const uint32_t s0 = c_o - c_d + m;
          if (m + 3u < c_d) {  // four consecutive sources: one unaligned word
            const uint32_t* wsrc = reinterpret_cast<const uint32_t*>(base + (s0 & ~3u));
            const uint32_t lo = wsrc[0];
            const uint32_t hi = (s0 & 3u) ? wsrc[1] : 0u;
            v = lz_funnel(lo, hi, 8u * (s0 & 3u));
          } else {  // the period wraps inside my word (at most once: d >= 4)
            v = 0;
#pragma unroll
            for (uint32_t b = 0; b < 4; ++b) {
              uint32_t mb = m + b;
              if (mb >= c_d) mb -= c_d;
              v |= static_cast<uint32_t>(base[c_o - c_d + mb]) << (8u * b);
            }
          }
        }
        *reinterpret_cast<uint32_t*>(base + wp) = v;
        __syncwarp();
        cw = ncw;
        ncw = nncw;
        mw = nmw;
        nmw = nnmw;
        continue;
      }
      // ---- walk my 4 bytes, switching to my own heads as I pass them -------------------------
      uint32_t src[4];
      uint32_t pend = 0;
#pragma unroll
      for (uint32_t b = 0; b < 4; ++b) {
        const uint32_t p = wp + b;
        if ((hb4 >> b) & 1u) {
          const uint32_t d = lz_funnel(cw, nx, 8u * b) & 0xffffffu;
          t_o = p;
          t_end = p + (d & 255u) + 3u;
          t_d = (d >> 8) + 1u;
        }
        const bool cov = ((vm >> b) & 1u) && p < t_end;
        uint32_t k = p - t_o;
        if (cov && k >= t_d) k = lz_mod_small(k, t_d);  // overlapping copy: period t_d
        src[b] = t_o - t_d + k;  // = start - distance + (k mod distance) >= q (pass 1 checked)
        if (cov) pend |= 1u << b;
      }
      // resolution rounds
      uint32_t res = cw;
      for (;;) {
        // F = first unresolved byte of the chunk (P + 128 if none)
        const uint32_t pm_any = __ballot_sync(FULL, pend != 0);
        if (pm_any == 0) break;
        const int fl = __ffs(static_cast<int>(pm_any)) - 1;
        const uint32_t fp = __shfl_sync(FULL, pend, fl);
        const uint32_t F = P + 4u * static_cast<uint32_t>(fl) + static_cast<uint32_t>(__ffs(static_cast<int>(fp)) - 1);
#pragma unroll
        for (uint32_t b = 0; b < 4; ++b) {
          if (((pend >> b) & 1u) && src[b] < F) {
            const uint32_t byte = base[src[b]];
            res = lz_prmt(res, byte, 0x3210u ^ ((0x4u ^ b) << (4u * b)));  // byte b <- `byte`
            pend &= ~(1u << b);
          }
        }
        if (vm == 15u) {
          *reinterpret_cast<uint32_t*>(base + wp) = res;
        } else {  // first / last word of the stream: only our bytes
#pragma unroll
          for (uint32_t b = 0; b < 4; ++b)
            if ((vm >> b) & 1u) base[wp + b] = static_cast<uint8_t>(res >> (8u * b));
        }
        __syncwarp();
      }
      cw = ncw;
      ncw = nncw;
      mw = nmw;
      nmw = nnmw;
    }
  }
}

// Position-weighted checksum (see starflate_b200.h): one warp per stream.
__global__ void checksum_kernel(const uint8_t* base, const uint64_t* off, const uint64_t* len,
                                uint64_t* out, uint64_t n)
{
  const uint64_t w = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const unsigned lane = threadIdx.x & 31u;
  if (w >= n) return;
  const uint8_t* p = base + off[w];
  const uint64_t L = len[w];
  uint64_t acc = 0;
  for (uint64_t j = lane; j < L; j += 32)
    acc += (static_cast<uint64_t>(p[j]) + 1ull) * ((0x9E3779B97F4A7C15ull * (j + 1ull)) | 1ull);
  for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if (lane == 0) out[w] = acc;
}

}  // namespace sfb
