// gzip FILES: a series of members (RFC 1952 §2.2) — `cat a.gz b.gz`, and above all BGZF (BAM,
// bgzip'd .vcf.gz / .fastq.gz), whose members hold <= 64 KiB of output each and carry their own
// compressed size in the header (extra subfield 'B','C', SLEN 2: BSIZE = member length - 1).
// One BGZF file is a batch of small independent streams; these kernels turn it into the member
// table of the container batch path (container.cuh), on the device and without a serial walk:
//
//   gzf_count_kernel / gzf_exscan_kernel / gzf_scatter_kernel
//        every byte offset that starts a valid BGZF header is a candidate; count per tile, scan,
//        scatter: cpos[] ascending, cnext[] = cpos + BSIZE + 1
//   gzf_succ_kernel, gzf_jump_kernel (ceil(log2(m + 1)) tables)
//        J_0[c] = the candidate that starts at cnext[c] (m: none), J_{r+1}[c] = J_r[J_r[c]].  A false
//        candidate inside compressed data may point onto a real member, so chains MERGE: list
//        ranking by "same tail" is not enough, but succ^k(head) from the binary digits of k is exact
//   gzf_chain_kernel / gzf_expand_kernel
//        one thread finds the chain's length from the head (binary lifting); thread k writes member
//        k = succ^k(head).  O(m log m) work, O(log m) launches.
//   gzf_walk_kernel
//        one thread hops J_0 member by member: the fallback when the tables do not fit (slower, same
//        results)
//   gzf_skip_kernel   zero bytes behind a member are padding (as gzip(1) and Python skip them)
//   gzf_place_kernel  exclusive scan of ISIZE along the chain: each member's dst offset and room
//   gzf_result_kernel the first failing member in file order decides the file's status / written
//
// A member without the BGZF field (plain gzip) is found by the host (capi.cu): its header is parsed
// by container_parse_kernel, its payload decoded over the rest of the file (either single-stream
// route reports the bit behind the final block), and the walk resumes behind its trailer with the
// same tables.
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#define SFB_GZF_SMEM __shared__
#else
#define SFB_GZF_SMEM static  // (tests/cpu_emu: one block at a time, its threads share it)
#endif
#include "container.cuh"

namespace sfb {

constexpr int GZF_THREADS = 256;        // byte-parallel kernels: a block is a tile of GZF_THREADS * GZF_BYTES bytes
constexpr uint32_t GZF_BYTES = 64;      // bytes per thread (four 16-byte loads)
constexpr int GZF_SCAN_THREADS = 1024;  // the single-block scans
constexpr uint32_t GZF_DST_TOO_SMALL = 4;  // DecompressStatus DstTooSmall (deflate_lane.cuh: ST_DST_TOO_SMALL)

// one step of the walk (host <-> device, see capi.cu: gzip_file_impl)
struct GzfStep {
  uint64_t start;      // in: where the walk continues
  uint64_t skip;       // in: != 0: zero bytes at `start` are padding behind a member
  uint64_t first;      // in: members in the table so far (this step's go behind them)
  uint64_t out_total;  // in/out: sum of ISIZE of the members so far
  uint64_t head;       // first byte at or after `start` that is not padding (init: src_len)
  uint64_t head_idx;   // the candidate that starts there (m: none)
  uint64_t count;      // members found by this step
  uint64_t stop;       // the byte behind them (head when count == 0)
  uint64_t next;       // first byte at or after `stop` that is not padding (init: src_len)
  uint64_t pad[7];
};

struct GzfArgs {
  const uint8_t* src;
  uint64_t len;
  uint64_t* tile_count;  // count -> exscan -> scatter
  uint64_t* cpos;
  uint64_t* cnext;
  uint64_t m;            // candidates
  uint32_t* jump;        // n_tables tables of m + 1 entries (entry m: the "none" sentinel)
  uint32_t n_tables;
  GzfStep* step;
  // the member table
  uint64_t* mpos;
  uint64_t* mlen;
  uint64_t* moff;
  uint64_t* mcap;
  uint64_t dst_cap;
};

__device__ __forceinline__ uint32_t gzf_u16(const uint8_t* s) { return static_cast<uint32_t>(s[0]) | (static_cast<uint32_t>(s[1]) << 8); }

// Does a BGZF member header start at byte p?  *next = p + BSIZE + 1.
// 1f 8b 08, FLG with FEXTRA and no reserved bit, an XLEN whose subfields are walked within bounds,
// one of them 'B' 'C' with SLEN 2, and BSIZE + 1 >= header + trailer that fits in the bytes left.
__device__ __forceinline__ bool gzf_candidate(const uint8_t* s, uint64_t len, uint64_t p, uint64_t* next)
{
  if (len - p < 12 || s[p] != 0x1f || s[p + 1] != 0x8b || s[p + 2] != 8u) return false;
  const uint32_t flg = s[p + 3];
  if ((flg & 4u) == 0 || (flg & 0xe0u) != 0) return false;
  const uint64_t xlen = gzf_u16(s + p + 10);
  const uint64_t e = p + 12 + xlen;
  if (e > len) return false;
  for (uint64_t q = p + 12; q + 4 <= e;) {
    const uint64_t slen = gzf_u16(s + q + 2);
    if (q + 4 + slen > e) return false;
    if (s[q] == 'B' && s[q + 1] == 'C' && slen == 2) {
      const uint64_t total = static_cast<uint64_t>(gzf_u16(s + q + 4)) + 1;
      if (total < 12 + xlen + 8 || total > len - p) return false;
      *next = p + total;
      return true;
    }
    q += 4 + slen;
  }
  return false;
}

// Candidates among this thread's GZF_BYTES bytes (offsets x of the 16-byte aligned base `al`; the
// file starts at x = phase).  `out` == nullptr: count only.
// The loads are whole aligned 16-byte blocks that hold at least one byte of the file, so up to 15
// bytes before src and after src + len are read on purpose and never used: CUDA allocations are
// aligned and sized in far larger units, so such a block lies inside the allocation that holds the
// file, whatever view of it the caller passes (a memory checker does flag these bytes).
__device__ __forceinline__ uint32_t gzf_thread_scan(const uint8_t* s, uint64_t len, uint64_t x0, uint64_t* cpos,
                                                    uint64_t* cnext, uint64_t out)
{
  const uint8_t* const al = s - (reinterpret_cast<uintptr_t>(s) & 15u);
  const uint64_t phase = reinterpret_cast<uintptr_t>(s) & 15u;
  uint32_t c = 0;
#pragma unroll
  for (uint32_t v = 0; v < GZF_BYTES / 16; ++v) {
    const uint64_t xb = x0 + 16u * v;
    if (xb >= len + phase) break;
    const uint4 q = *reinterpret_cast<const uint4*>(al + xb);
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t t = w[k] ^ 0x1f1f1f1fu;
      if (((t - 0x01010101u) & ~t & 0x80808080u) == 0) continue;  // no 0x1f byte in this word
      for (uint32_t b = 0; b < 4; ++b) {
        if (((w[k] >> (8 * b)) & 0xffu) != 0x1fu) continue;
        const uint64_t x = xb + 4u * k + b;
        if (x < phase || x - phase >= len) continue;
        uint64_t nx = 0;
        if (!gzf_candidate(s, len, x - phase, &nx)) continue;
        if (cpos) {
          cpos[out + c] = x - phase;
          cnext[out + c] = nx;
        }
        ++c;
      }
    }
  }
  return c;
}

// exclusive prefix sum over the block; *total = the block's sum.  Every thread of the block calls it.
__device__ __forceinline__ uint64_t gzf_block_exscan(uint64_t v, uint64_t* total)
{
  constexpr unsigned FULL = 0xffffffffu;
  SFB_GZF_SMEM uint64_t s_warp[32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31u) >> 5;
  uint64_t incl = v;
  for (uint32_t o = 1; o < 32; o <<= 1) {
    const uint64_t y = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31u) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = lane < nwarps ? s_warp[lane] : 0;
    for (uint32_t o = 1; o < 32; o <<= 1) {
      const uint64_t y = __shfl_up_sync(FULL, w, o);
      if (lane >= o) w += y;
    }
    if (lane < nwarps) s_warp[lane] = w;
  }
  __syncthreads();
  const uint64_t base = warp ? s_warp[warp - 1] : 0;
  *total = s_warp[nwarps - 1];
  __syncthreads();  // (s_warp is reused by the next call)
  return base + incl - v;
}

// grid: one block per tile of blockDim.x * GZF_BYTES bytes (of the aligned base)
__global__ void __launch_bounds__(GZF_THREADS) gzf_count_kernel(const GzfArgs a)
{
  const uint64_t x0 = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * GZF_BYTES;
  const uint32_t c = gzf_thread_scan(a.src, a.len, x0, nullptr, nullptr, 0);
  uint64_t total = 0;
  gzf_block_exscan(c, &total);
  if (threadIdx.x == 0) a.tile_count[blockIdx.x] = total;
}

__global__ void __launch_bounds__(GZF_THREADS) gzf_scatter_kernel(const GzfArgs a)
{
  const uint64_t x0 = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * GZF_BYTES;
  const uint32_t c = gzf_thread_scan(a.src, a.len, x0, nullptr, nullptr, 0);
  uint64_t total = 0;
  const uint64_t at = a.tile_count[blockIdx.x] + gzf_block_exscan(c, &total);
  if (c) gzf_thread_scan(a.src, a.len, x0, a.cpos, a.cnext, at);
}

// one block: in-place exclusive scan of v[0 .. n); v[n] = the sum
__global__ void __launch_bounds__(GZF_SCAN_THREADS) gzf_exscan_kernel(uint64_t* v, uint64_t n)
{
  const uint64_t per = (n + blockDim.x - 1) / blockDim.x;
  const uint64_t lo = per * threadIdx.x < n ? per * threadIdx.x : n, hi = lo + per < n ? lo + per : n;
  uint64_t sum = 0;
  for (uint64_t i = lo; i < hi; ++i) sum += v[i];
  uint64_t total = 0;
  uint64_t run = gzf_block_exscan(sum, &total);
  for (uint64_t i = lo; i < hi; ++i) {
    const uint64_t x = v[i];
    v[i] = run;
    run += x;
  }
  if (threadIdx.x == 0) v[n] = total;
}

// the candidate that starts at byte p, or m
__device__ __forceinline__ uint64_t gzf_find(const uint64_t* cpos, uint64_t m, uint64_t p)
{
  uint64_t lo = 0, hi = m;
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (cpos[mid] < p) lo = mid + 1;
    else hi = mid;
  }
  return lo < m && cpos[lo] == p ? lo : m;
}

__global__ void gzf_succ_kernel(const GzfArgs a)
{
  const uint64_t c = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c > a.m) return;
  a.jump[c] = static_cast<uint32_t>(c == a.m ? a.m : gzf_find(a.cpos, a.m, a.cnext[c]));
}

// table r + 1 from table r
__global__ void gzf_jump_kernel(const GzfArgs a, uint32_t r)
{
  const uint64_t c = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c > a.m) return;
  uint32_t* const jr = a.jump + static_cast<uint64_t>(r) * (a.m + 1);
  jr[a.m + 1 + c] = jr[jr[c]];
}

// the first byte of [*from, len) that is not zero -> atomicMin(*out) (enable == 0: *from itself).
// A fixed grid walks the tiles in order and stops at tiles behind what was found already.
__global__ void __launch_bounds__(GZF_THREADS) gzf_skip_kernel(const GzfArgs a, const uint64_t* from,
                                                               const uint64_t* enable, unsigned long long* out)
{
  const uint64_t f = *from;
  if (*enable == 0) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicMin(out, static_cast<unsigned long long>(f));
    return;
  }
  const uint64_t tile = static_cast<uint64_t>(blockDim.x) * GZF_BYTES;
  for (uint64_t t = f / tile + blockIdx.x; t * tile < a.len; t += gridDim.x) {
    if (t * tile > *reinterpret_cast<volatile unsigned long long*>(out)) return;
    const uint64_t lo0 = t * tile + static_cast<uint64_t>(threadIdx.x) * GZF_BYTES;
    const uint64_t lo = lo0 > f ? lo0 : f;
    const uint64_t hi = lo0 + GZF_BYTES < a.len ? lo0 + GZF_BYTES : a.len;
    for (uint64_t p = lo; p < hi; ++p)
      if (a.src[p] != 0) {
        atomicMin(out, static_cast<unsigned long long>(p));
        break;
      }
  }
}

// one thread: the chain from the step's head — its length by binary lifting over the tables
__global__ void gzf_chain_kernel(const GzfArgs a)
{
  GzfStep* const st = a.step;
  const uint64_t h = gzf_find(a.cpos, a.m, st->head);
  st->head_idx = h;
  if (h == a.m) {
    st->count = 0;
    st->stop = st->head;
    return;
  }
  uint64_t cur = h, hops = 0;
  for (uint32_t r = a.n_tables; r-- > 0;) {
    const uint32_t nx = a.jump[static_cast<uint64_t>(r) * (a.m + 1) + cur];
    if (nx != a.m) {
      cur = nx;
      hops += 1ull << r;
    }
  }
  st->count = hops + 1;
  st->stop = a.cnext[cur];
}

// thread k: member k of the chain = succ^k(head), from the binary digits of k
__global__ void gzf_expand_kernel(const GzfArgs a)
{
  const GzfStep* const st = a.step;
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= st->count) return;
  uint64_t cur = st->head_idx;
  for (uint32_t r = 0; (k >> r) != 0; ++r)
    if ((k >> r) & 1u) cur = a.jump[static_cast<uint64_t>(r) * (a.m + 1) + cur];
  a.mpos[st->first + k] = a.cpos[cur];
  a.mlen[st->first + k] = a.cnext[cur] - a.cpos[cur];
}

// one thread: the same chain member by member on J_0 (when the other tables do not fit)
__global__ void gzf_walk_kernel(const GzfArgs a)
{
  GzfStep* const st = a.step;
  uint64_t cur = gzf_find(a.cpos, a.m, st->head), k = 0;
  st->head_idx = cur;
  uint64_t stop = st->head;
  for (; cur != a.m; cur = a.jump[cur], ++k) {
    a.mpos[st->first + k] = a.cpos[cur];
    a.mlen[st->first + k] = a.cnext[cur] - a.cpos[cur];
    stop = a.cnext[cur];
  }
  st->count = k;
  st->stop = stop;
}

// one block: members [first, first + count): dst offset = exclusive scan of ISIZE (the trailer's
// last four bytes) behind out_total, room = min(ISIZE, what is left of dst)
__global__ void __launch_bounds__(GZF_SCAN_THREADS) gzf_place_kernel(const GzfArgs a)
{
  GzfStep* const st = a.step;
  const uint64_t n = st->count, first = st->first, base = st->out_total;
  auto isize = [&](uint64_t i) {
    const uint8_t* t = a.src + a.mpos[i] + a.mlen[i] - 4;
    return static_cast<uint64_t>(gzf_u16(t)) | (static_cast<uint64_t>(gzf_u16(t + 2)) << 16);
  };
  const uint64_t per = (n + blockDim.x - 1) / blockDim.x;
  const uint64_t lo = per * threadIdx.x < n ? per * threadIdx.x : n, hi = lo + per < n ? lo + per : n;
  uint64_t sum = 0;
  for (uint64_t i = lo; i < hi; ++i) sum += isize(first + i);
  uint64_t total = 0;
  uint64_t run = base + gzf_block_exscan(sum, &total);
  for (uint64_t i = lo; i < hi; ++i) {
    const uint64_t sz = isize(first + i);
    const uint64_t off = run < a.dst_cap ? run : a.dst_cap;
    a.moff[first + i] = off;
    a.mcap[first + i] = sz < a.dst_cap - off ? sz : a.dst_cap - off;
    run += sz;
  }
  __syncthreads();
  if (threadIdx.x == 0) st->out_total = base + total;
}

// one block: the file's result.  The first member (file order) whose status is not Success decides:
// status (DstTooSmall where the room was ISIZE, not the end of dst, is SizeMismatch) and written =
// its dst offset + what it produced.  Without one: tail_status, written = end of the last member +
// tail_written (what a failing plain member behind them produced).  out[0] status, out[1] written.
__global__ void __launch_bounds__(GZF_SCAN_THREADS) gzf_result_kernel(const GzfArgs a, const uint8_t* status,
                                                                      const uint64_t* written, uint64_t n,
                                                                      uint32_t tail_status, uint64_t tail_written,
                                                                      uint64_t* out)
{
  constexpr unsigned FULL = 0xffffffffu;
  SFB_GZF_SMEM uint64_t s_min[32];
  uint64_t k = n;
  for (uint64_t i = threadIdx.x; i < n; i += blockDim.x)
    if (status[i] != 0) {
      k = i;
      break;
    }
  for (int o = 16; o; o >>= 1) {
    const uint64_t y = __shfl_down_sync(FULL, k, o);
    k = y < k ? y : k;
  }
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31u) >> 5;
  if (lane == 0) s_min[warp] = k;
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (uint32_t w = 0; w < nwarps; ++w) k = s_min[w] < k ? s_min[w] : k;
  if (k < n) {
    uint32_t s = status[k];
    if (s == GZF_DST_TOO_SMALL && a.mcap[k] < a.dst_cap - a.moff[k]) s = ST_SIZE_MISMATCH;
    out[0] = s;
    out[1] = a.moff[k] + written[k];
  } else {
    out[0] = tail_status;
    out[1] = (n ? a.moff[n - 1] + written[n - 1] : 0) + tail_written;
  }
}

}  // namespace sfb
