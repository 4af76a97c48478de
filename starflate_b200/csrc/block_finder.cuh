// Block finder and block chain for ONE LARGE stream on sm_100a (BASELINE.json's single-stream
// mode): lets the blocks of a stream be decoded side by side although a block's start is only
// KNOWN once the block before it has been decoded.
//
// DEFLATE has no block index, but a dynamic-Huffman block header (RFC 1951 §3.2.7, parsed by the
// reference in src/decompress.cpp:314-367) is highly redundant.  Every bit position of the input
// is tested, cheapest test first:
//   find_candidates_kernel  BTYPE == 2, HLIT <= 29, HDIST <= 29 (17 bits, 22 % pass), then the
//                           3-bit code-length-code lengths must form a COMPLETE prefix code
//                           (Kraft sum exactly 1; about 1 in 150 of the rest);
//   verify_candidates_kernel decodes the HLIT + HDIST code lengths with that code: no repeat
//                           without a previous length, no run past the end, the literal/length
//                           code complete and with an end-of-block symbol, the distance code
//                           complete (or at most one code).  Random bits practically never pass.
// What passes becomes a JOB: a warp decodes the block that starts there, counting only
// (huff_stream.cuh, mode 1), and records where it ends and what it would produce.
//
// THE FINDER IS ONLY A HINT; what is decoded is decided by the chain.  chain_kernel starts at bit 0
// (job 0, always there), and follows "this block ends at bit e" -> "the job that starts at bit
// e".  A job is used only if the block before it ends exactly at its start, i.e. only if a
// front-to-back decoder would have begun a block there too; its result then does not depend on
// how its start was found.  Where the chain cannot go on — the next block is a stored or fixed
// one (nothing to find), its header is one the finder is too strict for (zlib never writes one:
// incomplete or over-subscribed codes, which the reference accepts), the block is the last, or it
// fails — the job reached last becomes the TAIL: in the writing pass (mode 2) it decodes its
// block and then simply carries on, block after block, to the end of the stream, like the plain
// one-warp kernel.  So every input gives exactly the bytes, status and count of the front-to-back
// decode; the finder only decides how much of it runs in parallel.
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#endif

namespace sfb {

constexpr uint64_t JOB_NONE = ~0ull;
constexpr uint32_t JOB_ENDS = 1u;   // the stream ends in (or right after) this block, or it failed
constexpr uint32_t JOB_CLEAN = 2u;  // mode 1: a Huffman block decoded up to its end-of-block symbol
constexpr uint32_t JOB_RECS = 4u;   // mode 1: ... and all its windows are on record (WinRec)
constexpr uint32_t JOB_USE = 8u;    // chain: on the chain, sizes and distances fit: mode 2 may write from the records

struct BlockJob {
  uint64_t start_bit;  // where the block's header starts
  uint64_t end_bit;    // mode 1: where the next header starts
  uint64_t out;        // mode 1: bytes the block produces
  uint64_t base;       // chain: the block's output position, JOB_NONE: not on the chain
  uint32_t need;       // mode 1: the smallest base at which all its distances are in range
  uint32_t flags;      // mode 1: JOB_ENDS
  uint32_t next;       // mode 1: the job that starts at end_bit (0: none)
  uint32_t first_rec;  // mode 1: 1 + index of its first window record (0: none)
};

// What the counting job found out about one window of 32 spans, so that the writing job need not
// find it out again: where each lane's span really starts and where its output goes.
struct WinRec {
  uint64_t b0;         // the window's first bit
  uint32_t cut;        // first lane that meets the end of the block (32: none)
  uint32_t next;       // 1 + index of the block's next window (0: none)
  uint32_t s_rel[32];  // lane's true start, bits after b0
  uint32_t start[32];  // lane's output position, bytes after the block's
};

struct FindArgs {
  const uint8_t* src_base;
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint64_t idx;          // the stream
  uint64_t* cand;        // bit positions that passed the quick tests
  uint32_t* cand_count;  // zeroed
  uint32_t cand_cap;
  BlockJob* jobs;
  uint32_t* job_count;   // set to 1 (job 0 = bit 0) by find_candidates_kernel
  uint32_t job_cap;
  uint32_t* job_tab;     // zeroed; open-addressing hash table start_bit -> job (see job_find)
  uint32_t tab_mask;     // its size - 1 (a power of two, at least twice job_cap)
  uint32_t* tail_job;    // chain: the job that runs to the end of the stream
  const uint64_t* dst_cap;
};

// start_bit -> job: linear probing, a slot holds a job index (0: empty), the key is the job's
// start_bit.  Two jobs with the same start are the same block twice: whichever is found will do.
__device__ __forceinline__ uint32_t job_slot(uint64_t p, uint32_t mask)
{
  return static_cast<uint32_t>((p * 0x9E3779B97F4A7C15ull) >> 40) & mask;
}
__device__ __forceinline__ uint32_t job_find(const uint32_t* tab, uint32_t mask, const BlockJob* jobs,
                                             uint32_t n_jobs, uint64_t p)
{
  uint32_t s = job_slot(p, mask);
  for (uint32_t tries = 0; tries <= mask; ++tries) {
    const uint32_t k = tab[s];
    if (k == 0u) return 0u;
    if (k < n_jobs && jobs[k].start_bit == p) return k;
    s = (s + 1u) & mask;
  }
  return 0u;
}

// Follow the blocks from bit 0 (see the head of this file).  One thread: a step is one 48-byte
// record, the links were looked up by the counting jobs.
__global__ void chain_kernel(const FindArgs a)
{
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint64_t cap = a.dst_cap[a.idx];
  uint32_t n_jobs = *a.job_count;
  if (n_jobs > a.job_cap) n_jobs = a.job_cap;
  uint32_t j = 0;
  uint64_t base = 0;
  for (;;) {
    const BlockJob jb = a.jobs[j];
    a.jobs[j].base = base;
    if ((jb.flags & JOB_RECS) && jb.need <= base && base + jb.out <= cap) a.jobs[j].flags = jb.flags | JOB_USE;
    if ((jb.flags & JOB_ENDS) || jb.need > base || base + jb.out > cap || jb.next == 0u || jb.next >= n_jobs) break;
    base += jb.out;
    j = jb.next;
  }
  *a.tail_job = j;
}

constexpr int FIND_THREADS = 256;

// 32-bit word i of the 4-byte aligned view of the stream, zero outside [src, src + slen)
__device__ __forceinline__ uint32_t find_word(const uint8_t* src, uint64_t slen, uint32_t sh, uint64_t i)
{
  const int64_t b0 = static_cast<int64_t>(4ull * i) - static_cast<int64_t>(sh);  // stream offset of its first byte
  if (b0 >= 0 && static_cast<uint64_t>(b0) + 4u <= slen) return *reinterpret_cast<const uint32_t*>(src + b0);
  uint32_t w = 0;
  for (int k = 0; k < 4; ++k) {
    const int64_t b = b0 + k;
    if (b >= 0 && static_cast<uint64_t>(b) < slen) w |= static_cast<uint32_t>(src[b]) << (8 * k);
  }
  return w;
}

__global__ void __launch_bounds__(FIND_THREADS) find_candidates_kernel(const FindArgs a)
{
  const uint8_t* const src = a.src_base + a.src_off[a.idx];
  const uint64_t slen = a.src_len[a.idx];
  const uint64_t gtid = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gtid == 0) {
    BlockJob j0;
    j0.start_bit = 0;
    j0.end_bit = 0;
    j0.out = 0;
    j0.base = JOB_NONE;
    j0.need = 0;
    j0.flags = JOB_ENDS;
    j0.next = 0;
    j0.first_rec = 0;
    a.jobs[0] = j0;
    *a.job_count = 1u;
  }
  // three code-length-code lengths (9 bits) -> their Kraft sum in units of 2^-7 | number of codes << 16
  __shared__ uint32_t s_kraft[512];
  for (uint32_t x = threadIdx.x; x < 512u; x += blockDim.x) {
    uint32_t e = 0;
    for (uint32_t c = 0; c < 3; ++c) {
      const uint32_t len = (x >> (3u * c)) & 7u;
      if (len) e += (128u >> len) + 0x10000u;
    }
    s_kraft[x] = e;
  }
#ifndef SFB_CPU_EMU
  __syncthreads();
#endif
  if (slen >= 0xffffff00ull) return;
  const uint32_t sh = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(src) & 3u);
  const uint64_t total_bits = 8ull * slen;
  const uint64_t n_words = (slen + sh + 3u) / 4u;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (uint64_t i = gtid; i < n_words; i += stride) {
    const uint32_t w0 = find_word(src, slen, sh, i), w1 = find_word(src, slen, sh, i + 1);
    // quick tests on the 32 positions that start in w0, all at once: bit j of A(k) is bit k of
    // position j's header.  BTYPE == 2: bit 1 clear, bit 2 set; HLIT (bits 3-7) and HDIST (bits
    // 8-12) <= 29: their upper four bits not all set.
    auto A = [&](uint32_t k) { return __funnelshift_r(w0, w1, k); };
    uint32_t pass = ~A(1) & A(2) & ~(A(4) & A(5) & A(6) & A(7)) & ~(A(9) & A(10) & A(11) & A(12));
    if (pass == 0) continue;
    const uint32_t w2 = find_word(src, slen, sh, i + 2), w3 = find_word(src, slen, sh, i + 3);
    const uint64_t lo64 = (static_cast<uint64_t>(w1) << 32) | w0, hi64 = (static_cast<uint64_t>(w3) << 32) | w2;
    while (pass) {
      const uint32_t j = static_cast<uint32_t>(__ffs(static_cast<int>(pass)) - 1);
      pass &= pass - 1u;
      const int64_t p = static_cast<int64_t>(32ull * i + j) - 8 * static_cast<int64_t>(sh);
      if (p <= 0) continue;  // (bit 0 is job 0 anyway)
      const uint32_t hclen = (__funnelshift_r(w0, w1, j) >> 13) & 15u;
      const uint32_t ncl = hclen + 4u;
      if (static_cast<uint64_t>(p) + 17u + 3u * ncl > total_bits) continue;
      const uint32_t s = j + 17u;  // 17 .. 48
      // the ncl 3-bit lengths, three at a time through the table: Kraft sum and number of codes
      const uint64_t v = ((lo64 >> s) | (hi64 << (64u - s))) & ((1ull << (3u * ncl)) - 1ull);
      uint32_t acc = 0;
#pragma unroll
      for (uint32_t c = 0; c < 7; ++c) acc += s_kraft[static_cast<uint32_t>(v >> (9u * c)) & 511u];
      if ((acc & 0xffffu) != 128u || (acc >> 16) < 2u) continue;
      const uint32_t at = atomicAdd(a.cand_count, 1u);
      if (at < a.cand_cap) a.cand[at] = static_cast<uint64_t>(p);
    }
  }
}

// n <= 16 bits at bit position p (zero past the end)
__device__ __forceinline__ uint32_t find_bits(const uint8_t* src, uint64_t slen, uint64_t p, uint32_t n)
{
  const uint64_t b = p >> 3;
  uint32_t w = 0;
  for (uint32_t k = 0; k < 3; ++k)
    if (b + k < slen) w |= static_cast<uint32_t>(src[b + k]) << (8u * k);
  return (w >> (p & 7u)) & ((1u << n) - 1u);
}

__global__ void __launch_bounds__(FIND_THREADS) verify_candidates_kernel(const FindArgs a)
{
  // per thread a 128-entry table for the code-length code: 7 input bits -> symbol << 3 | length;
  // entry k of thread t at byte k * FIND_THREADS + t (threads of a warp never meet in a bank)
  __shared__ uint8_t s_cl[128 * FIND_THREADS];
  uint8_t* const lut = s_cl + (threadIdx.x % FIND_THREADS);
  const uint8_t* const src = a.src_base + a.src_off[a.idx];
  const uint64_t slen = a.src_len[a.idx];
  const uint64_t total_bits = 8ull * slen;
  const uint32_t sh = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(src) & 3u);
  uint32_t n_cand = *a.cand_count;
  if (n_cand > a.cand_cap) n_cand = a.cand_cap;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t ci = blockIdx.x * blockDim.x + threadIdx.x; ci < n_cand; ci += stride) {
    const uint64_t p0 = a.cand[ci];
    // bit buffer over the 4-byte aligned view of the stream (zero past its end): `have` valid bits
    // in `buf`, the next word to append is `wi`; `p` counts the bits taken
    uint64_t p = p0 + 3u;
    uint64_t wi = (p + 8u * sh) >> 5;
    uint64_t buf = static_cast<uint64_t>(find_word(src, slen, sh, wi)) >> ((p + 8u * sh) & 31u);
    uint32_t have = 32u - static_cast<uint32_t>((p + 8u * sh) & 31u);
    ++wi;
    auto take = [&](uint32_t n) -> uint32_t {  // n <= 16
      if (have < n + 16u) {                     // (keeps >= 16 bits for the peek below: have + 32 <= 64)
        buf |= static_cast<uint64_t>(find_word(src, slen, sh, wi)) << have;
        have += 32u;
        ++wi;
      }
      const uint32_t v = static_cast<uint32_t>(buf) & ((1u << n) - 1u);
      buf >>= n;
      have -= n;
      p += n;
      return v;
    };
    const uint32_t n_lit = take(5) + 257u;
    const uint32_t n_dist = take(5) + 1u;
    const uint32_t ncl = take(4) + 4u;
    // the code-length code: lengths in the order of RFC 1951 §3.2.7, canonical codes (§3.2.2),
    // the table filled with every 7-bit input whose low bits are a (bit-reversed) code
    uint32_t cl[19];
#pragma unroll
    for (uint32_t c = 0; c < 19; ++c) cl[c] = 0;
    uint64_t bl_count = 0;  // byte l: number of codes of length l
#pragma unroll
    for (uint32_t c = 0; c < 19; ++c) {
      constexpr uint32_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
      if (c < ncl) {
        const uint32_t l = take(3);
        cl[order[c]] = l;
        if (l) bl_count += 1ull << (8u * l);
      }
    }
    uint64_t next_code = 0;  // byte l: the next code of length l
    {
      uint32_t code = 0;
      for (uint32_t l = 1; l <= 7; ++l) {
        code = (code + static_cast<uint32_t>((bl_count >> (8u * (l - 1u))) & 255u) * (l > 1u)) << 1;
        next_code |= static_cast<uint64_t>(code & 255u) << (8u * l);
      }
    }
#pragma unroll
    for (uint32_t c = 0; c < 19; ++c) {
      const uint32_t l = cl[c];
      if (l) {
        const uint32_t code = static_cast<uint32_t>(next_code >> (8u * l)) & 255u;
        next_code += 1ull << (8u * l);
        const uint32_t rev = __brev(code) >> (32u - l);
        for (uint32_t k = rev; k < 128u; k += 1u << l) lut[k * FIND_THREADS] = static_cast<uint8_t>((c << 3) | l);
      }
    }
    // the HLIT + HDIST lengths
    const uint32_t total = n_lit + n_dist;
    uint32_t i = 0, prev = 0, kraft_lit = 0, kraft_dist = 0, dist_codes = 0, eob_len = 0;
    bool ok = true;
    while (ok && i < total) {
      if (have < 16u) {
        buf |= static_cast<uint64_t>(find_word(src, slen, sh, wi)) << have;
        have += 32u;
        ++wi;
      }
      const uint32_t e = lut[(static_cast<uint32_t>(buf) & 127u) * FIND_THREADS];
      const uint32_t len = e & 7u, sym = e >> 3;
      buf >>= len;
      have -= len;
      p += len;
      uint32_t rep = 1, val = sym;
      if (sym == 16u) {
        if (i == 0) {
          ok = false;
          break;
        }
        rep = 3u + take(2);
        val = prev;
      } else if (sym == 17u) {
        rep = 3u + take(3);
        val = 0;
      } else if (sym == 18u) {
        rep = 11u + take(7);
        val = 0;
      }
      if (i + rep > total) {
        ok = false;
        break;
      }
      if (val) {
        const uint32_t lit_end = i + rep < n_lit ? i + rep : n_lit;
        const uint32_t in_lit = lit_end > i ? lit_end - i : 0u;
        kraft_lit += in_lit * (32768u >> val);
        kraft_dist += (rep - in_lit) * (32768u >> val);
        dist_codes += rep - in_lit;
        if (i <= 256u && 256u < i + rep) eob_len = val;
      }
      prev = val;
      i += rep;
      if (kraft_lit > 32768u || kraft_dist > 32768u) {  // over-subscribed already (random bits mostly are, early)
        ok = false;
        break;
      }
    }
    if (!ok || p > total_bits) continue;
    if (kraft_lit != 32768u || eob_len == 0u) continue;
    if (!(kraft_dist == 32768u || dist_codes <= 1u)) continue;
    const uint32_t j = atomicAdd(a.job_count, 1u);
    if (j >= a.job_cap) continue;
    BlockJob jb;
    jb.start_bit = p0;
    jb.end_bit = p0;
    jb.out = 0;
    jb.base = JOB_NONE;
    jb.need = 0;
    jb.flags = JOB_ENDS;
    jb.next = 0;
    jb.first_rec = 0;
    a.jobs[j] = jb;
    __threadfence();  // the record before the table entry
    uint32_t slot = job_slot(p0, a.tab_mask);
    while (atomicCAS(a.job_tab + slot, 0u, j) != 0u) slot = (slot + 1u) & a.tab_mask;
  }
}

#if !defined(SFB_CPU_EMU) || defined(SFB_EMU_BLOCK)  // (tests/cpu_emu: emu_block.cpp runs this on 1024 host threads)

// The same chain, in parallel, by ONE block (the walk above takes 0.5 us per block of the stream:
// 6 ms for the 12 000 blocks of a 1 GiB stream).  Pointer jumping over the jobs: J[j] = the job 2^k
// blocks after j, W[j] = the bytes of those 2^k blocks.  In round k every job already known to be on
// the chain (those up to 2^k - 1 blocks from job 0) marks J[j] and gives it its position base[j] +
// W[j], then J and W double.  What the walk decides on the way — stop at a block whose distances or
// size do not fit — is decided afterwards: among the marked jobs that do not fit, the one that
// starts first is the tail, and everything after it is taken off the chain again.
constexpr int CHAIN_THREADS = 1024;
struct ChainScratch {
  uint32_t* ja;  // [job_cap] each
  uint32_t* jb;
  uint64_t* wa;
  uint64_t* wb;
  uint32_t* mark;
};

__global__ void __launch_bounds__(CHAIN_THREADS) chain_parallel_kernel(const FindArgs a, const ChainScratch c)
{
  constexpr uint32_t NONE = 0xffffffffu;
  __shared__ unsigned long long s_first_bad;  // smallest start_bit among the chain jobs that do not fit
  __shared__ uint32_t s_tail;
  const uint32_t tid = threadIdx.x;
  const uint64_t cap = a.dst_cap[a.idx];
  uint32_t n = *a.job_count;
  if (n > a.job_cap) n = a.job_cap;
  uint32_t* J = c.ja;
  uint32_t* Jn = c.jb;
  uint64_t* W = c.wa;
  uint64_t* Wn = c.wb;
  for (uint32_t j = tid; j < n; j += CHAIN_THREADS) {
    const BlockJob jb = a.jobs[j];
    const bool ends = (jb.flags & JOB_ENDS) || jb.next == 0u || jb.next >= n;
    J[j] = ends ? NONE : jb.next;
    W[j] = jb.out;
    c.mark[j] = j == 0u ? 1u : 0u;  // 0: not on the chain, else 2 + the round that found it (job 0: 1)
    if (j == 0u) a.jobs[0].base = 0;
  }
  if (tid == 0) {
    s_first_bad = ~0ull;
    s_tail = 0;
  }
  __syncthreads();
  uint32_t rounds = 1;
  while ((1u << rounds) < n && rounds < 31u) ++rounds;
  for (uint32_t k = 0; k <= rounds; ++k) {
    for (uint32_t j = tid; j < n; j += CHAIN_THREADS) {
      const uint32_t t = J[j];
      const uint32_t stamp = c.mark[j];
      if (stamp != 0u && stamp < k + 2u && t != NONE) {  // on the chain since an EARLIER round (its base is settled)
        a.jobs[t].base = a.jobs[j].base + W[j];
        c.mark[t] = k + 2u;
      }
      Jn[j] = t == NONE ? NONE : J[t];
      Wn[j] = t == NONE ? W[j] : W[j] + W[t];
    }
    __syncthreads();
    uint32_t* tj = J;
    J = Jn;
    Jn = tj;
    uint64_t* tw = W;
    W = Wn;
    Wn = tw;
  }
  // the first job on the chain that does not fit (or, if all fit, the one the chain ends with)
  for (uint32_t j = tid; j < n; j += CHAIN_THREADS) {
    if (!c.mark[j]) continue;
    const BlockJob jb = a.jobs[j];
    if (jb.need > jb.base || jb.base + jb.out > cap) atomicMin(&s_first_bad, static_cast<unsigned long long>(jb.start_bit));
  }
  __syncthreads();
  const uint64_t first_bad = s_first_bad;
  for (uint32_t j = tid; j < n; j += CHAIN_THREADS) {
    if (!c.mark[j]) continue;
    const BlockJob jb = a.jobs[j];
    if (jb.start_bit > first_bad) {  // behind the tail: not decoded by a job of its own after all
      a.jobs[j].base = JOB_NONE;
      continue;
    }
    const bool fits = jb.need <= jb.base && jb.base + jb.out <= cap;
    if ((jb.flags & JOB_RECS) && fits) a.jobs[j].flags = jb.flags | JOB_USE;
    const bool ends = (jb.flags & JOB_ENDS) || jb.next == 0u || jb.next >= n;
    if (jb.start_bit == first_bad || (first_bad == ~0ull && ends)) s_tail = j;
  }
  __syncthreads();
  if (tid == 0) *a.tail_job = s_tail;
}

#endif  // SFB_CPU_EMU

}  // namespace sfb
