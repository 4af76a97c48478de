// Batched raw-DEFLATE COMPRESSION for sm_100a, ONE WARP PER STREAM (SURVEY.md §8 f4: the step on the
// other side of the hot path, which the reference's README names as the parallelisable direction
// it has not built, README.md:5-7).  LZ77 by hashing + ONE Huffman block per stream — DYNAMIC
// (RFC 1951 §3.2.7) where that is smaller, else FIXED (§3.2.6; the reference's fixed tables are
// src/decompress.cpp:25-40) — or stored blocks when neither beats the input.  What it writes is
// what the decoder of this repository, zlib and the reference decompress() all accept; the tests
// round-trip through all three.
//
// The dynamic block takes the parse TWICE (the hash table starts from zero both times, so the two
// passes see the same tokens): pass A only counts symbols (shared-memory histograms), the warp then
// derives the code lengths, pass B emits.  Code lengths are not built from a Huffman tree but from
// the Kraft sum, which is what a warp can do in parallel (cmp_build_lengths): Shannon lengths
// ceil(log2(total / f)) clamped to the limit, then one symbol at a time is lengthened (only if the
// clamp pushed the sum over 1) or shortened — always the one with the best bits-saved per
// code-space ratio f * 2^len that still fits, found by a warp arg-max — until the sum is EXACTLY 1:
// a complete prefix code (zlib refuses incomplete ones), within ~1 % of Huffman's on text.  The
// two alphabets' lengths are run-length coded separately (the reference has undefined behaviour on
// a repeat that crosses from the literal/length lengths into the distance lengths).
//
// Per step the warp looks at 32 consecutive positions, one per lane:
//   1. hash of the 4 bytes at the position -> candidate (the last earlier position with that hash:
//      a 4 096-entry table of 16-bit positions per warp in shared memory); the highest lane of every
//      hash value then enters its own position (deterministic: __match_any_sync);
//   2. each lane measures its match against the candidate, 4 bytes per comparison (unaligned words
//      put together from aligned ones; never a byte past the stream);
//   3. greedy parse, front to back, by the whole warp: the token at the cursor is the lane's match if
//      it is at least 4 bytes long, else a literal; the cursor moves by its length (possibly past
//      the 32 positions: the next step starts where the cursor stands, positions inside a match are
//      not entered in the table);
//   4. every token lane builds its bits — fixed literal/length code MSB first, extra bits, 5-bit
//      distance code, extra bits: at most 31 — an exclusive scan of the bit counts places them, and
//      the lanes OR them into a 64-word staging window in shared memory that is written out to dst
//      in whole words (bytes where dst is not word-aligned or the capacity ends inside a word).
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#endif

#include "deflate_lane.cuh"

namespace sfb {

struct CompressArgs {
  const uint8_t* src_base;
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint8_t* dst_base;
  const uint64_t* dst_off;
  const uint64_t* dst_cap;
  uint8_t* status;       // ST_SUCCESS, ST_DST_TOO_SMALL (neither form fits dst_cap), ST_ERROR (src_len >= 4 GiB - 256)
  uint64_t* written;
  uint64_t n;
  unsigned long long* counter;  // zeroed before launch
  int fixed_only;               // != 0: one pass, fixed-Huffman blocks only (the first generation; A/B runs)
};

constexpr int CMP_WARPS = 4;   // 43 KiB of shared memory per CTA: five CTAs, 20 warps per SM
constexpr int CMP_HASH_BITS = 12;
constexpr int CMP_STAGE_WORDS = 128;   // flushed from 1 024 bits on; one step adds at most 32 x 48 bits
constexpr int CMP_NLL = 288;           // literal/length symbols (286 used)
constexpr int CMP_ND = 32;             // distance symbols (30 used)
constexpr int CMP_NCL = 32;            // code-length symbols (19 used)
constexpr int CMP_NSEQ = 320;          // run-length coded code lengths: at most 286 + 30 entries
// per warp: hash table | bit staging | u32 tables (frequencies, then codes) | u8 lengths | u16 RLE sequence
constexpr int CMP_TAB_WORDS = CMP_NLL + CMP_ND + CMP_NCL;
constexpr int CMP_WARP_BYTES = (1 << CMP_HASH_BITS) * 2 + CMP_STAGE_WORDS * 4 + CMP_TAB_WORDS * 4 +
                               (CMP_NLL + CMP_ND + CMP_NCL) + CMP_NSEQ * 2;
constexpr int CMP_SMEM_BYTES = CMP_WARPS * CMP_WARP_BYTES;
constexpr uint32_t CMP_MIN_MATCH = 4;
#ifndef SFB_CMP_LAZY
#define SFB_CMP_LAZY 1
#endif
constexpr bool CMP_LAZY = SFB_CMP_LAZY != 0;
constexpr uint32_t CMP_MAX_MATCH = 258;
constexpr uint32_t CMP_MAX_DIST = 32768;

// bytes [p, p + 4) of the stream at `s` as a little-endian word, from aligned words that each hold
// at least one of them (p + 4 <= stream length is the caller's business)
__device__ __forceinline__ uint32_t cmp_load32(const uint8_t* s, uint32_t p)
{
  const uintptr_t a = reinterpret_cast<uintptr_t>(s + p);
  const uint32_t r = static_cast<uint32_t>(a & 3u);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a - r);
  const uint32_t lo = w[0];
  const uint32_t hi = r ? w[1] : 0u;
  return funnel_r(lo, hi, 8u * r);
}

__device__ __forceinline__ uint32_t cmp_ctz(uint32_t v)
{
#ifdef SFB_CPU_EMU
  return static_cast<uint32_t>(__builtin_ctz(v));
#else
  return static_cast<uint32_t>(__ffs(static_cast<int>(v)) - 1);
#endif
}

// length 3..258 -> length symbol 257 + k, extra bits (RFC 1951 §3.2.5)
__device__ __forceinline__ void cmp_len_sym(uint32_t len, uint32_t* k, uint32_t* eb, uint32_t* ev)
{
  const uint32_t l = len - 3u;
  if (len == 258u) {
    *k = 28u;
    *eb = 0u;
    *ev = 0u;
  } else if (l < 8u) {
    *k = l;
    *eb = 0u;
    *ev = 0u;
  } else {
    const uint32_t n = 31u - static_cast<uint32_t>(__clz(static_cast<int>(l)));
    *eb = n - 2u;
    *k = 4u * (n - 2u) + 4u + ((l >> (n - 2u)) & 3u);
    *ev = l & ((1u << (n - 2u)) - 1u);
  }
}
// distance 1..32768 -> distance symbol, extra bits
__device__ __forceinline__ void cmp_dist_sym(uint32_t dist, uint32_t* ds, uint32_t* eb, uint32_t* ev)
{
  const uint32_t x = dist - 1u;
  if (x < 4u) {
    *ds = x;
    *eb = 0u;
    *ev = 0u;
  } else {
    const uint32_t n = 31u - static_cast<uint32_t>(__clz(static_cast<int>(x)));
    *eb = n - 1u;
    *ds = 2u * n + ((x >> (n - 1u)) & 1u);
    *ev = x & ((1u << (n - 1u)) - 1u);
  }
}
// fixed-Huffman code lengths (RFC 1951 §3.2.6)
__device__ __forceinline__ uint32_t cmp_fixed_ll_len(uint32_t sym)
{
  return sym < 144u ? 8u : sym < 256u ? 9u : sym < 280u ? 7u : 8u;
}

// fixed-Huffman bits of one token, LSB = first bit of the stream; *nb = how many (<= 31)
__device__ __forceinline__ uint32_t cmp_literal_bits(uint32_t lit, uint32_t* nb)
{
  // 0-143: 8 bits 00110000.. ; 144-255: 9 bits 110010000..  (codes go out MSB first)
  const bool small = lit < 144u;
  const uint32_t code = small ? 0x30u + lit : 0x190u + (lit - 144u);
  const uint32_t n = small ? 8u : 9u;
  *nb = n;
  return __brev(code) >> (32u - n);
}
__device__ __forceinline__ uint32_t cmp_match_bits(uint32_t len, uint32_t dist, uint32_t* nb)
{
  uint32_t k, leb, lev;
  cmp_len_sym(len, &k, &leb, &lev);
  // fixed code of 257 + k: 256-279 are 7 bits 0000000.., 280-287 8 bits 11000000..
  const uint32_t sym = 257u + k;
  const bool seven = sym < 280u;
  const uint32_t lcode = seven ? sym - 256u : 0xC0u + (sym - 280u);
  const uint32_t ln = seven ? 7u : 8u;
  uint32_t bits = __brev(lcode) >> (32u - ln);
  uint32_t at = ln;
  bits |= lev << at;
  at += leb;
  // distance symbol, 5-bit fixed code, extra bits
  uint32_t ds, deb, dev;
  cmp_dist_sym(dist, &ds, &deb, &dev);
  bits |= (__brev(ds) >> 27) << at;
  at += 5u;
  bits |= dev << at;
  at += deb;
  *nb = at;
  return bits;
}

// The warp's bit writer: a window of CMP_STAGE_WORDS words over the output, starting at word `wbase`.
struct CmpWriter {
  uint32_t* stage;   // shared
  uint8_t* d;        // dst of the stream
  uint32_t cap;      // its capacity in bytes
  uint32_t wbase;    // output words already written out
  uint32_t cur;      // bits in the window
  uint32_t lane;

  __device__ __forceinline__ void open(uint32_t* stage_, uint8_t* d_, uint32_t cap_, uint32_t lane_)
  {
    stage = stage_;
    d = d_;
    cap = cap_;
    wbase = 0;
    cur = 0;
    lane = lane_;
    for (uint32_t j = lane; j < static_cast<uint32_t>(CMP_STAGE_WORDS); j += 32u) stage[j] = 0;
    __syncwarp();
  }
  // word j of the window -> dst (only bytes inside the capacity)
  __device__ __forceinline__ void store_word(uint32_t j, uint32_t nbytes)
  {
    const uint32_t at = 4u * (wbase + j);
    const uint32_t v = stage[j];
    uint8_t* p = d + at;
    if (nbytes == 4u && at + 4u <= cap && (reinterpret_cast<uintptr_t>(p) & 3u) == 0u) {
      *reinterpret_cast<uint32_t*>(p) = v;
    } else {
      for (uint32_t b = 0; b < nbytes; ++b)
        if (at + b < cap) p[b] = static_cast<uint8_t>(v >> (8u * b));
    }
  }
  // every lane brings `nb` bits (0: none; at most 48), in lane order
  __device__ __forceinline__ void put(uint64_t bits, uint32_t nb)
  {
    constexpr unsigned FULL = 0xffffffffu;
    uint32_t off = nb;  // inclusive scan
#pragma unroll
    for (int dlt = 1; dlt < 32; dlt <<= 1) {
      const uint32_t t = __shfl_up_sync(FULL, off, static_cast<unsigned>(dlt));
      if (lane >= static_cast<uint32_t>(dlt)) off += t;
    }
    const uint32_t total = __shfl_sync(FULL, off, 31);
    off -= nb;
    if (nb) {
      const uint32_t at = cur + off, w = at >> 5, sh = at & 31u;
      const uint64_t lo = bits << sh;   // (bits < 2^48, sh < 32: what is shifted out is bits >> (64 - sh))
      atomicOr(&stage[w], static_cast<uint32_t>(lo));
      if (sh + nb > 32u) atomicOr(&stage[w + 1], static_cast<uint32_t>(lo >> 32));
      if (sh + nb > 64u) atomicOr(&stage[w + 2], static_cast<uint32_t>(bits >> (64u - sh)));
    }
    cur += total;
    __syncwarp();
    if (cur >= 32u * 32u) flush_words();
  }
  // write the complete words out and move the open one to the front
  __device__ __forceinline__ void flush_words()
  {
    const uint32_t nw = cur >> 5;   // < CMP_STAGE_WORDS
    for (uint32_t j = lane; j < nw; j += 32u) store_word(j, 4u);
    __syncwarp();
    const uint32_t open_word = stage[nw];
    __syncwarp();
    for (uint32_t j = lane; j < static_cast<uint32_t>(CMP_STAGE_WORDS); j += 32u) stage[j] = j == 0u ? open_word : 0u;
    wbase += nw;
    cur &= 31u;
    __syncwarp();
  }
  // the end of the stream: everything out; -> total bytes
  __device__ __forceinline__ uint64_t close()
  {
    const uint32_t nw = cur >> 5, rest = (cur & 31u) + 7u >> 3;
    for (uint32_t j = lane; j < nw; j += 32u) store_word(j, 4u);
    if (lane == 0u && rest) store_word(nw, rest);
    __syncwarp();
    return 4ull * (static_cast<uint64_t>(wbase) + nw) + rest;
  }
};

// stored blocks (src/decompress.cpp:416-436 reads them): 5 header bytes per <= 65 535 payload bytes
__device__ __forceinline__ uint64_t cmp_stored_size(uint64_t n) { return n + 5ull * (n ? (n + 65534ull) / 65535ull : 1ull); }

__device__ __forceinline__ void cmp_write_stored(const uint8_t* s, uint32_t n, uint8_t* d, uint32_t lane)
{
  uint32_t done = 0;
  uint64_t at = 0;
  do {
    const uint32_t blk = n - done < 65535u ? n - done : 65535u;
    const bool fin = done + blk == n;
    if (lane == 0u) {
      d[at] = fin ? 1u : 0u;
      d[at + 1] = static_cast<uint8_t>(blk);
      d[at + 2] = static_cast<uint8_t>(blk >> 8);
      d[at + 3] = static_cast<uint8_t>(~blk);
      d[at + 4] = static_cast<uint8_t>((~blk) >> 8);
    }
    for (uint32_t i = lane; i < blk; i += 32u) d[at + 5 + i] = s[done + i];
    at += 5ull + blk;
    done += blk;
  } while (done < n);
}

// ---------------------------------------------------------------------------------------------
// Code lengths of a complete prefix code for the symbols with freq != 0 (at least two: the caller
// sees to it), none longer than `maxlen` (<= 15), by the whole warp; lane l owns symbols l, l + 32, ..
// Kraft sum in units of 2^-15: a symbol of length len takes 2^(15 - len), a complete code 2^15.
// -> false if the loops hit their bound (the caller then does without a dynamic block).
__device__ __forceinline__ uint32_t cmp_shfl_down(uint32_t v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }

__device__ __forceinline__ bool cmp_build_lengths(const uint32_t* freq, uint32_t nsym, uint32_t maxlen, uint8_t* len,
                                                  uint32_t lane)
{
  constexpr unsigned FULL = 0xffffffffu;
  uint32_t tot = 0;
  for (uint32_t i = lane; i < nsym; i += 32u) tot += freq[i];
  tot = __reduce_add_sync(FULL, tot);
  uint32_t kraft = 0;
  for (uint32_t i = lane; i < nsym; i += 32u) {
    const uint32_t f = freq[i];
    uint32_t l = 0;
    if (f) {
      l = 1;
      while (l < maxlen && (static_cast<uint64_t>(f) << l) < tot) ++l;   // ceil(log2(tot / f)), clamped
      kraft += 1u << (15u - l);
    }
    len[i] = static_cast<uint8_t>(l);
  }
  kraft = __reduce_add_sync(FULL, kraft);
  __syncwarp();
  // One move per iteration.  Over 1 (only the clamp does that): lengthen the symbol that loses
  // the fewest bits per unit of code space it gives back, f * 2^len smallest.  Under 1: shorten
  // the symbol with the largest f * 2^len among those whose step still fits.  A sum below 1 is a
  // multiple of the smallest unit in use, so the longest code always fits: the loop ends at 1.
  for (uint32_t iter = 0; iter < 8192u; ++iter) {
    if (kraft == (1u << 15)) return true;
    const bool over = kraft > (1u << 15);
    const uint32_t slack = over ? 0u : (1u << 15) - kraft;
    uint64_t best = over ? ~0ull : 0ull;
    uint32_t besti = 0xffffffffu;
    for (uint32_t i = lane; i < nsym; i += 32u) {
      const uint32_t l = len[i];
      if (l == 0u) continue;
      const uint64_t key = static_cast<uint64_t>(freq[i]) << l;
      if (over) {
        if (l < maxlen && (key < best || besti == 0xffffffffu)) {
          best = key;
          besti = i;
        }
      } else {
        if (l > 1u && (1u << (15u - l)) <= slack && (key > best || besti == 0xffffffffu)) {
          best = key;
          besti = i;
        }
      }
    }
    // warp arg-min / arg-max (ties: the lower symbol, so that the result does not depend on timing)
#pragma unroll
    for (int dlt = 16; dlt >= 1; dlt >>= 1) {
      const uint32_t ohi = cmp_shfl_down(static_cast<uint32_t>(best >> 32), dlt);
      const uint32_t olo = cmp_shfl_down(static_cast<uint32_t>(best), dlt);
      const uint32_t oi = cmp_shfl_down(besti, dlt);
      const uint64_t ob = (static_cast<uint64_t>(ohi) << 32) | olo;
      bool take = false;
      if (oi != 0xffffffffu) {
        if (besti == 0xffffffffu) take = true;
        else if (ob == best) take = oi < besti;
        else take = over ? ob < best : ob > best;
      }
      if (take) {
        best = ob;
        besti = oi;
      }
    }
    besti = __shfl_sync(FULL, besti, 0);
    if (besti == 0xffffffffu) return false;   // (cannot happen with two or more symbols and maxlen >= 9 .. see caller)
    const uint32_t l = len[besti];
    __syncwarp();
    if (over) {
      if (lane == 0u) len[besti] = static_cast<uint8_t>(l + 1u);
      kraft -= 1u << (14u - l);
    } else {
      if (lane == 0u) len[besti] = static_cast<uint8_t>(l - 1u);
      kraft += 1u << (15u - l);
    }
    __syncwarp();
  }
  return false;
}

// canonical codes for `len` (RFC 1951 §3.2.2), bit-reversed (codes go out MSB first, the writer is
// LSB first) and packed as code | len << 16; one lane
__device__ __forceinline__ void cmp_assign_codes(const uint8_t* len, uint32_t nsym, uint32_t* code)
{
  uint32_t count[16], next[16];
  for (uint32_t l = 0; l < 16u; ++l) count[l] = 0;
  for (uint32_t i = 0; i < nsym; ++i) ++count[len[i]];
  count[0] = 0;
  uint32_t c = 0;
  next[0] = 0;
  for (uint32_t l = 1; l < 16u; ++l) {
    c = (c + count[l - 1u]) << 1;
    next[l] = c;
  }
  for (uint32_t i = 0; i < nsym; ++i) {
    const uint32_t l = len[i];
    code[i] = l ? ((__brev(next[l]++) >> (32u - l)) | (l << 16)) : 0u;
  }
}

// The parse: 32 consecutive positions per step (see the header of this file).  MODE 0 counts the
// symbols (atomic adds into freq_ll / freq_d, extra bits summed per lane into *xbits), MODE 1 emits
// fixed-Huffman bits, MODE 2 emits with the code tables code_ll / code_d.  The hash table starts
// from zero every time, so every mode sees the same tokens.
template <int MODE>
__device__ __forceinline__ void cmp_parse(const uint8_t* s, uint32_t n, uint16_t* tab, uint32_t lane, CmpWriter& w,
                                          uint32_t* tab_ll, uint32_t* tab_d, uint64_t* xbits)
{
  constexpr unsigned FULL = 0xffffffffu;
  for (uint32_t j = lane; j < (1u << CMP_HASH_BITS) / 2u; j += 32u) reinterpret_cast<uint32_t*>(tab)[j] = 0u;
  __syncwarp();
  uint32_t c = 0;                    // the cursor: everything before it is encoded
  while (c < n) {
    const uint32_t pos = c + lane;
    const bool can = pos + CMP_MIN_MATCH <= n;   // four bytes to hash
    uint32_t v = 0, h = 0xffffffffu - lane;      // (lanes without a hash never share one)
    uint32_t cand16 = 0;
    if (can) {
      v = cmp_load32(s, pos);
      h = (v * 0x9E3779B1u) >> (32 - CMP_HASH_BITS);
      cand16 = tab[h];
    }
    __syncwarp();
    {
      const uint32_t same = __match_any_sync(FULL, h);
      if (can && (same >> lane) <= 1u) tab[h] = static_cast<uint16_t>(pos);   // the highest lane with this hash
    }
    // candidate position: the table holds the low 16 bits of a position before this step
    uint32_t mlen = 0, dist = 0;
    if (can) {
      int64_t cand = static_cast<int64_t>((pos & ~0xffffu) | cand16);
      if (cand >= static_cast<int64_t>(c)) cand -= 65536;
      if (cand >= 0 && pos - static_cast<uint32_t>(cand) <= CMP_MAX_DIST) {
        const uint32_t cp = static_cast<uint32_t>(cand);
        const uint32_t maxlen = n - pos < CMP_MAX_MATCH ? n - pos : CMP_MAX_MATCH;
        uint32_t m = 0;
        bool open_end = true;
        while (m + 4u <= maxlen) {
          const uint32_t x = cmp_load32(s, pos + m) ^ cmp_load32(s, cp + m);
          if (x) {
            m += cmp_ctz(x) >> 3;
            open_end = false;
            break;
          }
          m += 4u;
        }
        if (open_end)
          while (m < maxlen && s[pos + m] == s[cp + m]) ++m;
        if (m >= CMP_MIN_MATCH) {
          mlen = m;
          dist = pos - cp;
        }
      }
    }
    // parse of the 32 positions, front to back, by the whole warp: greedy with one step of
    // laziness — a match gives way to a literal when the next position has a longer one (what
    // zlib's deflate_slow does; the next position's candidate is already there, so it costs a shuffle)
    // (the loop runs once per MATCH taken: the literals between two matches are found with the
    //  ballot of the positions that have one)
    const uint32_t lim = n - c < 32u ? n - c : 32u;
    const uint32_t mm = __ballot_sync(FULL, mlen != 0u);
    uint32_t start_mask = 0, lit_mask = 0;
    uint32_t t = 0;
    while (t < lim) {
      const uint32_t rest = mm & (0xffffffffu << t);                         // matches at or after t ..
      const uint32_t p = rest ? cmp_ctz(rest) : 32u;                         // .. the first of them
      if (p >= lim) {                                                        // literals to the end of the step
        start_mask |= (0xffffffffu << t) & (0xffffffffu >> (32u - lim));
        t = lim;
        break;
      }
      start_mask |= (0xffffffffu << t) & (0xffffffffu >> (31u - p));         // literals [t, p) and the token at p
      const uint32_t L = __shfl_sync(FULL, mlen, static_cast<int>(p));
      const uint32_t Ln = __shfl_sync(FULL, mlen, static_cast<int>((p + 1u) & 31u));
      const bool defer = CMP_LAZY && p + 1u < 32u && Ln > L;
      if (defer) {
        lit_mask |= 1u << p;
        t = p + 1u;
      } else {
        t = p + L;
      }
    }
    const bool start = ((start_mask >> lane) & 1u) != 0u, as_lit = ((lit_mask >> lane) & 1u) != 0u;
    if (as_lit) mlen = 0;
    if constexpr (MODE == 0) {
      if (start) {
        if (mlen) {
          uint32_t k, leb, lev, ds, deb, dev;
          cmp_len_sym(mlen, &k, &leb, &lev);
          cmp_dist_sym(dist, &ds, &deb, &dev);
          atomicAdd(&tab_ll[257u + k], 1u);
          atomicAdd(&tab_d[ds], 1u);
          *xbits += leb + deb;
        } else {
          atomicAdd(&tab_ll[s[pos]], 1u);
        }
      }
    } else if constexpr (MODE == 1) {
      uint32_t bits = 0, nb = 0;
      if (start) bits = mlen ? cmp_match_bits(mlen, dist, &nb) : cmp_literal_bits(s[pos], &nb);
      w.put(bits, nb);
    } else {
      uint64_t bits = 0;
      uint32_t nb = 0;
      if (start) {
        if (mlen) {
          uint32_t k, leb, lev, ds, deb, dev;
          cmp_len_sym(mlen, &k, &leb, &lev);
          cmp_dist_sym(dist, &ds, &deb, &dev);
          const uint32_t el = tab_ll[257u + k], ed = tab_d[ds];
          bits = el & 0xffffu;
          nb = el >> 16;
          bits |= static_cast<uint64_t>(lev) << nb;
          nb += leb;
          bits |= static_cast<uint64_t>(ed & 0xffffu) << nb;
          nb += ed >> 16;
          bits |= static_cast<uint64_t>(dev) << nb;
          nb += deb;   // <= 15 + 5 + 15 + 13
        } else {
          const uint32_t el = tab_ll[s[pos]];
          bits = el & 0xffffu;
          nb = el >> 16;
        }
      }
      w.put(bits, nb);
    }
    c += t;
  }
  __syncwarp();
}

// Piece mode (PIECES, compress_parallel.cuh): stream si is one piece of a larger buffer.  BFINAL is
// set only on stream `last`; nothing is written for a piece that falls back to a stored block (the
// stitch kernel writes it from the source at its final bit position); status is ST_SUCCESS or
// CMP_PIECE_STORED, written the block's exact size in BITS (0 when stored).
constexpr uint8_t CMP_PIECE_STORED = 0x80;

template <bool PIECES>
__device__ __forceinline__ void cmp_streams(const CompressArgs& a, uint64_t last)
{
#ifdef SFB_CPU_EMU
  uint8_t* const smem = reinterpret_cast<uint8_t*>(SFB_EMU_SMEM);
#else
  extern __shared__ __align__(16) uint8_t smem[];
#endif
  constexpr unsigned FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp = threadIdx.x >> 5;
  uint8_t* const wsm = smem + warp * CMP_WARP_BYTES;
  uint16_t* const tab = reinterpret_cast<uint16_t*>(wsm);
  uint32_t* const stage = reinterpret_cast<uint32_t*>(wsm + (1 << CMP_HASH_BITS) * 2);
  uint32_t* const t_ll = stage + CMP_STAGE_WORDS;   // frequencies, then codes
  uint32_t* const t_d = t_ll + CMP_NLL;
  uint32_t* const t_cl = t_d + CMP_ND;
  uint8_t* const l_ll = reinterpret_cast<uint8_t*>(t_cl + CMP_NCL);
  uint8_t* const l_d = l_ll + CMP_NLL;
  uint8_t* const l_cl = l_d + CMP_ND;
  uint16_t* const seq = reinterpret_cast<uint16_t*>(l_cl + CMP_NCL);   // symbol | extra value << 5
  for (;;) {
    unsigned long long si = 0;
    if (lane == 0) si = atomicAdd(a.counter, 1ull);
    si = __shfl_sync(FULL, si, 0);
    if (si >= a.n) break;
    const bool fin = !PIECES || si == last;   // BFINAL
    const uint64_t slen = a.src_len[si], cap64 = a.dst_cap[si];
    if (slen >= 0xffffff00ull) {
      if (lane == 0) {
        a.status[si] = ST_ERROR;
        a.written[si] = 0;
      }
      continue;
    }
    const uint8_t* const s = a.src_base + a.src_off[si];
    uint8_t* const d = a.dst_base + a.dst_off[si];
    const uint32_t n = static_cast<uint32_t>(slen);
    const uint32_t cap = cap64 > 0xffffffffull ? 0xffffffffu : static_cast<uint32_t>(cap64);
    CmpWriter w;
    w.open(stage, d, cap, lane);
    // ---- pass A: symbol statistics, code lengths, which kind of block ---------------------------
    bool dynamic = false;
    uint32_t hlit = 257, hdist = 1, hclen = 4, nseq = 0;
    if (!a.fixed_only && n != 0u) {
      for (uint32_t j = lane; j < static_cast<uint32_t>(CMP_TAB_WORDS); j += 32u) t_ll[j] = 0u;
      __syncwarp();
      uint64_t xb = 0;   // (extra bits: the same under both codes, not needed for the choice)
      cmp_parse<0>(s, n, tab, lane, w, t_ll, t_d, &xb);
      if (lane == 0u) {
        t_ll[256] = 1u;   // the end-of-block symbol
        // at least two symbols per alphabet (a one-symbol code cannot be complete)
        uint32_t used = 0;
        for (uint32_t i = 0; i < 30u; ++i) used += t_d[i] != 0u;
        if (used < 2u) {   // (what zlib does too: the decoders want a complete distance code)
          if (t_d[0] == 0u) t_d[0] = 1u;
          if (t_d[1] == 0u) t_d[1] = 1u;
        }
        used = 0;
        for (uint32_t i = 0; i < 286u; ++i) used += t_ll[i] != 0u;
        if (used < 2u) t_ll[0] += 1u;   // (only the end-of-block symbol: an empty parse cannot happen with n != 0, but stay safe)
      }
      __syncwarp();
      bool ok = cmp_build_lengths(t_ll, 286u, 15u, l_ll, lane);
      ok = cmp_build_lengths(t_d, 30u, 15u, l_d, lane) && ok;
      __syncwarp();
      // bits of the tokens under both codes (extra bits are the same in both)
      uint64_t dyn_bits = 0, fix_bits = 0;
      for (uint32_t i = lane; i < 286u; i += 32u) {
        dyn_bits += static_cast<uint64_t>(t_ll[i]) * l_ll[i];
        fix_bits += static_cast<uint64_t>(t_ll[i]) * cmp_fixed_ll_len(i);
      }
      for (uint32_t i = lane; i < 30u; i += 32u) {
        dyn_bits += static_cast<uint64_t>(t_d[i]) * l_d[i];
        fix_bits += static_cast<uint64_t>(t_d[i]) * 5u;
      }
#pragma unroll
      for (int dlt = 16; dlt >= 1; dlt >>= 1) {
        dyn_bits += __shfl_down_sync(FULL, dyn_bits, dlt);
        fix_bits += __shfl_down_sync(FULL, fix_bits, dlt);
      }
      // ---- the code-length sequence (lane 0): the two alphabets run-length coded one after the
      //      other (RFC 1951 §3.2.7: 16 = repeat the previous length 3-6 times, 17 / 18 = 3-10 /
      //      11-138 zeros), frequencies of the 19 symbols
      if (lane == 0u) {
        hlit = 286u;
        while (hlit > 257u && l_ll[hlit - 1u] == 0u) --hlit;
        hdist = 30u;
        while (hdist > 1u && l_d[hdist - 1u] == 0u) --hdist;
        for (uint32_t i = 0; i < static_cast<uint32_t>(CMP_NCL); ++i) t_cl[i] = 0u;
        uint32_t ns = 0;
        for (uint32_t which = 0; which < 2u; ++which) {
          const uint8_t* L = which ? l_d : l_ll;
          const uint32_t cnt = which ? hdist : hlit;
          uint32_t i = 0;
          while (i < cnt) {
            const uint32_t v = L[i];
            uint32_t run = 1;
            while (i + run < cnt && L[i + run] == v) ++run;
            uint32_t left = run;
            if (v == 0u) {
              while (left >= 11u) {
                const uint32_t r = left < 138u ? left : 138u;
                seq[ns++] = static_cast<uint16_t>(18u | ((r - 11u) << 5));
                ++t_cl[18];
                left -= r;
              }
              if (left >= 3u) {
                seq[ns++] = static_cast<uint16_t>(17u | ((left - 3u) << 5));
                ++t_cl[17];
                left = 0;
              }
              while (left) {
                seq[ns++] = 0;
                ++t_cl[0];
                --left;
              }
            } else {
              seq[ns++] = static_cast<uint16_t>(v);
              ++t_cl[v];
              --left;
              while (left >= 3u) {
                const uint32_t r = left < 6u ? left : 6u;
                seq[ns++] = static_cast<uint16_t>(16u | ((r - 3u) << 5));
                ++t_cl[16];
                left -= r;
              }
              while (left) {
                seq[ns++] = static_cast<uint16_t>(v);
                ++t_cl[v];
                --left;
              }
            }
            i += run;
          }
        }
        nseq = ns;
        uint32_t used = 0;
        for (uint32_t i = 0; i < 19u; ++i) used += t_cl[i] != 0u;
        if (used < 2u) t_cl[t_cl[0] ? 1u : 0u] += 1u;
      }
      __syncwarp();
      nseq = __shfl_sync(FULL, nseq, 0);
      hlit = __shfl_sync(FULL, hlit, 0);
      hdist = __shfl_sync(FULL, hdist, 0);
      ok = cmp_build_lengths(t_cl, 19u, 7u, l_cl, lane) && ok;
      __syncwarp();
      uint64_t head_bits = 0;
      if (lane == 0u) {
        // HCLEN: the code-length code's lengths go out in this order, trailing zeros dropped
        const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        hclen = 19u;
        while (hclen > 4u && l_cl[order[hclen - 1u]] == 0u) --hclen;
        head_bits = 3u + 5u + 5u + 4u + 3u * hclen;
        for (uint32_t i = 0; i < nseq; ++i) {
          const uint32_t sym = seq[i] & 31u;
          head_bits += l_cl[sym] + (sym == 16u ? 2u : sym == 17u ? 3u : sym == 18u ? 7u : 0u);
        }
      }
      head_bits = __shfl_sync(FULL, head_bits, 0);
      hclen = __shfl_sync(FULL, hclen, 0);
      dyn_bits = __shfl_sync(FULL, dyn_bits, 0) + head_bits;
      fix_bits = __shfl_sync(FULL, fix_bits, 0) + 3u;
      dynamic = ok && dyn_bits < fix_bits;
      if (dynamic) {   // the tables turn from frequencies into codes
        __syncwarp();
        if (lane == 0u) cmp_assign_codes(l_ll, 286u, t_ll);
        if (lane == 1u) cmp_assign_codes(l_d, 30u, t_d);
        if (lane == 2u) cmp_assign_codes(l_cl, 19u, t_cl);
        __syncwarp();
      }
    }
    // ---- pass B: the block ---------------------------------------------------------------------
    if (dynamic) {
      const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
      // BFINAL, BTYPE = 10, HLIT, HDIST, HCLEN
      w.put((fin ? 5u : 4u) | ((hlit - 257u) << 3) | ((hdist - 1u) << 8) | ((hclen - 4u) << 13), lane == 0u ? 17u : 0u);
      w.put(lane < hclen ? l_cl[order[lane < 19u ? lane : 0u]] : 0u, lane < hclen ? 3u : 0u);
      for (uint32_t base = 0; base < nseq; base += 32u) {
        uint64_t bits = 0;
        uint32_t nb = 0;
        if (base + lane < nseq) {
          const uint32_t e = seq[base + lane], sym = e & 31u, c = t_cl[sym];
          bits = (c & 0xffffu) | (static_cast<uint64_t>(e >> 5) << (c >> 16));
          nb = (c >> 16) + (sym == 16u ? 2u : sym == 17u ? 3u : sym == 18u ? 7u : 0u);
        }
        w.put(bits, nb);
      }
      uint64_t dummy = 0;
      cmp_parse<2>(s, n, tab, lane, w, t_ll, t_d, &dummy);
      w.put(t_ll[256] & 0xffffu, lane == 0u ? t_ll[256] >> 16 : 0u);   // end of block
    } else {
      uint64_t dummy = 0;
      w.put(fin ? 3u : 2u, lane == 0u ? 3u : 0u);   // BFINAL, BTYPE = 01
      cmp_parse<1>(s, n, tab, lane, w, t_ll, t_d, &dummy);
      w.put(0u, lane == 0u ? 7u : 0u);   // end of block: seven zero bits
    }
    const uint64_t bits = 32ull * w.wbase + w.cur;
    const uint64_t comp = w.close();
    const uint64_t stored = cmp_stored_size(n);
    if constexpr (PIECES) {   // the same choice of block as below (the stored size does not depend on where it lands)
      const bool as_stored = comp > stored || comp > cap;
      if (lane == 0) {
        a.status[si] = as_stored ? CMP_PIECE_STORED : static_cast<uint8_t>(ST_SUCCESS);
        a.written[si] = as_stored ? 0 : bits;
      }
      __syncwarp();
      continue;
    }
    uint64_t out = comp;
    int st = ST_SUCCESS;
    if (comp > stored || comp > cap) {
      if (stored <= cap) {
        __syncwarp();
        cmp_write_stored(s, n, d, lane);
        out = stored;
      } else {
        st = ST_DST_TOO_SMALL;
        out = 0;
      }
    }
    if (lane == 0) {
      a.status[si] = static_cast<uint8_t>(st);
      a.written[si] = out;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(CMP_WARPS * 32) deflate_compress_kernel(const CompressArgs a) { cmp_streams<false>(a, 0); }

// piece mode: `last` = the index of the stream that ends the buffer (none: ~0).  (Five CTAs per SM is
// what the shared memory allows anyway; without the hint ptxas takes 64 registers and spills.)
__global__ void __launch_bounds__(CMP_WARPS * 32, 5) deflate_compress_pieces_kernel(const CompressArgs a, uint64_t last)
{
  cmp_streams<true>(a, last);
}

}  // namespace sfb
