// ONE buffer as ONE raw-DEFLATE, zlib or gzip stream at batch speed (sfb200_compress_parallel_device):
// the buffer is cut into BGZF's pieces of BGZF_PIECE bytes, the pieces are compressed side by side as
// self-contained blocks (BFINAL only on the last), and the blocks are joined at BIT granularity, so the
// stream has no empty stored block between pieces and the decoder's block finder sees one dynamic
// block header per piece.  What pigz does on CPUs, without its 32 KiB priming.
//
// Piece k's block starts at bit B_k (B_0 = 8 x header bytes).  A Huffman piece of b bits moves it by b;
// a stored piece of L bytes (3 header bits, zero padding to a byte, LEN, NLEN, the bytes) maps it to
// align8(B_k + 3) + 32 + 8 L.  Both are maps  x -> x + c  and  x -> align8(x + a) + d,  which are closed
// under composition, so one exclusive scan of the pieces' maps places every piece.
//
// Per round of at most R pieces (BGZF's scratch and rounds), five launches and no host round trip:
//   bgzf_split_kernel               (container_write.cuh) a thread per piece: the compressor's arrays
//   deflate_compress_pieces_kernel  (deflate_compress.cuh) each piece's block into its scratch slot,
//                                   its exact size in bits, or "stored"
//   par_scan_kernel                 one block: the maps' exclusive scan from the carried base, in place:
//                                   pos[k] = B_k, pos[n] = the bit behind the round
//   par_stitch_kernel               a warp per piece: Adler-32 / CRC-32 of its source bytes, its bits
//                                   written at B_k (a Huffman piece shifted out of its slot, a stored
//                                   piece written from the source)
//   par_advance_kernel              one block: the round's checksums combined in order into the running
//                                   one, base and carry moved on; after the last round the final byte,
//                                   the trailer, the header and the call's result
// Byte ownership: byte j belongs to the piece that holds its first bit 8 j, so every byte of dst is
// written by exactly one warp.  That warp ORs in the next piece's first (at most 7) bits, read from the
// next piece's slot or known for a stored piece.  The byte that ends a round is carried to the next
// round's first piece in state[], and after the last round written by par_advance_kernel.
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#define SFB_PAR_SMEM __shared__
#else
#define SFB_PAR_SMEM static  // (tests/cpu_emu: one block at a time, its threads share it)
#endif
#include "container_write.cuh"
#include "deflate_compress.cuh"

namespace sfb {

constexpr int PAR_THREADS = 1024;  // the single-block kernels
// state[] of a call (u64 each)
constexpr int PAR_BASE = 0;       // bit where the round's first piece starts
constexpr int PAR_CARRY = 1;      // the bits of that byte below it
constexpr int PAR_STATUS = 2;     // the call's result: status ..
constexpr int PAR_WRITTEN = 3;    // .. and bytes written
constexpr int PAR_SUM = 4;        // running Adler-32 / CRC-32 of the source so far
constexpr int PAR_CARRY_OUT = 5;  // the round's last byte, left by its last piece
constexpr int PAR_LEN = 6;        // source bytes so far
constexpr int PAR_STATE_WORDS = 8;

struct ParArgs {
  const uint8_t* src;
  const uint64_t* src_off;  // per piece of the round (bgzf_split_kernel)
  const uint64_t* src_len;
  const uint8_t* slots;     // piece k's block at slots + k * BGZF_SLOT + BGZF_HEADER
  const uint8_t* kind;      // the compressor's status: ST_SUCCESS or CMP_PIECE_STORED
  uint64_t* pos;            // in: the compressor's bit counts; after the scan: B_k (n + 1 entries)
  uint32_t* sum;            // per piece: Adler-32 / CRC-32 of its source bytes
  uint8_t* dst;
  uint64_t dst_cap;
  uint64_t* state;          // PAR_*
  uint64_t n;               // pieces in the round
  uint64_t last;            // the round-local index of the buffer's last piece (none: ~0)
  uint32_t container;       // CT_RAW, CT_ZLIB or CT_GZIP
};

// ---- the placement maps: x -> x + d (align == 0) or x -> align8(x + a) + d (a < 8) ----------------
struct ParMap {
  uint64_t d;
  uint32_t a;  // bits 0-2: a, bit 3: align
};

__device__ __forceinline__ uint64_t par_apply(ParMap m, uint64_t x)
{
  return (m.a & 8u) ? ((x + (m.a & 7u) + 7u) & ~7ull) + m.d : x + m.d;
}

// g after f:  align8(align8(x + a) + d + a') + d' = align8(x + a) + align8(d + a') + d';
// x + c then align8(. + a') + d' = align8(x + r) + 8 q + d' with c + a' = 8 q + r
__device__ __forceinline__ ParMap par_then(ParMap f, ParMap g)
{
  if (!(g.a & 8u)) return ParMap{f.d + g.d, f.a};
  if (!(f.a & 8u)) {
    const uint64_t t = f.d + (g.a & 7u);
    return ParMap{(t & ~7ull) + g.d, 8u | static_cast<uint32_t>(t & 7u)};
  }
  return ParMap{((f.d + (g.a & 7u) + 7u) & ~7ull) + g.d, f.a};
}

__device__ __forceinline__ ParMap par_piece_map(const ParArgs& a, uint64_t k)
{
  if (a.kind[k] == CMP_PIECE_STORED) return ParMap{32u + 8u * a.src_len[k], 8u | 3u};
  return ParMap{a.pos[k], 0u};
}

__device__ __forceinline__ ParMap par_shfl_up(ParMap m, uint32_t o)
{
  constexpr unsigned FULL = 0xffffffffu;
  return ParMap{__shfl_up_sync(FULL, m.d, o), __shfl_up_sync(FULL, m.a, o)};
}

// one block: pos[k] = B_k for k <= n, from state[PAR_BASE]
__global__ void __launch_bounds__(PAR_THREADS) par_scan_kernel(const ParArgs a)
{
  SFB_PAR_SMEM ParMap s_warp[32];
  const uint64_t n = a.n;
  const uint64_t per = (n + blockDim.x - 1) / blockDim.x;
  const uint64_t lo = per * threadIdx.x < n ? per * threadIdx.x : n, hi = lo + per < n ? lo + per : n;
  ParMap mine{0, 0};  // the identity
  for (uint64_t k = lo; k < hi; ++k) mine = par_then(mine, par_piece_map(a, k));
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31u) >> 5;
  ParMap incl = mine;
  for (uint32_t o = 1; o < 32; o <<= 1) {
    const ParMap y = par_shfl_up(incl, o);
    if (lane >= o) incl = par_then(y, incl);
  }
  ParMap excl = par_shfl_up(incl, 1);
  if (lane == 0) excl = ParMap{0, 0};
  if (lane == 31u) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    ParMap w = lane < nwarps ? s_warp[lane] : ParMap{0, 0};
    for (uint32_t o = 1; o < 32; o <<= 1) {
      const ParMap y = par_shfl_up(w, o);
      if (lane >= o) w = par_then(y, w);
    }
    if (lane < nwarps) s_warp[lane] = w;
  }
  __syncthreads();
  const uint64_t base = a.state[PAR_BASE];
  uint64_t x = par_apply(warp ? par_then(s_warp[warp - 1], excl) : excl, base);
  for (uint64_t k = lo; k < hi; ++k) {
    const ParMap m = par_piece_map(a, k);  // (reads pos[k] before it is overwritten)
    a.pos[k] = x;
    x = par_apply(m, x);
  }
  if (threadIdx.x == 0) a.pos[n] = par_apply(s_warp[nwarps - 1], base);
}

// ---- the stitch ------------------------------------------------------------------------------------
// 32 bits of a slot's block from bit s on (aligned loads: a slot is 4-byte aligned, and the word
// behind the block is still inside it)
__device__ __forceinline__ uint32_t par_slot_bits(const uint8_t* blk, uint64_t s)
{
  const uintptr_t mis = reinterpret_cast<uintptr_t>(blk) & 3u;
  const uint32_t* const w = reinterpret_cast<const uint32_t*>(blk - mis);
  const uint64_t t = s + 8u * mis;
  return __funnelshift_r(w[t >> 5], w[(t >> 5) + 1], static_cast<uint32_t>(t & 31u));
}

__global__ void __launch_bounds__(CHECK_THREADS) par_stitch_kernel(const ParArgs a)
{
#ifdef SFB_CPU_EMU
  uint32_t* const crc_tab = SFB_EMU_CRC_SMEM;  // tests/cpu_emu: the block's shared memory
#else
  extern __shared__ uint32_t crc_tab[];
#endif
  if (a.container == CT_GZIP) crc_tables_init(crc_tab);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
  for (uint64_t i = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; i < a.n; i += warps) {
    const uint8_t* const s = a.src + a.src_off[i];
    const uint64_t slen = a.src_len[i];
    if (a.container == CT_ZLIB) {
      const uint32_t c = warp_adler32(s, slen, lane);
      if (lane == 0) a.sum[i] = c;
    } else if (a.container == CT_GZIP) {
      const uint32_t c = warp_crc32(s, slen, lane, crc_tab);
      if (lane == 0) a.sum[i] = c;
    }
    const uint64_t b0 = a.pos[i], b1 = a.pos[i + 1];
    if (((b1 + 7) >> 3) > a.dst_cap) continue;  // past the end of dst: the call fails, write nothing
    const bool first = i == 0, round_last = i + 1 == a.n;
    const uint32_t carry = first ? static_cast<uint32_t>(a.state[PAR_CARRY]) : 0u;
    // bytes [j0, j1): the first one only when it starts here or carries the previous round's bits;
    // the last, partial one of a round goes to state[PAR_CARRY_OUT] instead
    const uint64_t j0 = (first || (b0 & 7u) == 0) ? b0 >> 3 : (b0 + 7) >> 3;
    const uint64_t j1 = round_last ? b1 >> 3 : (b1 + 7) >> 3;
    uint8_t* const d = a.dst;
    if (a.kind[i] == CMP_PIECE_STORED) {
      // BFINAL, BTYPE 00, zero padding to the byte at q, LEN, NLEN, the bytes (ends on a byte boundary)
      const uint64_t q = (b0 + 3 + 7) >> 3;
      const uint32_t fin = i == a.last ? 1u : 0u;
      for (uint64_t j = j0 + lane; j < q; j += 32) {
        uint32_t v = 0;
        if (8 * j < b0) v = carry & ((1u << (b0 - 8 * j)) - 1u);
        if (b0 >= 8 * j) v |= fin << (b0 - 8 * j);
        d[j] = static_cast<uint8_t>(v);
      }
      if (lane < 4) {
        const uint32_t len = static_cast<uint32_t>(slen), v = lane < 2 ? len : ~len;
        d[q + lane] = static_cast<uint8_t>(v >> (8 * (lane & 1u)));
      }
      warp_move(d + q + 4, s, slen, lane);
      continue;
    }
    const uint8_t* const blk = a.slots + i * BGZF_SLOT + BGZF_HEADER;
    // the next piece's first bits, where they share this piece's last byte
    uint32_t next = 0;
    if (!round_last && (b1 & 7u))
      next = a.kind[i + 1] == CMP_PIECE_STORED ? (i + 1 == a.last ? 1u : 0u) : blk[BGZF_SLOT];
    // byte j of the stream: the carried bits below b0, this block's bits, `nx` from b1 on
    auto byte_at = [&](uint64_t j, uint32_t nx) -> uint32_t {
      const uint64_t p = 8 * j;
      uint32_t v;
      if (p >= b0) {
        v = par_slot_bits(blk, p - b0) & 0xffu;
      } else {
        const uint32_t k = static_cast<uint32_t>(b0 - p);
        v = ((par_slot_bits(blk, 0) << k) & 0xffu) | (carry & ((1u << k) - 1u));
      }
      if (p + 8 > b1) {
        const uint32_t k = static_cast<uint32_t>(b1 - p);
        const uint32_t hm = (0xffu << k) & 0xffu;
        v = (v & ~hm) | ((nx << k) & hm);
      }
      return v;
    };
    // whole aligned words where every bit is this block's, bytes around them
    const uint64_t f0 = (b0 + 7) >> 3, f1 = b1 >> 3;
    uint64_t w0 = j1, w1 = j1;
    if (f1 >= f0 + 8) {
      w0 = f0 + ((4u - (reinterpret_cast<uintptr_t>(d + f0) & 3u)) & 3u);
      w1 = f1 - (reinterpret_cast<uintptr_t>(d + f1) & 3u);
    }
    for (uint64_t j = j0 + lane; j < w0; j += 32) d[j] = static_cast<uint8_t>(byte_at(j, next));
    for (uint64_t j = w0 + 4 * lane; j < w1; j += 128)
      *reinterpret_cast<uint32_t*>(d + j) = par_slot_bits(blk, 8 * j - b0);
    for (uint64_t j = w1 + lane; j < j1; j += 32) d[j] = static_cast<uint8_t>(byte_at(j, next));
    if (round_last && lane == 0) a.state[PAR_CARRY_OUT] = (b1 & 7u) ? byte_at(b1 >> 3, 0u) : 0u;
  }
}

// ---- the checksums: (sum, len) pairs combined in source order ------------------------------------
struct ParSum {
  uint32_t s;
  uint64_t len;
};

// zlib's adler32_combine
__device__ __forceinline__ uint32_t adler32_combine(uint32_t a1, uint32_t a2, uint64_t len2)
{
  constexpr uint32_t BASE = 65521u;
  const uint32_t rem = static_cast<uint32_t>(len2 % BASE);
  uint32_t s1 = a1 & 0xffffu;
  uint32_t s2 = static_cast<uint32_t>((static_cast<uint64_t>(rem) * s1) % BASE);
  s1 += (a2 & 0xffffu) + BASE - 1u;
  s2 += ((a1 >> 16) & 0xffffu) + ((a2 >> 16) & 0xffffu) + BASE - rem;
  if (s1 >= BASE) s1 -= BASE;
  if (s1 >= BASE) s1 -= BASE;
  if (s2 >= (BASE << 1)) s2 -= (BASE << 1);
  if (s2 >= BASE) s2 -= BASE;
  return s1 | (s2 << 16);
}

__device__ __forceinline__ ParSum par_combine(uint32_t container, ParSum x, ParSum y)
{
  if (container == CT_ZLIB) return ParSum{adler32_combine(x.s, y.s, y.len), x.len + y.len};
  return ParSum{crc_mulmod(crc_x8n(y.len), x.s) ^ y.s, x.len + y.len};  // crc(A || B) = crc(A) x^(8 |B|) + crc(B)
}

// one block after each round: the round's checksums into state[PAR_SUM], base and carry moved on;
// after the last round (last != 0) the final byte (zero padding), trailer and header, and the result
__global__ void __launch_bounds__(PAR_THREADS) par_advance_kernel(const ParArgs a, int last)
{
  constexpr unsigned FULL = 0xffffffffu;
  SFB_PAR_SMEM ParSum s_warp[32];
  const uint32_t kind = a.container;
  if (kind != CT_RAW) {
    const uint64_t n = a.n;
    const uint64_t per = (n + blockDim.x - 1) / blockDim.x;
    const uint64_t lo = per * threadIdx.x < n ? per * threadIdx.x : n, hi = lo + per < n ? lo + per : n;
    const ParSum id{kind == CT_ZLIB ? 1u : 0u, 0};
    ParSum acc = id;
    uint64_t xl = ~0ull;  // x^(8 len) of the last length seen (every piece but the buffer's last has the same)
    uint32_t xv = 0;
    for (uint64_t k = lo; k < hi; ++k) {
      const uint64_t len = a.src_len[k];
      if (kind == CT_ZLIB) {
        acc.s = adler32_combine(acc.s, a.sum[k], len);
      } else {
        if (len != xl) {
          xl = len;
          xv = crc_x8n(len);
        }
        acc.s = crc_mulmod(xv, acc.s) ^ a.sum[k];
      }
      acc.len += len;
    }
    // in order: after the step with offset o, lane l holds lanes [l, l + 2 o)
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31u) >> 5;
    for (uint32_t o = 1; o < 32; o <<= 1) {
      const ParSum y{__shfl_down_sync(FULL, acc.s, o), __shfl_down_sync(FULL, acc.len, o)};
      if (lane + o < 32u) acc = par_combine(kind, acc, y);
    }
    if (lane == 0) s_warp[warp] = acc;
    __syncthreads();
    if (warp == 0) {
      acc = lane < nwarps ? s_warp[lane] : id;
      for (uint32_t o = 1; o < 32; o <<= 1) {
        const ParSum y{__shfl_down_sync(FULL, acc.s, o), __shfl_down_sync(FULL, acc.len, o)};
        if (lane + o < 32u) acc = par_combine(kind, acc, y);
      }
      if (lane == 0) {
        const ParSum run{static_cast<uint32_t>(a.state[PAR_SUM]), 0};
        a.state[PAR_SUM] = par_combine(kind, run, acc).s;
        a.state[PAR_LEN] += acc.len;
      }
    }
  }
  if (threadIdx.x != 0) return;
  const uint64_t end_bit = a.pos[a.n];
  a.state[PAR_BASE] = end_bit;
  a.state[PAR_CARRY] = a.state[PAR_CARRY_OUT];
  if (!last) return;
  const uint64_t hb = kind == CT_RAW ? 0 : container_header_bytes(kind);
  const uint64_t tb = kind == CT_RAW ? 0 : container_trailer_bytes(kind);
  const uint64_t end = (end_bit + 7) >> 3, total = end + tb;
  if (total > a.dst_cap) {
    a.state[PAR_STATUS] = CW_ST_DST_TOO_SMALL;
    a.state[PAR_WRITTEN] = 0;
    return;
  }
  uint8_t* const d = a.dst;
  if (end_bit & 7u) d[end_bit >> 3] = static_cast<uint8_t>(a.state[PAR_CARRY]);  // (zero above the last bit)
  const uint32_t sum = static_cast<uint32_t>(a.state[PAR_SUM]);
  if (kind == CT_ZLIB) {  // as container_seal_kernel writes them
    d[0] = 0x78;
    d[1] = 0x9c;
    d[end] = static_cast<uint8_t>(sum >> 24);
    d[end + 1] = static_cast<uint8_t>(sum >> 16);
    d[end + 2] = static_cast<uint8_t>(sum >> 8);
    d[end + 3] = static_cast<uint8_t>(sum);
  } else if (kind == CT_GZIP) {
    const uint8_t hdr[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 0xff};
    for (uint64_t b = 0; b < hb; ++b) d[b] = hdr[b];
    put_le32(d + end, sum);
    put_le32(d + end + 4, static_cast<uint32_t>(a.state[PAR_LEN]));  // ISIZE: the length mod 2^32
  }
  a.state[PAR_STATUS] = 0;
  a.state[PAR_WRITTEN] = total;
}

}  // namespace sfb
