// zlib (RFC 1950) and gzip (RFC 1952) containers around the raw-DEFLATE path, with the Adler-32 /
// CRC-32 of the output verified on the device — SURVEY.md §8(f1), the wire formats real callers
// hold.  The reference is raw-DEFLATE only (its tools/deflate_compress.py:10-12 strips the
// wrapper with wbits = -MAX_WBITS), so there is no reference behaviour to match here: parity is
// against the RFCs and against zlib itself (tests use Python's zlib / gzip as the checker).
//
//   container_parse_kernel   a thread per stream: header -> where the DEFLATE payload lies, and the
//                            trailer's checksum (and ISIZE); a malformed header empties the stream
//   (the raw-DEFLATE batch path decodes the payloads)
//   container_check_kernel   a warp per stream: checksum of the produced bytes against the trailer
//
// One member per stream, and the trailer is taken from the END of the stream's bytes: trailing
// bytes after the member (or a second gzip member) are not supported and show up as a checksum
// mismatch — a file of several gzip members (BGZF, `cat a.gz b.gz`) goes through
// sfb200_decompress_gzip_file* (gzip_file.cuh), which finds the members and hands them to this path
// one stream each.  A preset dictionary (zlib FDICT) is not supported.
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#endif

namespace sfb {

// values of `kind` (per stream) and of the `container` argument of the C ABI
constexpr uint32_t CT_RAW = 0, CT_ZLIB = 1, CT_GZIP = 2, CT_AUTO = 3, CT_BAD = 0xffu;
// statuses beyond the reference's DecompressStatus (src/decompress.hpp:13-23 ends at 7)
constexpr uint8_t ST_BAD_CONTAINER = 8, ST_CHECKSUM_MISMATCH = 9, ST_SIZE_MISMATCH = 10;

struct ContainerArgs {
  const uint8_t* src_base;
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint32_t container;  // CT_*
  uint64_t n;
  // parse -> decode
  uint64_t* pay_off;
  uint64_t* pay_len;
  uint32_t* kind;
  uint32_t* expect;  // Adler-32 / CRC-32 from the trailer
  uint32_t* isize;   // gzip: size modulo 2^32
  // decode -> check
  const uint8_t* dst_base;
  const uint64_t* dst_off;
  uint8_t* status;
  uint64_t* written;
};

constexpr uint32_t CRC_POLY = 0xedb88320u;  // reflected CRC-32 (RFC 1952 §8)

__device__ __forceinline__ uint32_t crc_byte_table_entry(uint32_t i)
{
  uint32_t c = i;
  for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ CRC_POLY : c >> 1;
  return c;
}

// a(x) * b(x) mod P(x), reflected bit order (bit 31 = x^0)
__device__ inline uint32_t crc_mulmod(uint32_t a, uint32_t b)
{
  uint32_t p = 0;
  for (uint32_t m = 1u << 31; m; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1u) ? (b >> 1) ^ CRC_POLY : b >> 1;
  }
  return p;
}
// x^(8 n) mod P
__device__ inline uint32_t crc_x8n(uint64_t n)
{
  uint32_t sq = 1u << 23;  // x^8
  uint32_t p = 1u << 31;   // x^0
  for (; n; n >>= 1) {
    if (n & 1u) p = crc_mulmod(sq, p);
    sq = crc_mulmod(sq, sq);
  }
  return p;
}

__global__ void container_parse_kernel(const ContainerArgs a)
{
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const uint8_t* s = a.src_base + a.src_off[i];
  const uint64_t len = a.src_len[i];
  uint32_t kind = a.container;
  if (kind == CT_AUTO) {
    if (len >= 2 && s[0] == 0x1f && s[1] == 0x8b) kind = CT_GZIP;
    else if (len >= 2 && (s[0] & 15u) == 8u && (s[0] >> 4) <= 7u && ((static_cast<uint32_t>(s[0]) << 8) | s[1]) % 31u == 0u)
      kind = CT_ZLIB;
    else kind = CT_RAW;
  }
  uint64_t hdr = 0, trl = 0;
  uint32_t expect = 0, isize = 0;
  bool ok = true;
  if (kind == CT_ZLIB) {
    // CMF FLG [DICTID] ... ADLER32 (big endian)
    ok = len >= 6 && (s[0] & 15u) == 8u && (s[0] >> 4) <= 7u &&
         ((static_cast<uint32_t>(s[0]) << 8) | s[1]) % 31u == 0u && (s[1] & 0x20u) == 0u;
    hdr = 2;
    trl = 4;
    if (ok)
      expect = (static_cast<uint32_t>(s[len - 4]) << 24) | (static_cast<uint32_t>(s[len - 3]) << 16) |
               (static_cast<uint32_t>(s[len - 2]) << 8) | s[len - 1];
  } else if (kind == CT_GZIP) {
    // ID1 ID2 CM FLG MTIME(4) XFL OS [XLEN extra] [name 0] [comment 0] [HCRC(2)] ... CRC32 ISIZE (little endian)
    ok = len >= 18 && s[0] == 0x1f && s[1] == 0x8b && s[2] == 8u && (s[3] & 0xe0u) == 0u;
    uint64_t p = 10;
    if (ok) {
      const uint32_t flg = s[3];
      const uint64_t lim = len - 8;  // the header must end before the trailer
      if (flg & 4u) {                // FEXTRA
        if (p + 2 <= lim) p += 2u + (static_cast<uint32_t>(s[p]) | (static_cast<uint32_t>(s[p + 1]) << 8));
        else ok = false;
      }
      for (uint32_t bit = 8u; ok && bit <= 16u; bit <<= 1)  // FNAME, FCOMMENT: zero-terminated
        if (flg & bit) {
          while (p < lim && s[p] != 0) ++p;
          if (p < lim) ++p;
          else ok = false;
        }
      if (ok && (flg & 2u)) {  // FHCRC: the low 16 bits of the CRC-32 of the header so far
        if (p + 2 <= lim) {
          uint32_t c = 0xffffffffu;
          for (uint64_t k = 0; k < p; ++k) c = crc_byte_table_entry((c ^ s[k]) & 0xffu) ^ (c >> 8);
          c = ~c;
          ok = (c & 0xffffu) == (static_cast<uint32_t>(s[p]) | (static_cast<uint32_t>(s[p + 1]) << 8));
          p += 2;
        } else {
          ok = false;
        }
      }
      ok = ok && p <= lim;
    }
    hdr = p;
    trl = 8;
    if (ok) {
      const uint8_t* t = s + len - 8;
      expect = static_cast<uint32_t>(t[0]) | (static_cast<uint32_t>(t[1]) << 8) | (static_cast<uint32_t>(t[2]) << 16) |
               (static_cast<uint32_t>(t[3]) << 24);
      isize = static_cast<uint32_t>(t[4]) | (static_cast<uint32_t>(t[5]) << 8) | (static_cast<uint32_t>(t[6]) << 16) |
              (static_cast<uint32_t>(t[7]) << 24);
    }
  }
  a.kind[i] = ok ? kind : CT_BAD;
  a.pay_off[i] = a.src_off[i] + (ok ? hdr : 0);
  a.pay_len[i] = ok ? len - hdr - trl : 0;
  a.expect[i] = expect;
  a.isize[i] = isize;
}

constexpr int CHECK_THREADS = 1024;
constexpr int CHECK_SMEM_BYTES = 4 * 256 * 32 * 4;  // the per-lane CRC tables

// CRC-32, four bytes per step: T(k, b) = CRC of byte b followed by k zero bytes.  The four tables
// are kept once PER LANE (entry (k, b) of lane l at word (k * 256 + b) * 32 + l: bank = lane), so
// the 32 lanes' look-ups at 32 unrelated indices never meet in a bank: 128 KiB, one block per SM.
// Every thread of the block calls it; a __syncthreads() must follow before the tables are read.
__device__ __forceinline__ void crc_tables_init(uint32_t* crc_tab)
{
  for (uint32_t e = threadIdx.x; e < 1024u; e += blockDim.x) {
    uint32_t c = crc_byte_table_entry(e & 255u);
    for (uint32_t k = 0; k < (e >> 8); ++k) c = crc_byte_table_entry(c & 0xffu) ^ (c >> 8);
    for (uint32_t l = 0; l < 32u; ++l) crc_tab[e * 32u + l] = c;
  }
}

// Adler-32 (RFC 1950 §8.2) of d[0 .. n) by the whole warp; every lane returns it.
// s1 = 1 + sum b_j, s2 = n + sum (n - j) b_j, both mod 65521 (a lane takes aligned words, 128 bytes
// per warp and step; the weight n - j is kept modulo 65521 by subtracting 128 per step, so the inner
// loop has no division)
__device__ __forceinline__ uint32_t warp_adler32(const uint8_t* d, uint64_t n, uint32_t lane)
{
  constexpr unsigned FULL = 0xffffffffu;
  uint64_t s1 = 0, s2 = 0;
  const uint32_t mis = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(d)) & 3u;
  const uint64_t head = mis ? (4u - mis < n ? 4u - mis : n) : 0u;  // bytes before the first aligned word
  const uint64_t words = (n - head) >> 2;
  const uint64_t tail0 = head + 4u * words;
  if (lane == 0) {  // the few bytes around the aligned part
    for (uint64_t j = 0; j < head; ++j) {
      s1 += d[j];
      s2 += ((n - j) % 65521u) * d[j];
    }
    for (uint64_t j = tail0; j < n; ++j) {
      s1 += d[j];
      s2 += ((n - j) % 65521u) * d[j];
    }
  }
  const uint32_t* const dw = reinterpret_cast<const uint32_t*>(d + head);
  // weight of the first byte of my first word, then 128 less every step (mod 65521)
  uint32_t wm = static_cast<uint32_t>((n - head - 4u * lane) % 65521u);
  for (uint64_t k = lane; k < words; k += 32) {
    const uint32_t w = dw[k];
    const uint32_t b0 = w & 0xffu, b1 = (w >> 8) & 0xffu, b2 = (w >> 16) & 0xffu, b3 = w >> 24;
    const uint32_t bs = b0 + b1 + b2 + b3;
    s1 += bs;
    // sum (wm - i) b_i  =  wm * bs - (b1 + 2 b2 + 3 b3); wm may be < 3: add 65521 first (same residue)
    s2 += static_cast<uint64_t>(wm + 65521u) * bs - (b1 + 2u * b2 + 3u * b3);
    wm = wm >= 128u ? wm - 128u : wm + 65521u - 128u;
  }
  for (int o = 16; o; o >>= 1) {
    s1 += __shfl_down_sync(FULL, s1, o);
    s2 += __shfl_down_sync(FULL, s2, o);
  }
  s1 = (1u + s1) % 65521u;
  s2 = (n % 65521u + s2) % 65521u;
  return __shfl_sync(FULL, static_cast<uint32_t>((s2 << 16) | s1), 0);
}

// CRC-32 of d[0 .. n) by the whole warp over the lane-private tables of crc_tables_init; every lane
// returns it.  64 contiguous pieces, two per lane (two independent chains hide the look-up latency),
// then  crc(A || B) = crc(A) * x^(8 |B|) + crc(B)  front to back.
__device__ __forceinline__ uint32_t warp_crc32(const uint8_t* d, uint64_t n, uint32_t lane, const uint32_t* crc_tab)
{
  constexpr unsigned FULL = 0xffffffffu;
  const uint32_t* const tl = crc_tab + lane;
  auto step1 = [&](uint32_t c, uint32_t byte) { return tl[((c ^ byte) & 0xffu) * 32u] ^ (c >> 8); };
  auto step4 = [&](uint32_t c, uint32_t word) {
    c ^= word;
    return tl[(768u + (c & 0xffu)) * 32u] ^ tl[(512u + ((c >> 8) & 0xffu)) * 32u] ^
           tl[(256u + ((c >> 16) & 0xffu)) * 32u] ^ tl[(c >> 24) * 32u];
  };
  const uint64_t piece = ((n + 63) / 64 + 15) & ~15ull;
  auto lo_of = [&](uint32_t pc) { return piece * pc < n ? piece * pc : n; };
  auto hi_of = [&](uint32_t pc) { return lo_of(pc) + piece < n ? lo_of(pc) + piece : n; };
  uint64_t j0 = lo_of(lane), j1 = lo_of(lane + 32u);
  const uint64_t h0 = hi_of(lane), h1 = hi_of(lane + 32u);
  uint32_t c0 = 0xffffffffu, c1 = 0xffffffffu;
  // bytes up to a 16-byte boundary, 16-byte loads (a lane walks its own piece: a 32-byte
  // sector then serves two loads instead of eight), the bytes left over
  for (; j0 < h0 && ((reinterpret_cast<uintptr_t>(d + j0)) & 15u); ++j0) c0 = step1(c0, d[j0]);
  for (; j1 < h1 && ((reinterpret_cast<uintptr_t>(d + j1)) & 15u); ++j1) c1 = step1(c1, d[j1]);
  while (j0 + 16 <= h0 && j1 + 16 <= h1) {
    const uint4 v0 = *reinterpret_cast<const uint4*>(d + j0);
    const uint4 v1 = *reinterpret_cast<const uint4*>(d + j1);
    c0 = step4(c0, v0.x);
    c1 = step4(c1, v1.x);
    c0 = step4(c0, v0.y);
    c1 = step4(c1, v1.y);
    c0 = step4(c0, v0.z);
    c1 = step4(c1, v1.z);
    c0 = step4(c0, v0.w);
    c1 = step4(c1, v1.w);
    j0 += 16;
    j1 += 16;
  }
  for (; j0 + 4 <= h0; j0 += 4) c0 = step4(c0, *reinterpret_cast<const uint32_t*>(d + j0));
  for (; j1 + 4 <= h1; j1 += 4) c1 = step4(c1, *reinterpret_cast<const uint32_t*>(d + j1));
  for (; j0 < h0; ++j0) c0 = step1(c0, d[j0]);
  for (; j1 < h1; ++j1) c1 = step1(c1, d[j1]);
  c0 = ~c0;  // each piece's own CRC-32 (of an empty piece: 0)
  c1 = ~c1;
  const uint32_t shift_full = crc_x8n(piece);
  uint32_t acc = 0;
  for (uint32_t pc = 0; pc < 64u; ++pc) {
    const uint32_t cl = __shfl_sync(FULL, pc < 32u ? c0 : c1, static_cast<int>(pc & 31u));
    const uint64_t l_len = hi_of(pc) - lo_of(pc);
    if (lane == 0 && l_len) acc = crc_mulmod(l_len == piece ? shift_full : crc_x8n(l_len), acc) ^ cl;
  }
  return __shfl_sync(FULL, acc, 0);
}

__global__ void __launch_bounds__(CHECK_THREADS) container_check_kernel(const ContainerArgs a)
{
#ifdef SFB_CPU_EMU
  uint32_t* const crc_tab = SFB_EMU_CRC_SMEM;  // tests/cpu_emu: the block's shared memory
#else
  extern __shared__ uint32_t crc_tab[];
#endif
  crc_tables_init(crc_tab);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
  for (uint64_t i = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; i < a.n; i += warps) {
    const uint32_t kind = a.kind[i];
    if (kind == CT_BAD) {
      if (lane == 0) {
        a.status[i] = ST_BAD_CONTAINER;
        a.written[i] = 0;
      }
      continue;
    }
    if (kind == CT_RAW || a.status[i] != 0) continue;  // raw: nothing to check; failed: the decoder's status stands
    const uint8_t* d = a.dst_base + a.dst_off[i];
    const uint64_t n = a.written[i];
    const uint32_t got = kind == CT_ZLIB ? warp_adler32(d, n, lane) : warp_crc32(d, n, lane, crc_tab);
    if (lane == 0) {
      if (got != a.expect[i]) a.status[i] = ST_CHECKSUM_MISMATCH;
      else if (kind == CT_GZIP && a.isize[i] != static_cast<uint32_t>(n)) a.status[i] = ST_SIZE_MISMATCH;
    }
  }
}

}  // namespace sfb
