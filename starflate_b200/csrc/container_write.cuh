// WRITING zlib (RFC 1950), gzip (RFC 1952) and BGZF around what deflate_compress_kernel produces,
// with the checksum of the source bytes computed on the device — the other half of container.cuh.
//
// Per stream (sfb200_compress_container_batch_device):
//   container_frame_kernel  a thread per stream: the compressor's dst region = the caller's region
//                           minus header and trailer (capacity 0 where they alone do not fit)
//   (deflate_compress_kernel, unchanged, writes the payload in place)
//   container_seal_kernel   a warp per stream: Adler-32 / CRC-32 of the source, header in front of the
//                           payload, trailer behind it, written = header + payload + trailer
//
// BGZF (sfb200_compress_bgzf_device): the input is cut into pieces of BGZF_PIECE bytes (bgzip's), each
// compressed into a scratch slot of BGZF_SLOT bytes, its payload at +BGZF_HEADER; rounds of at most R
// pieces bound the scratch.  Per round, a constant number of launches and no host round trip:
//   bgzf_split_kernel      a thread per piece: the compressor's four arrays
//   deflate_compress_kernel
//   gzf_exscan_kernel      (gzip_file.cuh) written[] in place: member k starts at
//                          base + scan[k] + BGZF_FRAME * k
//   container_seal_kernel  a warp per member: CRC-32 of the piece, header, payload moved from its slot
//                          to its place in dst, trailer — only members that end inside dst are written
//   bgzf_advance_kernel    one thread: base += the round's bytes; after the last round the EOF marker
//                          and the call's result
// A stored piece is the worst case (BGZF_PIECE + 5 payload bytes), so every piece fits its slot and
// BSIZE fits 16 bits: with dst_cap >= ceil(len / BGZF_PIECE) * (BGZF_PIECE + 31) + 28 the call succeeds.
#pragma once

#include <cstdint>
#ifndef SFB_CPU_EMU
#include <cuda_runtime.h>
#endif
#include "container.cuh"

namespace sfb {

constexpr uint32_t CT_BGZF = 4;                  // container_seal_kernel only: members moved from scratch slots
constexpr uint64_t BGZF_PIECE = 0xff00;           // input bytes per member (bgzip's block size)
constexpr uint64_t BGZF_SLOT = 65536;             // scratch per piece
constexpr uint64_t BGZF_HEADER = 18;              // 1f 8b 08 04 MTIME XFL OS XLEN 'B' 'C' SLEN BSIZE
constexpr uint64_t BGZF_FRAME = BGZF_HEADER + 8;  // header + CRC-32 + ISIZE
constexpr uint64_t BGZF_EOF_BYTES = 28;
constexpr uint8_t CW_ST_DST_TOO_SMALL = 4;        // DecompressStatus DstTooSmall

__device__ __forceinline__ uint64_t container_header_bytes(uint32_t kind) { return kind == CT_ZLIB ? 2u : 10u; }
__device__ __forceinline__ uint64_t container_trailer_bytes(uint32_t kind) { return kind == CT_ZLIB ? 4u : 8u; }

struct SealArgs {
  const uint8_t* src_base;  // the source bytes the checksum is over
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint8_t* dst_base;
  const uint64_t* dst_off;  // per stream: the framed stream's region (BGZF: unused)
  const uint64_t* dst_cap;
  uint8_t* status;          // the compressor's (a frame that does not fit has already failed there)
  uint64_t* written;        // per stream: in the payload's size, out the framed size; BGZF: the scan (n + 1 entries)
  uint64_t n;
  uint32_t container;       // CT_ZLIB, CT_GZIP or CT_BGZF
  // BGZF
  const uint8_t* slots;     // payload of member k at slots + k * BGZF_SLOT + BGZF_HEADER
  uint64_t* state;          // [0] bytes of dst before this round, [1] the call's status (max), [2] written
  uint64_t dst_bytes;       // size of dst
};

// a thread per stream: where the compressor writes the payload, and how much room it has
__global__ void container_frame_kernel(uint32_t kind, const uint64_t* dst_off, const uint64_t* dst_cap, uint64_t* pay_off,
                                       uint64_t* pay_cap, uint64_t n)
{
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t frame = container_header_bytes(kind) + container_trailer_bytes(kind);
  const bool fits = dst_cap[i] >= frame;
  pay_off[i] = dst_off[i] + (fits ? container_header_bytes(kind) : 0);
  pay_cap[i] = fits ? dst_cap[i] - frame : 0;  // (no room: the compressor reports DstTooSmall)
}

// a thread per piece of the round that starts at piece `first`
__global__ void bgzf_split_kernel(uint64_t src_len, uint64_t piece, uint64_t first, uint64_t n, uint64_t* src_off,
                                  uint64_t* piece_len, uint64_t* dst_off, uint64_t* dst_cap)
{
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint64_t at = (first + k) * piece;
  src_off[k] = at;
  piece_len[k] = src_len - at < piece ? src_len - at : piece;
  dst_off[k] = k * BGZF_SLOT + BGZF_HEADER;
  dst_cap[k] = BGZF_SLOT - BGZF_FRAME;
}

__device__ __forceinline__ void put_le32(uint8_t* p, uint32_t v)
{
  p[0] = static_cast<uint8_t>(v);
  p[1] = static_cast<uint8_t>(v >> 8);
  p[2] = static_cast<uint8_t>(v >> 16);
  p[3] = static_cast<uint8_t>(v >> 24);
}

// the warp copies s[0 .. n) to d[0 .. n): aligned 4-byte stores into d, each word put together from two
// aligned loads of s (up to 3 bytes past s + n are read: inside the scratch slot, whose trailer room
// follows the payload)
__device__ __forceinline__ void warp_move(uint8_t* d, const uint8_t* s, uint64_t n, uint32_t lane)
{
  const uint64_t head = (4u - (reinterpret_cast<uintptr_t>(d) & 3u)) & 3u;
  const uint64_t h = head < n ? head : n;
  if (lane < h) d[lane] = s[lane];
  const uint64_t words = (n - h) >> 2;
  const uint8_t* const sw = s + h;
  const uint32_t sh = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(sw) & 3u) * 8u;
  const uint32_t* const sa = reinterpret_cast<const uint32_t*>(sw - (reinterpret_cast<uintptr_t>(sw) & 3u));
  uint32_t* const dw = reinterpret_cast<uint32_t*>(d + h);
  for (uint64_t k = lane; k < words; k += 32) dw[k] = sh ? __funnelshift_r(sa[k], sa[k + 1], sh) : sa[k];
  const uint64_t t = h + 4 * words;
  if (t + lane < n) d[t + lane] = s[t + lane];
}

__global__ void __launch_bounds__(CHECK_THREADS) container_seal_kernel(const SealArgs a)
{
#ifdef SFB_CPU_EMU
  uint32_t* const crc_tab = SFB_EMU_CRC_SMEM;  // tests/cpu_emu: the block's shared memory
#else
  extern __shared__ uint32_t crc_tab[];
#endif
  if (a.container != CT_ZLIB) crc_tables_init(crc_tab);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
  for (uint64_t i = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; i < a.n; i += warps) {
    const uint8_t* const s = a.src_base + a.src_off[i];
    const uint64_t slen = a.src_len[i];
    if (a.container == CT_BGZF) {
      const uint64_t plen = a.written[i + 1] - a.written[i];
      const uint64_t off = a.state[0] + a.written[i] + BGZF_FRAME * i;
      if (a.status[i] != 0) {  // (cannot happen: a stored piece fits its slot)
        if (lane == 0) atomicMax(reinterpret_cast<unsigned long long*>(&a.state[1]), a.status[i]);
        continue;
      }
      if (off + BGZF_FRAME + plen > a.dst_bytes) continue;  // past the end of dst: the call fails, write nothing
      const uint32_t crc = warp_crc32(s, slen, lane, crc_tab);
      uint8_t* const d = a.dst_base + off;
      warp_move(d + BGZF_HEADER, a.slots + i * BGZF_SLOT + BGZF_HEADER, plen, lane);
      if (lane == 0) {
        const uint32_t bsize = static_cast<uint32_t>(plen + BGZF_FRAME - 1);
        const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
        for (int b = 0; b < 16; ++b) d[b] = hdr[b];
        d[16] = static_cast<uint8_t>(bsize);
        d[17] = static_cast<uint8_t>(bsize >> 8);
        put_le32(d + BGZF_HEADER + plen, crc);
        put_le32(d + BGZF_HEADER + plen + 4, static_cast<uint32_t>(slen));
      }
      continue;
    }
    if (a.status[i] != 0) continue;  // the compressor's DstTooSmall / Error stands (written 0)
    const uint32_t kind = a.container;
    const uint64_t hb = container_header_bytes(kind), plen = a.written[i];
    uint8_t* const d = a.dst_base + a.dst_off[i];
    const uint32_t sum = kind == CT_ZLIB ? warp_adler32(s, slen, lane) : warp_crc32(s, slen, lane, crc_tab);
    if (lane == 0) {
      uint8_t* const t = d + hb + plen;
      if (kind == CT_ZLIB) {  // CMF 78 (deflate, 32 KiB window), FLG 9c (default level, FCHECK); Adler-32 big endian
        d[0] = 0x78;
        d[1] = 0x9c;
        t[0] = static_cast<uint8_t>(sum >> 24);
        t[1] = static_cast<uint8_t>(sum >> 16);
        t[2] = static_cast<uint8_t>(sum >> 8);
        t[3] = static_cast<uint8_t>(sum);
      } else {  // ID1 ID2 CM FLG, MTIME 0, XFL 0, OS 255 (unknown); CRC-32 and ISIZE little endian
        const uint8_t hdr[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 0xff};
        for (int b = 0; b < 10; ++b) d[b] = hdr[b];
        put_le32(t, sum);
        put_le32(t + 4, static_cast<uint32_t>(slen));
      }
      a.written[i] = hb + plen + container_trailer_bytes(kind);
    }
  }
}

// one thread, after each round: base += the round's members; after the last round (last != 0) the EOF
// marker behind them and the call's result: state[1] status, state[2] written
__global__ void bgzf_advance_kernel(uint64_t* state, const uint64_t* scan, uint64_t n, uint8_t* dst, uint64_t dst_bytes,
                                    int last)
{
  if (n) state[0] += scan[n] + BGZF_FRAME * n;
  if (!last) return;
  const uint64_t end = state[0] + BGZF_EOF_BYTES;
  if (state[1] == 0 && end > dst_bytes) state[1] = CW_ST_DST_TOO_SMALL;
  if (state[1] != 0) {
    state[2] = 0;
    return;
  }
  // the empty member of the SAM/BAM specification §4.1.2: BSIZE 27, a fixed block with no symbols
  const uint8_t eof[BGZF_EOF_BYTES] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0,
                                       0,    0,    0, 0, 0, 0, 0, 0};
  for (uint64_t b = 0; b < BGZF_EOF_BYTES; ++b) dst[state[0] + b] = eof[b];
  state[2] = end;
}

}  // namespace sfb
