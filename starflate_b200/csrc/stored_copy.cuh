// Streams made of STORED blocks only, ONE WARP PER STREAM: the stored-block branch of the
// reference's decompress() (src/decompress.cpp:416-436) with read_header (:370-385) in front of
// every block, as a wide copy instead of a lane of pass 1.
//
// Why: in the lane kernel a stored block is copied by the whole warp, one block at a time, after a
// lane-local header parse — 32 pages one after the other, each behind the 31 others' headers.  A
// third of BASELINE config 3 (1 M x 4 KiB pages, stored / fixed / dynamic by turns) is such pages:
// 5.2 of its 22.8 ms of pass 1 went into what is a 1.4 GB memcpy.  The batch is already ordered by
// the type of each stream's first block (lz_warp.cuh: prep kernels); this kernel walks the class
// "first block stored" with a warp per stream and 16 bytes per lane and iteration:
//
//   * a chain of stored blocks is followed to its final block (every header of such a chain starts
//     at a byte boundary); the checks, their order and their statuses are the lane kernel's
//     (deflate_lane.cuh: parse_block_header) — no header byte: InvalidBlockHeader; BTYPE 3:
//     InvalidBlockHeader; fewer than 4 bytes for LEN / NLEN: SrcTooSmall (the reference's unchecked
//     pop_16, class U); LEN != ~NLEN: NoCompressionLenMismatch; payload past the input: SrcTooSmall;
//     payload larger than the room left: DstTooSmall; bytes of earlier blocks stay written;
//   * a stream that turns out to hold a Huffman block after its stored ones is NOT finished here:
//     handled[i] stays 0 and the lane kernel decodes it from the start (it rewrites the same bytes).
// Streams done here have handled[i] = 1 and final status[i] / written[i]; they contain no match, so
// pass 2 finds an empty bitmap for them.
#pragma once

#include "deflate_lane.cuh"
#include "lz_warp.cuh"

namespace sfb {

struct StoredArgs {
  const uint8_t* src_base;
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint8_t* dst_base;
  const uint64_t* dst_off;   // relative to dst_base
  const uint64_t* dst_cap;
  uint8_t* status;
  uint64_t* written;
  uint8_t* handled;                       // out: 1 for every stream finished here (zeroed before launch)
  const uint32_t* order;                  // the batch in type order (prep_scatter_kernel)
  const unsigned long long* type_count;   // [4]: dynamic, fixed, invalid, stored
  unsigned long long* counter;            // work counter, zeroed before launch
};

constexpr int STORED_THREADS = 256;

// n bytes from s to d, any alignment, by one warp.  Reads only [s - 3, s + n): the 16-byte slots are
// dst-aligned and assembled from aligned 32-bit src words; a slot whose last word would reach past
// the payload is left to the byte loop.
__device__ __forceinline__ void stored_warp_copy(const uint8_t* s, uint8_t* d, uint32_t n, uint32_t lane)
{
  const uint32_t head = min(n, static_cast<uint32_t>(-reinterpret_cast<intptr_t>(d)) & 15u);
  if (lane < head) d[lane] = s[lane];
  const uint8_t* sb = s + head;
  uint8_t* db = d + head;
  const uint32_t sh = 8u * (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(sb)) & 3u);
  uint32_t slots = (n - head) >> 4;
  if (sh != 0u && slots != 0u) --slots;   // (its fifth word holds bytes past the payload)
  const uint32_t* sw = reinterpret_cast<const uint32_t*>(sb - (sh >> 3));
  if (sh == 0u && (reinterpret_cast<uintptr_t>(sb) & 15u) == 0u) {
    for (uint32_t i = lane; i < slots; i += 32u)
      reinterpret_cast<uint4*>(db)[i] = reinterpret_cast<const uint4*>(sb)[i];
  } else {
    for (uint32_t i = lane; i < slots; i += 32u) {
      const uint32_t w0 = sw[4u * i], w1 = sw[4u * i + 1u], w2 = sw[4u * i + 2u], w3 = sw[4u * i + 3u];
      const uint32_t w4 = sh ? sw[4u * i + 4u] : 0u;
      uint4 v;
      v.x = lz_funnel(w0, w1, sh);
      v.y = lz_funnel(w1, w2, sh);
      v.z = lz_funnel(w2, w3, sh);
      v.w = lz_funnel(w3, w4, sh);
      reinterpret_cast<uint4*>(db)[i] = v;
    }
  }
  for (uint32_t i = head + 16u * slots + lane; i < n; i += 32u) d[i] = s[i];
}

#if !defined(SFB_CPU_EMU) || defined(SFB_EMU_BLOCK)
__global__ void __launch_bounds__(STORED_THREADS) stored_streams_kernel(const StoredArgs a)
{
  constexpr unsigned FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31u;
  const unsigned long long first = a.type_count[0] + a.type_count[1] + a.type_count[2];
  const unsigned long long count = a.type_count[3];
  for (;;) {
    unsigned long long k = 0;
    if (lane == 0) k = atomicAdd(a.counter, 1ull);
    k = __shfl_sync(FULL, k, 0);
    if (k >= count) break;
    const uint64_t idx = a.order[first + k];
    const uint64_t slen = a.src_len[idx], cap = a.dst_cap[idx];
    if (slen >= 0xffffff00ull || cap >= 0xffffff00ull) continue;  // outside the batch precondition: the lane kernel says so
    const uint8_t* const s = a.src_base + a.src_off[idx];
    uint8_t* const d = a.dst_base + a.dst_off[idx];
    const uint32_t len = static_cast<uint32_t>(slen), room0 = static_cast<uint32_t>(cap);
    uint32_t p = 0, wr = 0;
    int status = -1;   // DecompressStatus once the stream ends here; -2: not ours
    while (status == -1) {
      if (p >= len) {
        status = ST_INVALID_BLOCK_HEADER;   // fewer than 3 bits left (src/decompress.cpp:372-375)
        break;
      }
      // the (up to) five header bytes, one per lane
      const uint32_t hb = (lane < 5u && p + lane < len) ? s[p + lane] : 0u;
      const uint32_t h0 = __shfl_sync(FULL, hb, 0);
      const uint32_t b1 = __shfl_sync(FULL, hb, 1), b2 = __shfl_sync(FULL, hb, 2), b3 = __shfl_sync(FULL, hb, 3),
                     b4 = __shfl_sync(FULL, hb, 4);
      const uint32_t type = (h0 >> 1) & 3u;
      if (type == 3u) {
        status = ST_INVALID_BLOCK_HEADER;
      } else if (type != 0u) {
        status = -2;
      } else if (len - (p + 1u) < 4u) {
        status = ST_SRC_TOO_SMALL;
      } else {
        const uint32_t blen = b1 | (b2 << 8), nlen = b3 | (b4 << 8);
        if (blen != ((~nlen) & 0xffffu)) {
          status = ST_LEN_MISMATCH;
        } else if (len - (p + 5u) < blen) {
          status = ST_SRC_TOO_SMALL;
        } else if (room0 - wr < blen) {
          status = ST_DST_TOO_SMALL;
        } else {
          stored_warp_copy(s + p + 5u, d + wr, blen, lane);
          wr += blen;
          p += 5u + blen;
          if (h0 & 1u) status = ST_SUCCESS;
        }
      }
    }
    if (status >= 0 && lane == 0) {
      a.status[idx] = static_cast<uint8_t>(status);
      a.written[idx] = wr;
      a.handled[idx] = 1;
    }
  }
}
#endif

}  // namespace sfb
