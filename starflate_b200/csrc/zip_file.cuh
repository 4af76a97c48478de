// ZIP archives (PKWARE APPNOTE 6.3, as Python's zipfile reads them): a table of independent DEFLATE
// (method 8) or stored (method 0) entries, whose central directory (CD) gives every entry's sizes and
// CRC-32 up front.  Listing and extraction run on the device:
//
//   zip_eocd_kernel      one block: the last end-of-central-directory record (EOCD) whose 22 bytes lie
//                        in the file, the ZIP64 records in front of it, and the shift of every offset
//                        by prepended bytes (Python's `concat`)
//   zip_count_kernel / gzf_exscan_kernel / zip_scatter_kernel
//                        every offset of the CD that starts a plausible CD record (46 + n + m + k bytes
//                        inside the CD) is a candidate; cpos / cnext relative to the CD's start
//   gzf_succ_kernel, gzf_jump_kernel, gzf_chain_kernel / gzf_expand_kernel (or gzf_walk_kernel)
//                        the chain of records from the CD's start, exactly as for BGZF members: a
//                        name that contains PK\1\2 is a false candidate whose chain merges or ends
//   zip_entry_kernel     a thread per entry: CD record, ZIP64 extra field, local header -> the row
//   gzf_exscan_kernel    over the sizes: the packed dst offsets and the total; zip_offsets_kernel
//                        writes them into the rows
//
//   zip_split_kernel     a thread per row to extract: validation, decoder group (deflated entries below
//                        ZipExArgs::large, or the others), piece counts; gzf_exscan_kernel over them
//   zip_slot_kernel      the deflated rows' decoder arrays, in row order, each group packed
//   (the raw batch path decodes the deflated entries)
//   zip_piece_kernel     a warp per piece of at most ZIP_PIECE bytes of an entry's output: stored bytes
//                        copied, then the piece's CRC-32 (the lane-private tables of container.cuh)
//   zip_result_kernel    a thread per row: piece CRCs combined in order, sizes and CRC compared
#pragma once

#include <cstdint>
#include "gzip_file.cuh"
#include "stored_copy.cuh"

namespace sfb {

constexpr uint64_t ZIP_PIECE = 1ull << 20;  // bytes of output per warp of the piece kernel
constexpr uint64_t ZIP_MAX_DEFLATE = 0xffffff00ull;  // the batch precondition on src_len / dst_cap
constexpr uint64_t ZIP_TAIL = 22 + 65535;          // where the EOCD can start: the record + its longest comment
constexpr uint8_t ZIP_KIND_DEFLATE = 0, ZIP_KIND_STORED = 1, ZIP_KIND_DONE = 2;

// One row of the entry table (include/starflate_b200.h: sfb200_zip_entry)
struct ZipEntry {
  uint64_t name_off, data_off, comp_size, size, dst_off, written;
  uint32_t crc32;
  uint16_t method, flags, name_len;
  uint8_t status;
  uint8_t pad[5];
};
static_assert(sizeof(ZipEntry) == 64, "sfb200_zip_entry is 64 bytes");

// what zip_eocd_kernel found (status != 0: not an archive this library reads)
struct ZipInfo {
  uint64_t status;
  uint64_t n;         // entries
  uint64_t cd_begin;  // the CD: src[cd_begin .. cd_end)
  uint64_t cd_end;
  int64_t concat;     // prepended bytes: added to every local-header offset
  uint64_t pad[3];
};

struct ZipArgs {
  const uint8_t* src;
  uint64_t len;
  ZipInfo* info;
  const GzfStep* step;    // the chain of CD records (gzip_file.cuh)
  const uint64_t* mpos;   // record k at src[cd_begin + mpos[k]]
  ZipEntry* rows;
  uint64_t cap;           // rows written: min(n, cap)
  uint64_t* size;         // n + 1: the sizes, then their exclusive scan
};

__device__ __forceinline__ uint64_t zip_u32(const uint8_t* s)
{
  return static_cast<uint64_t>(gzf_u16(s)) | (static_cast<uint64_t>(gzf_u16(s + 2)) << 16);
}
__device__ __forceinline__ uint64_t zip_u64(const uint8_t* s) { return zip_u32(s) | (zip_u32(s + 4) << 32); }
__device__ __forceinline__ bool zip_sig(const uint8_t* s, uint32_t a, uint32_t b)
{
  return s[0] == 'P' && s[1] == 'K' && s[2] == a && s[3] == b;
}

// one block: the EOCD, the ZIP64 records, the CD's place.  Python's _EndRecData / _EndRecData64 /
// _RealGetContents, with a split archive (disk numbers), a CD outside the file and a negative shift
// rejected.
__global__ void __launch_bounds__(GZF_SCAN_THREADS) zip_eocd_kernel(const uint8_t* s, uint64_t len, ZipInfo* out)
{
  constexpr unsigned FULL = 0xffffffffu;
  SFB_GZF_SMEM uint64_t s_max[32];
  // the last p in [lo, len - 22] with PK\5\6, as p + 1 (0: none)
  uint64_t best = 0;
  if (len >= 22) {
    const uint64_t lo = len - 22 > ZIP_TAIL - 22 ? len - ZIP_TAIL : 0;
    for (uint64_t i = threadIdx.x; i <= len - 22 - lo; i += blockDim.x)  // (backwards: the first hit is the thread's last)
      if (zip_sig(s + len - 22 - i, 5, 6)) {
        best = len - 22 - i + 1;
        break;
      }
  }
  for (int o = 16; o; o >>= 1) {
    const uint64_t y = __shfl_down_sync(FULL, best, o);
    best = y > best ? y : best;
  }
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31u) >> 5;
  if (lane == 0) s_max[warp] = best;
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (uint32_t w = 0; w < nwarps; ++w) best = s_max[w] > best ? s_max[w] : best;
  ZipInfo r{};
  r.status = 1;
  if (best == 0) {
    *out = r;
    return;
  }
  const uint64_t e = best - 1;
  uint64_t disk = gzf_u16(s + e + 4) | gzf_u16(s + e + 6);
  uint64_t n = gzf_u16(s + e + 10), cd_size = zip_u32(s + e + 12), cd_off = zip_u32(s + e + 16);
  int64_t loc = static_cast<int64_t>(e);
  if (e >= 20 && zip_sig(s + e - 20, 6, 7)) {  // ZIP64 locator
    const uint64_t loc_disk = zip_u32(s + e - 16), reloff = zip_u64(s + e - 12), disks = zip_u32(s + e - 4);
    if (loc_disk != 0 || disks > 1 || e < 20 + 56 || reloff > e - 20 - 56) {
      *out = r;
      return;
    }
    const uint64_t at = e - 20 - 56;  // where the record lies without prepended bytes or extensible data
    uint64_t z = reloff, extra = at - reloff;
    if (!zip_sig(s + z, 6, 6) && reloff != at) {
      z = at;
      extra = 0;
    }
    if (!zip_sig(s + z, 6, 6)) {
      *out = r;
      return;
    }
    const uint64_t sz = zip_u64(s + z + 4);
    disk = zip_u32(s + z + 16) | zip_u32(s + z + 20);
    n = zip_u64(s + z + 32);
    cd_size = zip_u64(s + z + 40);
    cd_off = zip_u64(s + z + 48);
    if (cd_off + cd_size != reloff || sz + 12 != 56 + extra) {
      *out = r;
      return;
    }
    loc = static_cast<int64_t>(at - extra);
  }
  const int64_t concat = loc - static_cast<int64_t>(cd_size) - static_cast<int64_t>(cd_off);
  if (disk != 0 || cd_size > static_cast<uint64_t>(loc) || concat < 0) {
    *out = r;
    return;
  }
  r.status = 0;
  r.n = n;
  r.cd_begin = cd_off + static_cast<uint64_t>(concat);
  r.cd_end = r.cd_begin + cd_size;
  r.concat = concat;
  *out = r;
}

// Does a CD record start at byte p of the CD s[0 .. len)?  *next = p + 46 + n + m + k.
__device__ __forceinline__ bool zip_candidate(const uint8_t* s, uint64_t len, uint64_t p, uint64_t* next)
{
  if (len - p < 46 || !zip_sig(s + p, 1, 2)) return false;
  const uint64_t total = 46 + static_cast<uint64_t>(gzf_u16(s + p + 28)) + gzf_u16(s + p + 30) + gzf_u16(s + p + 32);
  if (total > len - p) return false;
  *next = p + total;
  return true;
}

// gzf_thread_scan for CD records (same tiles, same aligned 16-byte loads), 'P' as the trigger byte
__device__ __forceinline__ uint32_t zip_thread_scan(const uint8_t* s, uint64_t len, uint64_t x0, uint64_t* cpos,
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
      const uint32_t t = w[k] ^ 0x50505050u;
      if (((t - 0x01010101u) & ~t & 0x80808080u) == 0) continue;  // no 'P' in this word
      for (uint32_t b = 0; b < 4; ++b) {
        if (((w[k] >> (8 * b)) & 0xffu) != 0x50u) continue;
        const uint64_t x = xb + 4u * k + b;
        if (x < phase || x - phase >= len) continue;
        uint64_t nx = 0;
        if (!zip_candidate(s, len, x - phase, &nx)) continue;
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

// a.src / a.len: the CD
__global__ void __launch_bounds__(GZF_THREADS) zip_count_kernel(const GzfArgs a)
{
  const uint64_t x0 = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * GZF_BYTES;
  const uint32_t c = zip_thread_scan(a.src, a.len, x0, nullptr, nullptr, 0);
  uint64_t total = 0;
  gzf_block_exscan(c, &total);
  if (threadIdx.x == 0) a.tile_count[blockIdx.x] = total;
}

__global__ void __launch_bounds__(GZF_THREADS) zip_scatter_kernel(const GzfArgs a)
{
  const uint64_t x0 = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * GZF_BYTES;
  const uint32_t c = zip_thread_scan(a.src, a.len, x0, nullptr, nullptr, 0);
  uint64_t total = 0;
  const uint64_t at = a.tile_count[blockIdx.x] + gzf_block_exscan(c, &total);
  if (c) zip_thread_scan(a.src, a.len, x0, a.cpos, a.cnext, at);
}

// a thread per entry.  Nothing is written unless the chain holds exactly the EOCD's count and ends at
// the CD's end (the host then rejects the archive).
__global__ void zip_entry_kernel(const ZipArgs z)
{
  const ZipInfo inf = *z.info;
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= inf.n || z.step->count != inf.n || z.step->stop != inf.cd_end - inf.cd_begin) return;
  const uint8_t* const s = z.src;
  const uint64_t p = inf.cd_begin + z.mpos[k];
  const uint8_t* const c = s + p;
  const uint64_t name_len = gzf_u16(c + 28), extra_len = gzf_u16(c + 30);
  uint64_t csize = zip_u32(c + 20), usize = zip_u32(c + 24), lh = zip_u32(c + 42);
  bool ok = true;
  // the extra field: subfields (id, length) that must stay inside it; ZIP64 (id 1) holds the
  // uncompressed size, compressed size and local-header offset, each only where the 32-bit one is ~0
  const uint8_t* x = c + 46 + name_len;
  for (uint64_t rem = extra_len; rem >= 4;) {
    const uint64_t ln = gzf_u16(x + 2);
    if (ln + 4 > rem) {
      ok = false;
      break;
    }
    if (gzf_u16(x) == 1u) {
      const uint8_t* d = x + 4;
      uint64_t left = ln;
      auto take = [&](uint64_t* v) {
        if (left < 8) {
          ok = false;
          return;
        }
        *v = zip_u64(d);
        d += 8;
        left -= 8;
      };
      if (usize == 0xffffffffull) take(&usize);
      if (ok && csize == 0xffffffffull) take(&csize);
      if (ok && lh == 0xffffffffull) take(&lh);
    }
    x += 4 + ln;
    rem -= 4 + ln;
  }
  lh += static_cast<uint64_t>(inf.concat);
  uint64_t data_off = 0;
  if (ok && lh < z.len && z.len - lh >= 30 && zip_sig(s + lh, 3, 4)) {
    data_off = lh + 30 + gzf_u16(s + lh + 26) + gzf_u16(s + lh + 28);
    ok = data_off <= z.len && csize <= z.len - data_off;
  } else {
    ok = false;
  }
  const uint32_t method = gzf_u16(c + 10), flags = gzf_u16(c + 8);
  ok = ok && (method == 0 || method == 8) && (flags & 0x41u) == 0;  // no encryption (bits 0 and 6)
  z.size[k] = usize;
  if (k >= z.cap) return;
  ZipEntry r{};
  r.name_off = p + 46;
  r.data_off = data_off;
  r.comp_size = csize;
  r.size = usize;
  r.crc32 = static_cast<uint32_t>(zip_u32(c + 16));
  r.method = static_cast<uint16_t>(method);
  r.flags = static_cast<uint16_t>(flags);
  r.name_len = static_cast<uint16_t>(name_len);
  r.status = ok ? 0 : ST_BAD_CONTAINER;
  z.rows[k] = r;
}

__global__ void zip_offsets_kernel(const ZipArgs z)
{
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const ZipInfo inf = *z.info;
  const uint64_t n = inf.n < z.cap ? inf.n : z.cap;
  if (k < n && z.step->count == inf.n && z.step->stop == inf.cd_end - inf.cd_begin) z.rows[k].dst_off = z.size[k];
}

// ---- extraction ---------------------------------------------------------------------------------
// The deflated rows form two decoder groups, g = 0 below `large` bytes and g = 1 the others, each in
// row order (slots from exclusive scans, so the decoder sees the directory's order).  A group's
// outputs are packed at `pos` in a window of its own: dst itself when the rows' regions already lie
// there back to back (off - pos the same for all of them), else scratch, from which the piece kernel
// copies each row to its region.  Either way the decoder sees only the group's own bytes, whatever
// else dst holds.
constexpr uint64_t ZIP_BIAS = 1ull << 63;  // off - pos is kept as off + ZIP_BIAS - pos (unsigned)

struct ZipExArgs {
  const uint8_t* src;
  uint64_t len;
  ZipEntry* rows;
  uint64_t n;
  uint8_t* dst;
  uint64_t dst_cap;
  uint64_t large;  // deflated entries of at least this size form group 1
  // the decoder's arrays (n slots: group 0 from slot 0, group 1 behind it)
  uint64_t* d_off;
  uint64_t* d_len;
  uint64_t* d_pos;     // place in the group's window
  uint64_t* d_room;
  uint64_t* d_written;
  uint64_t* d_dst;     // the row's region in dst
  uint8_t* d_status;
  uint32_t* slot;      // per row: its decoder slot
  uint8_t* kind;       // per row: ZIP_KIND_*
  uint64_t* pieces;    // n + 1: pieces per row, then their exclusive scan
  uint64_t* group;     // 4 columns of n + 1: g0 count, g0 room, g1 count, g1 room; then their scans
  unsigned long long* span;  // [0..1] min / max of off + ZIP_BIAS - pos per group, [2] largest g1 room
  const uint8_t* scratch[2];  // per group: its window when the outputs are copied from there (else null)
  uint32_t* pcrc;      // per piece: CRC-32 of its output
};

// where row r writes and how much of it fits
__device__ __forceinline__ void zip_region(const ZipExArgs& a, const ZipEntry& r, uint64_t* off, uint64_t* room)
{
  *off = r.dst_off < a.dst_cap ? r.dst_off : a.dst_cap;
  *room = r.size < a.dst_cap - *off ? r.size : a.dst_cap - *off;
}

// a thread per row: status decided here, or stored, or deflated in group 0 / 1; piece and group counts
__global__ void zip_split_kernel(const ZipExArgs a)
{
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= a.n) return;
  ZipEntry& r = a.rows[k];
  uint64_t off = 0, room = 0;
  zip_region(a, r, &off, &room);
  uint32_t done = 0xffffffffu;  // a status decided here
  if (r.status == ST_BAD_CONTAINER || (r.method != 0 && r.method != 8) || (r.flags & 0x41u) != 0 ||
      r.data_off > a.len || r.comp_size > a.len - r.data_off)
    done = ST_BAD_CONTAINER;
  else if (r.method == 8 && (r.size >= ZIP_MAX_DEFLATE || r.comp_size >= ZIP_MAX_DEFLATE))
    done = ST_ERROR;
  else if (r.method == 0 && r.comp_size != r.size)
    done = ST_SIZE_MISMATCH;
  uint64_t pc = 0, in0 = 0, in1 = 0;  // deflated in group 0 / 1
  if (done != 0xffffffffu) {
    a.kind[k] = ZIP_KIND_DONE;
    r.status = static_cast<uint8_t>(done);
    r.written = 0;
  } else {
    pc = (room + ZIP_PIECE - 1) / ZIP_PIECE;
    a.kind[k] = r.method == 0 ? ZIP_KIND_STORED : ZIP_KIND_DEFLATE;
    if (r.method == 8) (r.size >= a.large ? in1 : in0) = 1;
  }
  const uint64_t m = a.n + 1;
  a.pieces[k] = pc;
  a.group[k] = in0;
  a.group[m + k] = in0 * room;
  a.group[2 * m + k] = in1;
  a.group[3 * m + k] = in1 * room;
}

// a thread per row, after the scans: the deflated rows' decoder slots
__global__ void zip_slot_kernel(const ZipExArgs a)
{
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= a.n || a.kind[k] != ZIP_KIND_DEFLATE) return;
  const ZipEntry& r = a.rows[k];
  uint64_t off = 0, room = 0;
  zip_region(a, r, &off, &room);
  const uint64_t m = a.n + 1;
  const int g = r.size >= a.large ? 1 : 0;
  const uint64_t i = (g ? a.group[m - 1] : 0) + a.group[2 * g * m + k];
  const uint64_t pos = a.group[(2 * g + 1) * m + k];
  a.slot[k] = static_cast<uint32_t>(i);
  a.d_off[i] = r.data_off;
  a.d_len[i] = r.comp_size;
  a.d_pos[i] = pos;
  a.d_room[i] = room;
  a.d_dst[i] = off;
  const unsigned long long b = off + ZIP_BIAS - pos;
  atomicMin(a.span + 2 * g, b);
  atomicMax(a.span + 2 * g + 1, b);
  if (g) atomicMax(a.span + 4, static_cast<unsigned long long>(room));
}

// the row whose pieces hold piece q: the last k with pieces[k] <= q (pieces: the exclusive scan)
__device__ __forceinline__ uint64_t zip_piece_row(const uint64_t* base, uint64_t n, uint64_t q)
{
  uint64_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const uint64_t mid = (lo + hi) >> 1;
    if (base[mid] <= q) lo = mid;
    else hi = mid;
  }
  return lo;
}

// grid: one CHECK_THREADS block per SM (the lane-private CRC tables); a warp per piece
__global__ void __launch_bounds__(CHECK_THREADS) zip_piece_kernel(const ZipExArgs a)
{
#ifdef SFB_CPU_EMU
  uint32_t* const crc_tab = SFB_EMU_CRC_SMEM;
#else
  extern __shared__ uint32_t crc_tab[];
#endif
  crc_tables_init(crc_tab);
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t total = a.pieces[a.n];
  const uint64_t warps = (static_cast<uint64_t>(gridDim.x) * blockDim.x) >> 5;
  for (uint64_t q = (static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; q < total; q += warps) {
    const uint64_t k = zip_piece_row(a.pieces, a.n, q);
    const ZipEntry& r = a.rows[k];
    uint64_t off = 0, room = 0;
    zip_region(a, r, &off, &room);
    const uint64_t lo = (q - a.pieces[k]) * ZIP_PIECE;
    uint64_t end = room;  // the bytes of the entry's output that exist
    const uint8_t* d = a.dst + off;
    if (a.kind[k] == ZIP_KIND_STORED) {
      const uint64_t hi = lo + ZIP_PIECE < room ? lo + ZIP_PIECE : room;
      stored_warp_copy(a.src + r.data_off + lo, a.dst + off + lo, static_cast<uint32_t>(hi - lo), lane);
      d = a.src + r.data_off;  // (the same bytes: no need to wait for the copy)
    } else {
      const uint32_t i = a.slot[k];
      const uint64_t w = a.d_written[i];
      end = a.d_status[i] == 0 ? w : 0;
      const uint8_t* const win = a.scratch[i < a.group[a.n] ? 0 : 1];
      if (win) {  // decoded in scratch: every byte produced goes to the row's region
        const uint64_t hi = lo + ZIP_PIECE < w ? lo + ZIP_PIECE : w;
        if (hi > lo) stored_warp_copy(win + a.d_pos[i] + lo, a.dst + off + lo, static_cast<uint32_t>(hi - lo), lane);
        d = win + a.d_pos[i];
      }
    }
    const uint64_t hi = lo + ZIP_PIECE < end ? lo + ZIP_PIECE : end;
    const uint32_t c = warp_crc32(d + lo, hi > lo ? hi - lo : 0, lane, crc_tab);
    if (lane == 0) a.pcrc[q] = c;
  }
}

// a thread per row: the entry's result
__global__ void zip_result_kernel(const ZipExArgs a)
{
  const uint64_t k = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= a.n || a.kind[k] == ZIP_KIND_DONE) return;
  ZipEntry& r = a.rows[k];
  uint64_t off = 0, room = 0;
  zip_region(a, r, &off, &room);
  uint32_t st = 0;
  uint64_t w = room;
  if (a.kind[k] == ZIP_KIND_DEFLATE) {
    const uint32_t i = a.slot[k];
    st = a.d_status[i];
    w = a.d_written[i];
    if (st == GZF_DST_TOO_SMALL && room < a.dst_cap - off) st = ST_SIZE_MISMATCH;  // the CD's size was the limit
    else if (st == 0 && w != r.size) st = ST_SIZE_MISMATCH;
  } else if (room < r.size) {
    st = GZF_DST_TOO_SMALL;
  }
  if (st == 0) {  // crc(A || B) = crc(A) * x^(8 |B|) + crc(B), piece by piece
    const uint32_t full = crc_x8n(ZIP_PIECE);
    uint32_t crc = 0;
    for (uint64_t q = a.pieces[k], lo = 0; q < a.pieces[k + 1]; ++q, lo += ZIP_PIECE) {
      const uint64_t l = w - lo < ZIP_PIECE ? w - lo : ZIP_PIECE;
      crc = crc_mulmod(l == ZIP_PIECE ? full : crc_x8n(l), crc) ^ a.pcrc[q];
    }
    if (crc != r.crc32) st = ST_CHECKSUM_MISMATCH;
  }
  r.status = static_cast<uint8_t>(st);
  r.written = w;
}

}  // namespace sfb
