// TEST INFRASTRUCTURE ONLY — the zip-archive kernels (zip_file.cuh) on the host, in the order of
// capi.cu's zip_list_impl / zip_extract_impl.  A block is one warp of 32 host threads in lock-step
// (cuda_shim_warp.h); the kernels that need no barrier run their threads one after the other.  The
// extraction's DEFLATE decode is not run here: the caller places each deflated entry's output in dst
// and says what the decoder reported.
#define SFB_CPU_EMU 1
#include "cuda_shim_warp.h"

#include <thread>
#include <vector>

static inline unsigned long long atomicMin(unsigned long long* p, unsigned long long v)  // (gzf_skip_kernel)
{
  unsigned long long cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v < cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return cur;
}

static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v)  // (zip_slot_kernel)
{
  unsigned long long cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v > cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return cur;
}

static uint32_t emu_zip_crc_smem[4 * 256 * 32];  // the piece kernel's CRC tables (one block at a time)
#define SFB_EMU_CRC_SMEM emu_zip_crc_smem
#include "../../starflate_b200/csrc/zip_file.cuh"

namespace {
constexpr unsigned kThreads = 32;

template <class F> void run_blocks_sync(unsigned grid, F&& body)
{
  for (unsigned b = 0; b < grid; ++b) {
    EmuWarp warp;
    emu_warp = &warp;
    std::vector<std::thread> th;
    for (unsigned t = 0; t < kThreads; ++t)
      th.emplace_back([&, b, t] {
        threadIdx.x = t;
        blockIdx.x = b;
        blockDim.x = kThreads;
        gridDim.x = grid;
        body();
      });
    for (auto& x : th) x.join();
    emu_warp = nullptr;
  }
}

template <class F> void run_threads(unsigned grid, unsigned threads, F&& body)
{
  blockDim.x = threads;
  gridDim.x = grid;
  for (unsigned b = 0; b < grid; ++b)
    for (unsigned t = 0; t < threads; ++t) {
      blockIdx.x = b;
      threadIdx.x = t;
      body();
    }
}

// src at the caller's address phase mod 16, with guard bytes around it
struct Staged {
  std::vector<uint8_t> buf;
  uint8_t* p;
  Staged(const uint8_t* src, uint64_t len) : buf(len + 64, 0xEE)
  {
    p = buf.data() + 16;
    while ((reinterpret_cast<uintptr_t>(p) & 15u) != (reinterpret_cast<uintptr_t>(src) & 15u)) ++p;
    if (len) std::memcpy(p, src, len);
  }
};
}  // namespace

// The listing.  info[0..4] = the EOCD kernel's status, n, cd_begin, cd_end, concat.  Returns the
// archive's status (0, or 8: rejected); *count / *total as sfb200_zip_list reports them.
extern "C" int emu_zip_list(const uint8_t* src, uint64_t len, int walk, sfb::ZipEntry* rows, uint64_t cap,
                            int64_t* info_out, uint64_t* count, uint64_t* total)
{
  *count = *total = 0;
  Staged s(src, len);
  sfb::ZipInfo info{};
  run_blocks_sync(1, [&] { sfb::zip_eocd_kernel(s.p, len, &info); });
  const int64_t iv[5] = {static_cast<int64_t>(info.status), static_cast<int64_t>(info.n),
                         static_cast<int64_t>(info.cd_begin), static_cast<int64_t>(info.cd_end), info.concat};
  for (int k = 0; k < 5; ++k) info_out[k] = iv[k];
  if (info.status) return sfb::ST_BAD_CONTAINER;
  const uint64_t n = info.n, cd = info.cd_end - info.cd_begin;
  sfb::GzfArgs a{};
  a.src = s.p + info.cd_begin;
  a.len = cd;
  a.dst_cap = ~0ull;
  const uint64_t tile = static_cast<uint64_t>(kThreads) * sfb::GZF_BYTES;
  const uint64_t tiles = cd ? (cd + (reinterpret_cast<uintptr_t>(a.src) & 15u) + tile - 1) / tile : 0;
  std::vector<uint64_t> tc(tiles + 1, 0);
  a.tile_count = tc.data();
  uint64_t m = 0;
  if (tiles) {
    run_blocks_sync(static_cast<unsigned>(tiles), [&] { sfb::zip_count_kernel(a); });
    run_blocks_sync(1, [&] { sfb::gzf_exscan_kernel(tc.data(), tiles); });
    m = tc[tiles];
  }
  if (n > m) return sfb::ST_BAD_CONTAINER;
  uint32_t tables = 1;
  while ((1ull << tables) < m + 1) ++tables;
  if (walk) tables = 1;
  std::vector<uint64_t> cpos(m + 1), cnext(m + 1), mpos(m + 1), mlen(m + 1), sizes(n + 1);
  std::vector<uint32_t> jump((m + 1) * tables, 0xDEADBEEFu);
  a.cpos = cpos.data();
  a.cnext = cnext.data();
  a.jump = jump.data();
  a.m = m;
  a.n_tables = tables;
  a.mpos = mpos.data();
  a.mlen = mlen.data();
  sfb::GzfStep st{};
  a.step = &st;
  const unsigned cgrid = static_cast<unsigned>((m + 1 + 255) / 256);
  if (tiles) run_blocks_sync(static_cast<unsigned>(tiles), [&] { sfb::zip_scatter_kernel(a); });
  run_threads(cgrid, 256, [&] { sfb::gzf_succ_kernel(a); });
  for (uint32_t r = 0; r + 1 < tables; ++r) run_threads(cgrid, 256, [&] { sfb::gzf_jump_kernel(a, r); });
  if (tables == 1) {
    run_threads(1, 1, [&] { sfb::gzf_walk_kernel(a); });
  } else {
    run_threads(1, 1, [&] { sfb::gzf_chain_kernel(a); });
    run_threads(cgrid, 256, [&] { sfb::gzf_expand_kernel(a); });
  }
  sfb::ZipArgs z{};
  z.src = s.p;
  z.len = len;
  z.info = &info;
  z.step = &st;
  z.mpos = mpos.data();
  z.rows = rows;
  z.cap = cap;
  z.size = sizes.data();
  run_threads(static_cast<unsigned>((n + 255) / 256), 256, [&] { sfb::zip_entry_kernel(z); });
  run_blocks_sync(1, [&] { sfb::gzf_exscan_kernel(sizes.data(), n); });
  const uint64_t shown = n < cap ? n : cap;
  run_threads(static_cast<unsigned>((shown + 255) / 256), 256, [&] { sfb::zip_offsets_kernel(z); });
  if (st.count != n || st.stop != cd) return sfb::ST_BAD_CONTAINER;
  *count = n;
  *total = sizes[n];
  return 0;
}

// The extraction without the decoder, in the order of capi.cu's zip_extract_impl: rows [0, n) as
// given; what the decoder produced for deflated row k is dec[dec_at[k] .. + dec_written[k]) with
// status dec_status[k], placed where the decoder would have written it (its group's window, or with
// `alone` the row's region for group 1).  `grid` blocks of one warp run the piece kernel.
// in_place[2] receives whether each group was decoded in dst.
extern "C" void emu_zip_extract(const uint8_t* src, uint64_t len, sfb::ZipEntry* rows, uint64_t n, uint8_t* dst,
                                uint64_t dst_cap, const uint8_t* dec_status, const uint64_t* dec_written,
                                const uint8_t* dec, const uint64_t* dec_at, uint64_t large, int alone, unsigned grid,
                                int* in_place)
{
  if (n == 0) return;
  Staged s(src, len);
  std::vector<uint64_t> d(6 * n), pieces(n + 1), group(4 * (n + 1));
  std::vector<uint32_t> slot(n);
  std::vector<uint8_t> kind(n), d_status(n);
  unsigned long long span[5] = {~0ull, 0, ~0ull, 0, 0};
  sfb::ZipExArgs x{};
  x.src = s.p;
  x.len = len;
  x.rows = rows;
  x.n = n;
  x.dst = dst;
  x.dst_cap = dst_cap;
  x.large = large;
  x.d_off = d.data();
  x.d_len = x.d_off + n;
  x.d_pos = x.d_len + n;
  x.d_room = x.d_pos + n;
  x.d_written = x.d_room + n;
  x.d_dst = x.d_written + n;
  x.d_status = d_status.data();
  x.slot = slot.data();
  x.kind = kind.data();
  x.pieces = pieces.data();
  x.group = group.data();
  x.span = span;
  const unsigned rgrid = static_cast<unsigned>((n + 255) / 256);
  run_threads(rgrid, 256, [&] { sfb::zip_split_kernel(x); });
  run_blocks_sync(1, [&] { sfb::gzf_exscan_kernel(pieces.data(), n); });
  for (int c = 0; c < 4; ++c) run_blocks_sync(1, [&] { sfb::gzf_exscan_kernel(group.data() + c * (n + 1), n); });
  run_threads(rgrid, 256, [&] { sfb::zip_slot_kernel(x); });
  const uint64_t cnt[2] = {group[n], group[2 * (n + 1) + n]}, bytes[2] = {group[(n + 1) + n], group[3 * (n + 1) + n]};
  std::vector<uint8_t> scratch[2];
  uint8_t* win[2] = {nullptr, nullptr};
  for (int g = 0; g < 2; ++g) {
    in_place[g] = cnt[g] && span[2 * g] == span[2 * g + 1];
    if (!cnt[g] || (g == 1 && alone)) continue;
    if (in_place[g]) {
      win[g] = dst + (span[2 * g] - sfb::ZIP_BIAS);
    } else {
      scratch[g].assign(bytes[g] + 16, 0xCD);
      win[g] = scratch[g].data();
      x.scratch[g] = win[g];
    }
  }
  for (uint64_t k = 0; k < n; ++k)  // the decoder
    if (kind[k] == sfb::ZIP_KIND_DEFLATE) {
      const uint32_t i = slot[k];
      const int g = i < cnt[0] ? 0 : 1;
      uint8_t* const at = (g == 1 && alone) ? dst + x.d_dst[i] : win[g] + x.d_pos[i];
      std::memcpy(at, dec + dec_at[k], dec_written[k]);
      d_status[i] = dec_status[k];
      x.d_written[i] = dec_written[k];
    }
  std::vector<uint32_t> pcrc(pieces[n] + 1);
  x.pcrc = pcrc.data();
  if (pieces[n]) run_blocks_sync(grid, [&] { sfb::zip_piece_kernel(x); });
  run_threads(rgrid, 256, [&] { sfb::zip_result_kernel(x); });
}
