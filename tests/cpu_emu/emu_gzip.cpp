// TEST INFRASTRUCTURE ONLY — the gzip-file kernels (gzip_file.cuh) on the host: the candidate
// scan (count / scan / scatter), the jump tables, the chain from a start offset and the one-thread
// walk.  A block is one warp of 32 host threads in lock-step (cuda_shim_warp.h); the kernels that
// need no barrier run their threads one after the other.
#define SFB_CPU_EMU 1
#include "cuda_shim_warp.h"

#include <thread>
#include <vector>

static inline unsigned long long atomicMin(unsigned long long* p, unsigned long long v)
{
  unsigned long long cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v < cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return cur;
}

static uint32_t* emu_gzip_crc_smem = nullptr;  // (container.cuh's check kernel is not run here)
#define SFB_EMU_CRC_SMEM emu_gzip_crc_smem
#include "../../starflate_b200/csrc/gzip_file.cuh"

namespace {
constexpr unsigned kThreads = 32;  // one warp per block here

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
}  // namespace

// Candidates of src (kept at the caller's address phase mod 16) and the chain of members from
// `start` (zero padding at `start` skipped when skip != 0), by the jump tables (walk == 0) or the
// one-thread walk.  Returns the number of members; *m = candidates, *stop = the byte behind the
// chain (*head: where it starts), *next = the first non-zero byte behind it.
extern "C" uint64_t emu_gzip_chain(const uint8_t* src, uint64_t len, uint64_t start, int skip, int walk,
                                   uint64_t* cand_pos, uint64_t* cand_next, uint64_t cand_cap, uint64_t* m_out,
                                   uint64_t* mem_pos, uint64_t* mem_len, uint64_t mem_cap, uint64_t* head,
                                   uint64_t* stop, uint64_t* next)
{
  std::vector<uint8_t> sbuf(len + 64, 0xEE);
  uint8_t* sp = sbuf.data() + 16;
  while ((reinterpret_cast<uintptr_t>(sp) & 15u) != (reinterpret_cast<uintptr_t>(src) & 15u)) ++sp;
  if (len) std::memcpy(sp, src, len);
  const uint64_t tile = static_cast<uint64_t>(kThreads) * sfb::GZF_BYTES;
  const uint64_t tiles = (len + (reinterpret_cast<uintptr_t>(sp) & 15u) + tile - 1) / tile;
  std::vector<uint64_t> tc(tiles + 1, 0);
  sfb::GzfArgs a{};
  a.src = sp;
  a.len = len;
  a.tile_count = tc.data();
  a.dst_cap = ~0ull;
  run_blocks_sync(static_cast<unsigned>(tiles), [&] { sfb::gzf_count_kernel(a); });
  run_blocks_sync(1, [&] { sfb::gzf_exscan_kernel(tc.data(), tiles); });
  const uint64_t m = tc[tiles];
  *m_out = m;
  uint32_t tables = 1;
  while ((1ull << tables) < m + 1) ++tables;
  if (walk) tables = 1;
  std::vector<uint64_t> cpos(m + 1), cnext(m + 1);
  std::vector<uint32_t> jump((m + 1) * tables, 0xDEADBEEFu);
  a.cpos = cpos.data();
  a.cnext = cnext.data();
  a.m = m;
  a.jump = jump.data();
  a.n_tables = tables;
  run_blocks_sync(static_cast<unsigned>(tiles), [&] { sfb::gzf_scatter_kernel(a); });
  for (uint64_t c = 0; c < m && c < cand_cap; ++c) {
    cand_pos[c] = cpos[c];
    cand_next[c] = cnext[c];
  }
  const unsigned cgrid = static_cast<unsigned>((m + 1 + 255) / 256);
  run_threads(cgrid, 256, [&] { sfb::gzf_succ_kernel(a); });
  for (uint32_t r = 0; r + 1 < tables; ++r) run_threads(cgrid, 256, [&] { sfb::gzf_jump_kernel(a, r); });
  std::vector<uint64_t> mpos(m + 1), mlen(m + 1), moff(m + 1), mcap(m + 1);
  a.mpos = mpos.data();
  a.mlen = mlen.data();
  a.moff = moff.data();
  a.mcap = mcap.data();
  sfb::GzfStep st{};
  st.start = start;
  st.skip = static_cast<uint64_t>(skip);
  st.head = st.next = len;
  a.step = &st;
  auto* const hd = reinterpret_cast<unsigned long long*>(&st.head);
  auto* const nx = reinterpret_cast<unsigned long long*>(&st.next);
  run_threads(4, 256, [&] { sfb::gzf_skip_kernel(a, &st.start, &st.skip, hd); });
  if (tables == 1) {
    run_threads(1, 1, [&] { sfb::gzf_walk_kernel(a); });
  } else {
    run_threads(1, 1, [&] { sfb::gzf_chain_kernel(a); });
    run_threads(cgrid, 256, [&] { sfb::gzf_expand_kernel(a); });
  }
  run_blocks_sync(1, [&] { sfb::gzf_place_kernel(a); });
  run_threads(4, 256, [&] { sfb::gzf_skip_kernel(a, &st.stop, &st.count, nx); });
  for (uint64_t k = 0; k < st.count && k < mem_cap; ++k) {
    mem_pos[k] = mpos[k];
    mem_len[k] = mlen[k];
  }
  *head = st.head;
  *stop = st.stop;
  *next = st.next;
  return st.count;
}
