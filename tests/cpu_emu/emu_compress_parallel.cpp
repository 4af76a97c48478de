// TEST INFRASTRUCTURE ONLY — one buffer as one raw-DEFLATE / zlib / gzip stream (compress_parallel.cuh)
// on the host: the split kernel, the compressor's piece mode, the scan, stitch and advance kernels and
// the round driver of capi.cu (sfb200_compress_parallel_device), in the same order, with a piece size
// and a round size of the caller's choosing.  A block is one warp of 32 host threads in lock-step
// (cuda_shim_warp.h); the split kernel's threads run one after the other.
#define SFB_CPU_EMU 1
#include "cuda_shim_warp.h"

#include <algorithm>
#include <thread>
#include <vector>

static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v)  // (container_seal_kernel)
{
  unsigned long long cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v > cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return cur;
}

static uint8_t* emu_cmp_smem = nullptr;        // the compressing warp's shared memory
static uint32_t* emu_seal_crc_smem = nullptr;  // the stitching block's CRC tables
#define SFB_EMU_SMEM emu_cmp_smem
#define SFB_EMU_CRC_SMEM emu_seal_crc_smem
#include "../../starflate_b200/csrc/compress_parallel.cuh"

namespace {
template <class F> void run_warp(F&& body)
{
  EmuWarp warp;
  emu_warp = &warp;
  std::vector<std::thread> th;
  for (unsigned t = 0; t < 32; ++t)
    th.emplace_back([&, t] {
      threadIdx.x = t;
      blockIdx.x = 0;
      blockDim.x = 32;
      gridDim.x = 1;
      body();
    });
  for (auto& x : th) x.join();
  emu_warp = nullptr;
}

template <class F> void run_threads(uint64_t n, F&& body)
{
  blockDim.x = 256;
  gridDim.x = static_cast<unsigned>((n + 255) / 256);
  for (uint64_t i = 0; i < n; ++i) {
    blockIdx.x = static_cast<unsigned>(i / 256);
    threadIdx.x = static_cast<unsigned>(i % 256);
    body();
  }
}
}  // namespace

// sfb200_compress_parallel_device with pieces of `piece` bytes and rounds of at most `round` pieces.
// -> the status; *written the stream's size; bits[0 .. pieces] = B_0 .. B_pieces (where each piece's
// block starts, and the bit behind the last)
extern "C" int emu_compress_parallel(int container, const uint8_t* src, uint64_t len, uint64_t piece, uint64_t round,
                                     uint8_t* dst, uint64_t dst_cap, uint64_t* written, uint64_t* bits)
{
  std::vector<uint8_t> cmp_smem(sfb::CMP_WARP_BYTES + 64, 0xDD);
  std::vector<uint32_t> crc_smem(sfb::CHECK_SMEM_BYTES / 4, 0xDDDDDDDDu);
  emu_cmp_smem = cmp_smem.data();
  emu_seal_crc_smem = crc_smem.data();
  const uint64_t pieces = std::max<uint64_t>(1, (len + piece - 1) / piece);
  const uint64_t r = std::min(pieces, std::max<uint64_t>(1, round));  // (as capi.cu sizes a round)
  std::vector<uint8_t> slots(r * sfb::BGZF_SLOT + 16, 0xCC), kinds(r);
  std::vector<uint64_t> so(r), sl(r), dof(r), dc(r), pos(r + 1), state(sfb::PAR_STATE_WORDS, 0);
  std::vector<uint32_t> sums(r);
  const uint64_t hb = container == sfb::CT_ZLIB ? 2 : container == sfb::CT_GZIP ? 10 : 0;
  state[sfb::PAR_BASE] = 8 * hb;
  state[sfb::PAR_SUM] = container == sfb::CT_ZLIB ? 1 : 0;
  sfb::CompressArgs c;
  unsigned long long counter = 0;
  c.src_base = src;
  c.src_off = so.data();
  c.src_len = sl.data();
  c.dst_base = slots.data();
  c.dst_off = dof.data();
  c.dst_cap = dc.data();
  c.status = kinds.data();
  c.written = pos.data();
  c.counter = &counter;
  c.fixed_only = 0;
  sfb::ParArgs a{};
  a.src = src;
  a.src_off = so.data();
  a.src_len = sl.data();
  a.slots = slots.data();
  a.kind = kinds.data();
  a.pos = pos.data();
  a.sum = sums.data();
  a.dst = dst;
  a.dst_cap = dst_cap;
  a.state = state.data();
  a.container = static_cast<uint32_t>(container);
  uint64_t first = 0;
  do {
    const uint64_t n = std::min(r, pieces - first);
    const bool last = first + n >= pieces;
    run_threads(n, [&] { sfb::bgzf_split_kernel(len, piece, first, n, so.data(), sl.data(), dof.data(), dc.data()); });
    counter = 0;
    c.n = n;
    a.n = n;
    a.last = last ? n - 1 : ~0ull;
    run_warp([&] { sfb::deflate_compress_pieces_kernel(c, a.last); });
    run_warp([&] { sfb::par_scan_kernel(a); });
    std::copy(pos.begin(), pos.begin() + static_cast<std::ptrdiff_t>(n + 1), bits + first);
    run_warp([&] { sfb::par_stitch_kernel(a); });
    run_warp([&] { sfb::par_advance_kernel(a, last ? 1 : 0); });
    first += n;
  } while (first < pieces);
  emu_cmp_smem = nullptr;
  emu_seal_crc_smem = nullptr;
  *written = state[sfb::PAR_WRITTEN];
  return static_cast<int>(state[sfb::PAR_STATUS]);
}
