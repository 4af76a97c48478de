// TEST INFRASTRUCTURE ONLY — writing zlib / gzip / BGZF (container_write.cuh) on the host: the frame
// kernel, the unchanged compression kernel, the scan of gzip_file.cuh, the seal kernel and the BGZF
// round driver of capi.cu, in the same order.  A block is one warp of 32 host threads in lock-step
// (cuda_shim_warp.h); the kernels that need no barrier run their threads one after the other.
#define SFB_CPU_EMU 1
#include "cuda_shim_warp.h"

#include <algorithm>
#include <thread>
#include <vector>

static inline unsigned long long atomicMin(unsigned long long* p, unsigned long long v)
{
  unsigned long long cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v < cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return cur;
}
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v)
{
  unsigned long long cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (v > cur && !__atomic_compare_exchange_n(p, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return cur;
}

static uint8_t* emu_cmp_smem = nullptr;        // the compressing warp's shared memory
static uint32_t* emu_seal_crc_smem = nullptr;  // the sealing block's CRC tables
#define SFB_EMU_SMEM emu_cmp_smem
#define SFB_EMU_CRC_SMEM emu_seal_crc_smem
#include "../../starflate_b200/csrc/deflate_compress.cuh"
#include "../../starflate_b200/csrc/gzip_file.cuh"
#include "../../starflate_b200/csrc/container_write.cuh"

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

struct Smem {
  std::vector<uint8_t> cmp = std::vector<uint8_t>(sfb::CMP_WARP_BYTES + 64, 0xDD);
  std::vector<uint32_t> crc = std::vector<uint32_t>(sfb::CHECK_SMEM_BYTES / 4, 0xDDDDDDDDu);
  Smem()
  {
    emu_cmp_smem = cmp.data();
    emu_seal_crc_smem = crc.data();
  }
};

void compress(const uint8_t* src, const uint64_t* so, const uint64_t* sl, uint8_t* dst, const uint64_t* dof,
              const uint64_t* dc, uint8_t* status, uint64_t* written, uint64_t n)
{
  unsigned long long counter = 0;
  sfb::CompressArgs a;
  a.src_base = src;
  a.src_off = so;
  a.src_len = sl;
  a.dst_base = dst;
  a.dst_off = dof;
  a.dst_cap = dc;
  a.status = status;
  a.written = written;
  a.n = n;
  a.counter = &counter;
  a.fixed_only = 0;
  run_warp([&] { sfb::deflate_compress_kernel(a); });
}
}  // namespace

// sfb200_compress_container_batch_device (ZLIB or GZIP) on host memory; src and dst must have 16
// readable bytes before and after every stream's region
extern "C" void emu_compress_container(int container, const uint8_t* src, const uint64_t* src_off,
                                       const uint64_t* src_len, uint8_t* dst, const uint64_t* dst_off,
                                       const uint64_t* dst_cap, uint8_t* status, uint64_t* written, uint64_t n)
{
  Smem smem;
  std::vector<uint64_t> pay_off(n), pay_cap(n);
  run_threads(n, [&] {
    sfb::container_frame_kernel(static_cast<uint32_t>(container), dst_off, dst_cap, pay_off.data(), pay_cap.data(), n);
  });
  compress(src, src_off, src_len, dst, pay_off.data(), pay_cap.data(), status, written, n);
  sfb::SealArgs s{};
  s.src_base = src;
  s.src_off = src_off;
  s.src_len = src_len;
  s.dst_base = dst;
  s.dst_off = dst_off;
  s.dst_cap = dst_cap;
  s.status = status;
  s.written = written;
  s.n = n;
  s.container = static_cast<uint32_t>(container);
  run_warp([&] { sfb::container_seal_kernel(s); });
}

// sfb200_compress_bgzf_device with pieces of `piece` bytes and rounds of at most `round` pieces
extern "C" int emu_compress_bgzf(const uint8_t* src, uint64_t len, uint64_t piece, uint64_t round, uint8_t* dst,
                                 uint64_t dst_cap, uint64_t* written, uint64_t* members)
{
  Smem smem;
  const uint64_t pieces = (len + piece - 1) / piece;
  const uint64_t r = std::max<uint64_t>(1, std::min(pieces, round));  // (as capi.cu sizes a round)
  std::vector<uint8_t> slots(r * sfb::BGZF_SLOT + 16, 0xCC), pst(r);
  std::vector<uint64_t> so(r), sl(r), dof(r), dc(r), wr(r + 1), state(4, 0);
  sfb::SealArgs s{};
  s.src_base = src;
  s.src_off = so.data();
  s.src_len = sl.data();
  s.dst_base = dst;
  s.status = pst.data();
  s.written = wr.data();
  s.container = sfb::CT_BGZF;
  s.slots = slots.data();
  s.state = state.data();
  s.dst_bytes = dst_cap;
  uint64_t first = 0;
  do {
    const uint64_t n = r < pieces - first ? r : pieces - first;
    const bool last = first + n >= pieces;
    if (n) {
      run_threads(n, [&] { sfb::bgzf_split_kernel(len, piece, first, n, so.data(), sl.data(), dof.data(), dc.data()); });
      compress(src, so.data(), sl.data(), slots.data(), dof.data(), dc.data(), pst.data(), wr.data(), n);
      run_warp([&] { sfb::gzf_exscan_kernel(wr.data(), n); });
      s.n = n;
      run_warp([&] { sfb::container_seal_kernel(s); });
    }
    sfb::bgzf_advance_kernel(state.data(), wr.data(), n, dst, dst_cap, last ? 1 : 0);
    first += n;
  } while (first < pieces);
  *written = state[2];
  *members = state[1] == 0 ? pieces + 1 : 0;
  return static_cast<int>(state[1]);
}
