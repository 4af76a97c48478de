// TEST INFRASTRUCTURE ONLY — the block-level kernels run on the host (see cuda_shim_block.h):
// pass 2 of the single-stream route (lz_jump.cuh), the parallel block chain (block_finder.cuh),
// batch preparation (lz_warp.cuh: prep kernels) and the stored-stream copy (stored_copy.cuh).
#define SFB_CPU_EMU 1
#define SFB_EMU_BLOCK 1
#include "cuda_shim_block.h"

#include "../../starflate_b200/csrc/lz_jump.cuh"
#include "../../starflate_b200/csrc/stored_copy.cuh"
#include "../../starflate_b200/csrc/block_finder.cuh"

#include <algorithm>
#include <cstdlib>

// Pointer-jumping pass 2 over streams 0 .. n-1, in the order and with the buffers of the launch
// sequence of capi.cu (the `jump` branch of pass 2), which this mirrors: per stream tile_done and
// the round flags are cleared, `ptr` and `open` keep what the stream before left; the pointers of
// stripe sp + 1 are set up before the rounds of stripe sp; as many rounds as a chain inside the
// stripe can need.  The tile arrays are sized for `dst_bytes` bytes from dst_base (128-byte
// aligned).  stripe_tiles 0: one stripe.  A launch has `warps` warps in blocks of `block_warps`,
// run in block order or (reverse) last block first.  rounds[0] = the most rounds any stripe used.
extern "C" void emu_jump_resolve(uint8_t* dst_base, const uint64_t* dst_off, const uint64_t* written,
                                 const uint32_t* match_bits, uint64_t n, uint64_t dst_bytes, uint64_t stripe_tiles,
                                 uint32_t warps, uint32_t block_warps, int reverse, uint32_t* rounds)
{
  if (stripe_tiles == 0) stripe_tiles = 1ull << 23;
  const uint64_t jump_tiles = (dst_bytes + 128 + sfb::JUMP_TILE - 1) / sfb::JUMP_TILE + 1;
  const uint64_t stripes = (jump_tiles + stripe_tiles - 1) / stripe_tiles;
  // (on the device these are left over from earlier calls: not zeroed here either)
  std::vector<uint32_t> ptr(jump_tiles * sfb::JUMP_TILE, 0u), open(jump_tiles * (sfb::JUMP_TILE / 128), 0x5A5A5A5Au);
  std::vector<uint32_t> tile_done(jump_tiles), todo(stripes * (sfb::JUMP_MAX_ROUNDS + 1));
  const unsigned grid = (warps + block_warps - 1) / block_warps, threads = 32u * block_warps;
  sfb::JumpArgs j{};
  j.dst_base = dst_base;
  j.dst_delta = 0;
  j.dst_off = dst_off;
  j.written = written;
  j.match_bits = match_bits;
  j.ptr = ptr.data();
  j.tile_done = tile_done.data();
  j.open = open.data();
  uint32_t most = 0;
  auto launch = [&](void (*k)(sfb::JumpArgs)) { emu_launch(grid, threads, reverse != 0, [&] { k(j); }); };
  for (uint64_t si = 0; si < n; ++si) {
    j.idx = si;
    std::fill(tile_done.begin(), tile_done.end(), 0u);
    std::fill(todo.begin(), todo.end(), 0u);
    auto set_stripe = [&](uint64_t sp) {
      j.tile_lo = static_cast<uint32_t>(sp * stripe_tiles);
      j.tile_hi = static_cast<uint32_t>(std::min<uint64_t>(jump_tiles, (sp + 1) * stripe_tiles));
      j.todo = todo.data() + sp * (sfb::JUMP_MAX_ROUNDS + 1);
    };
    set_stripe(0);
    j.round = 0;
    launch(sfb::lz_jump_init_kernel);
    for (uint64_t sp = 0; sp < stripes; ++sp) {
      if (sp + 1 < stripes) {
        set_stripe(sp + 1);
        j.round = 0;
        launch(sfb::lz_jump_init_kernel);
      }
      set_stripe(sp);
      int max_rounds = 2;
      for (uint64_t reach = 3; reach < static_cast<uint64_t>(j.tile_hi - j.tile_lo) * sfb::JUMP_TILE; reach *= 3)
        ++max_rounds;
      if (max_rounds > sfb::JUMP_MAX_ROUNDS) max_rounds = sfb::JUMP_MAX_ROUNDS;
      for (int r = 1; r <= max_rounds; ++r) {
        j.round = static_cast<uint32_t>(r);
        launch(sfb::lz_jump_round_kernel);
        if (j.todo[r - 1]) most = std::max<uint32_t>(most, static_cast<uint32_t>(r));
      }
    }
  }
  if (rounds) rounds[0] = most;
}

// The chain of block jobs (block_finder.cuh) over jobs[0 .. count): chain_parallel_kernel on one
// block of CHAIN_THREADS threads (parallel != 0) or the sequential walk chain_kernel.
static void chain_parallel(const sfb::FindArgs& f)
{
  const uint32_t cap = f.job_cap;
  std::vector<uint32_t> ja(cap, 0xDEADBEEFu), jb(cap, 0xDEADBEEFu), mark(cap, 0xDEADBEEFu);
  std::vector<uint64_t> wa(cap, ~0ull), wb(cap, ~0ull);
  const sfb::ChainScratch cs{ja.data(), jb.data(), wa.data(), wb.data(), mark.data()};
  emu_launch(1, sfb::CHAIN_THREADS, false, [&] { sfb::chain_parallel_kernel(f, cs); });
}

// The chain for the stream route of emu_route.cpp (emu_set_chain): chain_parallel_kernel, checked
// against chain_kernel on a copy of the same job table — every job's base and flags, and the tail.
// emu_chain_checks(out): out[0] = chains compared, out[1] = chains that differed.
static uint64_t emu_chain_compared = 0, emu_chain_differed = 0;
extern "C" void emu_chain_parallel_args(const sfb::FindArgs* f)
{
  const uint32_t n = *f->job_count < f->job_cap ? *f->job_count : f->job_cap;
  std::vector<sfb::BlockJob> walk(f->jobs, f->jobs + n);
  uint32_t walk_tail = 0;
  sfb::FindArgs w = *f;
  w.jobs = walk.data();
  w.tail_job = &walk_tail;
  threadIdx.x = 0;
  blockIdx.x = 0;
  sfb::chain_kernel(w);
  chain_parallel(*f);
  bool same = *f->tail_job == walk_tail;
  for (uint32_t j = 0; j < n; ++j) same = same && f->jobs[j].base == walk[j].base && f->jobs[j].flags == walk[j].flags;
  ++emu_chain_compared;
  emu_chain_differed += !same;
}
extern "C" void emu_chain_checks(uint64_t* out)
{
  out[0] = emu_chain_compared;
  out[1] = emu_chain_differed;
}

extern "C" void emu_chain(sfb::BlockJob* jobs, uint32_t job_count, uint32_t job_cap, uint64_t dst_cap,
                          uint32_t* tail, int parallel)
{
  sfb::FindArgs f{};
  f.idx = 0;
  f.jobs = jobs;
  f.job_count = &job_count;
  f.job_cap = job_cap;
  f.tail_job = tail;
  f.dst_cap = &dst_cap;
  if (parallel) {
    chain_parallel(f);
  } else {
    threadIdx.x = 0;
    blockIdx.x = 0;
    sfb::chain_kernel(f);
  }
}

// A sorted batch's preparation and stored-stream copy, as capi.cu launches them: prep_count_kernel
// and prep_scatter_kernel on a grid of PREP_THREADS-thread blocks, then stored_streams_kernel with
// `warps` warps in blocks of up to STORED_THREADS threads.  Stream i is src_len[i] bytes at
// src + src_at[i]; it is copied into an allocation of its own that ends at its last byte (so that
// AddressSanitizer sees a read past it) and starts src_phase[i] bytes before it (the stream's
// address mod 16).  Its output goes to dst_base + dst_off[i].  status / written are only written
// for the streams the copy finished.
extern "C" void emu_prep_stored(const uint8_t* src, const uint64_t* src_at, const uint64_t* src_len,
                                const uint32_t* src_phase, uint8_t* dst_base, const uint64_t* dst_off,
                                const uint64_t* dst_cap, uint64_t n, uint8_t* status, uint64_t* written,
                                uint8_t* handled, uint32_t* order, unsigned long long* type_count, uint32_t warps,
                                int reverse)
{
  std::vector<void*> own(n);
  uintptr_t lo = ~uintptr_t{0};
  for (uint64_t i = 0; i < n; ++i) {
    if (posix_memalign(&own[i], 16, src_phase[i] + src_len[i])) return;
    uint8_t* const p = static_cast<uint8_t*>(own[i]);
    std::memset(p, 0xEE, src_phase[i]);
    if (src_len[i]) std::memcpy(p + src_phase[i], src + src_at[i], src_len[i]);
    lo = std::min(lo, reinterpret_cast<uintptr_t>(p));
  }
  std::vector<uint64_t> src_off(n);
  for (uint64_t i = 0; i < n; ++i) src_off[i] = reinterpret_cast<uintptr_t>(own[i]) + src_phase[i] - lo;
  const uint8_t* const src_base = reinterpret_cast<const uint8_t*>(lo);
  unsigned long long cursor[4] = {0, 0, 0, 0}, counter = 0;
  std::fill(type_count, type_count + 4, 0ull);
  sfb::PrepArgs pa{};
  pa.src_base = src_base;
  pa.src_off = src_off.data();
  pa.src_len = src_len;
  pa.n = n;
  pa.type_count = type_count;
  pa.type_cursor = cursor;
  pa.order = order;
  const unsigned grid = static_cast<unsigned>((n + sfb::PREP_THREADS - 1) / sfb::PREP_THREADS);
  emu_launch(grid, sfb::PREP_THREADS, reverse != 0, [&] { sfb::prep_count_kernel(pa); });
  emu_launch(grid, sfb::PREP_THREADS, reverse != 0, [&] { sfb::prep_scatter_kernel(pa); });
  std::fill(handled, handled + n, uint8_t{0});
  sfb::StoredArgs sa{};
  sa.src_base = src_base;
  sa.src_off = src_off.data();
  sa.src_len = src_len;
  sa.dst_base = dst_base;
  sa.dst_off = dst_off;
  sa.dst_cap = dst_cap;
  sa.status = status;
  sa.written = written;
  sa.handled = handled;
  sa.order = order;
  sa.type_count = type_count;
  sa.counter = &counter;
  const unsigned per_block = std::min<uint32_t>(warps, sfb::STORED_THREADS / 32);
  emu_launch((warps + per_block - 1) / per_block, 32u * per_block, reverse != 0,
             [&] { sfb::stored_streams_kernel(sa); });
  for (void* p : own) free(p);
}
