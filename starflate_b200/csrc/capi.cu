// C ABI of the B200-native DEFLATE decompressor (include/starflate_b200.h).
// Host-side plumbing only: context, launch geometry, staging copies.  No CPU decode path
// exists anywhere in this library: without a CUDA device every call fails.
#include "../../include/starflate_b200.h"
#include "huff_lanes.cuh"
#include "huff_stream.cuh"
#include "lz_warp.cuh"
#include "stored_copy.cuh"
#include "lz_window.cuh"
#include "lz_jump.cuh"
#include "container.cuh"
#include "gzip_file.cuh"
#include "deflate_compress.cuh"
#include "container_write.cuh"
#include "compress_parallel.cuh"
#include "zip_file.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <new>
#include <string>
#include <thread>
#include <utility>
#include <vector>

namespace {

#ifndef SFB_ROOT_LIT
#define SFB_ROOT_LIT 8
#define SFB_ROOT_DIST 6
#define SFB_POOL 96
#define SFB_WARPS 4
#endif
#ifndef SFB_LANE_CTAS
#define SFB_LANE_CTAS 2
#endif
#ifndef SFB_LZ_CTAS_PER_SM
#define SFB_LZ_CTAS_PER_SM 6  /* pass-2 CTAs per SM (0 = as many as fit); see lz_warp.cuh */
#endif
// Two LUT geometries for pass 1 (DESIGN.md §3).  LaneCfg holds any block's codes (8/6-bit roots,
// 896 B of shared memory per lane, 8 warps per SM).  SmallCfg (6/5-bit roots, 448 B per lane,
// 16 warps per SM) is tried first: low-entropy alphabets — short codes — fit it, and twice the
// lanes in flight is twice the throughput of this latency-bound pass; a stream whose first
// block does not fit is handed to a LaneCfg launch.
using LaneCfg = sfb::Cfg<SFB_ROOT_LIT, SFB_ROOT_DIST, SFB_POOL, SFB_WARPS, SFB_LANE_CTAS>;
using SmallCfg = sfb::Cfg<6, 5, 96, 8, 2>;
// WideCfg (9/6-bit roots, a 256-entry sub-table pool, 1 728 B per lane, ONE CTA of 4 warps per SM) is
// for batches with no more streams than that has lanes (BASELINE config 4: 16 384 x 1 MiB) — such a
// batch cannot fill the SMs anyway, and its blocks are the ones whose alphabets overflow the tables
// of LaneCfg (C4: one 1-bit code for length 258 and 256 literals of 9-10 bits, 15 % of the tokens,
// which took the canonical long-code path through global scratch one lane at a time).
using WideCfg = sfb::Cfg<9, 6, 256, 4, 1>;
// single-stream mode (huff_stream.cuh): one warp per CTA, the large geometry
// (7/5-bit roots: 18.5 KiB of shared memory per warp, 8 warps per SM instead of 7 — this kernel has one
//  warp per CTA and is latency-bound too; measured 12 % faster on a 256 MiB stream and 24 % on 1 184 x
//  64 KiB streams than with the 8/6-bit roots of the lane kernel, which in turn loses with them)
#ifndef SFB_STREAM_ROOT_LIT
#define SFB_STREAM_ROOT_LIT 7
#define SFB_STREAM_ROOT_DIST 5
#endif
using StreamCfg = sfb::Cfg<SFB_STREAM_ROOT_LIT, SFB_STREAM_ROOT_DIST, SFB_POOL, 1>;
// work counters per call, four per wave k: [4k] small pass 1, [4k+1] large pass 1, [4k+2] pass 2,
// [4k+3] number of streams handed from the small to the large geometry
constexpr uint64_t kMaxWaves = 256;
constexpr uint64_t kCountersPerWave = 4;
// d_order per stream: its place in the processing order (u32); behind all of those, one byte each,
// "stored_streams_kernel finished it"
constexpr uint64_t kOrderBytes = sizeof(uint32_t) + 1;

// Device memory owned by a context or an inflate stream, freed with its owner (which is deleted
// while a DeviceGuard for its device is alive).  reserve() grows it.
struct DevBuf {
  uint8_t* p = nullptr;
  uint64_t cap = 0;  // bytes
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release()
  {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  void swap(DevBuf& o)
  {
    std::swap(p, o.p);
    std::swap(cap, o.cap);
  }
  template <class T>
  T* as() const
  {
    return reinterpret_cast<T*>(p);
  }
};

}  // namespace

struct sfb200_ctx {
  int device = -1;
  int sm_count = 0;
  int ctas_per_sm = 0;
  int regs_per_thread = 0;
  int lz_ctas_per_sm = 0;
  int lz_regs_per_thread = 0;
  int lzw_minb = 5;            // lz_window_kernel instantiation (register budget for 4 / 5 / 6 CTAs per SM;
                               // measured with the long periodic fill in: 5 (48 registers) beats 6 (40, spills
                               // in the chunk loop) on C2 8.5 / 8.9 ms and C4 5.0 / 5.5 ms — SFB200_LZW_CTAS)
  bool lzw_pf = false;         // SFB200_LZW_PF=1: lz_window_kernel with the source prefetch (measured slower; 5 CTAs per SM only)
  DevBuf d_queue;              // hand-over queue of the overlapped mode (QueueArgs): counters, turns, states, items
  int queue_mode = 0;          // SFB200_QUEUE=1: pass 2 runs beside pass 1 (lz_window_queue_kernel)
  int queue_ctas = 4;          // ... with this many of its CTAs per SM on the second stream (SFB200_QUEUE_CTAS)
  int compress_ctas_per_sm = 0;
  bool no_stored = false;      // SFB200_NO_STORED=1: stored streams go through the lane kernel like the others (A/B runs)
  uint32_t no_pair = 0;        // SFB200_NO_PAIR=1: pass 1 takes one token per iteration (A/B runs)
  bool lz_v1 = false;          // SFB200_LZ_V1=1: the first-generation pass 2 (lz_warp.cuh), kept for A/B runs
  int small_ctas_per_sm = 0;   // SmallCfg pass 1 (0: not usable)
  int wide_ctas_per_sm = 0;    // WideCfg pass 1 (0: not usable; SFB200_NO_WIDE=1 turns it off)
  int small_regs_per_thread = 0;
  int stream_ctas_per_sm = 0;  // huff_stream_kernel (0: not usable)
  int stream_regs_per_thread = 0;
  DevBuf d_defer;    // streams handed from the small to the large geometry
  DevBuf d_order;    // processing order (streams sorted by first block type), kOrderBytes per stream
  DevBuf d_counter;  // 2 * kMaxWaves work counters
  DevBuf d_lens;     // per-resident-lane code-length scratch
  DevBuf d_bits;     // match-head bitmap: 1 bit per dst byte (bitmap_bytes)
  DevBuf d_cont;     // container route: payload offsets / sizes, kinds, trailer values, written
  DevBuf d_gzf;      // gzip files (gzip_file.cuh): the walk's step, result, probe metadata, tile counts
  DevBuf d_gzc;      // ... candidates and jump tables
  DevBuf d_gzm;      // ... the member table (kGzfMemberBytes per member, gzm_members)
  DevBuf d_zip;      // zip archives (zip_file.cuh): ZipInfo, the chain's step, tile counts
  DevBuf d_zipl;     // ... listing: CD record positions and lengths, sizes and their scan
  DevBuf d_zipx;     // ... extraction: the decoder's arrays, slots, kinds, piece counts
  DevBuf d_zipc;     // ... the piece CRCs
  DevBuf d_zips;     // ... windows of decoder groups whose regions are not back to back in dst
  DevBuf d_wrap;     // writing containers (container_write.cuh): the payloads' offsets and capacities
  DevBuf d_bgzf;     // writing BGZF: a round's scratch slots, the compressor's arrays, the call's state
  DevBuf d_find;     // single-stream pass 1 (block_finder.cuh): counters, hash table, jobs, candidates
  DevBuf d_jump;     // single-stream pass 2 (lz_jump.cuh): pointers, tile flags, round flags
  DevBuf d_written;  // pass-1 -> pass-2 sizes when the caller passes written == NULL
  uint64_t launches = 0;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // call start | pass 1 start | pass 1 end | pass 2 end
  bool ev_valid = false;
  std::string err;
  // staging for the host-buffer entry points: a ring of kStageSlots sub-batch slots in device memory
  // (bounded whatever the batch: SFB200_HOST_STAGING_MB), plus the single-buffer calls' buffers
  DevBuf d_src, d_dst;  // (single-buffer calls: host_buffer_call)
  DevBuf d_meta;        // ... their metadata block
  DevBuf st_src[3], st_dst[3];             // exactly st_src_cap + 64 and st_dst_cap + 64 bytes each
  uint64_t st_src_cap = 0, st_dst_cap = 0;  // per slot
  int st_slots = 0;                         // slots allocated so far (a small call needs one)
  DevBuf st_meta[3];  // per slot: src_off, src_len, dst_off, dst_cap, written (u64 x st_meta_n), status (u8 x st_meta_n)
  uint64_t* st_hmeta[3] = {nullptr, nullptr, nullptr};  // pinned mirror: the four input arrays (rebased) + written + status
  uint64_t st_meta_n = 0;
  cudaStream_t s_meta = nullptr;                // status / written read-back
  cudaEvent_t st_ev[3][4] = {};                 // per slot: in_done | run_done | meta_done | out_done
  cudaStream_t hs[3] = {nullptr, nullptr, nullptr};  // H2D | kernels | D2H
  cudaStream_t ps[2] = {nullptr, nullptr};           // pass-1 chain | pass-2 chain (wave overlap)
  std::vector<cudaEvent_t> wave_ev;
};

namespace {

int fail(sfb200_ctx* ctx, cudaError_t e, const char* what)
{
  if (ctx) ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
  return e == cudaErrorMemoryAllocation ? SFB200_RC_OUT_OF_MEMORY : SFB200_RC_CUDA_ERROR;
}

// Every entry point works on its context's device and leaves the calling thread's current
// device as it found it (a process with one context per GPU — or PyTorch beside us — must not
// see its current device change under it).
struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int device)
  {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    ok = prev == device || cudaSetDevice(device) == cudaSuccess;
    if (prev == device) prev = -1;  // nothing to restore
  }
  ~DeviceGuard()
  {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define SFB_ENTER(ctx)                                                   \
  DeviceGuard guard_((ctx)->device);                                     \
  if (!guard_.ok) return fail((ctx), cudaGetLastError(), "cudaSetDevice"); \
  (ctx)->err.clear()

#define SFB_TRY(ctx, call)                                   \
  do {                                                       \
    const cudaError_t e_ = (call);                           \
    if (e_ != cudaSuccess) return fail((ctx), e_, #call);    \
  } while (0)

// Room for `need` bytes in b: grown to need + need / 8 + 256 bytes (exactly `need` when `exact`),
// never shrunk.  keep == 0: the old memory is freed first, so that a failed allocation returns
// SFB200_RC_OUT_OF_MEMORY with b empty and valid, and the caller may take a route that needs less.
// keep > 0: the first `keep` bytes move to the new memory.
int reserve(sfb200_ctx* ctx, DevBuf& b, uint64_t need, uint64_t keep = 0, bool exact = false)
{
  if (need <= b.cap) return SFB200_RC_OK;
  if (!keep) b.release();
  DevBuf q;
  const uint64_t want = exact ? need : need + need / 8 + 256;
  SFB_TRY(ctx, cudaMalloc(reinterpret_cast<void**>(&q.p), want));
  q.cap = want;
  if (keep) SFB_TRY(ctx, cudaMemcpy(q.p, b.p, keep, cudaMemcpyDeviceToDevice));
  b.swap(q);  // (q frees the old memory)
  return SFB200_RC_OK;
}

// The kernel's function attributes (they are per device: set once, by sfb200_create): the dynamic
// shared memory it may take (smem > 0) and, with `carveout`, the largest shared-memory carve-out.
// per_sm / regs (if given) receive its resident CTAs per SM at `threads` and `smem`, and its
// registers per thread.
template <class Kernel>
cudaError_t setup_kernel(Kernel kern, int smem, bool carveout, int threads = 0, int* per_sm = nullptr,
                         int* regs = nullptr)
{
  cudaError_t e = cudaSuccess;
  if (smem > 0 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess)
    return e;
  if (carveout && (e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout,
                                            cudaSharedmemCarveoutMaxShared)) != cudaSuccess)
    return e;
  if (per_sm && (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kern, threads, smem)) != cudaSuccess)
    return e;
  cudaFuncAttributes fa;
  if (regs && (e = cudaFuncGetAttributes(&fa, kern)) != cudaSuccess) return e;
  if (regs) *regs = fa.numRegs;
  return cudaSuccess;
}

// CTAs of a launch that pulls its work dynamically: what the work wants, at most what is resident
unsigned grid_size(uint64_t want, uint64_t resident) { return static_cast<unsigned>(std::min(want, resident)); }

// pass 2's match-head bitmap: one bit per byte of dst (counted from its 128-byte aligned base,
// `delta` bytes in front of dst_base) and eight guard words
uint64_t bitmap_bytes(uint64_t dst_bytes, uint64_t delta) { return ((dst_bytes + delta) / 32 + 8) * sizeof(uint32_t); }

// The single-buffer host calls.  src is staged in the context's d_src, `device(d_src, d_dst, meta, &wr)`
// makes the device call into d_dst on the legacy default stream, and of dst only the `wr` bytes it
// produced come back.  meta is the context's block {src_off = 0, src_len, dst_off = 0, dst_cap}, then
// written and status (u8) for the call to fill: a batch of one stream, whose results read_meta() returns.
template <class Device>
int host_buffer_call(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, uint8_t* dst, uint64_t dst_cap,
                     uint64_t* written, Device device)
{
  int rc = reserve(ctx, ctx->d_src, src_len + 64);
  if (rc == SFB200_RC_OK) rc = reserve(ctx, ctx->d_dst, dst_cap + 64);
  if (rc == SFB200_RC_OK) rc = reserve(ctx, ctx->d_meta, 6 * sizeof(uint64_t), 0, true);
  if (rc != SFB200_RC_OK) return rc;
  const uint64_t h[6] = {0, src_len, 0, dst_cap, 0, 0};
  uint64_t* const meta = ctx->d_meta.as<uint64_t>();
  if (src_len) SFB_TRY(ctx, cudaMemcpyAsync(ctx->d_src.p, src, src_len, cudaMemcpyHostToDevice, nullptr));
  SFB_TRY(ctx, cudaMemcpyAsync(meta, h, sizeof h, cudaMemcpyHostToDevice, nullptr));
  uint64_t wr = 0;
  rc = device(ctx->d_src.p, ctx->d_dst.p, meta, &wr);
  if (rc != SFB200_RC_OK) return rc;
  if (wr > dst_cap) return SFB200_RC_CUDA_ERROR;  // (cannot happen)
  if (wr) SFB_TRY(ctx, cudaMemcpy(dst, ctx->d_dst.p, wr, cudaMemcpyDeviceToHost));  // only what was produced
  if (written) *written = wr;
  return SFB200_RC_OK;
}

int read_meta(sfb200_ctx* ctx, const uint64_t* meta, uint64_t* written, uint8_t* status)
{
  SFB_TRY(ctx, cudaMemcpyAsync(written, meta + 4, 8, cudaMemcpyDeviceToHost, nullptr));
  SFB_TRY(ctx, cudaMemcpyAsync(status, meta + 5, 1, cudaMemcpyDeviceToHost, nullptr));
  SFB_TRY(ctx, cudaStreamSynchronize(nullptr));
  return SFB200_RC_OK;
}

}  // namespace

extern "C" {

void sfb200_destroy(sfb200_ctx* ctx);

int sfb200_abi_version(void) { return SFB200_ABI_VERSION; }

int sfb200_create(int device, sfb200_ctx** out)
{
  if (!out) return SFB200_RC_BAD_ARGUMENT;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return SFB200_RC_NO_DEVICE;
  }
  if (device < 0 || device >= count) return SFB200_RC_BAD_ARGUMENT;
  sfb200_ctx* ctx = new (std::nothrow) sfb200_ctx;
  if (!ctx) return SFB200_RC_OUT_OF_MEMORY;
  ctx->device = device;
  auto bail = [&](int rc) {
    delete ctx;
    return rc;
  };
  DeviceGuard guard_(device);
  if (!guard_.ok) return bail(SFB200_RC_NO_DEVICE);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(SFB200_RC_CUDA_ERROR);
  ctx->sm_count = prop.multiProcessorCount;
  if (const char* e = std::getenv("SFB200_LZ_V1")) ctx->lz_v1 = e[0] == '1';
  if (const char* e = std::getenv("SFB200_NO_PAIR")) ctx->no_pair = e[0] == '1';
  if (const char* e = std::getenv("SFB200_NO_STORED")) ctx->no_stored = e[0] == '1';
  if (const char* e = std::getenv("SFB200_QUEUE")) ctx->queue_mode = std::atoi(e);
  if (const char* e = std::getenv("SFB200_LZW_PF")) ctx->lzw_pf = e[0] == '1';
  if (const char* e = std::getenv("SFB200_QUEUE_CTAS")) ctx->queue_ctas = std::max(1, std::atoi(e));
  if (const char* e = std::getenv("SFB200_LZW_CTAS")) {
    const int v = std::atoi(e);
    if (v == 4 || v == 5 || v == 6) ctx->lzw_minb = v;
  }
  static_assert(sfb::LZ_THREADS == sfb::LZW_THREADS, "one launch geometry for both pass-2 kernels");
  static_assert(LaneCfg::WARPS == WideCfg::WARPS, "the wide launch takes the CTA count computed for the large one");
  const void* lzw = ctx->lzw_minb == 4   ? reinterpret_cast<const void*>(sfb::lz_window_kernel<4>)
                    : ctx->lzw_minb == 5 ? reinterpret_cast<const void*>(sfb::lz_window_kernel<5>)
                                         : reinterpret_cast<const void*>(sfb::lz_window_kernel<6>);
  const void* lz = ctx->lz_v1 ? reinterpret_cast<const void*>(sfb::lz_resolve_kernel) : lzw;
  // the kernels the calls launch (pass 1, size discovery, the END decode of gzip members, the container
  // checksums and seal, compression and its piece mode, the parallel stream's stitch, pass 2): a
  // context has them all
  int lz_per_sm = 0;
  if (setup_kernel(sfb::huff_lanes_kernel<LaneCfg>, LaneCfg::SMEM_BYTES, true, LaneCfg::WARPS * 32, &ctx->ctas_per_sm,
                   &ctx->regs_per_thread) != cudaSuccess ||
      ctx->ctas_per_sm < 1 ||
      setup_kernel(sfb::huff_lanes_kernel<LaneCfg, true>, LaneCfg::SMEM_BYTES, true) != cudaSuccess ||
      setup_kernel(sfb::huff_lanes_kernel<LaneCfg, false, false, true>, LaneCfg::SMEM_BYTES, true) != cudaSuccess ||
      setup_kernel(sfb::container_check_kernel, sfb::CHECK_SMEM_BYTES, false) != cudaSuccess ||
      setup_kernel(sfb::container_seal_kernel, sfb::CHECK_SMEM_BYTES, false) != cudaSuccess ||
      setup_kernel(sfb::deflate_compress_kernel, sfb::CMP_SMEM_BYTES, false, sfb::CMP_WARPS * 32,
                   &ctx->compress_ctas_per_sm) != cudaSuccess ||
      setup_kernel(sfb::deflate_compress_pieces_kernel, sfb::CMP_SMEM_BYTES, false) != cudaSuccess ||
      setup_kernel(sfb::par_stitch_kernel, sfb::CHECK_SMEM_BYTES, false) != cudaSuccess ||
      setup_kernel(sfb::zip_piece_kernel, sfb::CHECK_SMEM_BYTES, false) != cudaSuccess ||
      setup_kernel(lz, 0, false, sfb::LZ_THREADS, &lz_per_sm, &ctx->lz_regs_per_thread) != cudaSuccess || lz_per_sm < 1)
    return bail(SFB200_RC_CUDA_ERROR);
  ctx->compress_ctas_per_sm = std::max(1, ctx->compress_ctas_per_sm);
  // The queue-mode pass 2 must be able to share an SM with pass 1: an SM changes its shared-memory
  // carve-out only when it is idle, so a kernel that asks for none of it, once resident, keeps
  // pass 1 (112 KiB per CTA) off that SM for as long as it runs — ask for pass 1's carve-out.
  if (ctx->queue_mode) {
    const void* lzq = ctx->lzw_minb == 4   ? reinterpret_cast<const void*>(sfb::lz_window_queue_kernel<4>)
                      : ctx->lzw_minb == 5 ? reinterpret_cast<const void*>(sfb::lz_window_queue_kernel<5>)
                                           : reinterpret_cast<const void*>(sfb::lz_window_queue_kernel<6>);
    if (setup_kernel(sfb::huff_lanes_kernel<LaneCfg, false, true>, LaneCfg::SMEM_BYTES, true) != cudaSuccess ||
        setup_kernel(lzq, 0, true) != cudaSuccess)
      return bail(SFB200_RC_CUDA_ERROR);
  }
  // fewer resident warps keep the streams' 32 KiB windows inside the L2 (DESIGN.md)
  int cap = SFB_LZ_CTAS_PER_SM;
  if (const char* e = std::getenv("SFB200_LZ_CTAS_PER_SM")) cap = std::atoi(e);
  ctx->lz_ctas_per_sm = (cap > 0 && cap < lz_per_sm) ? cap : lz_per_sm;
  // the other geometries: one that cannot be set up is not used (0 CTAs per SM)
  if (setup_kernel(sfb::huff_lanes_kernel<SmallCfg>, SmallCfg::SMEM_BYTES, true, SmallCfg::WARPS * 32,
                   &ctx->small_ctas_per_sm, &ctx->small_regs_per_thread) != cudaSuccess)
    ctx->small_ctas_per_sm = 0;
  bool no_wide = false;
  if (const char* e = std::getenv("SFB200_NO_WIDE")) no_wide = e[0] == '1';
  if (no_wide || setup_kernel(sfb::huff_lanes_kernel<WideCfg>, WideCfg::SMEM_BYTES, true, WideCfg::WARPS * 32,
                              &ctx->wide_ctas_per_sm) != cudaSuccess)
    ctx->wide_ctas_per_sm = 0;
  if (setup_kernel(sfb::huff_stream_kernel<StreamCfg>, StreamCfg::SMEM_BYTES, true, 32, &ctx->stream_ctas_per_sm,
                   &ctx->stream_regs_per_thread) != cudaSuccess)
    ctx->stream_ctas_per_sm = 0;
  cudaGetLastError();
  const size_t big_warps = std::max(static_cast<size_t>(ctx->ctas_per_sm) * LaneCfg::WARPS,
                                    static_cast<size_t>(ctx->stream_ctas_per_sm));
  const size_t small_warps = static_cast<size_t>(ctx->small_ctas_per_sm) * SmallCfg::WARPS;
  const size_t lens_bytes = static_cast<size_t>(ctx->sm_count) * std::max(big_warps, small_warps) *
                            sfb::SCRATCH_WORDS * 32 * sizeof(uint32_t);
  int rc = reserve(ctx, ctx->d_counter, (kCountersPerWave * kMaxWaves + 16) * sizeof(unsigned long long), 0, true);
  if (rc == SFB200_RC_OK) rc = reserve(ctx, ctx->d_lens, lens_bytes, 0, true);
  if (rc != SFB200_RC_OK) return bail(rc);
  for (auto& e : ctx->ev)
    if (cudaEventCreate(&e) != cudaSuccess) {
      sfb200_destroy(ctx);
      return SFB200_RC_CUDA_ERROR;
    }
  *out = ctx;
  return SFB200_RC_OK;
}

void sfb200_destroy(sfb200_ctx* ctx)
{
  if (!ctx) return;
  DeviceGuard guard_(ctx->device);  // (the context's device memory is freed with it, on its device)
  for (int k = 0; k < 3; ++k) {
    if (ctx->st_hmeta[k]) cudaFreeHost(ctx->st_hmeta[k]);
    for (auto& e : ctx->st_ev[k])
      if (e) cudaEventDestroy(e);
  }
  if (ctx->s_meta) cudaStreamDestroy(ctx->s_meta);
  for (auto& e : ctx->ev)
    if (e) cudaEventDestroy(e);
  for (auto& st : ctx->hs)
    if (st) cudaStreamDestroy(st);
  for (auto& st : ctx->ps)
    if (st) cudaStreamDestroy(st);
  for (auto& e : ctx->wave_ev) cudaEventDestroy(e);
  delete ctx;
}

const char* sfb200_last_error(const sfb200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

// Diagnostic of the experimental queue mode (SFB200_QUEUE=1; not part of the declared ABI): waits for
// the device and copies the queue's eight counters — tail, head, final_tail, done, dbg[0..3].
int sfb200_debug_queue(sfb200_ctx* ctx, unsigned long long* out8)
{
  if (!ctx || !out8 || !ctx->d_queue.p) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  SFB_TRY(ctx, cudaDeviceSynchronize());
  SFB_TRY(ctx, cudaMemcpy(out8, ctx->d_queue.p, 64, cudaMemcpyDeviceToHost));
  return SFB200_RC_OK;
}

int sfb200_get_launch_info(sfb200_ctx* ctx, sfb200_launch_info* out)
{
  if (!ctx || !out) return SFB200_RC_BAD_ARGUMENT;
  out->sm_count = ctx->sm_count;
  out->warps_per_cta = LaneCfg::WARPS;
  out->ctas_per_sm = ctx->ctas_per_sm;
  out->smem_bytes_per_cta = LaneCfg::SMEM_BYTES;
  out->regs_per_thread = ctx->regs_per_thread;
  out->lz_threads_per_cta = sfb::LZ_THREADS;
  out->lz_ctas_per_sm = ctx->lz_ctas_per_sm;
  out->lz_regs_per_thread = ctx->lz_regs_per_thread;
  out->small_warps_per_cta = SmallCfg::WARPS;
  out->small_ctas_per_sm = ctx->small_ctas_per_sm;
  out->small_regs_per_thread = ctx->small_regs_per_thread;
  out->stream_ctas_per_sm = ctx->stream_ctas_per_sm;
  out->stream_regs_per_thread = ctx->stream_regs_per_thread;
  out->kernel_launches = ctx->launches;
  return SFB200_RC_OK;
}

}  // extern "C"

namespace {
// chunked input (sfb200_inflate_stream_feed): where each stream starts, and where its decode got to.
// start_bit == nullptr: not a continued decode — only `end`, which either route can serve.
struct Resume {
  const uint64_t* start_bit = nullptr;
  const uint64_t* start_out = nullptr;
  uint64_t* blk_end = nullptr;
  bool end = false;  // blk_end[2 i] also receives the end of the final block (huff_lanes_kernel: END;
                     // huff_stream_kernel: StreamArgs::end_bit)
};

int batch_device_impl(sfb200_ctx* ctx, const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                      uint8_t* dst_base, uint64_t dst_bytes, const uint64_t* dst_off, const uint64_t* dst_cap,
                      uint8_t* status, uint64_t* written, uint64_t n, void* cuda_stream, const Resume* resume);
}  // namespace

extern "C" {

int sfb200_decompress_batch_device(sfb200_ctx* ctx, const uint8_t* src_base,
                                   const uint64_t* src_off, const uint64_t* src_len,
                                   uint8_t* dst_base, uint64_t dst_bytes, const uint64_t* dst_off,
                                   const uint64_t* dst_cap, uint8_t* status,
                                   uint64_t* written, uint64_t n, void* cuda_stream)
{
  return batch_device_impl(ctx, src_base, src_off, src_len, dst_base, dst_bytes, dst_off, dst_cap, status, written,
                           n, cuda_stream, nullptr);
}

}  // extern "C"

namespace {
int batch_device_impl(sfb200_ctx* ctx, const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                      uint8_t* dst_base, uint64_t dst_bytes, const uint64_t* dst_off, const uint64_t* dst_cap,
                      uint8_t* status, uint64_t* written, uint64_t n, void* cuda_stream, const Resume* resume)
{
  if (!ctx) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !dst_off || !dst_cap || !status) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  // the kernels index dst (and the bitmap) from a 128-byte aligned base
  const uint64_t delta = reinterpret_cast<uintptr_t>(dst_base) & 127u;
  dst_base -= delta;
  const uint64_t bits_bytes = bitmap_bytes(dst_bytes, delta);
  int rc = reserve(ctx, ctx->d_bits, bits_bytes);
  if (rc != SFB200_RC_OK) return rc;
  uint32_t* const match_bits = ctx->d_bits.as<uint32_t>();
  unsigned long long* const ctrs = ctx->d_counter.as<unsigned long long>();
  if (!written) {
    rc = reserve(ctx, ctx->d_written, n * sizeof(uint64_t));
    if (rc != SFB200_RC_OK) return rc;
    written = ctx->d_written.as<uint64_t>();
  }
  // Few streams: a lane per stream would leave the GPU empty, so each stream gets a warp that
  // decodes 32 spans of it speculatively (huff_stream.cuh).  Same results, by construction.
  // Measured on B200 with 64 KiB streams: 1 184 streams 1.8 ms against 4.7 ms lane per stream, 3 552
  // 4.5 against 4.8 ms, 4 736 5.8 against 5.0 ms: up to three streams per resident warp of the lane
  // kernel.  Small streams do not pay for a warp each (4 KiB pages are 7x slower that way): stream
  // sizes are only known on the device, so the room the caller gave them stands in (at least
  // 32 KiB of dst per stream on average).
  bool stream_mode = ctx->stream_ctas_per_sm > 0 &&
                     n * 32 <= 3 * static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->ctas_per_sm) *
                                       LaneCfg::WARPS * 32 &&
                     dst_bytes / n >= 32768;
  if (const char* e = std::getenv("SFB200_STREAM_MODE")) stream_mode = e[0] == '1' && ctx->stream_ctas_per_sm > 0;
  const bool chunked = resume && resume->start_bit;
  if (chunked) stream_mode = false;  // (a decode that continues at a block boundary: the lane kernel only)
  // One stream: pass 2 works on the whole output at once (lz_jump.cuh) instead of one warp walking it
  // (also a FEW large streams, one after the other: sizes are only known on the device, so "large" is
  //  judged by the room the caller gave them)
  bool jump = stream_mode && (n == 1 || (n <= 16 && dst_bytes / n >= (1ull << 20)));
  if (const char* e = std::getenv("SFB200_JUMP")) jump = jump && e[0] != '0';
  uint64_t jump_tiles = 0, stripe_tiles = 1ull << 23;  // (one stripe unless SFB200_JUMP_STRIPE_MB says otherwise)
  if (jump) {
    jump_tiles = (dst_bytes + delta + 128 + sfb::JUMP_TILE - 1) / sfb::JUMP_TILE + 1;
    if (const char* e = std::getenv("SFB200_JUMP_STRIPE_MB")) {
      const long mb = std::atol(e);
      if (mb > 0) stripe_tiles = static_cast<uint64_t>(mb) * ((1u << 20) / sfb::JUMP_TILE);
    }
    const uint64_t stripes = (jump_tiles + stripe_tiles - 1) / stripe_tiles;
    const uint64_t need = jump_tiles * sfb::JUMP_TILE * 4 + jump_tiles * 4 * (1 + sfb::JUMP_TILE / 128) +
                          stripes * (sfb::JUMP_MAX_ROUNDS + 1) * 4;
    rc = reserve(ctx, ctx->d_jump, need);
    if (rc == SFB200_RC_OUT_OF_MEMORY) {
      // no room for the pointer array (4 bytes per dst byte): a warp walks the stream instead —
      // slower, same results
      cudaGetLastError();
      ctx->err.clear();
      jump = false;
    } else if (rc != SFB200_RC_OK) {
      return rc;
    }
  }
  // ... and pass 1 decodes its blocks side by side (block_finder.cuh).  The input's size is only known
  // on the device; the scratch is sized for an input a little larger than the output, and block
  // starts that do not fit are simply not found (their blocks are then decoded by the tail job).
  bool blocks = jump;
  if (const char* e = std::getenv("SFB200_BLOCKS")) blocks = blocks && e[0] != '0';
  uint32_t cand_cap = 0, job_cap = 0, tab_size = 0, rec_cap = 0;
  if (blocks) {
    const uint64_t src_bits_max = 8 * (dst_bytes + dst_bytes / 32 + 65536);
    cand_cap = static_cast<uint32_t>(std::min<uint64_t>(src_bits_max / 128 + 4096, 1ull << 30));
    job_cap = static_cast<uint32_t>(std::min<uint64_t>(src_bits_max / 2048 + 1024, 1ull << 27));
    tab_size = 1024;
    while (tab_size < 2 * job_cap) tab_size *= 2;
    rec_cap = static_cast<uint32_t>(std::min<uint64_t>(src_bits_max / (16 * sfb::SPAN_BITS) + 65536, 1ull << 26));
    const uint64_t need = 64 + 4ull * tab_size + sizeof(sfb::BlockJob) * static_cast<uint64_t>(job_cap) +
                          8ull * cand_cap + sizeof(sfb::WinRec) * static_cast<uint64_t>(rec_cap) +
                          28ull * job_cap + 64;
    rc = reserve(ctx, ctx->d_find, need);
    if (rc == SFB200_RC_OUT_OF_MEMORY) {  // blocks one after the other instead of side by side
      cudaGetLastError();
      ctx->err.clear();
      blocks = false;
      jump = false;
    } else if (rc != SFB200_RC_OK) {
      return rc;
    }
  }
  // Geometry.  Measured on C2 (profiles/r01_small_geometry_c2.md): with 16 warps per SM the small
  // geometry makes pass 1 issue-bound (63 % of issue slots, 11.1 ms against 12.1 ms for the
  // large one), and the few percent of streams it hands on cost a whole extra stream latency
  // (4.5 ms) — so the large geometry is the default and the small one is opt-in
  // (SFB200_GEOMETRY=small) until the hand-over can overlap.
  bool use_small = false;
  if (const char* e = std::getenv("SFB200_GEOMETRY")) use_small = e[0] == 's' && ctx->small_ctas_per_sm > 0;
  if (resume) use_small = false;  // (the small geometry reports neither resume point nor end)
  if (use_small) {
    rc = reserve(ctx, ctx->d_defer, n * sizeof(uint32_t));
    if (rc != SFB200_RC_OK) return rc;
  }
  // Waves.  The two passes run BACK TO BACK over the whole batch: one launch each, inside which
  // warps pull groups of streams dynamically.  Cutting the batch into waves and running pass 2 of
  // wave k beside pass 1 of wave k+1 on two internal streams is kept for experiments
  // (SFB200_OVERLAP=1; wave size SFB200_WAVE_STREAMS) — measured at the end of round 2 it loses on
  // every shape: 65 536 x 64 KiB 19.4 against 18.6 ms, 131 072 x 64 KiB 39.7 against 37.0 ms,
  // 1 048 576 x 4 KiB 18.5 against 18.1 ms (DESIGN.md §3): pass 1 is latency-bound and slows down
  // by more than pass 2 gains when it shares its SMs.
  const uint64_t big_lanes = static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->ctas_per_sm) *
                             LaneCfg::WARPS * 32;
  const uint64_t small_lanes = static_cast<uint64_t>(ctx->sm_count) *
                               static_cast<uint64_t>(ctx->small_ctas_per_sm) * SmallCfg::WARPS * 32;
  // (a launch takes one wave of streams, or several when the batch has more than eight waves:
  //  inside a launch warps pull groups dynamically, which evens out unequal streams and lets a
  //  lane keep its fixed-Huffman tables from one stream to the next)
  const uint64_t lanes = use_small ? small_lanes : big_lanes;
  uint64_t wave = lanes * std::max<uint64_t>(1, (n + 8 * lanes - 1) / (8 * lanes));
  if (const char* e = std::getenv("SFB200_WAVE_STREAMS")) {  // (experiments: the size of a wave)
    const uint64_t v = std::strtoull(e, nullptr, 10);
    if (v >= 1024) wave = v;
  }
  uint64_t n_waves = (n + wave - 1) / wave;
  bool overlap_waves = false;
  if (const char* e = std::getenv("SFB200_OVERLAP")) overlap_waves = e[0] == '1';
  if (!overlap_waves) n_waves = 1;
  if (n_waves > kMaxWaves) n_waves = 1;  // (counters are a fixed array: enormous batches run unsplit)
  if (stream_mode) n_waves = 1;
  // Queue mode: ONE launch of pass 1, pass 2 beside it on the second stream, fed segment by segment
  // (deflate_lane.cuh: QueueArgs; lz_window.cuh: lz_window_queue_kernel).
  const bool qmode = ctx->queue_mode != 0 && !stream_mode && !use_small && !resume && !jump && !ctx->lz_v1;
  uint64_t qcap = 0;
  if (qmode) {
    n_waves = 1;
    qcap = 2 * n + ((dst_bytes + delta) >> sfb::Q_SEG_SHIFT) + 64;
    rc = reserve(ctx, ctx->d_queue, 64 + 24 * n + 8 * qcap + 64);
    if (rc != SFB200_RC_OK) return rc;
  }
  const uint64_t per_wave = n_waves == 1 ? n : wave;
  const bool overlap = n_waves > 1 || qmode;
  if (overlap) {
    if (!ctx->ps[0]) {  // pass 1's stream: the higher priority (its CTAs are placed first)
      int lo = 0, hi = 0;
      SFB_TRY(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
      SFB_TRY(ctx, cudaStreamCreateWithPriority(&ctx->ps[0], cudaStreamNonBlocking, hi));
    }
    for (auto& ps : ctx->ps)
      if (!ps) SFB_TRY(ctx, cudaStreamCreateWithFlags(&ps, cudaStreamNonBlocking));
    for (uint64_t k = ctx->wave_ev.size(); k < n_waves + 3; ++k) {
      cudaEvent_t e = nullptr;
      SFB_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ctx->wave_ev.push_back(e);
    }
  }
  cudaStream_t s1 = overlap ? ctx->ps[0] : st;  // pass-1 chain
  cudaStream_t s2 = overlap ? ctx->ps[1] : st;  // pass-2 chain
  ctx->ev_valid = false;
  SFB_TRY(ctx, cudaEventRecord(ctx->ev[0], st));
  SFB_TRY(ctx, cudaMemsetAsync(ctrs, 0,
                               kCountersPerWave * std::max<uint64_t>(n_waves, 1) * sizeof(unsigned long long), st));
  SFB_TRY(ctx, cudaMemsetAsync(ctrs + kCountersPerWave * kMaxWaves, 0, 16 * sizeof(unsigned long long), st));
  SFB_TRY(ctx, cudaMemsetAsync(match_bits, 0, bits_bytes, st));
  if (qmode) SFB_TRY(ctx, cudaMemsetAsync(ctx->d_queue.p, 0, 64 + 24 * n + 8 * qcap, st));
  // Order the streams by the type of their first block (see lz_warp.cuh: PrepArgs)
  uint8_t* handled = nullptr;
  bool sorted = n >= 64 && n < 0xffffffffull && !stream_mode && !resume;
  if (const char* e = std::getenv("SFB200_NO_SORT"))
    if (e[0] == '1') sorted = false;
  if (sorted) {
    rc = reserve(ctx, ctx->d_order, n * kOrderBytes);
    if (rc != SFB200_RC_OK) return rc;
    sfb::PrepArgs pa;
    pa.src_base = src_base;
    pa.src_off = src_off;
    pa.src_len = src_len;
    pa.n = n;
    pa.type_count = ctrs + kCountersPerWave * kMaxWaves;
    pa.type_cursor = pa.type_count + 4;
    pa.order = ctx->d_order.as<uint32_t>();
    const unsigned grid = static_cast<unsigned>((n + sfb::PREP_THREADS - 1) / sfb::PREP_THREADS);
    sfb::prep_count_kernel<<<grid, sfb::PREP_THREADS, 0, st>>>(pa);
    sfb::prep_scatter_kernel<<<grid, sfb::PREP_THREADS, 0, st>>>(pa);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 2;
    // Streams of stored blocks: a warp each, wide copies (stored_copy.cuh); the lane kernel skips
    // what this kernel finished.
    if (!ctx->no_stored) {
      handled = ctx->d_order.p + sizeof(uint32_t) * (ctx->d_order.cap / kOrderBytes);  // (behind the entries)
      SFB_TRY(ctx, cudaMemsetAsync(handled, 0, n, st));
      sfb::StoredArgs sa;
      sa.src_base = src_base;
      sa.src_off = src_off;
      sa.src_len = src_len;
      sa.dst_base = dst_base + delta;
      sa.dst_off = dst_off;
      sa.dst_cap = dst_cap;
      sa.status = status;
      sa.written = written;
      sa.handled = handled;
      sa.order = pa.order;
      sa.type_count = pa.type_count;
      sa.counter = pa.type_count + 8;
      const uint64_t warps = static_cast<uint64_t>(ctx->sm_count) * 8 * (sfb::STORED_THREADS / 32);
      const uint64_t want = (std::min<uint64_t>(n, warps) + sfb::STORED_THREADS / 32 - 1) / (sfb::STORED_THREADS / 32);
      sfb::stored_streams_kernel<<<static_cast<unsigned>(want), sfb::STORED_THREADS, 0, st>>>(sa);
      SFB_TRY(ctx, cudaGetLastError());
      ctx->launches += 1;
    }
  }
  SFB_TRY(ctx, cudaEventRecord(ctx->ev[1], st));
  if (overlap) {
    SFB_TRY(ctx, cudaEventRecord(ctx->wave_ev[n_waves], st));
    SFB_TRY(ctx, cudaStreamWaitEvent(s1, ctx->wave_ev[n_waves], 0));
    SFB_TRY(ctx, cudaStreamWaitEvent(s2, ctx->wave_ev[n_waves], 0));
  }
  for (uint64_t k = 0; k < n_waves; ++k) {
    const uint64_t first = k * per_wave;
    const uint64_t cnt = std::min(per_wave, n - first);
    unsigned long long* const ctr = ctrs + kCountersPerWave * k;
    const uint32_t* const order = sorted ? ctx->d_order.as<uint32_t>() + first : nullptr;
    // pass 1: Huffman layer, one lane per stream
    sfb::BatchArgs a{};
    a.src_base = src_base;
    a.src_off = src_off;
    a.src_len = src_len;
    a.dst_base = dst_base;
    a.dst_delta = delta;
    a.dst_off = dst_off;
    a.dst_cap = dst_cap;
    a.status = status;
    a.written = written;
    a.n = cnt;
    a.idx_base = first;
    a.lens_scratch = ctx->d_lens.as<uint32_t>();
    a.match_bits = match_bits;
    a.todo_list = order;
    a.no_pair = ctx->no_pair;
    a.handled = handled;
    a.start_bit = resume ? resume->start_bit : nullptr;
    a.start_out = resume ? resume->start_out : nullptr;
    a.blk_end = resume ? resume->blk_end : nullptr;
    if (qmode) {
      unsigned long long* const c = ctx->d_queue.as<unsigned long long>();
      a.q.tail = c + 0;
      a.q.head = c + 1;
      a.q.final_tail = c + 2;
      a.q.done = reinterpret_cast<unsigned int*>(c + 3);
      a.q.dbg = c + 4;
      a.q.turn = reinterpret_cast<unsigned int*>(ctx->d_queue.p + 64);
      a.q.state = reinterpret_cast<uint32_t*>(ctx->d_queue.p + 64 + 4 * n);
      a.q.items = reinterpret_cast<unsigned long long*>(ctx->d_queue.p + 64 + 24 * n);
      a.q.cap = qcap;
      a.q.seg_shift = sfb::Q_SEG_SHIFT;
      a.q.lag = sfb::Q_LAG;
    }
    const uint64_t groups = (cnt + 31) / 32;
    if (stream_mode) {
      sfb::StreamArgs sa{};
      sa.src_base = src_base;
      sa.src_off = src_off;
      sa.src_len = src_len;
      sa.dst_base = dst_base;
      sa.dst_delta = delta;
      sa.dst_off = dst_off;
      sa.dst_cap = dst_cap;
      sa.status = status;
      sa.written = written;
      sa.idx_base = first;
      sa.n = cnt;
      sa.stream_counter = ctr + 0;
      sa.lens_scratch = ctx->d_lens.as<uint32_t>();
      sa.match_bits = match_bits;
      sa.end_bit = resume && resume->end ? resume->blk_end : nullptr;
      const uint64_t resident =
          static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->stream_ctas_per_sm);
      if (blocks) {
        // find block starts | count each candidate block | chain | write the chained blocks
        uint32_t* const counters = ctx->d_find.as<uint32_t>();  // cand_count, job_count, tail_job
        sfb::FindArgs f;
        f.src_base = src_base;
        f.src_off = src_off;
        f.src_len = src_len;
        f.idx = 0;
        f.cand_count = counters + 0;
        f.job_count = counters + 1;
        f.tail_job = counters + 2;
        f.job_tab = counters + 16;
        f.tab_mask = tab_size - 1;
        f.jobs = reinterpret_cast<sfb::BlockJob*>(ctx->d_find.p + 64 + 4ull * tab_size);
        f.job_cap = job_cap;
        f.cand = reinterpret_cast<uint64_t*>(ctx->d_find.p + 64 + 4ull * tab_size +
                                             sizeof(sfb::BlockJob) * static_cast<uint64_t>(job_cap));
        f.cand_cap = cand_cap;
        f.dst_cap = dst_cap;
        sa.recs = reinterpret_cast<sfb::WinRec*>(reinterpret_cast<uint8_t*>(f.cand) + 8ull * cand_cap);
        sa.rec_count = counters + 3;
        sa.rec_cap = rec_cap;
        sfb::ChainScratch cs;  // behind the window records (8-byte aligned: WinRec is 272 bytes)
        cs.wa = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sa.recs) + sizeof(sfb::WinRec) * static_cast<uint64_t>(rec_cap));
        cs.wb = cs.wa + job_cap;
        cs.ja = reinterpret_cast<uint32_t*>(cs.wb + job_cap);
        cs.jb = cs.ja + job_cap;
        cs.mark = cs.jb + job_cap;
        bool seq_chain = false;
        if (const char* e = std::getenv("SFB200_CHAIN")) seq_chain = e[0] == 's';
        sa.jobs = f.jobs;
        sa.job_count = f.job_count;
        sa.job_cap = job_cap;
        sa.job_tab = f.job_tab;
        sa.tab_mask = f.tab_mask;
        sa.tail_job = f.tail_job;
        const unsigned grid = static_cast<unsigned>(resident);
        for (uint64_t si = 0; si < cnt; ++si) {
          f.idx = first + si;
          sa.idx_base = first + si;
          SFB_TRY(ctx, cudaMemsetAsync(ctx->d_find.p, 0, 64 + 4ull * tab_size, s1));
          if (si) SFB_TRY(ctx, cudaMemsetAsync(ctr, 0, 2 * sizeof(unsigned long long), s1));
          sfb::find_candidates_kernel<<<ctx->sm_count * 8, sfb::FIND_THREADS, 0, s1>>>(f);
          sfb::verify_candidates_kernel<<<ctx->sm_count * 4, sfb::FIND_THREADS, 0, s1>>>(f);
          sa.mode = 1;
          sa.stream_counter = ctr + 0;
          sfb::huff_stream_kernel<StreamCfg><<<grid, 32, StreamCfg::SMEM_BYTES, s1>>>(sa);
          if (seq_chain) sfb::chain_kernel<<<1, 32, 0, s1>>>(f);
          else sfb::chain_parallel_kernel<<<1, sfb::CHAIN_THREADS, 0, s1>>>(f, cs);
          sa.mode = 2;
          sa.stream_counter = ctr + 1;
          sfb::huff_stream_kernel<StreamCfg><<<grid, 32, StreamCfg::SMEM_BYTES, s1>>>(sa);
          SFB_TRY(ctx, cudaGetLastError());
        }
        ctx->launches += 5 * cnt;
      } else {
        const unsigned grid = grid_size(cnt, resident);
        sfb::huff_stream_kernel<StreamCfg><<<grid, 32, StreamCfg::SMEM_BYTES, s1>>>(sa);
        SFB_TRY(ctx, cudaGetLastError());
        ctx->launches += 1;
      }
    } else if (use_small) {
      a.group_counter = ctr + 0;
      a.defer_list = ctx->d_defer.as<uint32_t>() + first;
      a.defer_count = ctr + 3;
      const uint64_t want = (groups + SmallCfg::WARPS - 1) / SmallCfg::WARPS;
      const uint64_t resident =
          static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->small_ctas_per_sm);
      const unsigned grid = grid_size(want, resident);
      sfb::huff_lanes_kernel<SmallCfg><<<grid, SmallCfg::WARPS * 32, SmallCfg::SMEM_BYTES, s1>>>(a);
      SFB_TRY(ctx, cudaGetLastError());
      ctx->launches += 1;
      // the streams it handed on (none for low-entropy data: this launch then ends at once)
      a.defer_list = nullptr;
      a.defer_count = nullptr;
      a.todo_list = ctx->d_defer.as<uint32_t>() + first;
      a.todo_count = ctr + 3;
    }
    if (!stream_mode) {
      a.group_counter = ctr + 1;
      const uint64_t want = (groups + LaneCfg::WARPS - 1) / LaneCfg::WARPS;
      const uint64_t resident =
          static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->ctas_per_sm);
      const unsigned grid = grid_size(want, resident);
      // (a batch that fits the lanes of the wide geometry takes it: see WideCfg)
      const uint64_t wide_resident =
          static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->wide_ctas_per_sm);
      if (qmode) {
        sfb::huff_lanes_kernel<LaneCfg, false, true><<<grid, LaneCfg::WARPS * 32, LaneCfg::SMEM_BYTES, s1>>>(a);
      } else if (resume && resume->end) {
        sfb::huff_lanes_kernel<LaneCfg, false, false, true><<<grid, LaneCfg::WARPS * 32, LaneCfg::SMEM_BYTES, s1>>>(a);
      } else if (!use_small && n_waves == 1 && wide_resident != 0 && want <= wide_resident)
        sfb::huff_lanes_kernel<WideCfg><<<static_cast<unsigned>(want), WideCfg::WARPS * 32, WideCfg::SMEM_BYTES, s1>>>(a);
      else
        sfb::huff_lanes_kernel<LaneCfg><<<grid, LaneCfg::WARPS * 32, LaneCfg::SMEM_BYTES, s1>>>(a);
      SFB_TRY(ctx, cudaGetLastError());
      ctx->launches += 1;
    }
    if (overlap && !qmode) {
      SFB_TRY(ctx, cudaEventRecord(ctx->wave_ev[k], s1));
      SFB_TRY(ctx, cudaStreamWaitEvent(s2, ctx->wave_ev[k], 0));
    }
    if (k + 1 == n_waves) SFB_TRY(ctx, cudaEventRecord(ctx->ev[2], s1));  // end of all of pass 1
    // pass 2: LZ77 back-references, one warp per stream
    sfb::ResolveArgs r{};
    r.dst_base = dst_base;
    r.dst_delta = delta;
    r.dst_off = dst_off;
    r.written = written;
    r.match_bits = match_bits;
    r.n = cnt;
    r.idx_base = first;
    r.todo_list = order;
    r.stream_counter = ctr + 2;
    if (qmode) {
      // beside pass 1 (second stream), and the rest of the GPU's worth behind it (its own stream)
      // (beside pass 1: CTAs of 4 warps — 6 144 registers, what is left next to two CTAs of pass 1 —
      //  and few enough of them that pass 1 finds room on some SM whatever the order the two kernels
      //  start in: its stream has the higher priority, but nothing in CUDA promises the order)
      const unsigned per_sm = static_cast<unsigned>(ctx->lz_ctas_per_sm);
      const unsigned qa = std::min<unsigned>(static_cast<unsigned>(ctx->queue_ctas), 4u);
      const unsigned grid_a = static_cast<unsigned>(ctx->sm_count) * qa;
      const unsigned grid_b = static_cast<unsigned>(ctx->sm_count) * std::max(1u, per_sm - qa / 2u);
      if (ctx->lzw_minb == 4) {
        sfb::lz_window_queue_kernel<4><<<grid_a, 128, 0, s2>>>(r, a.q);
        sfb::lz_window_queue_kernel<4><<<grid_b, sfb::LZW_THREADS, 0, s1>>>(r, a.q);
      } else if (ctx->lzw_minb == 5) {
        sfb::lz_window_queue_kernel<5><<<grid_a, 128, 0, s2>>>(r, a.q);
        sfb::lz_window_queue_kernel<5><<<grid_b, sfb::LZW_THREADS, 0, s1>>>(r, a.q);
      } else {
        sfb::lz_window_queue_kernel<6><<<grid_a, 128, 0, s2>>>(r, a.q);
        sfb::lz_window_queue_kernel<6><<<grid_b, sfb::LZW_THREADS, 0, s1>>>(r, a.q);
      }
      SFB_TRY(ctx, cudaGetLastError());
      ctx->launches += 1;
    } else if (jump) {
      sfb::JumpArgs j;
      j.dst_base = dst_base;
      j.dst_delta = delta;
      j.dst_off = dst_off;
      j.written = written;
      j.match_bits = match_bits;
      j.ptr = ctx->d_jump.as<uint32_t>();
      j.tile_done = j.ptr + jump_tiles * sfb::JUMP_TILE;
      j.todo = j.tile_done + jump_tiles;
      const uint64_t stripes = (jump_tiles + stripe_tiles - 1) / stripe_tiles;
      uint32_t* const todo0 = j.todo;
      j.open = j.todo + stripes * (sfb::JUMP_MAX_ROUNDS + 1);
      constexpr uint64_t wpc = sfb::JUMP_THREADS / 32;
      const uint64_t resident = static_cast<uint64_t>(ctx->sm_count) * 8;
      for (uint64_t si = 0; si < cnt; ++si) {
        j.idx = first + si;
        SFB_TRY(ctx, cudaMemsetAsync(j.tile_done, 0, (jump_tiles + stripes * (sfb::JUMP_MAX_ROUNDS + 1)) * 4, s2));
        // pointers of stripe sp + 1 are set up BEFORE the rounds of stripe sp: the match that reaches
        // into a stripe from the left is read from its descriptor, which the rounds of the stripe
        // before replace by the final bytes
        auto set_stripe = [&](uint64_t sp) {
          j.tile_lo = static_cast<uint32_t>(sp * stripe_tiles);
          j.tile_hi = static_cast<uint32_t>(std::min<uint64_t>(jump_tiles, (sp + 1) * stripe_tiles));
          j.todo = todo0 + sp * (sfb::JUMP_MAX_ROUNDS + 1);
          const uint64_t want = (j.tile_hi - j.tile_lo + wpc - 1) / wpc;
          return grid_size(want, resident);
        };
        j.round = 0;
        sfb::lz_jump_init_kernel<<<set_stripe(0), sfb::JUMP_THREADS, 0, s2>>>(j);
        ctx->launches += 1;
        for (uint64_t sp = 0; sp < stripes; ++sp) {
          if (sp + 1 < stripes) {
            j.round = 0;
            sfb::lz_jump_init_kernel<<<set_stripe(sp + 1), sfb::JUMP_THREADS, 0, s2>>>(j);
            ctx->launches += 1;
          }
          const unsigned grid = set_stripe(sp);
          // a chain inside a stripe has fewer hops than the stripe has bytes, and a round divides
          // them by three: no more launches than that can need (+ 1 to see that nothing moved)
          int max_rounds = 2;
          for (uint64_t reach = 3; reach < static_cast<uint64_t>(j.tile_hi - j.tile_lo) * sfb::JUMP_TILE; reach *= 3)
            ++max_rounds;
          if (max_rounds > sfb::JUMP_MAX_ROUNDS) max_rounds = sfb::JUMP_MAX_ROUNDS;
          for (int r = 1; r <= max_rounds; ++r) {
            j.round = static_cast<uint32_t>(r);
            sfb::lz_jump_round_kernel<<<grid, sfb::JUMP_THREADS, 0, s2>>>(j);
            ctx->launches += 1;
          }
          SFB_TRY(ctx, cudaGetLastError());
        }
      }
    } else {
      constexpr uint64_t wpc = sfb::LZ_THREADS / 32;
      const uint64_t resident =
          static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->lz_ctas_per_sm);
      const uint64_t want = (cnt + wpc - 1) / wpc;
      const unsigned grid = grid_size(want, resident);
      if (ctx->lz_v1) sfb::lz_resolve_kernel<<<grid, sfb::LZ_THREADS, 0, s2>>>(r);
      else if (ctx->lzw_minb == 4) sfb::lz_window_kernel<4><<<grid, sfb::LZW_THREADS, 0, s2>>>(r);
      else if (ctx->lzw_minb == 5 && ctx->lzw_pf) sfb::lz_window_kernel<5, true><<<grid, sfb::LZW_THREADS, 0, s2>>>(r);
      else if (ctx->lzw_minb == 5) sfb::lz_window_kernel<5><<<grid, sfb::LZW_THREADS, 0, s2>>>(r);
      else sfb::lz_window_kernel<6><<<grid, sfb::LZW_THREADS, 0, s2>>>(r);
      SFB_TRY(ctx, cudaGetLastError());
    }
    if (qmode || !jump) ctx->launches += 1;   // (the jump route counted its launches one by one)
  }
  if (overlap) {
    SFB_TRY(ctx, cudaEventRecord(ctx->wave_ev[n_waves + 1], s1));
    SFB_TRY(ctx, cudaEventRecord(ctx->wave_ev[n_waves + 2], s2));
    SFB_TRY(ctx, cudaStreamWaitEvent(st, ctx->wave_ev[n_waves + 1], 0));
    SFB_TRY(ctx, cudaStreamWaitEvent(st, ctx->wave_ev[n_waves + 2], 0));
  }
  SFB_TRY(ctx, cudaEventRecord(ctx->ev[3], st));
  ctx->ev_valid = true;
  if (qmode) {
    // (experimental mode: synchronous, so that a consumer that gave up waiting — lz_window.cuh:
    //  lzq_give_up — fails the call instead of leaving matches unresolved behind a success)
    unsigned long long q8[8] = {0};
    SFB_TRY(ctx, cudaStreamSynchronize(st));
    SFB_TRY(ctx, cudaMemcpy(q8, ctx->d_queue.p, sizeof(q8), cudaMemcpyDeviceToHost));
    if (q8[4] != 0ull) {
      ctx->err = "queue mode: a pass-2 consumer gave up waiting (" + std::string(q8[4] == 1ull ? "for an item" : "for its turn") +
                 ", " + std::to_string(q8[5]) + " / " + std::to_string(q8[6]) + " / " + std::to_string(q8[7]) + ")";
      return SFB200_RC_CUDA_ERROR;
    }
  }
  return SFB200_RC_OK;
}

}  // namespace

extern "C" {

int sfb200_decompressed_size_batch_device(sfb200_ctx* ctx, const uint8_t* src_base,
                                          const uint64_t* src_off, const uint64_t* src_len,
                                          uint8_t* status, uint64_t* size, uint64_t n,
                                          void* cuda_stream)
{
  if (!ctx) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !status || !size) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  ctx->ev_valid = false;
  unsigned long long* const ctrs = ctx->d_counter.as<unsigned long long>();
  SFB_TRY(ctx, cudaMemsetAsync(ctrs, 0, kCountersPerWave * sizeof(unsigned long long), st));
  // (the counting writer never touches dst, its capacities or the bitmap: they stay null)
  sfb::BatchArgs a{};
  a.src_base = src_base;
  a.src_off = src_off;
  a.src_len = src_len;
  a.status = status;
  a.written = size;
  a.n = n;
  a.group_counter = ctrs + 1;
  a.lens_scratch = ctx->d_lens.as<uint32_t>();
  a.no_pair = ctx->no_pair;
  const uint64_t groups = (n + 31) / 32;
  const uint64_t want = (groups + LaneCfg::WARPS - 1) / LaneCfg::WARPS;
  const uint64_t resident = static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->ctas_per_sm);
  const unsigned grid = grid_size(want, resident);
  sfb::huff_lanes_kernel<LaneCfg, true><<<grid, LaneCfg::WARPS * 32, LaneCfg::SMEM_BYTES, st>>>(a);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  return SFB200_RC_OK;
}

int sfb200_last_pass_ms(sfb200_ctx* ctx, float* out3)
{
  if (!ctx || !out3 || !ctx->ev_valid) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  SFB_TRY(ctx, cudaEventSynchronize(ctx->ev[3]));
  for (int i = 0; i < 3; ++i) SFB_TRY(ctx, cudaEventElapsedTime(&out3[i], ctx->ev[i], ctx->ev[i + 1]));
  return SFB200_RC_OK;
}

int sfb200_checksum_batch_device(sfb200_ctx* ctx, const uint8_t* base, const uint64_t* off,
                                 const uint64_t* len, uint64_t* out, uint64_t n,
                                 void* cuda_stream)
{
  if (!ctx) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  SFB_ENTER(ctx);
  const unsigned threads = 128;
  const uint64_t blocks = (n * 32 + threads - 1) / threads;
  sfb::checksum_kernel<<<static_cast<unsigned>(blocks), threads, 0,
                         static_cast<cudaStream_t>(cuda_stream)>>>(base, off, len, out, n);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  return SFB200_RC_OK;
}

// Host buffers, in BOUNDED device memory.  The batch is cut into sub-batches of consecutive
// streams that flow through a ring of three staging slots (SFB200_HOST_STAGING_MB, default 3456:
// per slot 768 MiB of dst and 384 MiB of src) on four CUDA streams:
//   s_in   H2D of the sub-batch's compressed bytes and (rebased) offsets
//   s_run  the kernels (sfb200_decompress_batch_device on the slot's buffers)
//   s_meta status / written of the sub-batch -> pinned host memory
//   s_out  D2H of the bytes the decoder produced
// H2D of sub-batch k+2, the kernels of k+1 and the D2H of k overlap, so the call is bounded by the
// slower PCIe direction rather than by the sum of the stages, and a batch far larger than the GPU's
// memory decodes in the same ~3.4 GiB.  dst is NOT uploaded: only bytes the decoder produced are
// copied back (whole runs of adjacent, completely filled regions in one copy; for a stream that
// stopped early just its `written` prefix), so everything else in the caller's buffer keeps its
// value, as the reference guarantees.  A single stream larger than a slot makes the slots grow to
// hold it (one stream is one unit of work: SURVEY.md §8 f3 has the chunked single stream as next).
int sfb200_decompress_batch_host(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_bytes,
                                 const uint64_t* src_off, const uint64_t* src_len,
                                 uint8_t* dst, uint64_t dst_bytes, const uint64_t* dst_off,
                                 const uint64_t* dst_cap, uint8_t* status, uint64_t* written,
                                 uint64_t n)
{
  if (!ctx) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !dst_off || !dst_cap || !status) return SFB200_RC_BAD_ARGUMENT;
  if ((src_bytes && !src) || (dst_bytes && !dst)) return SFB200_RC_BAD_ARGUMENT;
  uint64_t max_src = 0, max_dst = 0;
  for (uint64_t i = 0; i < n; ++i) {
    if (src_off[i] > src_bytes || src_len[i] > src_bytes - src_off[i]) return SFB200_RC_BAD_ARGUMENT;
    if (dst_off[i] > dst_bytes || dst_cap[i] > dst_bytes - dst_off[i]) return SFB200_RC_BAD_ARGUMENT;
    max_src = std::max(max_src, src_len[i]);
    max_dst = std::max(max_dst, dst_cap[i]);
  }
  SFB_ENTER(ctx);
  constexpr int S = 3;
  // ---- slot sizes ------------------------------------------------------------------------------
  uint64_t budget = 3456ull << 20;
  if (const char* e = std::getenv("SFB200_HOST_STAGING_MB")) {
    const long v = std::atol(e);
    if (v > 0) budget = static_cast<uint64_t>(v) << 20;
  }
  if (const char* e = std::getenv("SFB200_HOST_STAGING_KB")) {  // (tests: force many sub-batches)
    const long v = std::atol(e);
    if (v > 0) budget = static_cast<uint64_t>(v) << 10;
  }
  uint64_t want_dst = std::max<uint64_t>(budget / S * 2 / 3, 4096), want_src = std::max<uint64_t>(budget / S / 3, 4096);
  // (a stream is staged whole; 256 bytes of slack for the 128-byte rebasing of the windows)
  want_dst = std::max(want_dst, max_dst + 256);
  want_src = std::max(want_src, max_src + 256);
  // no more than the batch needs
  want_dst = std::min(want_dst, dst_bytes + 256);
  want_src = std::min(want_src, src_bytes + 256);
  const uint64_t want_n = std::min<uint64_t>(n, 1ull << 22);  // streams per sub-batch
  auto sync_all = [&]() {
    for (auto& st : ctx->hs)
      if (st) cudaStreamSynchronize(st);
    if (ctx->s_meta) cudaStreamSynchronize(ctx->s_meta);
  };
  const uint64_t slot_src = want_src, slot_dst = want_dst;  // (what a sub-batch may span; the slots may be larger already)

  // ---- sub-batches of consecutive streams whose src and dst windows fit a slot -------------------
  struct Sub {
    uint64_t first, count, src_lo, src_hi, dst_lo, dst_hi;
  };
  std::vector<Sub> subs;
  // (the first sub-batches are an eighth, a quarter and a half of a slot: the download — the slower
  //  PCIe direction, which bounds the call — starts after the upload and the kernels of 1/8 of a
  //  slot instead of a whole one, and from then on never waits: a sub-batch's kernels take a
  //  quarter of the time its predecessor's download does even when it is twice as large)
  for (uint64_t i = 0; i < n;) {
    Sub sb{i, 0, ~0ull, 0, ~0ull, 0};
    const uint64_t ramp = subs.size() == 0 ? 8 : subs.size() == 1 ? 4 : subs.size() == 2 ? 2 : 1;
    const uint64_t lim_src = slot_src / ramp, lim_dst = slot_dst / ramp;
    while (i < n && sb.count < want_n) {
      const uint64_t slo = std::min(sb.src_lo, src_off[i]), shi = std::max(sb.src_hi, src_off[i] + src_len[i]);
      const uint64_t dlo = std::min(sb.dst_lo, dst_off[i]) & ~127ull, dhi = std::max(sb.dst_hi, dst_off[i] + dst_cap[i]);
      if (sb.count && (shi - slo > lim_src || dhi - dlo > lim_dst)) break;
      sb.src_lo = slo;
      sb.src_hi = shi;
      sb.dst_lo = dlo;  // (128-byte aligned: keeps the windows' alignment and the bitmap phase of the caller's layout)
      sb.dst_hi = dhi;
      ++sb.count;
      ++i;
    }
    subs.push_back(sb);
  }
  // ---- the slots this call needs (grown, never shrunk; a call with one sub-batch takes one) -----
  const int need_slots = static_cast<int>(std::min<size_t>(S, subs.size()));
  if (slot_dst > ctx->st_dst_cap || slot_src > ctx->st_src_cap) {
    sync_all();
    for (int k = 0; k < S; ++k) {
      ctx->st_src[k].release();
      ctx->st_dst[k].release();
    }
    ctx->st_slots = 0;
    ctx->st_src_cap = std::max(slot_src, ctx->st_src_cap);
    ctx->st_dst_cap = std::max(slot_dst, ctx->st_dst_cap);
  }
  int rc = SFB200_RC_OK;
  for (; ctx->st_slots < need_slots; ++ctx->st_slots) {
    const int k = ctx->st_slots;
    rc = reserve(ctx, ctx->st_src[k], ctx->st_src_cap + 64, 0, true);
    if (rc == SFB200_RC_OK) rc = reserve(ctx, ctx->st_dst[k], ctx->st_dst_cap + 64, 0, true);
    if (rc != SFB200_RC_OK) return rc;
  }
  if (want_n > ctx->st_meta_n) {
    sync_all();
    for (int k = 0; k < S; ++k) {
      ctx->st_meta[k].release();
      if (ctx->st_hmeta[k]) SFB_TRY(ctx, cudaFreeHost(ctx->st_hmeta[k]));
      ctx->st_hmeta[k] = nullptr;
    }
    ctx->st_meta_n = 0;
    const uint64_t cap = want_n + want_n / 8 + 64;
    for (int k = 0; k < S; ++k) {
      rc = reserve(ctx, ctx->st_meta[k], cap * (5 * 8 + 1) + 64, 0, true);
      if (rc != SFB200_RC_OK) return rc;
      SFB_TRY(ctx, cudaMallocHost(reinterpret_cast<void**>(&ctx->st_hmeta[k]), cap * (5 * 8 + 1) + 64));
    }
    ctx->st_meta_n = cap;
  }
  for (auto& st : ctx->hs)
    if (!st) SFB_TRY(ctx, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  if (!ctx->s_meta) SFB_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_meta, cudaStreamNonBlocking));
  for (int k = 0; k < S; ++k)
    for (auto& e : ctx->st_ev[k])
      if (!e) SFB_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  cudaStream_t s_in = ctx->hs[0], s_run = ctx->hs[1], s_out = ctx->hs[2], s_meta = ctx->s_meta;
  const uint64_t cap_n = ctx->st_meta_n;
  // the scratch of the device call is sized once, for the largest sub-batch (no reallocation —
  // cudaFree synchronises the device — while the pipeline runs)
  {
    uint64_t big = 0, big_n = 0;
    for (const Sub& sb : subs) {
      big = std::max(big, sb.dst_hi - sb.dst_lo);
      big_n = std::max(big_n, sb.count);
    }
    const uint64_t bits = bitmap_bytes(big, 127), order = big_n * kOrderBytes;
    if (bits > ctx->d_bits.cap || order > ctx->d_order.cap) sync_all();
    rc = reserve(ctx, ctx->d_bits, bits);
    if (rc == SFB200_RC_OK) rc = reserve(ctx, ctx->d_order, order);
    if (rc != SFB200_RC_OK) return rc;
  }
  auto cleanup = [&](int code) {
    sync_all();
    return code;
  };
#define SFB_TRYC(call)                                           \
  do {                                                           \
    const cudaError_t e_ = (call);                               \
    if (e_ != cudaSuccess) return cleanup(fail(ctx, e_, #call)); \
  } while (0)
  // slot k % S: device arrays and their pinned mirror
  auto d_arr = [&](int slot, int which) { return ctx->st_meta[slot].as<uint64_t>() + static_cast<uint64_t>(which) * cap_n; };
  auto h_arr = [&](int slot, int which) { return ctx->st_hmeta[slot] + static_cast<uint64_t>(which) * cap_n; };
  auto enqueue = [&](size_t k) -> int {
    const Sub& sb = subs[k];
    const int slot = static_cast<int>(k % S);
    const uint64_t f = sb.first, c = sb.count;
    // the slot is free once the bytes of its previous occupant have left for the host
    // (and the host has read that sub-batch's status / written from the pinned mirror: it has —
    //  sub-batch k - S was finished before this one is enqueued)
    if (k >= static_cast<size_t>(S)) SFB_TRYC(cudaStreamWaitEvent(s_in, ctx->st_ev[slot][3], 0));
    uint64_t* h_so = h_arr(slot, 0), * h_sl = h_arr(slot, 1), * h_do = h_arr(slot, 2), * h_dc = h_arr(slot, 3);
    for (uint64_t j = 0; j < c; ++j) {
      h_so[j] = src_off[f + j] - sb.src_lo;
      h_sl[j] = src_len[f + j];
      h_do[j] = dst_off[f + j] - sb.dst_lo;
      h_dc[j] = dst_cap[f + j];
    }
    if (sb.src_hi > sb.src_lo)
      SFB_TRYC(cudaMemcpyAsync(ctx->st_src[slot].p, src + sb.src_lo, sb.src_hi - sb.src_lo, cudaMemcpyHostToDevice, s_in));
    // (the four arrays are contiguous in both mirrors when c == cap_n; copy them one by one)
    for (int w = 0; w < 4; ++w)
      SFB_TRYC(cudaMemcpyAsync(d_arr(slot, w), h_arr(slot, w), c * 8, cudaMemcpyHostToDevice, s_in));
    SFB_TRYC(cudaEventRecord(ctx->st_ev[slot][0], s_in));
    SFB_TRYC(cudaStreamWaitEvent(s_run, ctx->st_ev[slot][0], 0));
    uint8_t* const d_status = reinterpret_cast<uint8_t*>(d_arr(slot, 5));
    const int r = sfb200_decompress_batch_device(ctx, ctx->st_src[slot].p, d_arr(slot, 0), d_arr(slot, 1),
                                                 ctx->st_dst[slot].p, sb.dst_hi - sb.dst_lo, d_arr(slot, 2),
                                                 d_arr(slot, 3), d_status, d_arr(slot, 4), c, s_run);
    if (r) return cleanup(r);
    SFB_TRYC(cudaEventRecord(ctx->st_ev[slot][1], s_run));
    SFB_TRYC(cudaStreamWaitEvent(s_meta, ctx->st_ev[slot][1], 0));
    SFB_TRYC(cudaMemcpyAsync(h_arr(slot, 4), d_arr(slot, 4), c * 8, cudaMemcpyDeviceToHost, s_meta));
    SFB_TRYC(cudaMemcpyAsync(h_arr(slot, 5), d_status, c, cudaMemcpyDeviceToHost, s_meta));
    SFB_TRYC(cudaEventRecord(ctx->st_ev[slot][2], s_meta));
    return SFB200_RC_OK;
  };
  size_t enq = 0;
  for (; enq < subs.size() && enq < static_cast<size_t>(S) - 1; ++enq) {
    rc = enqueue(enq);
    if (rc) return rc;
  }
  for (size_t k = 0; k < subs.size(); ++k) {
    // keep S - 1 sub-batches in flight behind this one (slot (k + S - 1) % S is the one sub-batch
    // k - 1 has just left)
    if (enq < subs.size()) {
      rc = enqueue(enq++);
      if (rc) return rc;
    }
    const Sub& sb = subs[k];
    const int slot = static_cast<int>(k % S);
    SFB_TRYC(cudaEventSynchronize(ctx->st_ev[slot][2]));
    const uint64_t* const wr_host = h_arr(slot, 4);
    const uint8_t* const st_host = reinterpret_cast<const uint8_t*>(h_arr(slot, 5));
    // bytes produced -> the caller's buffer, in as few copies as the layout allows
    SFB_TRYC(cudaStreamWaitEvent(s_out, ctx->st_ev[slot][1], 0));
    uint64_t run_lo = 0, run_hi = 0;  // pending run [run_lo, run_hi) of produced bytes (caller's offsets)
    auto flush_run = [&]() -> int {
      if (run_hi > run_lo)
        SFB_TRYC(cudaMemcpyAsync(dst + run_lo, ctx->st_dst[slot].p + (run_lo - sb.dst_lo), run_hi - run_lo,
                                 cudaMemcpyDeviceToHost, s_out));
      run_lo = run_hi = 0;
      return SFB200_RC_OK;
    };
    for (uint64_t j = 0; j < sb.count; ++j) {
      const uint64_t i = sb.first + j;
      const uint64_t w = wr_host[j];
      status[i] = st_host[j];
      if (written) written[i] = w;
      if (w == 0) continue;
      if (run_hi > run_lo && dst_off[i] == run_hi) {
        run_hi += w;
      } else {
        rc = flush_run();
        if (rc) return rc;
        run_lo = dst_off[i];
        run_hi = run_lo + w;
      }
      if (w != dst_cap[i]) {  // the rest of this region is not ours: the run ends here
        rc = flush_run();
        if (rc) return rc;
      }
    }
    rc = flush_run();
    if (rc) return rc;
    SFB_TRYC(cudaEventRecord(ctx->st_ev[slot][3], s_out));
  }
#undef SFB_TRYC
  return cleanup(SFB200_RC_OK);
}

uint64_t sfb200_staging_bytes(const sfb200_ctx* ctx)
{
  return ctx ? static_cast<uint64_t>(ctx->st_slots) * (ctx->st_src_cap + ctx->st_dst_cap + 128) : 0;
}

// One batch, several GPUs: the streams are cut into contiguous shards balanced by the bytes they
// move (sum of src_len + dst_cap, SURVEY.md §8e) and every context decodes its shard through
// sfb200_decompress_batch_host on a thread of its own.  No communication between the devices:
// streams are independent.  Returns the first non-zero infrastructure code, if any.
int sfb200_decompress_batch_host_multi(sfb200_ctx* const* ctxs, int n_ctx, const uint8_t* src, uint64_t src_bytes,
                                       const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst,
                                       uint64_t dst_bytes, const uint64_t* dst_off, const uint64_t* dst_cap,
                                       uint8_t* status, uint64_t* written, uint64_t n)
{
  if (!ctxs || n_ctx <= 0) return SFB200_RC_BAD_ARGUMENT;
  for (int k = 0; k < n_ctx; ++k)
    if (!ctxs[k]) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !dst_off || !dst_cap || !status) return SFB200_RC_BAD_ARGUMENT;
  if (n_ctx == 1)
    return sfb200_decompress_batch_host(ctxs[0], src, src_bytes, src_off, src_len, dst, dst_bytes, dst_off, dst_cap,
                                        status, written, n);
  std::vector<uint64_t> cut(static_cast<size_t>(n_ctx) + 1, n);
  sfb200_partition_streams(src_len, dst_cap, n, n_ctx, cut.data());
  std::vector<int> rcs(static_cast<size_t>(n_ctx), SFB200_RC_OK);
  std::vector<std::thread> th;
  for (int k = 0; k < n_ctx; ++k) {
    const uint64_t lo = cut[k], cnt = cut[k + 1] - cut[k];
    if (cnt == 0) continue;
    th.emplace_back([=, &rcs] {
      rcs[k] = sfb200_decompress_batch_host(ctxs[k], src, src_bytes, src_off + lo, src_len + lo, dst, dst_bytes,
                                            dst_off + lo, dst_cap + lo, status + lo, written ? written + lo : nullptr,
                                            cnt);
    });
  }
  for (auto& t : th) t.join();
  for (int r : rcs)
    if (r) return r;
  return SFB200_RC_OK;
}

// cut[0] = 0 <= cut[1] <= ... <= cut[parts] = n: contiguous shards with (nearly) equal sums of
// src_len + dst_cap.
void sfb200_partition_streams(const uint64_t* src_len, const uint64_t* dst_cap, uint64_t n, int parts, uint64_t* cut)
{
  long double total = 0;
  for (uint64_t i = 0; i < n; ++i) total += static_cast<long double>(src_len[i]) + static_cast<long double>(dst_cap[i]);
  cut[0] = 0;
  long double acc = 0;
  uint64_t i = 0;
  for (int k = 1; k < parts; ++k) {
    const long double goal = total * k / parts;
    while (i < n && acc + (static_cast<long double>(src_len[i]) + static_cast<long double>(dst_cap[i])) / 2 <= goal) {
      acc += static_cast<long double>(src_len[i]) + static_cast<long double>(dst_cap[i]);
      ++i;
    }
    cut[k] = i;
  }
  cut[parts] = n;
}

int sfb200_decompress(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst,
                      size_t dst_cap, uint8_t* status, uint64_t* written)
{
  if (!status) return SFB200_RC_BAD_ARGUMENT;
  const uint64_t zero = 0, sl = src_len, dc = dst_cap;
  return sfb200_decompress_batch_host(ctx, src, sl, &zero, &sl, dst, dc, &zero, &dc, status,
                                      written, 1);
}

// ---------------------------------------------------------------------------------------------
// Chunked input for ONE stream (SURVEY.md §8 f3; the reference anticipates it at
// src/decompress.cpp:214).  The unit of progress is the BLOCK: a call decodes, with the lane kernel,
// every block that is complete in the input fed so far, keeps what those blocks produced and
// carries three things to the next call — the bytes from the next block header on (device), the bit
// offset of that header, and the last 32 KiB of output (the LZ77 window, in front of the output
// buffer, so that distances reach into it as they would in one call).
struct sfb200_inflate_stream {
  sfb200_ctx* ctx = nullptr;
  DevBuf d_in[2];          // buffered input (the other one is the target of the next compaction)
  int cur = 0;
  uint64_t in_len = 0;     // bytes buffered
  uint64_t bit = 0;        // bit offset of the next block header inside the buffer (0..7 between calls)
  DevBuf d_out;            // [32 KiB window | output of one call]
  DevBuf d_tmp;            // 32 KiB (window moves that overlap)
  uint64_t hist = 0;       // valid window bytes, right-aligned in the first 32 KiB of d_out
  DevBuf d_meta;           // u64: src_off, src_len, dst_off, dst_cap, written, start_bit, start_out, blk_end[2], status
  bool finished = false;
  uint8_t final_status = 0;
};

namespace {
constexpr uint64_t kWindow = 32768;
}  // namespace

int sfb200_inflate_stream_create(sfb200_ctx* ctx, sfb200_inflate_stream** out)
{
  if (!ctx || !out) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  sfb200_inflate_stream* s = new (std::nothrow) sfb200_inflate_stream;
  if (!s) return SFB200_RC_OUT_OF_MEMORY;
  s->ctx = ctx;
  int rc = reserve(ctx, s->d_tmp, kWindow, 0, true);
  if (rc == SFB200_RC_OK) rc = reserve(ctx, s->d_meta, 16 * sizeof(uint64_t), 0, true);
  if (rc != SFB200_RC_OK) {
    delete s;
    cudaGetLastError();
    return rc;
  }
  *out = s;
  return SFB200_RC_OK;
}

void sfb200_inflate_stream_destroy(sfb200_inflate_stream* s)
{
  if (!s) return;
  DeviceGuard guard_(s->ctx->device);  // (its device memory is freed with it, on its device)
  delete s;
}

int sfb200_inflate_stream_feed(sfb200_inflate_stream* s, const uint8_t* src, size_t src_len, int last, uint8_t* dst,
                               size_t dst_cap, uint64_t* written, uint8_t* status, int* finished)
{
  if (!s || !status || !written || !finished || (src_len && !src) || (dst_cap && !dst)) return SFB200_RC_BAD_ARGUMENT;
  sfb200_ctx* const ctx = s->ctx;
  SFB_ENTER(ctx);
  *written = 0;
  if (s->finished) {
    *status = s->final_status;
    *finished = 1;
    return SFB200_RC_OK;
  }
  *finished = 0;
  *status = SFB200_SUCCESS;
  if (s->in_len + src_len >= 0xffffff00ull || kWindow + dst_cap >= 0xffffff00ull) return SFB200_RC_BAD_ARGUMENT;
  // the new input goes behind what is buffered
  int rc = reserve(ctx, s->d_in[s->cur], s->in_len + src_len + 64, s->in_len);
  if (rc != SFB200_RC_OK) return rc;
  if (src_len) SFB_TRY(ctx, cudaMemcpy(s->d_in[s->cur].p + s->in_len, src, src_len, cudaMemcpyHostToDevice));
  s->in_len += src_len;
  if (dst_cap == 0 && !last) return SFB200_RC_OK;  // (only buffering)
  rc = reserve(ctx, s->d_out, kWindow + dst_cap + 256, s->d_out.p ? kWindow : 0);
  if (rc != SFB200_RC_OK) return rc;
  // one lane-kernel decode from the pending block header, behind the window
  uint64_t h[16] = {0};
  h[0] = 0;                        // src_off
  h[1] = s->in_len;                // src_len
  h[2] = kWindow - s->hist;        // dst_off
  h[3] = s->hist + dst_cap;        // dst_cap
  h[4] = s->hist;                  // written (overwritten)
  h[5] = s->bit;                   // start_bit
  h[6] = s->hist;                  // start_out
  h[7] = s->bit;                   // blk_end: bit, output position (stay like this when no header is reached)
  h[8] = s->hist;
  h[9] = SFB200_ERROR;             // status (first byte)
  uint64_t* const m = s->d_meta.as<uint64_t>();
  SFB_TRY(ctx, cudaMemcpy(m, h, sizeof h, cudaMemcpyHostToDevice));
  Resume rs;
  rs.start_bit = m + 5;
  rs.start_out = m + 6;
  rs.blk_end = m + 7;
  rc = batch_device_impl(ctx, s->d_in[s->cur].p, m + 0, m + 1, s->d_out.p, kWindow + dst_cap, m + 2, m + 3,
                         reinterpret_cast<uint8_t*>(m + 9), m + 4, 1, nullptr, &rs);
  if (rc != SFB200_RC_OK) return rc;
  SFB_TRY(ctx, cudaMemcpy(h, m, sizeof h, cudaMemcpyDeviceToHost));
  const uint8_t st = static_cast<uint8_t>(h[9] & 0xffu);
  const uint64_t total = h[4], be_bit = h[7], be_out = h[8];
  uint64_t produced = 0;
  if (st == SFB200_SUCCESS || (last && st != SFB200_DST_TOO_SMALL)) {
    // the final block was decoded, or no more input will come: the stream ends as one call would end it
    produced = total - s->hist;
    s->finished = true;
    s->final_status = st;
    *status = st;
    *finished = 1;
  } else if (st == SFB200_DST_TOO_SMALL && be_out == s->hist) {
    *status = SFB200_DST_TOO_SMALL;  // not even the next block fits dst: call again with more room (nothing is lost)
    return SFB200_RC_OK;
  } else {
    // ran out of input (or of room) inside a block: keep the complete blocks, redo that one next time
    produced = be_out - s->hist;
    s->bit = be_bit;
  }
  if (produced) SFB_TRY(ctx, cudaMemcpy(dst, s->d_out.p + kWindow, produced, cudaMemcpyDeviceToHost));
  *written = produced;
  if (!s->finished) {
    // the window: the last 32 KiB of everything produced so far
    const uint64_t have = s->hist + produced;
    const uint64_t keep = have < kWindow ? have : kWindow;
    if (produced) {
      const uint8_t* from = s->d_out.p + kWindow + produced - keep;
      uint8_t* to = s->d_out.p + kWindow - keep;
      if (produced >= kWindow) {
        SFB_TRY(ctx, cudaMemcpy(to, from, keep, cudaMemcpyDeviceToDevice));
      } else {
        SFB_TRY(ctx, cudaMemcpy(s->d_tmp.p, from, keep, cudaMemcpyDeviceToDevice));
        SFB_TRY(ctx, cudaMemcpy(to, s->d_tmp.p, keep, cudaMemcpyDeviceToDevice));
      }
    }
    s->hist = keep;
    // the input: drop the bytes in front of the pending block header
    const uint64_t drop = s->bit >> 3;
    if (drop) {
      const int other = s->cur ^ 1;
      const uint64_t rest = s->in_len - drop;
      rc = reserve(ctx, s->d_in[other], rest + 64);
      if (rc != SFB200_RC_OK) return rc;
      if (rest) SFB_TRY(ctx, cudaMemcpy(s->d_in[other].p, s->d_in[s->cur].p + drop, rest, cudaMemcpyDeviceToDevice));
      s->cur = other;
      s->in_len = rest;
      s->bit &= 7u;
    }
  }
  return SFB200_RC_OK;
}


// ---------------------------------------------------------------------------------------------
// Batched compression (SURVEY.md §8 f4; deflate_compress.cuh)
uint64_t sfb200_compress_bound(uint64_t src_len)
{
  // stored blocks are the fallback: 5 header bytes per 65 535 payload bytes
  return src_len + 5ull * (src_len ? (src_len + 65534ull) / 65535ull : 1ull);
}

int sfb200_compress_batch_device(sfb200_ctx* ctx, const uint8_t* src_base, const uint64_t* src_off,
                                 const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                                 const uint64_t* dst_cap, uint8_t* status, uint64_t* written, uint64_t n,
                                 void* cuda_stream)
{
  if (!ctx) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !dst_off || !dst_cap || !status || !written) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  SFB_TRY(ctx, cudaMemsetAsync(ctx->d_counter.p, 0, sizeof(unsigned long long), st));
  sfb::CompressArgs a;
  a.src_base = src_base;
  a.src_off = src_off;
  a.src_len = src_len;
  a.dst_base = dst_base;
  a.dst_off = dst_off;
  a.dst_cap = dst_cap;
  a.status = status;
  a.written = written;
  a.n = n;
  a.counter = ctx->d_counter.as<unsigned long long>();
  a.fixed_only = 0;   // SFB200_COMPRESS_FIXED=1: the first generation (one pass, fixed-Huffman blocks only) for A/B runs
  if (const char* e = std::getenv("SFB200_COMPRESS_FIXED")) a.fixed_only = e[0] == '1';
  const uint64_t want = (n + sfb::CMP_WARPS - 1) / sfb::CMP_WARPS;
  const uint64_t resident = static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->compress_ctas_per_sm);
  sfb::deflate_compress_kernel<<<grid_size(want, resident), sfb::CMP_WARPS * 32, sfb::CMP_SMEM_BYTES, st>>>(a);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  return SFB200_RC_OK;
}

int sfb200_compress(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                    uint8_t* status, uint64_t* written)
{
  return sfb200_compress_container(ctx, SFB200_CONTAINER_RAW, src, src_len, dst, dst_cap, status, written);
}

int sfb200_decompress_container_batch_device(sfb200_ctx* ctx, int container, const uint8_t* src_base,
                                             const uint64_t* src_off, const uint64_t* src_len,
                                             uint8_t* dst_base, uint64_t dst_bytes,
                                             const uint64_t* dst_off, const uint64_t* dst_cap,
                                             uint8_t* status, uint64_t* written, uint64_t n,
                                             void* cuda_stream)
{
  if (!ctx || container < 0 || container > 3) return SFB200_RC_BAD_ARGUMENT;
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !dst_off || !dst_cap || !status) return SFB200_RC_BAD_ARGUMENT;
  if (container == SFB200_CONTAINER_RAW)
    return sfb200_decompress_batch_device(ctx, src_base, src_off, src_len, dst_base, dst_bytes, dst_off, dst_cap,
                                          status, written, n, cuda_stream);
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  int rc = reserve(ctx, ctx->d_cont, n * 36 + 64);
  if (rc != SFB200_RC_OK) return rc;
  sfb::ContainerArgs c;
  c.src_base = src_base;
  c.src_off = src_off;
  c.src_len = src_len;
  c.container = static_cast<uint32_t>(container);
  c.n = n;
  c.pay_off = ctx->d_cont.as<uint64_t>();
  c.pay_len = c.pay_off + n;
  uint64_t* const own_written = c.pay_len + n;
  c.kind = reinterpret_cast<uint32_t*>(own_written + n);
  c.expect = c.kind + n;
  c.isize = c.expect + n;
  c.dst_base = dst_base;
  c.dst_off = dst_off;
  c.status = status;
  c.written = written ? written : own_written;
  const unsigned pgrid = static_cast<unsigned>((n + 127) / 128);
  sfb::container_parse_kernel<<<pgrid, 128, 0, st>>>(c);
  SFB_TRY(ctx, cudaGetLastError());
  rc = sfb200_decompress_batch_device(ctx, src_base, c.pay_off, c.pay_len, dst_base, dst_bytes, dst_off, dst_cap,
                                      status, c.written, n, cuda_stream);
  if (rc != SFB200_RC_OK) return rc;
  const uint64_t want = (n * 32 + sfb::CHECK_THREADS - 1) / sfb::CHECK_THREADS;
  const uint64_t resident = static_cast<uint64_t>(ctx->sm_count);  // (one block per SM: 128 KiB of tables)
  sfb::container_check_kernel<<<grid_size(want, resident), sfb::CHECK_THREADS, sfb::CHECK_SMEM_BYTES, st>>>(c);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 2;
  return SFB200_RC_OK;
}

int sfb200_decompress_container(sfb200_ctx* ctx, int container, const uint8_t* src, size_t src_len,
                                uint8_t* dst, size_t dst_cap, uint8_t* status, uint64_t* written)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  return host_buffer_call(ctx, src, src_len, dst, dst_cap, written,
                          [&](uint8_t* s, uint8_t* d, uint64_t* m, uint64_t* wr) {
    const int rc = sfb200_decompress_container_batch_device(ctx, container, s, m, m + 1, d, dst_cap, m + 2, m + 3,
                                                            reinterpret_cast<uint8_t*>(m + 5), m + 4, 1, nullptr);
    return rc != SFB200_RC_OK ? rc : read_meta(ctx, m, wr, status);
  });
}

int sfb200_decompressed_size(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* status,
                             uint64_t* size)
{
  if (!ctx || !status || !size || (!src && src_len)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  // (the size goes to *size: no bytes of dst)
  return host_buffer_call(ctx, src, src_len, nullptr, 0, nullptr,
                          [&](uint8_t* s, uint8_t*, uint64_t* m, uint64_t*) {
    const int rc = sfb200_decompressed_size_batch_device(ctx, s, m, m + 1, reinterpret_cast<uint8_t*>(m + 5), m + 4, 1,
                                                         nullptr);
    return rc != SFB200_RC_OK ? rc : read_meta(ctx, m, size, status);
  });
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// gzip files of several members, BGZF at batch speed (gzip_file.cuh).  The members are found on the
// device: candidates, jump tables, then a walk in steps — one step per run of BGZF members (a whole
// BGZF file is one step), one more per plain member, whose length is known only after its payload
// was decoded (the "probe": a single-stream decode over the rest of the file on whichever route the
// size of dst selects; both report the bit behind the final block).  Then the member table goes
// through the container batch path, and one kernel reduces the members' results to the file's.
// (A plain member's probe has only the rest of dst as room, its ISIZE being unknown until its end is
//  found: one whose payload overruns a corrupt ISIZE AND does not fit the rest of dst reports
//  DstTooSmall, not SizeMismatch.)
namespace {
constexpr uint64_t kGzfMemberBytes = 5 * 8 + 1;    // pos, len, dst off, dst cap, written (u64); status (u8)
constexpr uint64_t kGzfMaxLen = 0xffffff00ull - 1;  // the batch precondition on src_len / dst_cap

struct GzfResult {
  uint8_t status = 0;
  uint64_t written = 0, members = 0, size = 0;
  bool complete = false;
};

// members the table has room for: its columns (five of u64, then status) are strided by this
uint64_t gzm_members(const sfb200_ctx* ctx) { return ctx->d_gzm.cap / kGzfMemberBytes; }

// room for `need` members in the table, keeping the first `keep`
int gzf_reserve(sfb200_ctx* ctx, uint64_t need, uint64_t keep, cudaStream_t st)
{
  const uint64_t old_n = gzm_members(ctx);
  if (need <= old_n) return SFB200_RC_OK;
  DevBuf q;
  const int rc = reserve(ctx, q, (need + need / 2 + 64) * kGzfMemberBytes, 0, true);
  if (rc != SFB200_RC_OK) return rc;
  const uint64_t cap = q.cap / kGzfMemberBytes;
  if (keep)
    for (int w = 0; w < 5; ++w)
      SFB_TRY(ctx, cudaMemcpyAsync(q.p + w * 8 * cap, ctx->d_gzm.p + w * 8 * old_n, keep * 8, cudaMemcpyDeviceToDevice,
                                   st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  ctx->d_gzm.swap(q);  // (q frees the old table)
  return SFB200_RC_OK;
}

// decode == false: discovery only (sizes of the BGZF members the walk reaches; a plain member ends it)
int gzip_file_impl(sfb200_ctx* ctx, const uint8_t* src, uint64_t len, uint8_t* dst, uint64_t dst_cap, bool decode,
                   cudaStream_t st, GzfResult* res)
{
  *res = GzfResult{};
  if (len == 0) {  // an empty file is an empty series of members (Python, gzip(1))
    res->complete = true;
    return SFB200_RC_OK;
  }
  const uint64_t tile = static_cast<uint64_t>(sfb::GZF_THREADS) * sfb::GZF_BYTES;
  const uint64_t tiles = (len + (reinterpret_cast<uintptr_t>(src) & 15u) + tile - 1) / tile;
  // step (128 B) | result (2 x u64) | probe metadata (16 x u64) | tile counts (tiles + 1)
  int rc = reserve(ctx, ctx->d_gzf, 128 + 16 + 128 + 8 * (tiles + 1));
  if (rc != SFB200_RC_OK) return rc;
  sfb::GzfArgs a{};
  a.src = src;
  a.len = len;
  a.step = ctx->d_gzf.as<sfb::GzfStep>();
  uint64_t* const d_result = reinterpret_cast<uint64_t*>(ctx->d_gzf.p + 128);
  uint64_t* const pm = d_result + 2;
  a.tile_count = pm + 16;
  a.dst_cap = decode ? dst_cap : ~0ull;
  // ---- candidates: count per tile, scan, then (with scratch for exactly that many) scatter ------
  sfb::gzf_count_kernel<<<static_cast<unsigned>(tiles), sfb::GZF_THREADS, 0, st>>>(a);
  sfb::gzf_exscan_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(a.tile_count, tiles);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 2;
  uint64_t m = 0;
  SFB_TRY(ctx, cudaMemcpyAsync(&m, a.tile_count + tiles, 8, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  if (m >= 0xffffffffull) {  // (candidate indices are 32-bit: only a file of > 8 GiB of header-like bytes gets here)
    ctx->err = "gzip file: more than 2^32 - 2 BGZF header candidates";
    return SFB200_RC_BAD_ARGUMENT;
  }
  uint32_t tables = 1;  // J_0 .. J_{tables-1}: enough that 2^tables > the longest chain (<= m members)
  while ((1ull << tables) < m + 1) ++tables;
  if (const char* e = std::getenv("SFB200_GZIP_CHAIN"))  // (tests: =walk takes the fallback)
    if (e[0] == 'w') tables = 1;
  auto cand_bytes = [&](uint32_t t) { return 16 * m + 4 * (m + 1) * static_cast<uint64_t>(t) + 64; };
  rc = reserve(ctx, ctx->d_gzc, cand_bytes(tables));
  if (rc == SFB200_RC_OUT_OF_MEMORY && tables > 1) {
    // no room for the jump tables: one thread walks the chain on J_0 instead — slower, same results
    cudaGetLastError();
    ctx->err.clear();
    tables = 1;
    rc = reserve(ctx, ctx->d_gzc, cand_bytes(tables));
  }
  if (rc != SFB200_RC_OK) return rc;
  a.cpos = ctx->d_gzc.as<uint64_t>();
  a.cnext = a.cpos + m;
  a.jump = reinterpret_cast<uint32_t*>(a.cnext + m);
  a.m = m;
  a.n_tables = tables;
  const unsigned cgrid = static_cast<unsigned>((m + 1 + 255) / 256);
  sfb::gzf_scatter_kernel<<<static_cast<unsigned>(tiles), sfb::GZF_THREADS, 0, st>>>(a);
  sfb::gzf_succ_kernel<<<cgrid, 256, 0, st>>>(a);
  for (uint32_t r = 0; r + 1 < tables; ++r) sfb::gzf_jump_kernel<<<cgrid, 256, 0, st>>>(a, r);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1 + tables;
  auto bind_members = [&]() {
    const uint64_t cap = gzm_members(ctx);
    a.mpos = ctx->d_gzm.as<uint64_t>();
    a.mlen = a.mpos + cap;
    a.moff = a.mlen + cap;
    a.mcap = a.moff + cap;
  };
  const unsigned skip_grid = static_cast<unsigned>(std::min<uint64_t>(tiles, static_cast<uint64_t>(ctx->sm_count) * 8));
  sfb::GzfStep h{};
  auto place = [&](uint64_t first, uint64_t count, uint64_t out_total) -> int {  // one member the host found
    h = sfb::GzfStep{};
    h.first = first;
    h.count = count;
    h.out_total = out_total;
    SFB_TRY(ctx, cudaMemcpyAsync(a.step, &h, sizeof h, cudaMemcpyHostToDevice, st));
    sfb::gzf_place_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(a);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 1;
    SFB_TRY(ctx, cudaMemcpyAsync(&h, a.step, sizeof h, cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaStreamSynchronize(st));
    return SFB200_RC_OK;
  };
  // ---- the walk ---------------------------------------------------------------------------------
  uint64_t pos = 0, skip = 0, members = 0, chained = 0, out_total = 0, tail_written = 0;
  uint32_t tail_status = SFB200_SUCCESS;
  bool complete = false;
  for (;;) {
    if (pos >= len) {
      complete = true;
      break;
    }
    // room for every member a chain can still bring: each candidate is on at most one chain
    rc = gzf_reserve(ctx, members + (m - chained) + 1, members, st);
    if (rc != SFB200_RC_OK) return rc;
    bind_members();
    h = sfb::GzfStep{};
    h.start = pos;
    h.skip = skip;
    h.first = members;
    h.out_total = out_total;
    h.head = h.next = len;
    SFB_TRY(ctx, cudaMemcpyAsync(a.step, &h, sizeof h, cudaMemcpyHostToDevice, st));
    auto* const head = reinterpret_cast<unsigned long long*>(&a.step->head);
    auto* const next = reinterpret_cast<unsigned long long*>(&a.step->next);
    sfb::gzf_skip_kernel<<<skip_grid, sfb::GZF_THREADS, 0, st>>>(a, &a.step->start, &a.step->skip, head);
    if (tables == 1) {
      sfb::gzf_walk_kernel<<<1, 1, 0, st>>>(a);
    } else {
      sfb::gzf_chain_kernel<<<1, 1, 0, st>>>(a);
      sfb::gzf_expand_kernel<<<cgrid, 256, 0, st>>>(a);
      ctx->launches += 1;
    }
    sfb::gzf_place_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(a);
    sfb::gzf_skip_kernel<<<skip_grid, sfb::GZF_THREADS, 0, st>>>(a, &a.step->stop, &a.step->count, next);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 4;
    SFB_TRY(ctx, cudaMemcpyAsync(&h, a.step, sizeof h, cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaStreamSynchronize(st));
    members += h.count;
    chained += h.count;
    out_total = h.out_total;
    if (h.count) {  // continue behind the members (and the zero padding behind them)
      pos = h.next;
      skip = 1;
      continue;
    }
    const uint64_t q = h.head;
    if (q >= len) {  // only padding is left
      complete = true;
      break;
    }
    if (!decode) break;  // a member without the BGZF field (or not a member at all) ends discovery
    // ---- a plain member at q: its header ---------------------------------------------------------
    uint64_t hp[16] = {q, len - q};
    SFB_TRY(ctx, cudaMemcpyAsync(pm, hp, 16, cudaMemcpyHostToDevice, st));
    sfb::ContainerArgs c{};
    c.src_base = src;
    c.src_off = pm + 0;
    c.src_len = pm + 1;
    c.container = sfb::CT_GZIP;
    c.n = 1;
    c.pay_off = pm + 2;
    c.pay_len = pm + 3;
    c.kind = reinterpret_cast<uint32_t*>(pm + 4);
    c.expect = c.kind + 1;
    c.isize = c.kind + 2;
    sfb::container_parse_kernel<<<1, 128, 0, st>>>(c);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 1;
    SFB_TRY(ctx, cudaMemcpyAsync(hp, pm, 6 * 8, cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaStreamSynchronize(st));
    if (static_cast<uint32_t>(hp[4]) == sfb::CT_BAD) {  // not a gzip member, or its header is cut short
      tail_status = sfb::ST_BAD_CONTAINER;
      break;
    }
    // ---- its payload, decoded over the rest of the file into its place in dst --------------------
    const uint64_t pay = hp[2];
    const uint64_t off = std::min(out_total, dst_cap), room = dst_cap - off;
    uint64_t pr[14] = {pay, std::min(len - pay, kGzfMaxLen), 0, 0, 0, 0,
                       0 /* dst_off */, std::min(room, kGzfMaxLen), 0 /* written */, 0, 0, 0, 0 /* blk_end */,
                       SFB200_ERROR /* status */};
    SFB_TRY(ctx, cudaMemcpyAsync(pm, pr, sizeof pr, cudaMemcpyHostToDevice, st));
    Resume rs;  // (not a continued decode: the route is chosen as for any single stream)
    rs.blk_end = pm + 11;
    rs.end = true;
    rc = batch_device_impl(ctx, src, pm + 0, pm + 1, dst + off, pr[7], pm + 6, pm + 7, reinterpret_cast<uint8_t*>(pm + 13),
                           pm + 8, 1, st, &rs);
    if (rc != SFB200_RC_OK) return rc;
    SFB_TRY(ctx, cudaMemcpyAsync(pr, pm, sizeof pr, cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaStreamSynchronize(st));
    const uint8_t pst = static_cast<uint8_t>(pr[13] & 0xffu);
    if (pst != SFB200_SUCCESS) {  // the payload's own status; what it produced counts
      tail_status = pst;
      tail_written = pr[8];
      break;
    }
    const uint64_t end = pay + (pr[11] + 7) / 8;  // the trailer starts at the byte behind the final block
    if (end + 8 > len) {                          // the file ends inside the trailer
      tail_status = sfb::ST_BAD_CONTAINER;
      break;
    }
    rc = gzf_reserve(ctx, members + 1, members, st);
    if (rc != SFB200_RC_OK) return rc;
    bind_members();
    const uint64_t ml[2] = {q, end + 8 - q};
    SFB_TRY(ctx, cudaMemcpyAsync(a.mpos + members, &ml[0], 8, cudaMemcpyHostToDevice, st));
    SFB_TRY(ctx, cudaMemcpyAsync(a.mlen + members, &ml[1], 8, cudaMemcpyHostToDevice, st));
    rc = place(members, 1, out_total);
    if (rc != SFB200_RC_OK) return rc;
    out_total = h.out_total;
    ++members;
    pos = end + 8;
    skip = 1;
  }
  res->members = members;
  res->size = out_total;
  res->complete = complete;
  if (!decode) return SFB200_RC_OK;
  // ---- the members side by side, then the file's result ------------------------------------------
  uint8_t* const m_status = ctx->d_gzm.p + 40 * gzm_members(ctx);
  uint64_t* const m_written = a.mcap + gzm_members(ctx);
  if (members) {
    rc = sfb200_decompress_container_batch_device(ctx, SFB200_CONTAINER_GZIP, src, a.mpos, a.mlen, dst, dst_cap, a.moff,
                                                  a.mcap, m_status, m_written, members, st);
    if (rc != SFB200_RC_OK) return rc;
  }
  sfb::gzf_result_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(a, m_status, m_written, members, tail_status, tail_written,
                                                              d_result);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  uint64_t out[2] = {0, 0};
  SFB_TRY(ctx, cudaMemcpyAsync(out, d_result, sizeof out, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  res->status = static_cast<uint8_t>(out[0]);
  res->written = out[1];
  return SFB200_RC_OK;
}
}  // namespace

extern "C" {

int sfb200_decompress_gzip_file_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, uint8_t* dst,
                                       uint64_t dst_cap, uint8_t* status, uint64_t* written, uint64_t* members,
                                       void* cuda_stream)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  GzfResult r;
  const int rc = gzip_file_impl(ctx, src, src_len, dst, dst_cap, true, static_cast<cudaStream_t>(cuda_stream), &r);
  if (rc != SFB200_RC_OK) return rc;
  *status = r.status;
  if (written) *written = r.written;
  if (members) *members = r.members;
  return SFB200_RC_OK;
}

int sfb200_decompress_gzip_file(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                                uint8_t* status, uint64_t* written, uint64_t* members)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  GzfResult r;
  const int rc = host_buffer_call(ctx, src, src_len, dst, dst_cap, written,
                                  [&](uint8_t* s, uint8_t* d, uint64_t*, uint64_t* wr) {
    const int e = gzip_file_impl(ctx, s, src_len, d, dst_cap, true, nullptr, &r);
    *wr = r.written;
    return e;
  });
  if (rc != SFB200_RC_OK) return rc;
  *status = r.status;
  if (members) *members = r.members;
  return SFB200_RC_OK;
}

int sfb200_gzip_file_size(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint64_t* size, uint64_t* members,
                          int* complete)
{
  if (!ctx || !size || (!src && src_len)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  GzfResult r;
  const int rc = host_buffer_call(ctx, src, src_len, nullptr, 0, nullptr,
                                  [&](uint8_t* s, uint8_t*, uint64_t*, uint64_t*) {
    return gzip_file_impl(ctx, s, src_len, nullptr, 0, false, nullptr, &r);
  });
  if (rc != SFB200_RC_OK) return rc;
  *size = r.size;
  if (members) *members = r.members;
  if (complete) *complete = r.complete ? 1 : 0;
  return SFB200_RC_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// zip archives (zip_file.cuh).  Listing: the EOCD (one small read-back), the CD's candidates (one
// more), then the chain, the rows and their packed offsets with one read-back at the end.
// Extraction: the split and slot kernels sort the rows; deflated entries go through the raw batch
// path — those of at least kZipLarge bytes apart from the rest, so that one large entry does not
// become one lane of the lane kernel (a lane decodes some 10 MB/s: a 1 GiB entry among 65 536 small
// ones would take the whole batch 100 s) —, each group on a window holding only its own outputs, so
// that the router's choice and its scratch follow the group and not what else dst holds; then the
// piece kernel copies stored entries (and groups decoded in scratch) and checksums every entry's
// output in pieces, and the result kernel combines the pieces' CRCs per row.
namespace {
constexpr uint64_t kZipLarge = 1ull << 20;  // DESIGN.md §3 "zip archives": the sweep that chose it
// Group 1 (entries >= kZipLarge) one call each or as one batch: a fixed cost per call and the
// single-stream rate, against one warp's rate for the largest entry.  Measured on B200 (DESIGN.md §3):
// 64 entries of 16 MiB one call each 117.9 ms, as one batch 258 ms; one 1 GiB entry alone 45.5 ms.
constexpr uint64_t kZipStage = 64ull << 20;  // host extract: produced regions this close come back in one copy
constexpr double kZipCallMs = 1.13;                     // per call, beside its bytes
constexpr double kZipStreamBpms = 23.6e6;               // bytes per ms, single-stream route
constexpr double kZipWarpBpms = 65.0e3;                 // bytes per ms, one warp per entry

struct ZipListResult {
  uint8_t status = sfb::ST_BAD_CONTAINER;
  uint64_t count = 0, total = 0;
};

int zip_list_impl(sfb200_ctx* ctx, const uint8_t* src, uint64_t len, sfb::ZipEntry* rows, uint64_t cap,
                  cudaStream_t st, ZipListResult* res)
{
  *res = ZipListResult{};
  // ZipInfo (64 B) | the chain's step (128 B) | tile counts
  int rc = reserve(ctx, ctx->d_zip, 64 + 128 + 64);
  if (rc != SFB200_RC_OK) return rc;
  sfb::zip_eocd_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(src, len, ctx->d_zip.as<sfb::ZipInfo>());
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  sfb::ZipInfo info{};
  SFB_TRY(ctx, cudaMemcpyAsync(&info, ctx->d_zip.p, sizeof info, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  if (info.status != 0) return SFB200_RC_OK;
  const uint64_t n = info.n, cd = info.cd_end - info.cd_begin;
  // ---- candidates over the CD (positions relative to its start) ------------------------------------
  sfb::GzfArgs a{};
  a.src = src + info.cd_begin;
  a.len = cd;
  a.dst_cap = ~0ull;
  const uint64_t tile = static_cast<uint64_t>(sfb::GZF_THREADS) * sfb::GZF_BYTES;
  const uint64_t tiles = cd ? (cd + (reinterpret_cast<uintptr_t>(a.src) & 15u) + tile - 1) / tile : 0;
  rc = reserve(ctx, ctx->d_zip, 64 + 128 + 8 * (tiles + 1), 64);
  if (rc != SFB200_RC_OK) return rc;
  sfb::ZipInfo* const d_info = ctx->d_zip.as<sfb::ZipInfo>();
  a.step = reinterpret_cast<sfb::GzfStep*>(ctx->d_zip.p + 64);
  a.tile_count = reinterpret_cast<uint64_t*>(ctx->d_zip.p + 192);
  uint64_t m = 0;
  if (tiles) {
    sfb::zip_count_kernel<<<static_cast<unsigned>(tiles), sfb::GZF_THREADS, 0, st>>>(a);
    sfb::gzf_exscan_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(a.tile_count, tiles);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 2;
    SFB_TRY(ctx, cudaMemcpyAsync(&m, a.tile_count + tiles, 8, cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaStreamSynchronize(st));
  }
  if (n > m) return SFB200_RC_OK;  // fewer records than the EOCD counts
  if (m >= 0xffffffffull) {         // (candidate indices are 32-bit: a CD of > 180 GiB)
    ctx->err = "zip archive: more than 2^32 - 2 central directory record candidates";
    return SFB200_RC_BAD_ARGUMENT;
  }
  uint32_t tables = 1;
  while ((1ull << tables) < m + 1) ++tables;
  if (const char* e = std::getenv("SFB200_GZIP_CHAIN"))  // (tests: =walk takes the fallback)
    if (e[0] == 'w') tables = 1;
  auto cand_bytes = [&](uint32_t t) { return 16 * m + 4 * (m + 1) * static_cast<uint64_t>(t) + 64; };
  rc = reserve(ctx, ctx->d_gzc, cand_bytes(tables));
  if (rc == SFB200_RC_OUT_OF_MEMORY && tables > 1) {  // one thread walks the chain instead
    cudaGetLastError();
    ctx->err.clear();
    tables = 1;
    rc = reserve(ctx, ctx->d_gzc, cand_bytes(tables));
  }
  if (rc != SFB200_RC_OK) return rc;
  a.cpos = ctx->d_gzc.as<uint64_t>();
  a.cnext = a.cpos + m;
  a.jump = reinterpret_cast<uint32_t*>(a.cnext + m);
  a.m = m;
  a.n_tables = tables;
  // record positions and lengths (m each), the sizes and their scan (n + 1)
  rc = reserve(ctx, ctx->d_zipl, 8 * (2 * m + n + 1) + 64);
  if (rc != SFB200_RC_OK) return rc;
  a.mpos = ctx->d_zipl.as<uint64_t>();
  a.mlen = a.mpos + m;
  uint64_t* const sizes = a.mlen + m;
  sfb::GzfStep h{};
  h.head = 0;  // the chain starts at the CD's first byte
  SFB_TRY(ctx, cudaMemcpyAsync(a.step, &h, sizeof h, cudaMemcpyHostToDevice, st));
  const unsigned cgrid = static_cast<unsigned>((m + 1 + 255) / 256);
  if (tiles) sfb::zip_scatter_kernel<<<static_cast<unsigned>(tiles), sfb::GZF_THREADS, 0, st>>>(a);
  sfb::gzf_succ_kernel<<<cgrid, 256, 0, st>>>(a);
  for (uint32_t r = 0; r + 1 < tables; ++r) sfb::gzf_jump_kernel<<<cgrid, 256, 0, st>>>(a, r);
  if (tables == 1) {
    sfb::gzf_walk_kernel<<<1, 1, 0, st>>>(a);
  } else {
    sfb::gzf_chain_kernel<<<1, 1, 0, st>>>(a);
    sfb::gzf_expand_kernel<<<cgrid, 256, 0, st>>>(a);
    ctx->launches += 1;
  }
  ctx->launches += (tiles ? 1 : 0) + tables + 1;
  // ---- the rows ----------------------------------------------------------------------------------
  sfb::ZipArgs z{};
  z.src = src;
  z.len = len;
  z.info = d_info;
  z.step = a.step;
  z.mpos = a.mpos;
  z.rows = rows;
  z.cap = cap;
  z.size = sizes;
  if (n) sfb::zip_entry_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(z);
  sfb::gzf_exscan_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(sizes, n);
  const uint64_t shown = std::min(n, cap);
  if (shown) sfb::zip_offsets_kernel<<<static_cast<unsigned>((shown + 255) / 256), 256, 0, st>>>(z);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1 + (n ? 1 : 0) + (shown ? 1 : 0);
  uint64_t total = 0;
  SFB_TRY(ctx, cudaMemcpyAsync(&h, a.step, sizeof h, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaMemcpyAsync(&total, sizes + n, 8, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  if (h.count != n || h.stop != cd) return SFB200_RC_OK;  // the records do not fill the CD as counted
  res->status = SFB200_SUCCESS;
  res->count = n;
  res->total = total;
  return SFB200_RC_OK;
}

int zip_extract_impl(sfb200_ctx* ctx, const uint8_t* src, uint64_t len, sfb::ZipEntry* rows, uint64_t n, uint8_t* dst,
                     uint64_t dst_cap, cudaStream_t st)
{
  if (n == 0) return SFB200_RC_OK;
  if (n >= 0xffffffffull) return SFB200_RC_BAD_ARGUMENT;  // (decoder slots are 32-bit)
  // six u64 arrays of the decoder, piece counts and four group columns (n + 1 each), five span words
  // | slots (u32) | kinds, decoder statuses (u8)
  const uint64_t words = 6 * n + 5 * (n + 1) + 5;
  int rc = reserve(ctx, ctx->d_zipx, 8 * words + 4 * n + 2 * n + 64);
  if (rc != SFB200_RC_OK) return rc;
  sfb::ZipExArgs x{};
  x.src = src;
  x.len = len;
  x.rows = rows;
  x.n = n;
  x.dst = dst;
  x.dst_cap = dst_cap;
  x.large = kZipLarge;
  x.d_off = ctx->d_zipx.as<uint64_t>();
  x.d_len = x.d_off + n;
  x.d_pos = x.d_len + n;
  x.d_room = x.d_pos + n;
  x.d_written = x.d_room + n;
  x.d_dst = x.d_written + n;
  x.pieces = x.d_dst + n;
  x.group = x.pieces + n + 1;
  x.span = reinterpret_cast<unsigned long long*>(x.group + 4 * (n + 1));
  x.slot = reinterpret_cast<uint32_t*>(x.span + 5);
  x.kind = reinterpret_cast<uint8_t*>(x.slot + n);
  x.d_status = x.kind + n;
  const unsigned long long span0[5] = {~0ull, 0, ~0ull, 0, 0};
  SFB_TRY(ctx, cudaMemcpyAsync(x.span, span0, sizeof span0, cudaMemcpyHostToDevice, st));
  const unsigned rgrid = static_cast<unsigned>((n + 255) / 256);
  sfb::zip_split_kernel<<<rgrid, 256, 0, st>>>(x);
  sfb::gzf_exscan_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(x.pieces, n);
  for (int c = 0; c < 4; ++c) sfb::gzf_exscan_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(x.group + c * (n + 1), n);
  sfb::zip_slot_kernel<<<rgrid, 256, 0, st>>>(x);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 7;
  uint64_t h[5], sp[5];  // g0 count, g0 bytes, g1 count, g1 bytes, pieces | spans, largest g1 room
  for (int c = 0; c < 4; ++c)
    SFB_TRY(ctx, cudaMemcpyAsync(h + c, x.group + c * (n + 1) + n, 8, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaMemcpyAsync(h + 4, x.pieces + n, 8, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaMemcpyAsync(sp, x.span, sizeof sp, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  const uint64_t cnt[2] = {h[0], h[2]}, bytes[2] = {h[1], h[3]}, pieces = h[4];
  // Group 1 one entry per call (each on its own window, on the single-stream route) or as one batch
  // (a warp per entry): the batch costs about its largest entry at one warp's rate, the calls a fixed
  // cost each plus their bytes at the single-stream rate (DESIGN.md §3 "zip archives", measured).
  const bool alone = cnt[1] && static_cast<double>(cnt[1]) * kZipCallMs + static_cast<double>(bytes[1]) / kZipStreamBpms <
                                   static_cast<double>(sp[4]) / kZipWarpBpms;
  // each batched group's window: dst where its regions lie back to back, else scratch
  bool in_place[2];
  uint64_t scratch_at[2] = {0, 0}, need = 0;
  for (int g = 0; g < 2; ++g) {
    in_place[g] = sp[2 * g] == sp[2 * g + 1];
    if (cnt[g] && !in_place[g] && !(g == 1 && alone)) {
      scratch_at[g] = need;
      need += bytes[g] + 16;
    }
  }
  if (need) {
    rc = reserve(ctx, ctx->d_zips, need);
    if (rc != SFB200_RC_OK) return rc;
  }
  for (int g = 0; g < 2; ++g) {
    if (!cnt[g] || (g == 1 && alone)) continue;
    const uint64_t b = g ? cnt[0] : 0;
    uint8_t* const win = in_place[g] ? dst + (sp[2 * g] - sfb::ZIP_BIAS) : ctx->d_zips.p + scratch_at[g];
    if (!in_place[g]) x.scratch[g] = win;
    rc = sfb200_decompress_batch_device(ctx, src, x.d_off + b, x.d_len + b, win, bytes[g], x.d_pos + b, x.d_room + b,
                                        x.d_status + b, x.d_written + b, cnt[g], st);
    if (rc != SFB200_RC_OK) return rc;
  }
  if (alone) {  // each on its own dst window: its scratch is in proportion to its size
    std::vector<uint64_t> doff(cnt[1]), room(cnt[1]);
    SFB_TRY(ctx, cudaMemcpyAsync(doff.data(), x.d_dst + cnt[0], 8 * cnt[1], cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaMemcpyAsync(room.data(), x.d_room + cnt[0], 8 * cnt[1], cudaMemcpyDeviceToHost, st));
    SFB_TRY(ctx, cudaStreamSynchronize(st));
    uint64_t* const d_zero = reinterpret_cast<uint64_t*>(x.span);  // (read back already: a zero dst offset)
    SFB_TRY(ctx, cudaMemsetAsync(d_zero, 0, 8, st));
    for (uint64_t j = 0, i = cnt[0]; j < cnt[1]; ++j, ++i) {
      rc = sfb200_decompress_batch_device(ctx, src, x.d_off + i, x.d_len + i, dst + doff[j], room[j], d_zero,
                                          x.d_room + i, x.d_status + i, x.d_written + i, 1, st);
      if (rc != SFB200_RC_OK) return rc;
    }
  }
  // ---- stored copies, copies out of scratch, CRCs, results ---------------------------------------
  rc = reserve(ctx, ctx->d_zipc, 4 * pieces + 64);
  if (rc != SFB200_RC_OK) return rc;
  x.pcrc = ctx->d_zipc.as<uint32_t>();
  if (pieces) {
    const uint64_t want = (pieces * 32 + sfb::CHECK_THREADS - 1) / sfb::CHECK_THREADS;
    const uint64_t resident = static_cast<uint64_t>(ctx->sm_count);  // (one block per SM: 128 KiB of tables)
    sfb::zip_piece_kernel<<<grid_size(want, resident), sfb::CHECK_THREADS, sfb::CHECK_SMEM_BYTES, st>>>(x);
    ctx->launches += 1;
  }
  sfb::zip_result_kernel<<<rgrid, 256, 0, st>>>(x);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  return SFB200_RC_OK;
}
}  // namespace

extern "C" {

int sfb200_zip_list_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, sfb200_zip_entry* entries,
                           uint64_t cap, uint8_t* status, uint64_t* count, uint64_t* total_size, void* cuda_stream)
{
  static_assert(sizeof(sfb200_zip_entry) == sizeof(sfb::ZipEntry), "one row layout");
  if (!ctx || !status || !count || (!src && src_len) || (!entries && cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  ZipListResult r;
  const int rc = zip_list_impl(ctx, src, src_len, reinterpret_cast<sfb::ZipEntry*>(entries), cap,
                               static_cast<cudaStream_t>(cuda_stream), &r);
  if (rc != SFB200_RC_OK) return rc;
  *status = r.status;
  *count = r.count;
  if (total_size) *total_size = r.total;
  return SFB200_RC_OK;
}

int sfb200_zip_list(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, sfb200_zip_entry* entries, uint64_t cap,
                    uint8_t* status, uint64_t* count, uint64_t* total_size)
{
  if (!ctx || !status || !count || (!src && src_len) || (!entries && cap) || cap > (1ull << 40))
    return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  ZipListResult r;
  const int rc = host_buffer_call(ctx, src, src_len, reinterpret_cast<uint8_t*>(entries), cap * sizeof(sfb200_zip_entry),
                                  nullptr, [&](uint8_t* s, uint8_t* d, uint64_t*, uint64_t* wr) {
    const int e = zip_list_impl(ctx, s, src_len, reinterpret_cast<sfb::ZipEntry*>(d), cap, nullptr, &r);
    *wr = std::min(r.count, cap) * sizeof(sfb200_zip_entry);
    return e;
  });
  if (rc != SFB200_RC_OK) return rc;
  *status = r.status;
  *count = r.count;
  if (total_size) *total_size = r.total;
  return SFB200_RC_OK;
}

int sfb200_zip_extract_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, sfb200_zip_entry* entries,
                              uint64_t n, uint8_t* dst, uint64_t dst_cap, void* cuda_stream)
{
  if (!ctx || (!src && src_len) || (!entries && n) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  return zip_extract_impl(ctx, src, src_len, reinterpret_cast<sfb::ZipEntry*>(entries), n, dst, dst_cap,
                          static_cast<cudaStream_t>(cuda_stream));
}

int sfb200_zip_extract(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, sfb200_zip_entry* entries, uint64_t n,
                       uint8_t* dst, size_t dst_cap)
{
  if (!ctx || (!src && src_len) || (!entries && n) || (!dst && dst_cap) || n > (1ull << 40))
    return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  return host_buffer_call(ctx, src, src_len, dst, dst_cap, nullptr,
                          [&](uint8_t* s, uint8_t* d, uint64_t*, uint64_t* wr) -> int {
    *wr = 0;  // (the rows' regions come back below, not a prefix of dst)
    const uint64_t bytes = n * sizeof(sfb200_zip_entry);
    int rc = reserve(ctx, ctx->d_zipl, bytes + 64);
    if (rc != SFB200_RC_OK) return rc;
    auto* const rows = ctx->d_zipl.as<sfb::ZipEntry>();
    if (n) SFB_TRY(ctx, cudaMemcpyAsync(rows, entries, bytes, cudaMemcpyHostToDevice, nullptr));
    rc = zip_extract_impl(ctx, s, src_len, rows, n, d, dst_cap, nullptr);
    if (rc != SFB200_RC_OK) return rc;
    if (n) SFB_TRY(ctx, cudaMemcpy(entries, rows, bytes, cudaMemcpyDeviceToHost));
    // only the bytes produced: the rows' [dst_off, + written) in dst order, adjacent ones merged into
    // runs; runs that lie within kZipStage bytes of each other come back in one copy through a host
    // staging buffer, so that a scattered subset costs one copy per kZipStage bytes, not one per row
    std::vector<std::pair<uint64_t, uint64_t>> runs;  // [lo, hi)
    {
      std::vector<uint64_t> order;
      order.reserve(n);
      for (uint64_t i = 0; i < n; ++i)
        if (entries[i].written) order.push_back(i);
      auto start = [&](uint64_t i) { return std::min<uint64_t>(entries[i].dst_off, dst_cap); };
      std::sort(order.begin(), order.end(), [&](uint64_t p, uint64_t q) { return start(p) < start(q); });
      for (const uint64_t i : order) {
        const uint64_t lo = start(i), hi = std::min<uint64_t>(lo + entries[i].written, dst_cap);
        if (!runs.empty() && lo <= runs.back().second) runs.back().second = std::max(runs.back().second, hi);
        else runs.emplace_back(lo, hi);
      }
    }
    std::vector<uint8_t> stage;
    for (size_t k = 0; k < runs.size();) {
      size_t e = k + 1;  // runs [k, e) share one staged copy
      while (e < runs.size() && runs[e].second - runs[k].first <= kZipStage) ++e;
      if (e == k + 1) {
        SFB_TRY(ctx, cudaMemcpy(dst + runs[k].first, d + runs[k].first, runs[k].second - runs[k].first,
                                cudaMemcpyDeviceToHost));
      } else {
        const uint64_t lo = runs[k].first, hi = runs[e - 1].second;
        stage.resize(hi - lo);
        SFB_TRY(ctx, cudaMemcpy(stage.data(), d + lo, hi - lo, cudaMemcpyDeviceToHost));
        for (size_t j = k; j < e; ++j)
          std::memcpy(dst + runs[j].first, stage.data() + (runs[j].first - lo), runs[j].second - runs[j].first);
      }
      k = e;
    }
    return SFB200_RC_OK;
  });
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Writing zlib, gzip and BGZF (container_write.cuh): the compressor writes the payloads, the seal
// kernel adds header and trailer with the checksum of the source bytes, all on the device.
namespace {
int seal_launch(sfb200_ctx* ctx, const sfb::SealArgs& s, cudaStream_t st)
{
  const uint64_t want = (s.n * 32 + sfb::CHECK_THREADS - 1) / sfb::CHECK_THREADS;
  const uint64_t resident = static_cast<uint64_t>(ctx->sm_count);  // (one block per SM: 128 KiB of tables)
  sfb::container_seal_kernel<<<grid_size(want, resident), sfb::CHECK_THREADS, sfb::CHECK_SMEM_BYTES, st>>>(s);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  return SFB200_RC_OK;
}
}  // namespace

extern "C" {

uint64_t sfb200_compress_container_bound(int container, uint64_t src_len)
{
  const uint64_t raw = sfb200_compress_bound(src_len);
  switch (container) {
    case SFB200_CONTAINER_RAW: return raw;
    case SFB200_CONTAINER_ZLIB: return raw + 6;
    case SFB200_CONTAINER_GZIP: return raw + 18;
    default: return 0;
  }
}

int sfb200_compress_container_batch_device(sfb200_ctx* ctx, int container, const uint8_t* src_base,
                                           const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base,
                                           const uint64_t* dst_off, const uint64_t* dst_cap, uint8_t* status,
                                           uint64_t* written, uint64_t n, void* cuda_stream)
{
  if (!ctx || container < SFB200_CONTAINER_RAW || container > SFB200_CONTAINER_GZIP) return SFB200_RC_BAD_ARGUMENT;
  if (container == SFB200_CONTAINER_RAW)
    return sfb200_compress_batch_device(ctx, src_base, src_off, src_len, dst_base, dst_off, dst_cap, status, written, n,
                                        cuda_stream);
  if (n == 0) return SFB200_RC_OK;
  if (!src_off || !src_len || !dst_off || !dst_cap || !status || !written) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  int rc = reserve(ctx, ctx->d_wrap, n * 16 + 64);
  if (rc != SFB200_RC_OK) return rc;
  uint64_t* const pay_off = ctx->d_wrap.as<uint64_t>();
  uint64_t* const pay_cap = pay_off + n;
  sfb::container_frame_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(
      static_cast<uint32_t>(container), dst_off, dst_cap, pay_off, pay_cap, n);
  SFB_TRY(ctx, cudaGetLastError());
  ctx->launches += 1;
  rc = sfb200_compress_batch_device(ctx, src_base, src_off, src_len, dst_base, pay_off, pay_cap, status, written, n,
                                    cuda_stream);
  if (rc != SFB200_RC_OK) return rc;
  sfb::SealArgs s{};
  s.src_base = src_base;
  s.src_off = src_off;
  s.src_len = src_len;
  s.dst_base = dst_base;
  s.dst_off = dst_off;
  s.dst_cap = dst_cap;
  s.status = status;
  s.written = written;
  s.n = n;
  s.container = static_cast<uint32_t>(container);
  return seal_launch(ctx, s, st);
}

int sfb200_compress_container(sfb200_ctx* ctx, int container, const uint8_t* src, size_t src_len, uint8_t* dst,
                              size_t dst_cap, uint8_t* status, uint64_t* written)
{
  if (!ctx || !status || !written || (src_len && !src) || (dst_cap && !dst)) return SFB200_RC_BAD_ARGUMENT;
  if (container < SFB200_CONTAINER_RAW || container > SFB200_CONTAINER_GZIP) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  return host_buffer_call(ctx, src, src_len, dst, dst_cap, written,
                          [&](uint8_t* s, uint8_t* d, uint64_t* m, uint64_t* wr) {
    const int rc = sfb200_compress_container_batch_device(ctx, container, s, m, m + 1, d, m + 2, m + 3,
                                                          reinterpret_cast<uint8_t*>(m + 5), m + 4, 1, nullptr);
    return rc != SFB200_RC_OK ? rc : read_meta(ctx, m, wr, status);
  });
}

uint64_t sfb200_compress_bgzf_bound(uint64_t src_len)
{
  return (src_len + sfb::BGZF_PIECE - 1) / sfb::BGZF_PIECE * (sfb::BGZF_PIECE + 5 + sfb::BGZF_FRAME) + sfb::BGZF_EOF_BYTES;
}

int sfb200_compress_bgzf_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, uint8_t* dst, uint64_t dst_cap,
                                uint8_t* status, uint64_t* written, uint64_t* members, void* cuda_stream)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  const uint64_t pieces = (src_len + sfb::BGZF_PIECE - 1) / sfb::BGZF_PIECE;
  uint64_t budget_mb = 8192;  // scratch of a round: 64 KiB per piece (SFB200_BGZF_SCRATCH_MB)
  if (const char* e = std::getenv("SFB200_BGZF_SCRATCH_MB")) budget_mb = std::max<long long>(1, std::atoll(e));
  const uint64_t slots = std::max<uint64_t>(1, (budget_mb << 20) / sfb::BGZF_SLOT);
  const uint64_t r = std::max<uint64_t>(1, std::min(pieces, slots));
  // slots (r x 64 KiB) | src_off, src_len, dst_off, dst_cap (r x u64 each) | written (r + 1) | state (4) | status (r)
  const uint64_t meta_at = r * sfb::BGZF_SLOT;
  int rc = reserve(ctx, ctx->d_bgzf, meta_at + 8 * (5 * r + 5) + r + 64);
  if (rc != SFB200_RC_OK) return rc;
  uint8_t* const slot = ctx->d_bgzf.p;
  uint64_t* const so = reinterpret_cast<uint64_t*>(ctx->d_bgzf.p + meta_at);
  uint64_t* const sl = so + r;
  uint64_t* const dof = sl + r;
  uint64_t* const dc = dof + r;
  uint64_t* const wr = dc + r;
  uint64_t* const state = wr + r + 1;
  uint8_t* const pst = reinterpret_cast<uint8_t*>(state + 4);
  SFB_TRY(ctx, cudaMemsetAsync(state, 0, 4 * sizeof(uint64_t), st));
  sfb::SealArgs s{};
  s.src_base = src;
  s.src_off = so;
  s.src_len = sl;
  s.dst_base = dst;
  s.status = pst;
  s.written = wr;
  s.container = sfb::CT_BGZF;
  s.slots = slot;
  s.state = state;
  s.dst_bytes = dst_cap;
  uint64_t first = 0;
  do {  // one round per r pieces (an empty input: one round without pieces, for the EOF marker)
    const uint64_t n = std::min(r, pieces - first);
    const bool last = first + n >= pieces;
    if (n) {
      sfb::bgzf_split_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(src_len, sfb::BGZF_PIECE, first, n,
                                                                                   so, sl, dof, dc);
      SFB_TRY(ctx, cudaGetLastError());
      ctx->launches += 1;
      rc = sfb200_compress_batch_device(ctx, src, so, sl, slot, dof, dc, pst, wr, n, st);
      if (rc != SFB200_RC_OK) return rc;
      sfb::gzf_exscan_kernel<<<1, sfb::GZF_SCAN_THREADS, 0, st>>>(wr, n);
      SFB_TRY(ctx, cudaGetLastError());
      ctx->launches += 1;
      s.n = n;
      rc = seal_launch(ctx, s, st);
      if (rc != SFB200_RC_OK) return rc;
    }
    sfb::bgzf_advance_kernel<<<1, 1, 0, st>>>(state, wr, n, dst, dst_cap, last ? 1 : 0);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 1;
    first += n;
  } while (first < pieces);
  uint64_t res[2] = {0, 0};
  SFB_TRY(ctx, cudaMemcpyAsync(res, state + 1, sizeof res, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  *status = static_cast<uint8_t>(res[0]);
  if (written) *written = res[1];
  if (members) *members = res[0] == SFB200_SUCCESS ? pieces + 1 : 0;
  return SFB200_RC_OK;
}

int sfb200_compress_bgzf(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                         uint8_t* status, uint64_t* written, uint64_t* members)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  return host_buffer_call(ctx, src, src_len, dst, dst_cap, written,
                          [&](uint8_t* s, uint8_t* d, uint64_t*, uint64_t* wr) {
    return sfb200_compress_bgzf_device(ctx, s, src_len, d, dst_cap, status, wr, members, nullptr);
  });
}


// One buffer as one raw-DEFLATE / zlib / gzip stream (compress_parallel.cuh): BGZF's pieces and rounds,
// the blocks joined at bit granularity.
//
// Bound: a piece of L bytes compressed as a Huffman block is kept only when ceil(bits / 8) <= L + 5,
// so it takes at most 8 (L + 5) bits.  A stored piece takes align8(B + 3) - B + 32 + 8 L bits, at most
// 10 + 32 + 8 L = 8 (L + 5) + 2 (when it starts at bit phase 6).  Over p pieces of n bytes in all that is
// at most 8 n + 42 p bits, which with the zero padding of the last byte is n + 5 p + ceil(2 p / 8) <=
// n + 6 p bytes, plus header and trailer.
uint64_t sfb200_compress_parallel_bound(int container, uint64_t src_len)
{
  if (container < SFB200_CONTAINER_RAW || container > SFB200_CONTAINER_GZIP) return 0;
  const uint64_t frame = container == SFB200_CONTAINER_ZLIB ? 6 : container == SFB200_CONTAINER_GZIP ? 18 : 0;
  const uint64_t pieces = std::max<uint64_t>(1, (src_len + sfb::BGZF_PIECE - 1) / sfb::BGZF_PIECE);
  return frame + src_len + 6 * pieces;
}

int sfb200_compress_parallel_device(sfb200_ctx* ctx, int container, const uint8_t* src, uint64_t src_len,
                                    uint8_t* dst, uint64_t dst_cap, uint8_t* status, uint64_t* written,
                                    void* cuda_stream)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  if (container < SFB200_CONTAINER_RAW || container > SFB200_CONTAINER_GZIP) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  const uint64_t pieces = std::max<uint64_t>(1, (src_len + sfb::BGZF_PIECE - 1) / sfb::BGZF_PIECE);
  uint64_t budget_mb = 8192;  // BGZF's scratch budget: 64 KiB per piece of a round (SFB200_BGZF_SCRATCH_MB)
  if (const char* e = std::getenv("SFB200_BGZF_SCRATCH_MB")) budget_mb = std::max<long long>(1, std::atoll(e));
  const uint64_t slots = std::max<uint64_t>(1, (budget_mb << 20) / sfb::BGZF_SLOT);
  const uint64_t r = std::min(pieces, slots);
  // slots (r x 64 KiB) | src_off, src_len, dst_off, dst_cap (r x u64 each) | pos (r + 1) | state |
  // sums (r x u32) | kinds (r)
  const uint64_t meta_at = r * sfb::BGZF_SLOT;
  int rc = reserve(ctx, ctx->d_bgzf, meta_at + 8 * (5 * r + 1 + sfb::PAR_STATE_WORDS) + 5 * r + 64);
  if (rc != SFB200_RC_OK) return rc;
  uint64_t* const so = reinterpret_cast<uint64_t*>(ctx->d_bgzf.p + meta_at);
  uint64_t* const sl = so + r;
  uint64_t* const dof = sl + r;
  uint64_t* const dc = dof + r;
  uint64_t* const pos = dc + r;
  uint64_t* const state = pos + r + 1;
  uint32_t* const sums = reinterpret_cast<uint32_t*>(state + sfb::PAR_STATE_WORDS);
  uint8_t* const kinds = reinterpret_cast<uint8_t*>(sums + r);
  const uint64_t hb = container == SFB200_CONTAINER_ZLIB ? 2 : container == SFB200_CONTAINER_GZIP ? 10 : 0;
  uint64_t init[sfb::PAR_STATE_WORDS] = {};
  init[sfb::PAR_BASE] = 8 * hb;
  init[sfb::PAR_SUM] = container == SFB200_CONTAINER_ZLIB ? 1 : 0;  // the Adler-32 / CRC-32 of nothing
  SFB_TRY(ctx, cudaMemcpyAsync(state, init, sizeof init, cudaMemcpyHostToDevice, st));
  sfb::CompressArgs c;
  c.src_base = src;
  c.src_off = so;
  c.src_len = sl;
  c.dst_base = ctx->d_bgzf.p;
  c.dst_off = dof;
  c.dst_cap = dc;
  c.status = kinds;
  c.written = pos;
  c.counter = ctx->d_counter.as<unsigned long long>();
  c.fixed_only = 0;
  sfb::ParArgs a{};
  a.src = src;
  a.src_off = so;
  a.src_len = sl;
  a.slots = ctx->d_bgzf.p;
  a.kind = kinds;
  a.pos = pos;
  a.sum = sums;
  a.dst = dst;
  a.dst_cap = dst_cap;
  a.state = state;
  a.container = static_cast<uint32_t>(container);
  const uint64_t resident = static_cast<uint64_t>(ctx->sm_count) * static_cast<uint64_t>(ctx->compress_ctas_per_sm);
  uint64_t first = 0;
  do {  // one round per r pieces (an empty input is one empty piece)
    const uint64_t n = std::min(r, pieces - first);
    const bool last = first + n >= pieces;
    sfb::bgzf_split_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(src_len, sfb::BGZF_PIECE, first, n,
                                                                                 so, sl, dof, dc);
    SFB_TRY(ctx, cudaGetLastError());
    SFB_TRY(ctx, cudaMemsetAsync(ctx->d_counter.p, 0, sizeof(unsigned long long), st));
    c.n = n;
    a.n = n;
    a.last = last ? n - 1 : ~0ull;
    const uint64_t want = (n + sfb::CMP_WARPS - 1) / sfb::CMP_WARPS;
    sfb::deflate_compress_pieces_kernel<<<grid_size(want, resident), sfb::CMP_WARPS * 32, sfb::CMP_SMEM_BYTES, st>>>(
        c, a.last);
    SFB_TRY(ctx, cudaGetLastError());
    sfb::par_scan_kernel<<<1, sfb::PAR_THREADS, 0, st>>>(a);
    SFB_TRY(ctx, cudaGetLastError());
    const uint64_t swant = (n * 32 + sfb::CHECK_THREADS - 1) / sfb::CHECK_THREADS;
    const uint64_t sresident = static_cast<uint64_t>(ctx->sm_count);  // (one block per SM: 128 KiB of tables)
    sfb::par_stitch_kernel<<<grid_size(swant, sresident), sfb::CHECK_THREADS, sfb::CHECK_SMEM_BYTES, st>>>(a);
    SFB_TRY(ctx, cudaGetLastError());
    sfb::par_advance_kernel<<<1, sfb::PAR_THREADS, 0, st>>>(a, last ? 1 : 0);
    SFB_TRY(ctx, cudaGetLastError());
    ctx->launches += 5;
    first += n;
  } while (first < pieces);
  uint64_t res[2] = {0, 0};
  SFB_TRY(ctx, cudaMemcpyAsync(res, state + sfb::PAR_STATUS, sizeof res, cudaMemcpyDeviceToHost, st));
  SFB_TRY(ctx, cudaStreamSynchronize(st));
  *status = static_cast<uint8_t>(res[0]);
  if (written) *written = res[1];
  return SFB200_RC_OK;
}

int sfb200_compress_parallel(sfb200_ctx* ctx, int container, const uint8_t* src, size_t src_len, uint8_t* dst,
                             size_t dst_cap, uint8_t* status, uint64_t* written)
{
  if (!ctx || !status || (!src && src_len) || (!dst && dst_cap)) return SFB200_RC_BAD_ARGUMENT;
  if (container < SFB200_CONTAINER_RAW || container > SFB200_CONTAINER_GZIP) return SFB200_RC_BAD_ARGUMENT;
  SFB_ENTER(ctx);
  return host_buffer_call(ctx, src, src_len, dst, dst_cap, written,
                          [&](uint8_t* s, uint8_t* d, uint64_t*, uint64_t* wr) {
    return sfb200_compress_parallel_device(ctx, container, s, src_len, d, dst_cap, status, wr, nullptr);
  });
}

}  // extern "C"
