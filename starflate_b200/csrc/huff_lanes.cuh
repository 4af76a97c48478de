// Pass 1 of the batched raw-DEFLATE decoder for sm_100a: the Huffman layer, ONE LANE PER STREAM.
//
// Replaces the reference's symbol loop decompress_block_huffman (src/decompress.cpp:197-242)
// together with read_header, the stored-block branch and the dynamic table decode (all via
// deflate_lane.cuh) — everything of decompress() except the bytes a back-reference copies, which
// pass 2 (lz_warp.cuh) fills in.  Per-stream status and `written` are final after this pass.
//
// Why a lane and not a warp per stream: Huffman decode of one stream is a serial dependency
// chain (bit window -> LUT -> code length -> next window).  A warp per stream spends one issue
// slot per instruction on ONE token; a lane per stream retires up to 32 tokens per issued
// instruction.  Why the LZ77 copy is NOT done here: with 32 streams per warp and 8 warps per SM
// there are ~38k streams in flight, whose 32 KiB windows (1.2 GB) cannot stay in the 126 MB L2;
// the one-pass lane kernel of earlier revisions spent its time waiting on DRAM for match
// sources (ncu: 6.4 of 11 stall cycles per issue on long scoreboard, 26 GB read for 0.75 GB of
// input).  The Huffman layer never reads the output, so this pass has no such dependency.
//
// Output of this pass, written IN PLACE into each stream's dst region (no token buffer, so the
// scratch memory is bounded by 1 bit per dst byte whatever the data):
//   * literal bytes and stored-block payload at their final positions;
//   * for a match (length L, distance D) that starts at output position p: a 3-byte descriptor
//     at dst[p..p+3):  byte0 = L - 3, byte1..2 = (D - 1) little endian  (L >= 3, so it fits);
//     dst[p+3..p+L) is left unspecified (pass 2 overwrites all of dst[p..p+L));
//   * bit (dst_off + p) of the match-head bitmap is set for every such p.
// The reference's output-side checks (distance > written -> InvalidDistance, room ->
// DstTooSmall; src/decompress.cpp:150-152,178-183) only need the output POSITION, which this
// pass tracks, so they are made here, in the reference's order.
//
// Each lane owns
//   * a register bit window (five 32-bit words, funnel-shift peeks, branch-free slide) fed from
//     a 64-byte ring in shared memory that cp.async fills 16 bytes at a time, several tokens
//     ahead of the reader (deflate_lane.cuh: BitReader),
//   * a two-level decode LUT in shared memory, interleaved so that element j of lane l sits at
//     u16 index j*32+l (lane pairs share a bank: at most 2-way conflicts on random lookups),
//   * an 8-byte write-combining register for its output window in HBM and a 32-bit
//     accumulator for its current bitmap word.
// The code lengths of the current block live in a per-lane slice of a global scratch buffer,
// which keeps the shared-memory footprint at LUT + ring: 896 B per lane -> 8 warps per SM.
// Scattered per-lane memory instructions are what bounds this pass (every lane touches its own
// 128-byte line, ~2 L1 cycles each), so the loop issues as few of them as it can: one 16-byte
// cp.async per ~9 tokens, one 8-byte store per ~1.5 tokens, one bitmap RED per 32 output bytes.
#pragma once

#include "deflate_lane.cuh"

namespace sfb {

// ---------------------------------------------------------------------------------------------
// Per-lane output window of pass 1.
// Invariant: bytes [vpos & ~7, vpos) of the output live in the low bytes of `obuf`, its higher
// bytes are zero; every byte below vpos & ~7 that pass 2 will not overwrite is in memory.
struct TokWin;
struct CountWin;
template <bool COUNT> struct WinOf { using type = TokWin; };
template <> struct WinOf<true> { using type = CountWin; };

struct TokWin {
  uint8_t* al;      // 8-byte aligned address of virtual position 0
  uint32_t lead;    // dst start within the first word (0..7): virtual position of byte 0
  uint32_t vpos;    // virtual position of the next byte to produce
  uint32_t vend;    // virtual position one past the capacity
  uint64_t obuf;
  uint64_t first;   // word 0 of an unaligned dst once the cursor has left it: its bytes before
                    // `lead` are not ours, so it is written bytewise at the end (flush_tail)
  bool first_out;   // word 0's own bytes are in memory already (publish()): flush_tail leaves them alone
  uint8_t* fbase;   // match-head bitmap, byte granular: the bits of word wv live in fbase[wv >> 3]
                    // (dst_base is 128-byte aligned, so address words and bitmap bytes line up)
  uint32_t fb;      // head bits of the open word

  __device__ __forceinline__ void open(uint8_t* dst_base, uint64_t off, uint32_t cap, uint32_t* bits)
  {
    uint8_t* d = dst_base + off;
    lead = static_cast<uint32_t>(off & 7u);
    al = d - lead;
    vpos = lead;
    vend = lead + cap;
    obuf = 0;
    first = 0;
    first_out = false;
    fbase = reinterpret_cast<uint8_t*>(bits) + ((off - lead) >> 3);
    fb = 0;
  }
  __device__ __forceinline__ void park()
  {
    al = nullptr;
    lead = vpos = vend = 0;
    obuf = first = 0;
    first_out = false;
    fbase = nullptr;
    fb = 0;
  }

  __device__ __forceinline__ uint32_t written() const { return vpos - lead; }
  __device__ __forceinline__ uint32_t room() const { return vend - vpos; }

  // merge the head bits of word wv into the bitmap with an atomic (words at the edges of a dst
  // region share their bitmap byte with the neighbouring stream)
  __device__ __forceinline__ void or_bits(uint32_t wv, uint32_t bits8) const
  {
    uint8_t* p = fbase + (wv >> 3);
    const uint32_t sh = 8u * (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(p)) & 3u);
    atomicOr(reinterpret_cast<uint32_t*>(p - (sh >> 3)), bits8 << sh);
  }

  // The one output step of a token: append the n (0..4) low bytes of `chunk` at the cursor —
  // the descriptor of a match iff `is_head` — then move the cursor `skipn` bytes further over
  // bytes pass 2 will produce (the body of a match).  A word the cursor leaves is stored whole:
  // its bytes past the appended ones all belong to the match body, so any value will do there;
  // its head bits go to the bitmap byte of that word.  No branches: predicated stores.
  // `hoff` (0 or 1): the descriptor starts that many bytes into the chunk — a literal paired with
  // the match that follows it (n <= 4 then; the caller keeps k + hoff <= 7, so the head bit stays
  // in this word).
  __device__ __forceinline__ void emit(uint32_t chunk, uint32_t n, uint32_t skipn, bool is_head, uint32_t hoff = 0u)
  {
#ifdef SFB_TRACE_EMIT
    SFB_TRACE_EMIT(vpos, chunk, n, skipn, obuf);
#endif
    const uint32_t k = vpos & 7u;
    const uint32_t sh = 8u * k;
    const uint64_t merged = obuf | (static_cast<uint64_t>(chunk) << sh);  // chunk < 2^(8n)
    const uint32_t hb = fb | (is_head ? 1u << (k + hoff) : 0u);
    const uint32_t np = vpos + n + skipn;
    const uint32_t wv = vpos & ~7u;
    const uint32_t nw = np & ~7u;
    const bool leaves = nw != wv;
    const bool spill = k + n > 8u;                         // the chunk reaches into the next word
    const uint32_t carry = chunk >> ((64u - sh) & 31u);    // ... with these bytes (sh >= 48 then)
    const bool stay = nw == wv + 8u;                       // the cursor ends in the next word
    const bool head = wv < lead;                           // word 0 of an unaligned dst
    const bool edge = head | (wv + 8u > vend);             // a word this region does not own alone
    if (leaves & !head) *reinterpret_cast<uint64_t*>(al + wv) = merged;
    if (leaves & head) first = merged;
    if (leaves & spill & !stay) *reinterpret_cast<uint64_t*>(al + wv + 8u) = carry;  // skipped past it too
    if (leaves & (hb != 0) & !edge) fbase[wv >> 3] = static_cast<uint8_t>(hb);
    if (leaves & (hb != 0) & edge) or_bits(wv, hb);
    fb = leaves ? 0u : hb;
    obuf = leaves ? ((spill & stay) ? carry : 0u) : merged;
    vpos = np;
  }

  // pending bytes of the open word -> memory, bytewise (the window stays as it is)
  __device__ __forceinline__ void spill_pending() const
  {
    const uint32_t wv = vpos & ~7u;
    uint32_t b = wv < lead ? lead : wv;
    for (; b < vpos; ++b) al[b] = static_cast<uint8_t>(obuf >> (8 * (b - wv)));
  }
  // the cursor was moved over bytes written straight to memory: re-read the open word
  __device__ __forceinline__ void jump(uint32_t n)
  {
    const uint32_t w0 = vpos & ~7u;
    const bool left0 = w0 < lead && ((vpos + n) & ~7u) != 0;  // leaving word 0
    vpos += n;
    const uint32_t wv = vpos & ~7u;
    if (wv != w0 && fb != 0) {  // head bits of the word left behind
      or_bits(w0, fb);
      fb = 0;
    }
    if (left0) {  // all of its bytes from `lead` on are in memory now: keep `first` consistent
      first = 0;
      for (uint32_t b = lead; b < 8; ++b) first |= static_cast<uint64_t>(al[b]) << (8 * b);
    }
    obuf = 0;
    for (uint32_t b = wv < lead ? lead : wv; b < vpos; ++b)
      obuf |= static_cast<uint64_t>(al[b]) << (8 * (b - wv));
  }
  // Everything below the open word is in memory — except word 0 of an unaligned dst, which is kept
  // back: before the first bytes of the stream are handed to a pass 2 that runs beside this one it
  // goes out too (pass 2 may rewrite those bytes: flush_tail must not put the old ones back).
  __device__ __forceinline__ void release_first()
  {
    if (lead != 0 && vpos >= 8u && !first_out) {
      for (uint32_t b = lead; b < 8; ++b) al[b] = static_cast<uint8_t>(first >> (8 * b));
      first_out = true;
    }
  }
  // called once, when the stream ends for any reason
  __device__ __forceinline__ void flush_tail()
  {
    spill_pending();
    if (lead != 0 && vpos >= 8u && !first_out)  // the cursor left word 0: its bytes from `lead` on are still pending
      for (uint32_t b = lead; b < 8; ++b) al[b] = static_cast<uint8_t>(first >> (8 * b));
    if (fb) or_bits(vpos & ~7u, fb);
    fb = 0;
  }
};

// The writer of the size-discovery mode (huff_lanes_kernel<C, true>): same interface, keeps only
// the position — nothing is stored, dst and the bitmap are never touched.
struct CountWin {
  uint8_t* al;
  uint32_t lead, vpos, vend;
  __device__ __forceinline__ void open(uint8_t*, uint64_t, uint32_t cap, uint32_t*)
  {
    al = nullptr;
    lead = 0;
    vpos = 0;
    vend = cap;
  }
  __device__ __forceinline__ void park()
  {
    al = nullptr;
    lead = vpos = vend = 0;
  }
  __device__ __forceinline__ uint32_t written() const { return vpos; }
  __device__ __forceinline__ uint32_t room() const { return vend - vpos; }
  __device__ __forceinline__ void emit(uint32_t, uint32_t n, uint32_t skipn, bool, uint32_t = 0u) { vpos += n + skipn; }
  __device__ __forceinline__ void spill_pending() const {}
  __device__ __forceinline__ void jump(uint32_t n) { vpos += n; }
  __device__ __forceinline__ void flush_tail() const {}
  __device__ __forceinline__ void release_first() const {}
};

__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src)
{
  const uint32_t lo = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v), src);
  const uint32_t hi = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), src);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

#ifdef SFB_CPU_EMU
constexpr uint32_t LANES = 1;   // tests/cpu_emu runs one lane per "warp"
#else
constexpr uint32_t LANES = 32;
#endif

// ---------------------------------------------------------------------------------------------
// The pass-1 kernel.  One lane per stream, 32 streams per warp, warps pull groups of 32
// consecutive streams from a global counter.
//
// Control structure (kept free of `break`s so that the warp reconverges after every stage):
//   rounds:  lanes that need a block header parse it (lock-step when several do); stored
//            blocks are then copied by the whole warp, one block at a time, coalesced; then
//   tokens:  while any lane is inside a Huffman block, every iteration each such lane decodes
//            exactly one token (literal | end of block | match) and emits it through the one
//            emit() site; lanes waiting for the next header (or finished) idle until the
//            round ends.
//
// COUNT = true is the size-discovery mode (SURVEY.md §8 f2: the reference returns no size and asks
// the caller to know it): the same decode with a writer that stores nothing and no capacity
// limit; status[i] / written[i] are what a decode into a large enough dst would return.
// END = true (a resumed decode, blk_end given): after the final block blk_end receives the bit behind
// its end-of-block code — where a gzip member's trailer starts (gzip_file.cuh) — and the output
// position.  A template parameter, so that the other instantiations keep their registers.
template <class C, bool COUNT = false, bool QUEUE = false, bool END = false>   // QUEUE: publish segments to a pass 2 that runs beside (QueueArgs)
__global__ void __launch_bounds__(C::WARPS * 32, C::CTAS)
huff_lanes_kernel(const BatchArgs a)
{
#ifdef SFB_CPU_EMU
  uint8_t* const smem = reinterpret_cast<uint8_t*>(SFB_EMU_SMEM);  // tests/cpu_emu: logic-only build
#else
  extern __shared__ __align__(16) uint8_t smem[];
#endif
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = static_cast<int>(threadIdx.x & 31u);
  const int warp = static_cast<int>(threadIdx.x >> 5);
  uint32_t* const s_dist_info = reinterpret_cast<uint32_t*>(smem + C::WARPS * C::WARP_BYTES);
  for (unsigned t = threadIdx.x; t < 32; t += blockDim.x) s_dist_info[t] = c_dist_info[t];
  __syncthreads();

  uint8_t* const warp_smem = smem + warp * C::WARP_BYTES;
  LaneMem m;
  m.lut = reinterpret_cast<uint16_t*>(warp_smem) + lane;
  m.lens = a.lens_scratch +
           (static_cast<size_t>(blockIdx.x) * C::WARPS + static_cast<size_t>(warp)) * (SCRATCH_WORDS * 32) +
           lane;
  const saddr_t lutb = to_saddr(m.lut);
  const saddr_t sdi = to_saddr(s_dist_info);
  const saddr_t ring = to_saddr(warp_smem + C::WARP_U16 * 2 + lane * 16);

  // the streams of this launch: all n, or the ones an earlier launch handed on
  const uint64_t n_todo = a.todo_count ? static_cast<uint64_t>(*a.todo_count) : a.n;
  const uint64_t n_groups = (n_todo + 31) / 32;
  const bool pair_on = a.no_pair == 0;
  constexpr bool qon = QUEUE && !COUNT;
  // per-lane table state that outlives a stream (see parse_block_header)
  bool tables_fixed = false;
  LongTab<C::ROOT_LIT> lt_lit;     // canonical first/count of the codes longer than the LUT roots
  LongTab<C::ROOT_DIST> lt_dist;
  lt_lit.usable = lt_dist.usable = false;
#pragma unroll
  for (int i = 0; i < 15 - C::ROOT_LIT; ++i) lt_lit.fc[i] = 0;
#pragma unroll
  for (int i = 0; i < 15 - C::ROOT_DIST; ++i) lt_dist.fc[i] = 0;
  lt_lit.off0 = lt_dist.off0 = 0;
  for (;;) {
    unsigned long long g = 0;
    if (lane == 0) g = atomicAdd(a.group_counter, 1ull);
    g = __shfl_sync(FULL, g, 0);
    if (g >= n_groups) break;
    const uint64_t slot = g * 32 + static_cast<uint64_t>(lane);
    const uint64_t idx = a.todo_list ? (slot < n_todo ? a.todo_list[slot] : 0) : a.idx_base + slot;

    int state = S_DONE;
    int status = ST_SUCCESS;
    BitReader br;
    typename WinOf<COUNT>::type ow;
    // lanes without a stream still run the (predicated-off) decode stage
    br.park(ring);
    ow.park();
    uint32_t final_block = 0;
    int n_lit = 0, n_dist = 0;
    const uint8_t* copy_src = nullptr;
    uint32_t copy_left = 0;
    bool live = slot < n_todo;
    bool first_header = true;  // nothing of this stream has been decided yet
    // hand-over to a pass 2 that runs beside this kernel (QueueArgs): the next segment to publish and
    // the cursor position from which it may be (never reached without a queue)
    uint32_t pub_k = 0, pub_at = 0xffffffffu;
    if (live && a.handled != nullptr && a.handled[idx] != 0) {  // (a stream of stored blocks: done already)
      live = false;
      if (qon) q_push(a.q, idx, 0u, true);
    }
    if (live) {
      const uint64_t slen = a.src_len[idx];
      const uint64_t cap = COUNT ? 0xfffffef0ull : a.dst_cap[idx];
      if (slen >= 0xffffff00ull || cap >= 0xffffff00ull) {
        a.status[idx] = ST_ERROR;  // outside the batch precondition
        a.written[idx] = 0;
        live = false;
        if (qon) q_push(a.q, idx, 0u, true);
      } else {
        br.open(a.src_base + a.src_off[idx], static_cast<uint32_t>(slen), ring);
        ow.open(a.dst_base, COUNT ? 0ull : a.dst_off[idx] + a.dst_delta, static_cast<uint32_t>(cap), a.match_bits);
        if (a.start_bit != nullptr) {  // chunked input: continue at a block header, behind earlier output
          br.seek_bit(a.start_bit[idx]);
          ow.jump(static_cast<uint32_t>(a.start_out[idx]));
        }
        state = S_HEADER;
        if (qon) pub_at = ow.lead + (1u << a.q.seg_shift) + a.q.lag + 8u;
      }
    }
    // every word below the open one is in memory: publish the segments that lie LAG bytes behind it
    auto publish = [&]() {
      ow.release_first();
      do {
        q_push(a.q, idx, pub_k, false);
        ++pub_k;
        pub_at += 1u << a.q.seg_shift;
      } while (ow.vpos >= pub_at);
    };

    while (__any_sync(FULL, state != S_DONE)) {
      if (state == S_HEADER) {
        if (a.blk_end != nullptr) {  // (chunked input) a block boundary: this far a later call need not redo
          a.blk_end[2 * idx] = static_cast<uint64_t>(br.bitpos());
          a.blk_end[2 * idx + 1] = ow.written();
        }
        uint32_t lost = 0;
        state = parse_block_header<C>(br, m, ow.room(), final_block, n_lit, n_dist, copy_src,
                                      copy_left, &status, &lost, lt_lit, lt_dist, tables_fixed);
        // A small-geometry launch hands the stream on when the codes of its FIRST block do not
        // fit the tables well (more than ~2^-9 of the code space would take the exact slow
        // path): nothing has been written for it yet.  Later blocks just live with it.
        if (a.defer_list != nullptr && first_header && state == S_DECODE && lost > C::DEFER_LOST) {
          a.defer_list[atomicAdd(a.defer_count, 1ull)] = static_cast<uint32_t>(idx);
          state = S_DONE;
          live = false;
        }
        first_header = false;
      }
      // ---- stored blocks (src/decompress.cpp:434): the warp copies them, one at a time ------
      for (unsigned sm = __ballot_sync(FULL, state == S_STORED); sm; sm &= sm - 1) {
        const int owner = __ffs(static_cast<int>(sm)) - 1;
        if (lane == owner) ow.spill_pending();
        const uint8_t* s = reinterpret_cast<const uint8_t*>(
            shfl_u64(reinterpret_cast<uint64_t>(copy_src), owner));
        uint8_t* d = reinterpret_cast<uint8_t*>(
            shfl_u64(reinterpret_cast<uint64_t>(ow.al + ow.vpos), owner));
        const uint32_t len = __shfl_sync(FULL, copy_left, owner);
        __syncwarp();
        if constexpr (!COUNT) {
          // dst-aligned 32-bit words, each funnelled from the two aligned src words it spans
          // (src words are only read where they hold at least one payload byte)
          const uint32_t head = min(len, static_cast<uint32_t>(-reinterpret_cast<intptr_t>(d)) & 3u);
          const uint8_t* sb0 = s + head;
          // (when src and dst are not congruent mod 4 a dst word spans two src words, and the
          //  second one of the LAST dst word could reach past the payload — i.e. past the end
          //  of the caller's buffer: leave that word to the byte loop)
          const bool skew = ((reinterpret_cast<uintptr_t>(sb0)) & 3u) != 0;
          uint32_t nwords = (len - head) >> 2;
          if (skew && nwords) --nwords;
          const uint32_t tail0 = head + 4u * nwords;
          for (uint32_t i = static_cast<uint32_t>(lane); i < head; i += LANES) d[i] = s[i];
          const uint8_t* sb = s + head;
          const uint32_t sh = 8u * (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(sb)) & 3u);
          const uint32_t* sw = reinterpret_cast<const uint32_t*>(sb - (sh >> 3));
          uint32_t* dw = reinterpret_cast<uint32_t*>(d + head);
#pragma unroll 4
          for (uint32_t i = static_cast<uint32_t>(lane); i < nwords; i += LANES) {
            const uint32_t lo = sw[i];
            const uint32_t hi = sh ? sw[i + 1] : 0u;
            dw[i] = funnel_r(lo, hi, sh);
          }
          for (uint32_t i = tail0 + static_cast<uint32_t>(lane); i < len; i += LANES) d[i] = s[i];
        }
        __syncwarp();
        if (lane == owner) {
          ow.jump(len);
          br.init_at(static_cast<uint32_t>(copy_src + len - br.base), 0);
          status = ST_SUCCESS;
          state = final_block ? S_DONE : S_HEADER;
        }
      }
      if constexpr (qon) { if (ow.vpos >= pub_at) publish(); }
      // ---- token iterations (all 32 lanes stay in this loop together) -----------------------
      uint32_t it = 0;
      // software pipeline: the output step of a token is deferred to the start of the next
      // iteration, where it is independent of everything around it and fills the latency of
      // the decode chain (window -> LUT -> length -> window)
      uint32_t p_chunk = 0, p_n = 0, p_skip = 0, p_hoff = 0;
      bool p_mt = false;
      while (__any_sync(FULL, state == S_DECODE)) {
        // ---- decode one token.  Straight-line and nearly branch-free (results are only used by
        //      lanes in S_DECODE, the others compute on stale data and discard): the two rare
        //      branches are the exact slow path and a token that does not fit the output. -----
        bool dec = state == S_DECODE;
        SFB_STAT(tokens);
        const uint32_t bo0 = br.bo;   // < 32
        // while no window word reaches past the end of the stream every bit the iteration can see
        // is real (a literal of <= ROOT_LIT bits and a token of <= 48 are at most 56 of the >= 65
        // window bits); otherwise go the exact way
        const bool tail = br.tail();
        uint32_t n0, n1;
        br.next2(n0, n1);
        // ---- a literal in front: when the next symbol is a literal whose code fits the LUT root
        //      (text: nearly every literal) it is taken together with the token behind it — one
        //      more root look-up on the chain, ~1.4 tokens per iteration on text.  Everything that
        //      can go wrong with the token behind it (exact path, distance / room checks) is not
        //      handled here: that token is then left for the next iteration, where it comes first.
        const uint32_t bits0 = br.peek();
        const uint32_t bits_hi = funnel_r(br.w1, br.w2, bo0);   // window bits [32, 64) from the token start
        const uint32_t e1 = lds16(lutb + (C::LIT_OFF * 64) + ((bits0 << 6) & (((1u << C::ROOT_LIT) - 1u) << 6)));
        ow.emit(p_chunk, p_n, p_skip, p_mt, p_hoff);   // (the previous iteration's output step)
        if constexpr (qon) { if (ow.vpos >= pub_at) publish(); }
        const bool pre1 = dec & !tail & (ow.room() != 0u) & ((ow.vpos & 7u) != 7u) & pair_on;
        // a literal entry has bits 12-15 clear and its code length (1 .. ROOT_LIT) in bits 0-3
        const uint32_t t1 = e1 & 0xf00fu;
        const bool lit1 = pre1 & (t1 - 1u < 15u);
        const uint32_t off = lit1 ? t1 : 0u;
        const uint32_t bo1 = bo0 + off;   // < 32 + ROOT_LIT
        const uint32_t bits = funnel_r(bits0, bits_hi, off);
        const uint32_t e = lut_lookup_s<C::ROOT_LIT, C::LIT_OFF, C::POOL_OFF, C::POOL>(lutb, bits);
        const uint32_t L = e & 15u;
        const uint32_t xb = (e >> 12) & 7u;               // 0 for literals
        bool is_match = (e & 0x8000u) != 0;               // (pointers were resolved: L != 0 then)
        uint32_t value = ((e >> 4) & 0xffu) + ((bits >> L) & ~(0xffffffffu << xb)) + (is_match ? 3u : 0u);
        const uint32_t used1 = L + xb;
        const uint32_t dbits = br.peek_at(bo1 + used1);   // bo1 + used1 <= 31 + 8 + 20
        const uint32_t de = lut_lookup_s<C::ROOT_DIST, C::DIST_OFF, C::POOL_OFF, C::POOL>(lutb, dbits);
        const uint32_t dL = de & 15u;
        const uint32_t dinfo = lds32(sdi + ((de >> 2) & 0x7cu));
        const uint32_t dxb = (de >> 9) & 15u;
        uint32_t dist = (dinfo & 0xffffu) + ((dbits >> dL) & ~(0xffffffffu << dxb));
        uint32_t used = used1 + (is_match ? dL + dxb : 0u);
        // anything that is not a plain literal / length+distance — end of block included — is
        // redone exactly, from the same 64 window bits
        // (near the end of the input the token must also fit into the real bits that are left)
        // (`tail`: a window word reaches past the end of the stream — the bits there are zeros, not
        //  input.  A plain token that ends inside the real bits is still exactly what the reference
        //  decodes bit by bit; one that does not goes the exact way, which names the status.  4 KiB
        //  pages spend their last ~10 tokens here: taking all of them the exact way, one lane at a
        //  time, was a fifth of pass 1 on BASELINE config 3.)
        const bool odd = (L == 0) | (is_match & (dL == 0));
        const int32_t left32 = static_cast<int32_t>(br.ebits - 32u * br.rp - bo0);   // real bits left (valid in `tail`)
        const bool past_end = tail & (static_cast<int32_t>(used) > left32);
        if (dec & !lit1 & (odd | past_end)) {
          // (a) a valid code longer than the tables hold: canonical decode in registers
          bool done = false;
          if (lt_lit.usable & lt_dist.usable) {
            const uint16_t* sorted = reinterpret_cast<const uint16_t*>(m.lens + SCR_SORTED * 32);
            bool ok = true, mt2 = is_match;
            uint32_t u1 = used1, val2 = value;
            if (L == 0) {
              uint32_t rank = 0;
              const uint32_t Lm = long_decode<C::ROOT_LIT>(lt_lit, bits, rank);
              const uint32_t sym = Lm ? sorted[(rank >> 1) * 64 + (rank & 1u)] : 999u;
              if (sym < 256u) {
                val2 = sym;
                mt2 = false;
                u1 = Lm;
              } else if (sym >= 257u && sym <= 285u) {
                const uint32_t info = c_len_info[sym - 257u];
                const uint32_t x = info >> 16;
                val2 = (info & 0xffffu) + ((bits >> Lm) & ~(0xffffffffu << x));
                mt2 = true;
                u1 = Lm + x;
              } else {
                ok = false;  // end of block, 286/287, or no code at all: the exact path decides
              }
            }
            uint32_t u2 = u1, dist2 = dist;
            if (ok & mt2) {
              const uint32_t db2 = br.peek_at(bo0 + u1);  // u1 <= 20
              const uint32_t de2 = lut_lookup_s<C::ROOT_DIST, C::DIST_OFF, C::POOL_OFF, C::POOL>(lutb, db2);
              uint32_t dl2 = de2 & 15u, dsym = (de2 >> 4) & 31u;
              if (dl2 == 0) {
                uint32_t rank = 0;
                dl2 = long_decode<C::ROOT_DIST>(lt_dist, db2, rank);
                const uint32_t r2 = 288u + rank;
                dsym = dl2 ? sorted[(r2 >> 1) * 64 + (r2 & 1u)] : 99u;
              }
              if (dl2 != 0 && dsym < 30u) {
                const uint32_t di = c_dist_info[dsym];
                const uint32_t x = di >> 16;
                dist2 = (di & 0xffffu) + ((db2 >> dl2) & ~(0xffffffffu << x));
                u2 = u1 + dl2 + x;
              } else {
                ok = false;
              }
            }
            if (ok && (!tail || static_cast<int32_t>(u2) <= left32)) {
              SFB_STAT(long_tokens);
              done = true;
              used = u2;
              is_match = mt2;
              value = val2;
              dist = dist2;
            }
          }
          // (b) everything else — end of block included — is redone exactly, bit by bit
          if (!done) {
            SFB_STAT(slow_tokens);
            const SlowToken t = slow_token(m.lens, (static_cast<uint64_t>(bits_hi) << 32) | bits,
                                           br.real_left());
            used = t.used;
            is_match = t.kind == 2;
            value = static_cast<uint32_t>(t.value);
            dist = static_cast<uint32_t>(t.dist);
            if (t.status != ST_SUCCESS || t.kind == 1) {  // failure, or end of block
              status = t.status;
              state = (t.status == ST_SUCCESS && !final_block) ? S_HEADER : S_DONE;
              dec = false;
              // (the end-of-block code is consumed: the next header starts right behind it)
              if (t.status == ST_SUCCESS) br.skip(used);
            }
          }
        }
        // ---- act on the token ----------------------------------------------------------------
        // (src/decompress.cpp:178-183 distance then room for a match, :150-152 room for a
        //  literal; nothing of a token that fails is written)
        const uint32_t lit1n = lit1 ? 1u : 0u;
        const bool drop2 = lit1 & odd;   // the token behind the literal waits for its own iteration
        if (dec) br.skip(off + (drop2 ? 0u : used));
        const bool bad_dist = is_match & (dist > ow.written() + lit1n);
        bool tok = dec & !drop2;
        if (tok & (bad_dist | (ow.room() - lit1n < (is_match ? value : 1u)))) {
          // (a literal in front of the failing token is still written: it came first)
          status = bad_dist ? ST_INVALID_DISTANCE : ST_DST_TOO_SMALL;
          state = S_DONE;
          tok = false;
        }
        br.norm2(n0, n1);
        if (it & 1u) br.stage_step();
        ++it;
        const bool mt = tok & is_match;
        const uint32_t desc = (value - 3u) | ((dist - 1u) << 8);
        const uint32_t chunk2 = tok ? (mt ? desc : value) : 0u;
        p_mt = mt;
        p_hoff = lit1n;
        p_chunk = lit1 ? (((e1 >> 4) & 0xffu) | (chunk2 << 8)) : chunk2;
        p_n = (tok ? (mt ? 3u : 1u) : 0u) + lit1n;
        p_skip = mt ? value - 3u : 0u;
      }
      ow.emit(p_chunk, p_n, p_skip, p_mt, p_hoff);  // drain the pipeline
      if (state == S_DONE && live) {
        if (END && status == ST_SUCCESS) {  // (see END above)
          a.blk_end[2 * idx] = static_cast<uint64_t>(br.bitpos());
          a.blk_end[2 * idx + 1] = ow.written();
        }
        ow.flush_tail();
        a.status[idx] = static_cast<uint8_t>(status);
        a.written[idx] = ow.written();
        live = false;
        if (qon) q_push(a.q, idx, pub_k, true);
        pub_at = 0xffffffffu;   // (the lane idles until its warp's other streams end: nothing more to publish)
      }
    }
  }
#ifndef SFB_CPU_EMU
  if (qon) {  // the last CTA to leave tells the consumers how many items there are
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(a.q.done, 1u) == gridDim.x - 1u) {
        *reinterpret_cast<volatile unsigned long long*>(a.q.final_tail) = atomicAdd(a.q.tail, 0ull);
        __threadfence();
        *reinterpret_cast<volatile unsigned int*>(a.q.done + 1) = 1u;
      }
    }
  }
#endif
}

}  // namespace sfb
