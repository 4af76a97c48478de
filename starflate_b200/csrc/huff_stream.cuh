// Pass 1 for FEW, LARGE streams on sm_100a: speculative, self-synchronising Huffman decode, ONE
// WARP PER STREAM — or, for a single large stream, per BLOCK of it (block_finder.cuh finds and
// chains the blocks; modes 1 and 2 below).  This is the first half of the single-stream mode of
// BASELINE.json's north_star; the second half, the LZ77 resolve, is lz_jump.cuh for one stream
// and lz_warp.cuh for a batch of them.
//
// A lane per stream (huff_lanes.cuh) leaves a batch of a few big streams on a few lanes.  Here
// the 32 lanes of a warp decode 32 consecutive bit ranges ("spans", SPAN_BITS each) of the SAME
// Huffman block at once.  Blocks are still taken one after the other — where a block starts is
// only known once the one before has been decoded — and every lane parses the block header
// itself (the same bits, so in lock-step: 32 identical copies of the tables, one per lane, at
// no extra cost in time).  Within a window of 32 spans:
//   1. lane 0 starts at the true position; lane i > 0 starts at the nominal boundary b0 + i*S,
//      which is almost never a token boundary.  Every lane decodes (counting only: output
//      bytes, and how far back its matches reach) until it crosses into the next span, and
//      reports where its last token ended;
//   2. that end is the true start of the next lane — if the lane before was right.  Lanes
//      whose start changed decode again; Huffman codes self-synchronise (a decoder started at
//      a wrong bit falls onto true token boundaries after a few tokens), so the ends stop
//      changing after typically two rounds, and by induction from lane 0 every start is then
//      the true one.  A lane that meets the end of the block (or a decode error) cuts off the
//      lanes after it;
//   3. a prefix sum of the byte counts gives every lane its output position, which also settles
//      the reference's output-side checks (distance > written, room) per lane before anything
//      is written;
//   4. the lanes decode their spans once more, now writing literals and match descriptors (the
//      in-place form of huff_lanes.cuh) at their positions.
// The same decode paths as in the batch kernel are used (LUT, canonical long codes in
// registers, exact bit-serial), so results — bytes, status, written — are identical to it and
// to the reference.
#pragma once

#include "huff_lanes.cuh"
#include "block_finder.cuh"

namespace sfb {

#ifndef SFB_SPAN_BITS
#define SFB_SPAN_BITS 1024
#endif
constexpr uint32_t SPAN_BITS = SFB_SPAN_BITS;

struct StreamArgs {
  const uint8_t* src_base;
  const uint64_t* src_off;
  const uint64_t* src_len;
  uint8_t* dst_base;  // 128-byte aligned
  uint64_t dst_delta;
  const uint64_t* dst_off;
  const uint64_t* dst_cap;
  uint8_t* status;
  uint64_t* written;
  const uint32_t* list;  // the streams to do (null: idx_base + 0 .. n)
  uint64_t idx_base;
  uint64_t n;
  unsigned long long* stream_counter;  // zeroed before launch
  uint32_t* lens_scratch;              // gridDim.x * SCRATCH_WORDS * 32 words
  uint32_t* match_bits;
  // Blocks of ONE stream (idx_base) side by side, see block_finder.cuh.  mode 0: whole streams as
  // above.  mode 1: a warp per job decodes the block at jobs[k].start_bit COUNTING ONLY and
  // records its end, size and reach.  mode 2: a warp per job that the chain gave a position
  // writes its block there; the tail job carries on to the end of the stream and reports.
  uint32_t mode;
  BlockJob* jobs;
  const uint32_t* job_count;
  uint32_t job_cap;
  const uint32_t* job_tab;
  uint32_t tab_mask;
  const uint32_t* tail_job;
  WinRec* recs;         // window records: written in mode 1, read in mode 2
  uint32_t* rec_count;  // zeroed
  uint32_t rec_cap;
  // (may be null) a stream that ends with Success: end_bit[2 * i] = the bit behind its final block's
  // end-of-block code — where a gzip member's trailer starts (gzip_file.cuh); the layout of
  // BatchArgs::blk_end
  uint64_t* end_bit;
};

struct Tok {
  uint32_t used, value, dist;
  bool is_match, eob;
  int status;  // ST_SUCCESS, or why the stream ends at this token
};

// One token at the reader's position (which is not advanced): the decode paths of the batch
// kernel's token loop, in one place.
template <class C>
__device__ __forceinline__ Tok decode_token(const BitReader& br, saddr_t lutb, saddr_t sdi, const LaneMem& m,
                                            const LongTab<C::ROOT_LIT>& lt_lit,
                                            const LongTab<C::ROOT_DIST>& lt_dist)
{
  Tok t;
  t.status = ST_SUCCESS;
  t.eob = false;
  const uint32_t bo0 = br.bo;
  const bool tail = br.tail();
  const uint32_t bits = br.peek();
  const uint32_t bits_hi = funnel_r(br.w1, br.w2, bo0);
  const uint32_t e = lut_lookup_s<C::ROOT_LIT, C::LIT_OFF, C::POOL_OFF, C::POOL>(lutb, bits);
  const uint32_t L = e & 15u;
  const uint32_t xb = (e >> 12) & 7u;
  t.is_match = (e & 0x8000u) != 0;
  t.value = ((e >> 4) & 0xffu) + ((bits >> L) & ~(0xffffffffu << xb)) + (t.is_match ? 3u : 0u);
  const uint32_t used1 = L + xb;
  const uint32_t dbits = br.peek_at(bo0 + used1);
  const uint32_t de = lut_lookup_s<C::ROOT_DIST, C::DIST_OFF, C::POOL_OFF, C::POOL>(lutb, dbits);
  const uint32_t dL = de & 15u;
  const uint32_t dinfo = lds32(sdi + ((de >> 2) & 0x7cu));
  const uint32_t dxb = dinfo >> 16;
  t.dist = (dinfo & 0xffffu) + ((dbits >> dL) & ~(0xffffffffu << dxb));
  t.used = used1 + (t.is_match ? dL + dxb : 0u);
  if ((L == 0) | (t.is_match & (dL == 0)) | tail) {
    const int32_t left32 = static_cast<int32_t>(br.ebits - 32u * br.rp - bo0);
    bool done = false;
    if (lt_lit.usable & lt_dist.usable) {
      const uint16_t* sorted = reinterpret_cast<const uint16_t*>(m.lens + SCR_SORTED * 32);
      bool ok = true, mt2 = t.is_match;
      uint32_t u1 = used1, val2 = t.value;
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
          ok = false;
        }
      }
      uint32_t u2 = u1, dist2 = t.dist;
      if (ok & mt2) {
        const uint32_t db2 = br.peek_at(bo0 + u1);
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
        done = true;
        t.used = u2;
        t.is_match = mt2;
        t.value = val2;
        t.dist = dist2;
      }
    }
    if (!done) {
      const SlowToken s = slow_token(m.lens, (static_cast<uint64_t>(bits_hi) << 32) | bits, br.real_left());
      t.used = s.used;
      t.is_match = s.kind == 2;
      t.eob = s.kind == 1;
      t.value = static_cast<uint32_t>(s.value);
      t.dist = static_cast<uint32_t>(s.dist);
      t.status = s.status;
    }
  }
  return t;
}

// what a lane found in its span
struct Span {
  uint32_t rel;   // bits from the span's start to the end of its last token
  uint32_t out;   // output bytes of its tokens
  int32_t need;   // max over its matches of (distance - bytes this span had produced before it)
  uint32_t flag;  // 0 ran into the next span, 1 end of block, 2 the stream ends here with `st`
  int st;
};

// Decode the tokens that START in [0, span_bits) from the reader's position.  `go` is false for
// lanes that only keep the warp company.  EMIT writes through `ow` (whose region starts at
// this span's output position `prefix`), else only counts.
template <class C, bool EMIT>
__device__ __forceinline__ Span run_span(BitReader& br, bool go, uint32_t span_bits, saddr_t lutb, saddr_t sdi,
                                         const LaneMem& m, const LongTab<C::ROOT_LIT>& lt_lit,
                                         const LongTab<C::ROOT_DIST>& lt_dist, TokWin& ow, uint64_t prefix)
{
  constexpr unsigned FULL = 0xffffffffu;
  Span r;
  r.rel = 0;
  r.out = 0;
  r.need = -0x7fffffff;
  r.flag = 0;
  r.st = ST_SUCCESS;
  uint32_t it = 0;
  while (__any_sync(FULL, go && r.flag == 0 && r.rel < span_bits)) {
    const bool act = go && r.flag == 0 && r.rel < span_bits;
    uint32_t n0, n1;
    br.next2(n0, n1);
    const Tok t = decode_token<C>(br, lutb, sdi, m, lt_lit, lt_dist);
    if (act) {
      if (t.status != ST_SUCCESS) {
        r.flag = 2;
        r.st = t.status;
      } else if (t.eob) {
        r.flag = 1;
        r.rel += t.used;
        br.skip(t.used);
      } else {
        const uint32_t size = t.is_match ? t.value : 1u;
        bool fail = false;
        if (EMIT) {
          // src/decompress.cpp:178-183 distance then room for a match, :150-152 room for a literal
          const bool bad_dist = t.is_match && static_cast<uint64_t>(t.dist) > prefix + ow.written();
          if (bad_dist || ow.room() < size) {
            r.flag = 2;
            r.st = bad_dist ? ST_INVALID_DISTANCE : ST_DST_TOO_SMALL;
            fail = true;
          } else if (t.is_match) {
            ow.emit((t.value - 3u) | ((t.dist - 1u) << 8), 3u, t.value - 3u, true);
          } else {
            ow.emit(t.value, 1u, 0u, false);
          }
        } else if (t.is_match) {
          const int32_t nd = static_cast<int32_t>(t.dist) - static_cast<int32_t>(r.out);
          r.need = nd > r.need ? nd : r.need;
        }
        if (!fail) {
          r.out += size;
          r.rel += t.used;
          br.skip(t.used);
        }
      }
    }
    br.norm2(n0, n1);
    if (it & 1u) br.stage_step();
    ++it;
  }
  return r;
}

__device__ __forceinline__ uint64_t shfl_up_u64(uint64_t v, unsigned d)
{
  const uint32_t lo = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(v), d);
  const uint32_t hi = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), d);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

template <class C>
__global__ void __launch_bounds__(32) huff_stream_kernel(const StreamArgs a)
{
#ifdef SFB_CPU_EMU
  uint8_t* const smem = reinterpret_cast<uint8_t*>(SFB_EMU_SMEM);
#else
  extern __shared__ __align__(16) uint8_t smem[];
#endif
  constexpr unsigned FULL = 0xffffffffu;
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t* const s_dist_info = reinterpret_cast<uint32_t*>(smem + C::WARP_BYTES);
  s_dist_info[lane] = c_dist_info[lane];
  __syncwarp();
  LaneMem m;
  m.lut = reinterpret_cast<uint16_t*>(smem) + lane;
  m.lens = a.lens_scratch + static_cast<size_t>(blockIdx.x) * (SCRATCH_WORDS * 32) + lane;
  const saddr_t lutb = to_saddr(m.lut);
  const saddr_t sdi = to_saddr(s_dist_info);
  const saddr_t ring = to_saddr(smem + C::WARP_U16 * 2 + lane * 16);
  bool tables_fixed = false;
  LongTab<C::ROOT_LIT> lt_lit;
  LongTab<C::ROOT_DIST> lt_dist;
  lt_lit.usable = lt_dist.usable = false;
#pragma unroll
  for (int i = 0; i < 15 - C::ROOT_LIT; ++i) lt_lit.fc[i] = 0;
#pragma unroll
  for (int i = 0; i < 15 - C::ROOT_DIST; ++i) lt_dist.fc[i] = 0;
  lt_lit.off0 = lt_dist.off0 = 0;

  const uint32_t mode = a.mode;  // (warp-uniform, like everything that steers the loops below)
  unsigned long long n_units = a.n;
  uint32_t tail = 0;
  if (mode) {
    const uint32_t nj = *a.job_count;
    n_units = nj < a.job_cap ? nj : a.job_cap;
    if (mode == 2u) tail = *a.tail_job;
  }
  for (;;) {
    unsigned long long si = 0;
    if (lane == 0) si = atomicAdd(a.stream_counter, 1ull);
    si = __shfl_sync(FULL, si, 0);
    if (si >= n_units) break;
    const uint64_t idx = mode ? a.idx_base : (a.list ? a.list[si] : a.idx_base + si);
    const uint64_t slen = a.src_len[idx];
    const uint64_t real_cap = a.dst_cap[idx];
    if (slen >= 0xffffff00ull || real_cap >= 0xffffff00ull) {
      if (lane == 0 && (mode == 0u || (mode == 2u && si == 0))) {
        a.status[idx] = ST_ERROR;  // outside the batch precondition
        a.written[idx] = 0;
      }
      continue;
    }
    const uint8_t* const src = a.src_base + a.src_off[idx];
    const uint64_t doff = a.dst_off[idx] + a.dst_delta;
    const uint64_t total_bits = 8ull * slen;
    uint64_t bitpos = 0;  // where the next block header starts (warp-uniform)
    uint64_t outpos = 0;  // bytes produced so far (warp-uniform)
    int status = -1;      // < 0: still going
    bool one_block = false, stop = false;
    uint64_t cap = real_cap;
    uint32_t job_need = 0;
    bool use_recs = false, recs_ok = true, clean = false;
    uint32_t first_rec = 0, prev_rec = 0;
    if (mode) {
      bitpos = a.jobs[si].start_bit;
      if (mode == 2u) {
        outpos = a.jobs[si].base;
        if (outpos == JOB_NONE) continue;  // not a block of the stream (or beyond its end)
        one_block = si != tail;
        use_recs = (a.jobs[si].flags & JOB_USE) != 0u;
      } else {
        one_block = true;
        cap = 0xfffffff0ull;  // sizes are settled by the chain
      }
    }
    const bool counting = mode == 1u;
    BitReader br;
    TokWin ow;
    ow.park();
    while (status < 0 && !stop) {
      if (one_block) stop = true;  // (every way round the loop below ends a block)
      if (outpos >= cap) {         // only a counting job that decodes garbage gets here
        if (counting) {
          status = ST_DST_TOO_SMALL;
          break;
        }
      }
      // ---- block header, by every lane --------------------------------------------------------
      br.open(src, static_cast<uint32_t>(slen), ring);
      br.seek_bit(bitpos < total_bits ? bitpos : total_bits);
      uint32_t final_block = 0, copy_left = 0, lost = 0;
      int n_lit = 0, n_dist = 0, st = ST_SUCCESS;
      const uint8_t* copy_src = nullptr;
      const int state = parse_block_header<C>(br, m, static_cast<uint32_t>(cap - outpos), final_block, n_lit,
                                              n_dist, copy_src, copy_left, &st, &lost, lt_lit, lt_dist,
                                              tables_fixed);
      if (state == S_DONE) {
        status = st;
        break;
      }
      if (state == S_HEADER) {  // an empty stored block that was not the last one
        bitpos = static_cast<uint64_t>(br.bitpos());
        continue;
      }
      if (state == S_STORED) {  // src/decompress.cpp:434, by the whole warp
        uint8_t* d = a.dst_base + doff + outpos;
        if (!counting)
          for (uint32_t i = lane; i < copy_left; i += 32u) d[i] = copy_src[i];
        outpos += copy_left;
        bitpos = 8ull * static_cast<uint64_t>(copy_src + copy_left - br.begin());
        if (final_block) status = ST_SUCCESS;
        continue;
      }
      // ---- Huffman block whose windows the counting job left on record: write, nothing else ----
      if (use_recs) {  // (warp-uniform; the job's first block only)
        use_recs = false;
        const BlockJob jb = a.jobs[si];
        for (uint32_t ri = jb.first_rec; ri != 0u;) {
          const WinRec* const rec = a.recs + (ri - 1u);
          const uint64_t wb0 = rec->b0;
          const uint64_t ws = wb0 + rec->s_rel[lane];
          const uint64_t wlim = wb0 + static_cast<uint64_t>(lane + 1u) * SPAN_BITS;
          const uint64_t wstart = outpos + rec->start[lane];
          const bool em = lane <= rec->cut;
          if (em) {
            br.seek_bit(ws < total_bits ? ws : total_bits);
            ow.open(a.dst_base, doff + wstart, static_cast<uint32_t>(cap - wstart), a.match_bits);
          }
          run_span<C, true>(br, em, static_cast<uint32_t>(wlim > ws ? wlim - ws : 0u), lutb, sdi, m, lt_lit, lt_dist,
                            ow, wstart);
          if (em) ow.flush_tail();
          ri = rec->next;
        }
        outpos += jb.out;
        bitpos = jb.end_bit;
        if (final_block) status = ST_SUCCESS;
        continue;
      }
      // ---- Huffman block: windows of 32 spans -------------------------------------------------
      uint64_t b0 = static_cast<uint64_t>(br.bitpos());
      for (;;) {
        uint64_t s = b0 + static_cast<uint64_t>(lane) * SPAN_BITS;
        const uint64_t lim = b0 + static_cast<uint64_t>(lane + 1u) * SPAN_BITS;
        // a span that starts at or past the end of the input has nothing in it (the lane before
        // it runs into the end and reports what the reference would)
        bool redo = true;
        Span r;
        r.rel = 0;
        r.out = 0;
        r.need = -0x7fffffff;
        r.flag = 0;
        r.st = ST_SUCCESS;
        uint32_t cut = 32;  // first lane that stops the block (end of block / error); 32: none
        for (;;) {
          const bool go = redo && lane <= cut && s < total_bits + 64u;
          if (go) br.seek_bit(s < total_bits ? s : total_bits);
          const Span nr = run_span<C, false>(br, go, static_cast<uint32_t>(lim > s ? lim - s : 0u), lutb, sdi, m,
                                             lt_lit, lt_dist, ow, 0);
          if (go) r = nr;
          const uint32_t stops = __ballot_sync(FULL, r.flag != 0);
          cut = stops ? static_cast<uint32_t>(__ffs(static_cast<int>(stops)) - 1) : 32u;
          const uint64_t prev_end = shfl_up_u64(s + r.rel, 1);
          redo = lane > 0 && lane <= cut && prev_end != s;
          if (redo) s = prev_end;
          if (!__any_sync(FULL, redo)) break;
        }
        // ---- output positions and the output-side checks ------------------------------------
        const bool live = lane <= cut;
        uint32_t inc = live ? r.out : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t v = __shfl_up_sync(FULL, inc, o);
          if (lane >= static_cast<uint32_t>(o)) inc += v;
        }
        const uint64_t my_start = outpos + (inc - (live ? r.out : 0u));
        const bool bad = live && ((r.need > 0 && static_cast<uint64_t>(r.need) > my_start) ||
                                  my_start + r.out > cap);
        const uint32_t bads = __ballot_sync(FULL, bad);
        const uint32_t last = bads ? static_cast<uint32_t>(__ffs(static_cast<int>(bads)) - 1) : cut;
        if (counting) {  // (warp-uniform) no writing pass: note the reach, take the count pass's verdict
          const uint32_t nd = live && r.need > 0 && static_cast<uint64_t>(r.need) > my_start
                                  ? static_cast<uint32_t>(static_cast<uint64_t>(r.need) - my_start)
                                  : 0u;
          const uint32_t wmax = __reduce_max_sync(FULL, nd);
          job_need = wmax > job_need ? wmax : job_need;
          if (recs_ok) {  // leave the window on record for the writing job
            uint32_t ri = 0;
            if (lane == 0) ri = atomicAdd(a.rec_count, 1u);
            ri = __shfl_sync(FULL, ri, 0);
            if (ri >= a.rec_cap) {
              recs_ok = false;
            } else {
              WinRec* const rec = a.recs + ri;
              rec->s_rel[lane] = static_cast<uint32_t>(s - b0);
              rec->start[lane] = static_cast<uint32_t>(my_start);
              if (lane == 0) {
                rec->b0 = b0;
                rec->cut = cut;
                rec->next = 0;
                if (prev_rec) a.recs[prev_rec - 1u].next = ri + 1u;
              }
              if (!prev_rec) first_rec = ri + 1u;
              prev_rec = ri + 1u;
            }
          }
          const uint32_t total_c = __shfl_sync(FULL, inc, 31);
          outpos += total_c;
          if (cut < 32u) {
            bitpos = shfl_u64(s + r.rel, static_cast<int>(cut));
            const uint32_t cflag = __shfl_sync(FULL, r.flag, static_cast<int>(cut));
            if (cflag == 2u) status = __shfl_sync(FULL, r.st, static_cast<int>(cut));
            else {
              clean = true;
              if (final_block) status = ST_SUCCESS;
            }
            break;
          }
          if (outpos >= cap) {
            status = ST_DST_TOO_SMALL;
            break;
          }
          b0 = shfl_u64(s + r.rel, 31);
          continue;
        }
        // ---- decode once more, writing --------------------------------------------------------
        const bool em = live && lane <= last;
        if (em) {
          br.seek_bit(s < total_bits ? s : total_bits);
          ow.open(a.dst_base, doff + my_start, static_cast<uint32_t>(cap - my_start), a.match_bits);
        }
        const Span er = run_span<C, true>(br, em, static_cast<uint32_t>(lim > s ? lim - s : 0u), lutb, sdi, m,
                                          lt_lit, lt_dist, ow, my_start);
        if (em) ow.flush_tail();
        // ---- what ended the window -----------------------------------------------------------
        const uint32_t errs = __ballot_sync(FULL, em && er.flag == 2);
        const uint32_t total = __shfl_sync(FULL, inc, 31);
        if (errs) {  // the stream ends inside this window
          const int f = __ffs(static_cast<int>(errs)) - 1;
          status = __shfl_sync(FULL, er.st, f);
          const uint64_t at = shfl_u64(my_start + er.out, f);
          outpos = at;
          break;
        }
        outpos += total;
        if (cut < 32u) {  // end of block in lane `cut`
          bitpos = shfl_u64(s + r.rel, static_cast<int>(cut));
          if (final_block) status = ST_SUCCESS;
          break;
        }
        b0 = shfl_u64(s + r.rel, 31);
      }
    }
    if (lane == 0) {
      if (counting) {
        BlockJob* const jb = a.jobs + si;
        jb->end_bit = bitpos;
        jb->out = outpos;
        jb->need = job_need;
        jb->flags = (status >= 0 ? JOB_ENDS : 0u) | (clean ? JOB_CLEAN : 0u) | (clean && recs_ok ? JOB_RECS : 0u);
        jb->first_rec = first_rec;
        jb->next = status < 0 ? job_find(a.job_tab, a.tab_mask, a.jobs, static_cast<uint32_t>(n_units), bitpos) : 0u;
      } else if (!one_block) {
        a.status[idx] = static_cast<uint8_t>(status);
        a.written[idx] = outpos;
        if (a.end_bit != nullptr && status == ST_SUCCESS) a.end_bit[2 * idx] = bitpos;
      }
    }
  }
}

}  // namespace sfb
