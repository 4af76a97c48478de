"""CPU: the block-level kernels the lane and warp emulations cannot run — pass 2 of the
single-stream route (lz_jump.cuh: pointer jumping), the parallel chain of block jobs
(block_finder.cuh: chain_parallel_kernel), batch preparation (lz_warp.cuh: prep kernels) and the
stored-stream copy (stored_copy.cuh) — on blocks of host threads (tests/cpu_emu/emu_block.cpp),
against the oracle, or against the sequential walk for the chain."""
import zlib

import numpy as np
import pytest

from tests import block_cases as B
from tests import deflate_tools as T
from tests import emu_block_bindings as E
from tests.emu_block_bindings import JOB_DTYPE, JOB_ENDS, JOB_NONE, JOB_RECS

FILL = 0xA5


@pytest.fixture(scope="module")
def route():
    return E.EmuRoute()


@pytest.fixture(scope="module")
def blk():
    return E.EmuBlock()


def _aligned(n, fill=FILL):
    raw = np.full(n + 128, fill, np.uint8)
    o = (-raw.ctypes.data) % 128
    return raw[o:o + n]


def _pass1(route, src, cap, q, cand=None):
    """the real single-stream pass 1 into a fresh 128-byte aligned buffer at phase q"""
    base = _aligned(q + cap + 1100)
    bits = np.zeros(len(base) // 32 + 8, np.uint32)
    st, wr, _, _ = route.stream_pass1(src, base, q, cap, bits, cand)
    return st, wr, base, bits


def _jump_one(route, blk, src, cap, q, **kw):
    """pass 1, then pointer-jumping pass 2 -> (status, written, dst region, rounds, outside intact)"""
    st, wr, base, bits = _pass1(route, src, cap, q)
    rounds = blk.jump_resolve(base, [q], [wr], bits, **kw)
    intact = bool((base[:q] == FILL).all() and (base[q + cap:] == FILL).all())
    return st, wr, base[q:q + cap].tobytes(), rounds, intact


# ------------------------------------------------------------------------------- pointer jumping
def test_jump_pass2_crafted_lz_shapes(route, blk, oracle):
    """tests.deflate_tools.crafted_lz_streams (runs, short periods, far copies, dense short matches,
    matches across chunk and word edges) through the single-stream route, dst phases (7k) mod 128."""
    for k, (name, src, n) in enumerate(T.crafted_lz_streams()):
        ost, odst, owr, _ = oracle.decompress(src, n)
        st, wr, dst, _, intact = _jump_one(route, blk, src, n, (7 * k) % 128, warps=2, block_warps=1,
                                           reverse=k % 2 == 1)
        assert (st, wr) == (ost, owr) == (0, n) and dst == odst and intact, name


def test_jump_pass2_golden_families(route, blk, oracle, golden):
    """The reference's answers: known answers, crafted dynamic headers, and a stride of the cut /
    cap / flip families — failed streams with written > 0 among them."""
    k = 0
    for name, fam in golden.families.items():
        if name == "known_answers":
            stride = 1
        elif name == "crafted_dynamic_headers":
            stride = 8
        elif name.startswith(("cut", "cap", "flip")):
            stride = max(1, len(fam["params"]) // 3 + 1)
        else:
            continue
        for i, src, cap in golden.cases(name, stride):
            want_st, want_wr, want_hash, cls = golden.expected(name, i)
            st, wr, dst, _, intact = _jump_one(route, blk, src, cap, (7 * k) % 128, warps=3, block_warps=1,
                                               reverse=k % 2 == 0)
            k += 1
            assert (st, wr) == (want_st, want_wr), (name, i, cls)
            assert "%016x" % oracle.fnv1a64(dst) == want_hash and intact, (name, i, cls)
    assert k > 150


def test_jump_pass2_match_carried_into_a_tile(route, blk):
    """tests.deflate_tools.tile_edge_lz_streams: one match whose head sits just before or at a 1 KiB
    tile edge, so that it reaches into the next tile or ends exactly at its edge (the 258-byte match
    at T - 258 must not be carried in, the one at T - 257 must).  Here the heads around the edge of
    the 288-byte window the tile searches and around the tile edge itself; the GPU test sweeps every
    offset."""
    offsets = list(range(-290, -250)) + list(range(-35, -29)) + list(range(-4, 2))
    cases = B.tile_edge_lz_streams(qs=(0, 1, 77, 127), lengths=(257, 258), dists=(1, 300), offsets=offsets)
    cases += B.tile_edge_lz_streams(qs=(0, 127), lengths=(3,), dists=(2,), offsets=range(-4, 2))
    cases += B.tile_edge_lz_streams(qs=(77,), lengths=(258,), dists=(32768,), offsets=(-258, -257, -256))
    for k, (name, q, src, plain) in enumerate(cases):
        st, wr, dst, _, intact = _jump_one(route, blk, src, len(plain), q, warps=1, block_warps=1)
        assert (st, wr) == (0, len(plain)) and dst == plain and intact, name


def test_jump_pass2_long_chains_any_order_any_stripes(route, blk):
    """Chains of many hops (a run of one byte, a period of 7, text): the same bytes whatever the
    number of warps, the order their blocks run in and the stripes (1, 2, 3 tiles, one stripe)."""
    inputs = [b"\x00" * 300000, b"abcdefg" * 43000, T.text_like(300000, 21)]
    seen_rounds = []
    for k, plain in enumerate(inputs):
        comp = T.raw_deflate(plain, 9)
        q = 37 * k + 5
        st, wr, base0, bits = _pass1(route, comp, len(plain), q)
        assert (st, wr) == (0, len(plain))
        for stripe, sizes in ((0, None), (1, 12000), (2, 30000), (3, 30000)):
            if sizes is not None:   # (small stripes on the first bytes only: a launch per stripe and round)
                st, wr, base0, bits = _pass1(route, T.raw_deflate(plain[:sizes], 9), sizes, q)
            for warps, block_warps, reverse in ((1, 1, False), (3, 1, True), (8, 8, False), (8, 1, True)):
                if sizes is not None and (warps, block_warps) == (8, 8):
                    continue
                base = _aligned(len(base0))
                base[:] = base0
                rounds = blk.jump_resolve(base, [q], [wr], bits.copy(), stripe_tiles=stripe, warps=warps,
                                          block_warps=block_warps, reverse=reverse)
                n = sizes or len(plain)
                assert base[q:q + n].tobytes() == plain[:n], (k, stripe, warps, block_warps, reverse)
                assert (base[:q] == FILL).all() and (base[q + n:] == FILL).all()
                if stripe == 0:
                    seen_rounds.append(rounds)
    assert max(seen_rounds) >= 6


def test_jump_pass2_several_streams_in_one_call(route, blk, oracle):
    """Several streams one after another through the same tables (pointers and open-group bits left
    by the stream before), their regions back to back so that they share 128-byte chunks and bitmap
    words, one with written = 0 between them: every region as the oracle has it, nothing else changed."""
    plains = [T.text_like(5000, 1), None, T.repetitive(7000, 2), b"xyz" * 1000, T.text_like(3000, 3)]
    srcs, caps = [], []
    for p in plains:
        if p is None:
            srcs.append(b"\x07")          # BTYPE 3 at once: written = 0
            caps.append(50)
        else:
            srcs.append(T.raw_deflate(p, 6))
            caps.append(len(p) - (100 if len(p) == 7000 else 0))   # (one destination too small)
    srcs.append(srcs[0])
    caps.append(caps[0] + 1)
    offs = np.cumsum([13] + caps[:-1]).astype(np.uint64)
    base = _aligned(int(offs[-1]) + caps[-1] + 1100)
    bits = np.zeros(len(base) // 32 + 8, np.uint32)
    wrs = []
    for src, off, cap in zip(srcs, offs, caps):
        st, wr, _, _ = route.stream_pass1(src, base, int(off), cap, bits)
        wrs.append(wr)
    assert wrs[1] == 0
    blk.jump_resolve(base, offs, wrs, bits, warps=3, block_warps=1, reverse=True)
    want = np.full(len(base), FILL, np.uint8)
    for src, off, cap, wr in zip(srcs, offs, caps, wrs):
        ost, odst, owr, _ = oracle.decompress(src, cap)
        assert owr == wr
        want[int(off):int(off) + cap] = np.frombuffer(odst, np.uint8)
    assert (base == want).all()


# ------------------------------------------------------------------------------- the chain of jobs
def _graph(rng, n, chain_len=None, cap_hit=None):
    """A job table: job 0 at bit 0, jobs at increasing starts; `chain_len` of them linked from job 0
    (the rest false starts, some linked among themselves), sizes, needs and flags at random"""
    starts = np.sort(rng.choice(np.arange(1, 200 * n + 2), n - 1, replace=False)) if n > 1 else np.zeros(0, np.int64)
    starts = np.concatenate([[0], starts]).astype(np.uint64)
    perm = np.concatenate([[0], 1 + rng.permutation(n - 1)]) if n > 1 else np.zeros(1, np.int64)
    jobs = np.zeros(n, JOB_DTYPE)
    jobs["start_bit"] = starts[perm]                 # job j starts at starts[perm[j]]
    jobs["base"] = JOB_NONE
    jobs["out"] = rng.integers(0, 5000, n)
    jobs["flags"] = np.where(rng.random(n) < 0.9, JOB_RECS, 0) | 2
    by_rank = np.argsort(perm)                       # job that holds the k-th start
    chain_len = n if chain_len is None else chain_len
    for k in range(n - 1):
        j = by_rank[k]
        if k + 1 < chain_len:
            jobs["next"][j] = by_rank[k + 1]
        elif rng.random() < 0.5:
            jobs["next"][j] = by_rank[rng.integers(k + 1, n)]
    jobs["end_bit"] = np.where(jobs["next"] > 0, jobs["start_bit"][jobs["next"]], jobs["start_bit"] + 5)
    return jobs, by_rank


def _same_chain(blk, jobs, cap, **kw):
    a, b = jobs.copy(), jobs.copy()
    ta = blk.chain(a, cap, parallel=False, **kw)
    tb = blk.chain(b, cap, parallel=True, **kw)
    assert ta == tb and (a["base"] == b["base"]).all() and (a["flags"] == b["flags"]).all(), (ta, tb)
    return a, ta


def test_parallel_chain_long_chains_around_round_counts(blk):
    """Chains through all jobs, n around CHAIN_THREADS and around the powers of two that set the
    number of rounds: every job's base and flags, and the tail, as the walk has them."""
    rng = np.random.default_rng(1)
    for n in (1, 2, 3, 1023, 1024, 1025, 2048, 2049, 3000):
        jobs, order = _graph(rng, n)
        a, tail = _same_chain(blk, jobs, 1 << 62)
        assert tail == order[-1] and (a["base"] != JOB_NONE).all()


def test_parallel_chain_stops_where_the_walk_stops(blk):
    """The first job that does not fit ends the chain: need > base at chosen positions, base + out
    equal to the capacity (fits) and one more (does not), JOB_ENDS in the middle, a `next` past the
    table, duplicate starts, a job count above the table's capacity."""
    rng = np.random.default_rng(2)
    for n in (2, 40, 1025, 2049):
        for pos in sorted({1, n // 3, n // 2, n - 1}):
            if pos >= n:
                continue
            jobs, order = _graph(rng, n)
            base_at = np.concatenate([[0], np.cumsum(jobs["out"][order])])   # base of the k-th job on the chain
            j = order[pos]
            # need > base at job `pos`, need == base one job before
            v = jobs.copy()
            v["need"][j] = base_at[pos] + 1
            v["need"][order[pos - 1]] = base_at[pos - 1]
            _, tail = _same_chain(blk, v, 1 << 62)
            assert tail == j
            # base + out == cap at job `pos` (fits: the chain goes on) and == cap + 1 (the tail)
            for extra, want in ((0, order[min(pos + 1, n - 1)]), (-1, j)):
                _, tail = _same_chain(blk, jobs, int(base_at[pos + 1]) + extra)
                if extra == 0 and pos + 1 < n and jobs["out"][order[pos + 1]] > 0:
                    assert tail == order[pos + 1]
                elif extra == -1:
                    assert tail == j
            # JOB_ENDS in the middle; next >= n; next == 0
            for how in ("ends", "past", "zero"):
                v = jobs.copy()
                if how == "ends":
                    v["flags"][j] |= JOB_ENDS
                elif how == "past":
                    v["next"][j] = n + int(rng.integers(0, 5))
                else:
                    v["next"][j] = 0
                a, tail = _same_chain(blk, v, 1 << 62)
                assert tail == j and (a["base"][order[pos + 1:]] == JOB_NONE).all()
        # duplicate starts: a false job with the start of a job on the chain
        jobs, order = _graph(rng, n)
        if n > 3:
            jobs["start_bit"][order[-1]] = jobs["start_bit"][order[n // 2]]
            jobs["next"][order[-2]] = 0
            _same_chain(blk, jobs, 1 << 62)
        # more jobs counted than the table holds
        _same_chain(blk, jobs, 1 << 62, count=n + 7, job_cap=n)
    # random graphs: partial chains, random needs and capacities
    for t in range(200):
        n = int(rng.integers(1, 60 if t < 100 else 2500))
        jobs, order = _graph(rng, n, chain_len=int(rng.integers(1, n + 1)))
        jobs["need"] = np.where(rng.random(n) < 0.05, rng.integers(0, 20000, n), 0)
        jobs["flags"] |= np.where(rng.random(n) < 0.01, JOB_ENDS, 0).astype(np.uint32)
        cap = int(rng.integers(0, 2500 * n + 1)) if t % 3 == 0 else 1 << 62
        _same_chain(blk, jobs, cap)


def test_parallel_chain_in_the_stream_route(route, blk, oracle):
    """The single-stream route with chain_parallel_kernel in place of the walk, on the job tables its
    counting jobs leave (every call also runs the walk on a copy of the table and compares every
    job's base and flags, and the tail): candidate block starts that are all true, with a gap, all
    wrong, true, wrong and duplicate mixed; complete, truncated and too-small-dst inputs; a distance
    out of range in a later block; the finder's own candidates on zlib output.  Then pass 2.  Bytes,
    status and count as the oracle has them, jobs on the chain and tail as with the walk."""
    rng = np.random.default_rng(99)
    chunks = [T.text_like(5000, 1), T.incompressible(300, 2), T.text_like(3000, 3), T.repetitive(8000, 4),
              T.text_like(2500, 5)]
    comp = T.raw_deflate_multiblock(chunks, [6, 0, 6, 9, 1], [zlib.Z_DEFAULT_STRATEGY, zlib.Z_DEFAULT_STRATEGY,
                                                            zlib.Z_FIXED, zlib.Z_DEFAULT_STRATEGY,
                                                            zlib.Z_DEFAULT_STRATEGY])
    plain = b"".join(chunks)
    starts = oracle.block_starts(comp, len(plain))
    assert len(starts) >= 9 and starts[0] == 0
    wrong = [int(x) for x in rng.integers(1, 8 * len(comp), 12)] + [starts[2] + 1, starts[3] - 1]
    cases = [
        (comp, len(plain), starts[1:]),
        (comp, len(plain), starts[1:4] + starts[6:]),
        (comp, len(plain), wrong),
        (comp, len(plain), starts[1:] + wrong + starts[2:4]),
        (comp, len(plain) - 4000, starts[1:]),
        (comp, 100, starts[1:]),
        (comp[: len(comp) * 2 // 3], len(plain), [s for s in starts[1:] if s < 8 * (len(comp) * 2 // 3)]),
        (comp[:40], len(plain), []),
    ]
    w = T.BitWriter()
    b = T.fixed_block(w, False)
    for ch in b"abcdefgh":
        b.literal(ch)
    b.eob()
    second = len(w)
    b = T.fixed_block(w, True)
    b.literal(ord("x"))
    b.match(5, 20)   # 9 bytes written so far: distance 20 is out of range
    b.eob()
    cases.append((w.tobytes(), 64, [second]))
    for plain_z in (T.text_like(150000, 11), T.text_like(40000, 14) + T.incompressible(3000, 15) + T.text_like(60000, 16)):
        cases.append((T.raw_deflate(plain_z, 6), len(plain_z), None))   # (the finder's candidates)
    before = blk.chain_checks()
    for k, (src, cap, cand) in enumerate(cases):
        q = (37 * k) % 128
        got = []
        for chain in (None, blk.chain_parallel_fn):
            route.set_chain(chain)
            try:
                base = _aligned(q + cap + 1100)
                bits = np.zeros(len(base) // 32 + 8, np.uint32)
                st, wr, on_chain, tail = route.stream_pass1(src, base, q, cap, bits, cand)
            finally:
                route.set_chain(None)
            blk.jump_resolve(base, [q], [wr], bits, warps=3, block_warps=1)
            got.append((st, wr, base[q:q + cap].tobytes(), on_chain, tail))
        ost, odst, owr, _ = oracle.decompress(src, cap)
        assert got[1] == got[0] and got[1][:3] == (ost, owr, odst), (k, got[1][:2], got[0][3:], got[1][3:])
        if k == 0:
            assert got[1][3] == len(starts)   # every block was decoded by a job of its own
    after = blk.chain_checks()
    assert after[0] - before[0] == len(cases) and after[1] == before[1]


# ------------------------------------------------------------------------------- prep + stored copy
def _rank(src):
    if len(src) == 0:
        return 2
    t = (src[0] >> 1) & 3
    return {2: 0, 1: 1, 3: 2, 0: 3}[t]


def _stored_batch():
    """(name, src, cap, src phase, dst phase): every payload length at all 16 x 16 phase pairs, the
    other stored shapes at a few"""
    out = []
    cases = B.stored_lz_streams()
    for name, src, cap in cases:
        if name.startswith("len"):
            out += [(name, src, cap, sp, dp) for sp in range(16) for dp in range(16)]
        else:
            out += [(name, src, cap, (5 * k) % 16, (11 * k + 3) % 16) for k in range(4)]
    return out


@pytest.mark.parametrize("warps,reverse", [(16, False), (3, True)])
def test_prep_and_stored_copy(blk, oracle, warps, reverse):
    """prep_count / prep_scatter_kernel, then stored_streams_kernel: `order` is a permutation of the
    batch grouped by first-block type and `type_count` counts the groups; the streams the copy
    finished have the oracle's status, count and bytes; the others keep status and count as they
    were and hold a prefix of the oracle's output followed by the fill; nothing outside the regions
    changes.  Every source lives in an allocation of its own (reads past it: AddressSanitizer)."""
    cases = _stored_batch()
    n = len(cases)
    caps = np.array([c[2] for c in cases], np.uint64)
    offs = np.zeros(n, np.uint64)
    at = 0
    for i, (_, _, cap, _, dp) in enumerate(cases):
        at = (at + 16 + 15) // 16 * 16 + dp           # >= 16 canary bytes in front of every region
        offs[i] = at
        at += cap
    dst = _aligned(at + 64)
    status = np.full(n, 0xEE, np.uint8)
    written = np.full(n, 0xDEAD, np.uint64)
    order, tc, handled = blk.prep_stored([(c[1], c[3]) for c in cases], dst, offs, caps, status, written,
                                         warps=warps, reverse=reverse)
    ranks = np.array([_rank(c[1]) for c in cases])
    assert sorted(order.tolist()) == list(range(n))
    assert tc.tolist() == [int((ranks == r).sum()) for r in range(4)]
    assert (np.diff(ranks[order]) >= 0).all()
    assert set(handled.tolist()) <= {0, 1} and (handled[ranks != 3] == 0).all()
    b = T.Batch([c[1] for c in cases], caps)
    dst_o = b.new_dst()
    ost, owr, _ = oracle.decompress_batch(b.src, b.src_off, b.src_len, dst_o, b.dst_off, b.dst_cap)
    mask = np.ones(len(dst), bool)
    done = 0
    for i, (name, src, cap, sp, dp) in enumerate(cases):
        region = dst[int(offs[i]):int(offs[i]) + cap]
        mask[int(offs[i]):int(offs[i]) + cap] = False
        want = b.dst_slice(dst_o, i)
        if handled[i]:
            done += 1
            assert (status[i], written[i]) == (ost[i], owr[i]) and (region == want).all(), (name, sp, dp)
        else:
            assert (status[i], written[i]) == (0xEE, 0xDEAD), name
            k = int(np.nonzero(region != FILL)[0][-1]) + 1 if (region != FILL).any() else 0
            assert (region[:k] == want[:k]).all(), (name, sp, dp)
    assert (dst[mask] == FILL).all()
    assert done >= 18 * 256 and (handled[ranks == 3] == 0).sum() >= 8
