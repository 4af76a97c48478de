"""GPU: the block-level kernels of the decoder through the C ABI, on the inputs made for them
(tests.block_cases; the same kernels run on host threads in tests/test_block_kernels_cpu.py):
pass 2 of the single-stream route (pointer jumping) on matches at every offset around a tile edge,
in stripes down to 1 MiB, behind streams that fail at once; the stored-stream copy of a sorted
batch.  The bar is bit-exact: status, written and every byte, against the oracle."""
import os

import numpy as np
import pytest

from tests import block_cases as B
from tests import deflate_tools as T
from tests import gpu_util
from tests.test_gpu_parity import _one_stream_per_call

pytestmark = pytest.mark.gpu


def test_single_stream_route_crafted_and_tile_edge_shapes(oracle, monkeypatch):
    """One call per stream (SFB200_STREAM_MODE=1: block finder, jobs, chain, pointer-jumping pass 2):
    LZ77 shapes (runs, periods, far copies, matches across chunk edges), and one match at every
    offset around a 1 KiB tile edge of pass 2, at the dst phase the stream is made for."""
    import starflate_b200 as S
    monkeypatch.setenv("SFB200_STREAM_MODE", "1")
    ctx = S.Context(0)
    try:
        k = 0
        for name, src, n in T.crafted_lz_streams():
            st, wr, dst, intact = _one_stream_per_call(ctx, src, n, phase=(7 * k) % 128, src_phase=k % 5)
            k += 1
            assert (st, wr) == (0, n) and intact, name
            assert dst == oracle.decompress(src, n)[1], name
        for name, q, src, plain in B.tile_edge_lz_streams():
            st, wr, dst, intact = _one_stream_per_call(ctx, src, len(plain), phase=q, src_phase=k % 5)
            k += 1
            assert (st, wr, dst) == (0, len(plain), plain) and intact, name
        assert k > 14000
    finally:
        ctx.close()


def _tile_edge_repeated(size):
    """A fixed-Huffman stream of `size` bytes or a little more, made of 2 KiB pairs: 767 literals and
    a 258-byte match (its head at 257 bytes before a 1 KiB edge: carried one byte into the next
    tile), 765 literals and a 258-byte match that ends exactly at the next edge. -> (compressed, plain)"""
    lits = np.random.default_rng(6).integers(32, 127, 767).astype(np.uint8).tobytes()
    w = T.BitWriter()
    blk = T.HuffBlock(w, T.FIXED_LIT_LENS, T.FIXED_DIST_LENS)
    pair = bytearray()
    for n in (767, 765):
        for b in lits[:n]:
            blk.literal(b)
            pair.append(b)
        blk.match(258, 300)
        for _ in range(258):
            pair.append(pair[-300])
    reps = (size + len(pair) - 1) // len(pair)
    head = T.BitWriter().header(True, 1).bits
    tail = T.BitWriter()
    T.HuffBlock(tail, T.FIXED_LIT_LENS, T.FIXED_DIST_LENS).eob()
    bits = np.concatenate([np.array(head, np.uint8), np.tile(np.array(w.bits, np.uint8), reps),
                           np.array(tail.bits, np.uint8)])
    return np.packbits(bits, bitorder="little").tobytes(), bytes(pair) * reps


@pytest.mark.parametrize("stripe_mb", ["0", "8", "1"])
def test_single_stream_route_tile_edges_across_pass2_stripes(monkeypatch, stripe_mb):
    """Pass 2 of the single-stream route in one piece, in 8 MiB and in 1 MiB stripes (the smallest
    SFB200_JUMP_STRIPE_MB takes): 20 MiB of matches that are carried one byte into a tile or end at
    its edge, at every tile; in 1 MiB stripes also a run of one byte, a period of 7, text."""
    import starflate_b200 as S
    monkeypatch.setenv("SFB200_JUMP_STRIPE_MB", stripe_mb)
    ctx = S.Context(0)
    try:
        size = 20 << 20
        comp, plain = _tile_edge_repeated(size)
        st, wr, dst, intact = _one_stream_per_call(ctx, comp, len(plain) + 7, phase=0, src_phase=3)
        assert (st, wr) == (0, len(plain)) and intact and dst[: len(plain)] == plain
        if stripe_mb == "1":
            for k, plain in enumerate([b"abcdefg" * (size // 7), b"\x00" * size, T.big_text(24 << 20, 31)]):
                comp = T.raw_deflate(plain, 9 if k != 2 else 6)
                st, wr, dst, intact = _one_stream_per_call(ctx, comp, len(plain) + 7, phase=(53 * k) % 128, src_phase=k)
                assert (st, wr) == (0, len(plain)) and intact, (k, st, wr)
                assert dst[: len(plain)] == plain and dst[len(plain):] == b"\xa5" * 7, k
    finally:
        ctx.close()


def test_few_large_streams_with_failed_and_crafted_ones(ctx, oracle):
    """The <= 16-stream route of pass 2 (pointer jumping, one stream after another through the same
    tables): large streams, and between them one that fails at its first header (written = 0), a
    truncated one, one with too small a destination and a crafted run of one distance."""
    streams, caps = [], []
    for kind, size, seed in (("dynamic", 3 << 20, 1), ("repetitive", 4 << 20, 3), ("dynamic", 1 << 20, 4)):
        plain, comp = T.make_stream(kind, size, 8800 + seed)
        streams.append(comp)
        caps.append(len(plain))
    streams.append(bytes.fromhex("0700"))                 # BTYPE 3 at once: written = 0
    caps.append(1 << 20)
    name, crafted, n = max(T.crafted_lz_streams(), key=lambda c: c[2])
    streams.append(crafted)
    caps.append(n)
    streams.append(streams[0][: len(streams[0]) // 2])   # truncated in the middle of a block
    caps.append(caps[0])
    streams.append(streams[2])                            # destination too small
    caps.append(caps[2] - 12345)
    b = T.Batch(streams, caps, dst_align=1)
    assert b.dst_total // b.n >= 1 << 20                  # (the large-stream route)
    st, wr, dst = gpu_util.run_device(ctx, b)
    dst_o = b.new_dst()
    ost, owr, _ = oracle.decompress_batch(b.src, b.src_off, b.src_len, dst_o, b.dst_off, b.dst_cap, 8)
    assert (st == ost).all() and (wr == owr).all()
    assert (dst == dst_o).all()
    assert list(st[:3]) == [0, 0, 0] and (st[3], wr[3]) == (2, 0) and (st[4], wr[4]) == (0, n) and st[6] == 4


@pytest.mark.parametrize("dst_align", [1, 16])
def test_stored_streams_copy_kernel(oracle, dst_align):
    """A sorted batch (>= 64 streams) of stored-block shapes (tests.block_cases.stored_lz_streams:
    every payload length, chains, stored blocks before a Huffman or BTYPE 3 header, truncations,
    LEN != ~NLEN, short destinations, an empty input) with the stored-stream copy kernel (default)
    and without it (SFB200_NO_STORED=1: the lane kernel decodes them): status, written and bytes
    the same three ways with the oracle, nothing outside the regions changed."""
    import starflate_b200 as S
    cases = B.stored_lz_streams() * 3
    b = T.Batch([c[1] for c in cases], [c[2] for c in cases], dst_align=dst_align)
    dst_o = b.new_dst()
    ost, owr, _ = oracle.decompress_batch(b.src, b.src_off, b.src_len, dst_o, b.dst_off, b.dst_cap)
    mask = np.ones(b.dst_total, dtype=bool)
    for k in range(b.n):
        mask[int(b.dst_off[k]):int(b.dst_off[k]) + int(b.dst_cap[k])] = False
    for env in ("0", "1"):
        os.environ["SFB200_NO_STORED"] = env
        try:
            c = S.Context(0)
        finally:
            del os.environ["SFB200_NO_STORED"]
        try:
            st, wr, dst = gpu_util.run_device(c, b)
        finally:
            c.close()
        bad = [cases[k][0] for k in range(b.n) if (st[k], wr[k]) != (ost[k], owr[k]) or
               not (b.dst_slice(dst, k) == b.dst_slice(dst_o, k)).all()]
        assert not bad, (env, bad[:5])
        assert (dst[mask] == 0xA5).all(), env
