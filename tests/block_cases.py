"""Test-side inputs for the block-level kernels (tests/test_block_kernels_cpu.py and
tests/test_gpu_block_kernels.py): DEFLATE streams written with tests.deflate_tools' bit writer."""
from __future__ import annotations

import numpy as np

from tests import deflate_tools as D


def tile_edge_lz_streams(qs=(0, 1, 77, 127), lengths=(3, 257, 258), dists=(1, 2, 300, 32768), offsets=range(-290, 2),
                         tile=1024):
    """Fixed-Huffman streams with ONE match, whose head sits at every offset in [T - 290, T + 2) of a
    tile edge T of pass 2 of the single-stream route (lz_jump.cuh: JUMP_TILE bytes of output per warp;
    a tile takes the match that reaches into it from the last head in the 288 bytes before it).  T
    counts from the 128-byte boundary below the stream's first byte, which lies q bytes after it: the
    stream is meant for a dst region at phase q.  A 258-byte match at T - 258 ends at T and must not
    be carried into the tile, one at T - 257 must.  `offsets`: a subset of [-290, 2), the head at T + offset.
    -> list of (name, q, compressed bytes, plain)"""
    out = []
    rng = np.random.default_rng(1024)
    for dist in dists:
        T = tile * ((dist + 290 + 127) // tile + 1)       # (room for the match's source before it)
        lits = rng.integers(32, 127, T + 300).astype(np.uint8).tobytes()
        w = D.BitWriter()
        blk = D.fixed_block(w, True)
        ends = [len(w)]
        for b in lits[:T + 2]:
            blk.literal(b)
            ends.append(len(w))
        prefix = np.array(w.bits, dtype=np.uint8)        # header + literals; literal k ends at ends[k + 1]
        for q in qs:
            for h in (T + o - q for o in offsets):
                for ln in lengths:
                    t = D.BitWriter()
                    tb = D.HuffBlock(t, D.FIXED_LIT_LENS, D.FIXED_DIST_LENS)
                    tb.match(ln, dist)
                    for b in lits[h:h + 40]:
                        tb.literal(b)
                    tb.eob()
                    bits = np.concatenate([prefix[:ends[h]], np.array(t.bits, dtype=np.uint8)])
                    plain = bytearray(lits[:h])
                    for j in range(ln):
                        plain.append(plain[-dist])
                    plain += lits[h:h + 40]
                    out.append((f"q{q}_h{h}_l{ln}_d{dist}", q, np.packbits(bits, bitorder="little").tobytes(),
                                bytes(plain)))
    return out


STORED_PAYLOAD_LENGTHS = (0, 1, 3, 4, 15, 16, 17, 31, 32, 33, 63, 64, 65, 511, 512, 513, 4096, 65535)


def stored_lz_streams():
    """Streams that start with a STORED block, for the sorted batch's stored-stream copy
    (stored_copy.cuh) and its preparation (lz_warp.cuh: prep kernels), with a few of the other
    first-block types around them: every payload length of STORED_PAYLOAD_LENGTHS as one final block,
    chains of 1-4 stored blocks, stored blocks followed by a fixed, a dynamic or a BTYPE 3 header,
    truncations inside LEN / NLEN and inside the payload, LEN != ~NLEN in block 2, input that ends
    after a non-final block, destinations that end at a block boundary or one byte short of it, an
    empty input.  -> list of (name, compressed bytes, dst capacity)"""
    rng = np.random.default_rng(16)
    pay = lambda n: rng.integers(0, 256, n).astype(np.uint8).tobytes()
    out = []
    for n in STORED_PAYLOAD_LENGTHS:
        out.append((f"len{n}", D.BitWriter().stored(True, pay(n)).tobytes(), n + 3))
    chains = ((5,), (100, 17), (3, 0, 4096), (1, 2, 33, 513), (0, 0), (64, 65, 63, 16))
    for lens in chains:
        w = D.BitWriter()
        for k, n in enumerate(lens):
            w.stored(k == len(lens) - 1, pay(n))
        total = sum(lens)
        out.append((f"chain{'_'.join(map(str, lens))}", w.tobytes(), total))
        bounds = np.cumsum(lens)
        for k in range(len(lens) - 1):                   # dst at a block boundary, one byte short of it
            if bounds[k] > 0:
                out.append((f"chain{'_'.join(map(str, lens))}_cap{bounds[k]}", w.tobytes(), int(bounds[k])))
                out.append((f"chain{'_'.join(map(str, lens))}_cap{bounds[k] - 1}", w.tobytes(), int(bounds[k]) - 1))
    text = D.text_like(3000, 16)
    for n_stored in (1, 2):
        head = D.BitWriter()
        for k in range(n_stored):
            head.stored(False, pay(37 * k + 20))
        before = sum(37 * k + 20 for k in range(n_stored))
        w = D.BitWriter()
        w.bits = list(head.bits)
        blk = D.fixed_block(w, True)
        for b in b"fixed block":
            blk.literal(b)
        blk.match(20, 5)
        blk.eob()
        out.append((f"stored{n_stored}_fixed", w.tobytes(), before + 31))
        out.append((f"stored{n_stored}_dynamic", head.tobytes() + D.raw_deflate(text, 6), before + len(text)))
        out.append((f"stored{n_stored}_btype3", head.tobytes() + bytes([0x07, 0x12]), before + 10))
        out.append((f"stored{n_stored}_ends", head.tobytes(), before + 10))    # input ends after a non-final block
    one = D.BitWriter().stored(False, pay(40)).tobytes()
    two = D.BitWriter().stored(True, pay(300)).tobytes()
    for cut in range(1, 5):                              # inside LEN / NLEN of block 1 and of block 2
        out.append((f"cut_lennlen1_{cut}", two[:cut], 400))
        out.append((f"cut_lennlen2_{cut}", one + two[:cut], 400))
    for cut in (5, 6, 100, len(two) - 1):                # inside the payload
        out.append((f"cut_payload1_{cut}", two[:cut], 400))
        out.append((f"cut_payload2_{cut}", one + two[:cut], 400))
    bad = D.BitWriter().stored(True, pay(9), nlen=0x1234).tobytes()
    out.append(("nlen_mismatch2", one + bad, 100))
    out.append(("empty", b"", 10))
    # the other first-block types, so that the batch has all four classes
    out.append(("dynamic", D.raw_deflate(text, 6), len(text)))
    out.append(("fixed", D.raw_deflate(text, 6, 4), len(text)))   # (zlib.Z_FIXED)
    out.append(("btype3", bytes([0x07, 0x00]), 10))
    return out
