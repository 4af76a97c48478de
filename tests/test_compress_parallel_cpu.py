"""CPU emulation of compressing one buffer to one raw-DEFLATE / zlib / gzip stream
(starflate_b200/csrc/compress_parallel.cuh with the compressor's piece mode, built for the host by
tests/cpu_emu/emu_compress_parallel.cpp) with a small piece size: the stream must decode with Python's
zlib, its header and trailer must be byte-exact, a buffer of one piece must be exactly what the
one-stream container path writes, every Huffman piece must sit bit for bit at its B_k, stored pieces
must land at every bit phase, the round size must not change a byte, DstTooSmall must leave the bytes
past dst_cap alone, and the decoder's block finder must see every piece."""
import ctypes as C
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from tests.emu_bindings import Emu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)
RAW, ZLIB, GZIP = 0, 1, 2
OK, DST_SMALL = 0, 4
FRAME = {RAW: (0, 0), ZLIB: (2, 4), GZIP: (10, 8)}
WBITS = {RAW: -15, ZLIB: 15, GZIP: 31}
P = 500  # the piece size in these tests (the library's is 65 280)


@pytest.fixture(scope="module")
def par():
    out = os.path.join(HERE, "cpu_emu", "libemu_compress_parallel.so")
    csrc = os.path.join(ROOT, "starflate_b200", "csrc")
    srcs = [os.path.join(HERE, "cpu_emu", f) for f in ("emu_compress_parallel.cpp", "cuda_shim_warp.h")] + \
           [os.path.join(csrc, f) for f in ("compress_parallel.cuh", "container_write.cuh", "container.cuh",
                                            "deflate_compress.cuh", "deflate_lane.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-w", "-o", out, srcs[0]])
    lib = C.CDLL(out)
    lib.emu_compress_parallel.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p,
                                          C.c_uint64, _u64p, _u64p]
    lib.emu_compress_parallel.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def emu():
    return Emu()


@pytest.fixture(scope="module")
def cont():
    """the one-stream container path (tests/cpu_emu/emu_compress_container.cpp)"""
    out = os.path.join(HERE, "cpu_emu", "libemu_compress_container.so")
    csrc = os.path.join(ROOT, "starflate_b200", "csrc")
    srcs = [os.path.join(HERE, "cpu_emu", f) for f in ("emu_compress_container.cpp", "cuda_shim_warp.h")] + \
           [os.path.join(csrc, f) for f in ("container_write.cuh", "container.cuh", "deflate_compress.cuh",
                                            "deflate_lane.cuh", "gzip_file.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-w", "-o", out, srcs[0]])
    lib = C.CDLL(out)
    lib.emu_compress_container.argtypes = [C.c_int, C.c_void_p, _u64p, _u64p, C.c_void_p, _u64p, _u64p, _u8p, _u64p,
                                           C.c_uint64]
    lib.emu_compress_container.restype = None
    return lib


def container_one(lib, container, data: bytes):
    """one stream through the container path -> (status, bytes)"""
    hb, tb = FRAME[container]
    cap = len(data) + 5 * max(1, -(-len(data) // 65535)) + hb + tb
    src = np.zeros(len(data) + 64, np.uint8)
    src[16:16 + len(data)] = np.frombuffer(data, np.uint8)
    dst = np.zeros(cap + 64, np.uint8)
    arr = lambda v: np.array([v], np.uint64)
    so, sl, do, dc, wr = arr(16), arr(len(data)), arr(16), arr(cap), arr(0)
    st = np.zeros(1, np.uint8)
    p = lambda a: a.ctypes.data_as(_u64p)
    lib.emu_compress_container(container, src.ctypes.data, p(so), p(sl), dst.ctypes.data, p(do), p(dc),
                               st.ctypes.data_as(_u8p), p(wr), 1)
    return int(st[0]), dst[16:16 + int(wr[0])].tobytes()


def text(n: int, seed: int) -> bytes:
    rnd = np.random.default_rng(seed)
    words = [b"alpha ", b"beta ", b"gamma ", b"delta\n", b"epsilon ", b"zeta, ", b"eta. "]
    out = b"".join(words[i] for i in rnd.integers(0, len(words), size=n // 4 + 1))
    return out[:n]


def noise(n: int, seed: int) -> bytes:
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8).tobytes()


def bound(container, n, piece=P):
    hb, tb = FRAME[container]
    return hb + tb + n + 6 * max(1, -(-n // piece))


def parallel(lib, container, data: bytes, piece=P, round_=1 << 20, cap=None, phase=0):
    """-> (status, stream bytes, [B_0 .. B_pieces]); src at `phase` mod 16, guard bytes around dst."""
    buf = np.zeros(len(data) + 48, np.uint8)
    s = buf[16 + phase:16 + phase + len(data)]
    s[:] = np.frombuffer(data, np.uint8)
    if cap is None:
        cap = bound(container, len(data), piece)
    dbuf = np.full(cap + 64, 0x5A, np.uint8)
    pieces = max(1, -(-len(data) // piece))
    bits = np.zeros(pieces + 1, np.uint64)
    wr = np.zeros(1, np.uint64)
    st = lib.emu_compress_parallel(container, s.ctypes.data, len(data), piece, round_, dbuf[16:].ctypes.data, cap,
                                   wr.ctypes.data_as(_u64p), bits.ctypes.data_as(_u64p))
    assert (dbuf[16 + cap:] == 0x5A).all() and (dbuf[:16] == 0x5A).all()  # nothing outside dst
    return st, dbuf[16:16 + int(wr[0])].tobytes(), [int(b) for b in bits]


def check_frame(container, data: bytes, out: bytes):
    if container == ZLIB:
        assert out[:2] == b"\x78\x9c" and out[-4:] == struct.pack(">I", zlib.adler32(data))
    elif container == GZIP:
        assert out[:10] == bytes.fromhex("1f8b08000000000000ff")
        assert out[-8:] == struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff)
    assert zlib.decompress(out, WBITS[container]) == data


def bits_of(b: bytes, lo: int, hi: int) -> int:
    return (int.from_bytes(b, "little") >> lo) & ((1 << (hi - lo)) - 1)


@pytest.mark.parametrize("container", [RAW, ZLIB, GZIP])
def test_sizes_every_phase(par, container):
    for n in (0, 1, P - 1, P, P + 1, 3 * P, 10 * P + 7):
        data = text(n, n + 1)
        want = None
        for phase in range(16):
            st, out, bits = parallel(par, container, data, phase=phase)
            assert st == OK
            if want is None:
                check_frame(container, data, out)
                assert bits[0] == 8 * FRAME[container][0] and len(bits) == max(1, -(-n // P)) + 1
                assert len(out) == (bits[-1] + 7) // 8 + FRAME[container][1] <= bound(container, n)
                want = out
            assert out == want, (n, phase)


def test_one_piece_is_the_container_path(par, emu, cont):
    """n <= P: byte-identical to the one-stream path (RAW: the raw compressor; ZLIB / GZIP: the
    container path), including the empty input (03 00) and a stored fallback (01 LEN NLEN ..)"""
    for data in (b"", b"x", text(17, 2), text(P - 1, 3), text(P, 4), noise(P, 5), noise(37, 6)):
        st, raw = emu.compress(data, len(data) + 5)
        assert st == OK
        if not data:
            assert raw == b"\x03\x00"
        if data == noise(P, 5):
            assert raw[:5] == b"\x01" + struct.pack("<HH", P, P ^ 0xffff)
        st, out, bits = parallel(par, RAW, data)
        assert (st, out) == (OK, raw) and bits[0] == 0 and (bits[1] + 7) // 8 == len(raw)
        for container in (ZLIB, GZIP):
            cst, cout = container_one(cont, container, data)
            st, out, _ = parallel(par, container, data)
            assert cst == OK and (st, out) == (OK, cout)
            check_frame(container, data, out)


def test_huffman_pieces_are_the_raw_streams(par, emu):
    data = text(2 * P, 7) + noise(P, 8) + text(3 * P + 123, 9)
    pieces = [data[i:i + P] for i in range(0, len(data), P)]
    for container in (RAW, GZIP):
        st, out, bits = parallel(par, container, data)
        assert st == OK
        check_frame(container, data, out)
        for k, piece in enumerate(pieces):
            lo, hi = bits[k], bits[k + 1]
            st, raw = emu.compress(piece, len(piece) + 5)
            assert st == OK
            if raw[0] & 6 == 0:  # stored: BFINAL, BTYPE 00, padding, LEN, NLEN, bytes
                assert hi == ((lo + 3 + 7) & ~7) + 32 + 8 * len(piece)
                assert bits_of(out, lo, lo + 3) == (1 if k == len(pieces) - 1 else 0)
                q = (lo + 3 + 7) // 8
                assert out[q:q + 4 + len(piece)] == struct.pack("<HH", len(piece), len(piece) ^ 0xffff) + piece
                continue
            b = hi - lo
            assert 8 * len(raw) - 7 <= b <= 8 * len(raw)
            want = int.from_bytes(raw, "little") & ((1 << b) - 1)
            if k != len(pieces) - 1:
                want &= ~1  # BFINAL only on the last piece
            assert bits_of(out, lo, hi) == want, k
        # the padding of the last byte is zero
        end = bits[-1]
        hb, tb = FRAME[container]
        assert len(out) == (end + 7) // 8 + tb and (end % 8 == 0 or out[end // 8] >> (end % 8) == 0)


def test_stored_pieces_at_every_bit_phase(par):
    parts, kinds = [], []
    for k in range(48):
        if k % 2:
            parts.append(noise(P, 100 + k))
            kinds.append("stored")
        else:
            parts.append(text(P, 200 + k)[: P - (k * 7) % 40] + text((k * 7) % 40, 300 + k))
            kinds.append("text")
    data = b"".join(parts)
    for container in (RAW, ZLIB, GZIP):
        st, out, bits = parallel(par, container, data)
        assert st == OK
        check_frame(container, data, out)
        phases = {bits[k] % 8 for k, kd in enumerate(kinds) if kd == "stored"}
        assert phases == set(range(8)), phases
        for k, kd in enumerate(kinds):
            if kd == "stored":
                assert bits[k + 1] == ((bits[k] + 3 + 7) & ~7) + 32 + 8 * P


def test_rounds_give_the_same_bytes(par):
    data = text(3 * P, 1) + noise(P + 11, 2) + text(4 * P, 3) + noise(5, 4)
    for container in (RAW, ZLIB, GZIP):
        want = parallel(par, container, data)
        assert want[0] == OK
        check_frame(container, data, want[1])
        for r in (1, 2, 3, 5, 8):
            assert parallel(par, container, data, round_=r, phase=r) == want, (container, r)


def test_dst_too_small(par):
    data = text(3 * P + 9, 5)
    for container in (RAW, ZLIB, GZIP):
        st, out, _ = parallel(par, container, data)
        assert st == OK
        assert parallel(par, container, data, cap=len(out))[:2] == (OK, out)
        hb, tb = FRAME[container]
        for cap in (len(out) - 1, hb + tb - 1 if hb else 0, 0):
            for r in (1, 1 << 20):
                assert parallel(par, container, data, cap=cap, round_=r)[:2] == (DST_SMALL, b"")
    # incompressible input: every piece stored, within the bound
    rnd = noise(7 * P + 3, 6)
    for container in (RAW, ZLIB, GZIP):
        st, out, _ = parallel(par, container, rnd)
        assert st == OK and len(out) <= bound(container, len(rnd))
        check_frame(container, rnd, out)


def test_the_block_finder_sees_every_piece(par, emu):
    """text pieces of 8 KiB are dynamic blocks: the decoder's finder accepts every B_k, and the
    blocks-side-by-side route decodes the stream with every piece on the chain"""
    piece = 8192
    data = text(9 * piece + 1234, 77)
    st, out, bits = parallel(par, RAW, data, piece=piece)
    assert st == OK and zlib.decompress(out, -15) == data
    starts = bits[:-1]
    assert all(((out[b >> 3] | out[(b >> 3) + 1] << 8) >> (b & 7) >> 1) & 3 == 2 for b in starts)  # dynamic
    found = emu.find_blocks(out)
    assert set(starts[1:]) <= set(found), sorted(set(starts[1:]) - set(found))
    st, dst, wr, on_chain, tail = emu.stream_decompress_jobs(out, len(data), found)
    assert (st, wr) == (OK, len(data)) and dst == data
    assert on_chain == len(starts) and tail == len(starts) - 1
