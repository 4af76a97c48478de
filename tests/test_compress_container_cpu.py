"""CPU emulation of writing zlib, gzip and BGZF (starflate_b200/csrc/container_write.cuh with the
unchanged compression kernel, built for the host by tests/cpu_emu/emu_compress_container.cpp): the
output must decode with Python's zlib / gzip, its headers and trailers must be byte-exact, and a
BGZF file must be the same whatever the round size — at every input phase mod 16 and at the sizes
around the piece size."""
import ctypes as C
import gzip
import io
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from tests import gzip_file_tools as G

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)
ZLIB, GZIP = 1, 2
OK, DST_SMALL = 0, 4
GZIP_HEADER = bytes.fromhex("1f8b08000000000000ff")
BGZF_HEADER = bytes.fromhex("1f8b08040000000000ff060042430200")  # up to BSIZE
P = 500  # the piece size in these tests (the library's is 65 280): many members from small inputs


@pytest.fixture(scope="module")
def emu():
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
    lib.emu_compress_bgzf.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, _u64p,
                                      _u64p]
    lib.emu_compress_bgzf.restype = C.c_int
    return lib


def gzipfile_header(s: bytes) -> bytes:
    """The first 10 bytes of what Python's GzipFile writes at level 6 with MTIME 0 (OS 255, unknown)."""
    b = io.BytesIO()
    with gzip.GzipFile(fileobj=b, mode="wb", compresslevel=6, mtime=0) as g:
        g.write(s)
    return b.getvalue()[:10]


def text(n: int, seed: int) -> bytes:
    rnd = np.random.default_rng(seed)
    words = [b"alpha ", b"beta ", b"gamma ", b"delta\n", b"epsilon ", b"zeta, ", b"eta. "]
    out = b"".join(words[i] for i in rnd.integers(0, len(words), size=n // 4 + 1))
    return out[:n]


def payload_bound(n: int) -> int:
    return n + 5 * max(1, (n + 65534) // 65535)


def containers(lib, container, streams, caps=None, phase=0):
    """-> [(status, bytes written)] for a batch; every stream at `phase` mod 16 in src and dst."""
    hb, tb = (2, 4) if container == ZLIB else (10, 8)
    if caps is None:
        caps = [payload_bound(len(s)) + hb + tb for s in streams]
    so, at = [], 16 + phase
    for s in streams:
        so.append(at)
        at += (len(s) + 47) // 16 * 16
    src = np.zeros(at + 32, np.uint8)
    for o, s in zip(so, streams):
        src[o:o + len(s)] = np.frombuffer(s, np.uint8)
    do, at = [], 16 + (phase * 7) % 16
    for c in caps:
        do.append(at)
        at += (c + 47) // 16 * 16
    dst = np.full(at + 32, 0xA5, np.uint8)
    n = len(streams)
    arr = lambda v: np.array(v, np.uint64)
    so, sl, do_, dc = arr(so), arr([len(s) for s in streams]), arr(do), arr(caps)
    st, wr = np.full(n, 0xEE, np.uint8), np.zeros(n, np.uint64)
    p = lambda a: a.ctypes.data_as(_u64p)
    lib.emu_compress_container(container, src.ctypes.data, p(so), p(sl), dst.ctypes.data, p(do_), p(dc),
                               st.ctypes.data_as(_u8p), p(wr), n)
    out = []
    for i in range(n):
        w = int(wr[i])
        assert w <= caps[i]
        out.append((int(st[i]), dst[do[i]:do[i] + w].tobytes()))
        assert (dst[do[i] - 16:do[i]] == 0xA5).all()  # nothing written in front of the region
    return out


def bgzf(lib, data: bytes, piece=P, round_=1 << 20, cap=None, phase=0):
    buf = np.zeros(len(data) + 48, np.uint8)
    s = buf[16 + phase:16 + phase + len(data)]
    s[:] = np.frombuffer(data, np.uint8)
    if cap is None:
        cap = -(-len(data) // piece) * (piece + 31) + 28
    dbuf = np.full(cap + 64, 0x5A, np.uint8)
    wr, nm = np.zeros(1, np.uint64), np.zeros(1, np.uint64)
    st = lib.emu_compress_bgzf(s.ctypes.data, len(data), piece, round_, dbuf[16:].ctypes.data, cap,
                               wr.ctypes.data_as(_u64p), nm.ctypes.data_as(_u64p))
    assert (dbuf[16 + cap:] == 0x5A).all() and (dbuf[:16] == 0x5A).all()  # nothing outside dst
    return st, dbuf[16:16 + int(wr[0])].tobytes(), int(nm[0])


def members_of(f: bytes):
    out, p = [], 0
    while p < len(f):
        assert f[p:p + 16] == BGZF_HEADER
        bsize = struct.unpack_from("<H", f, p + 16)[0]
        out.append(f[p:p + bsize + 1])
        p += bsize + 1
    assert p == len(f)
    return out


def test_zlib_and_gzip_every_phase(emu):
    streams = [text(0, 0), text(1, 1), text(3, 2), text(4, 3), text(15, 4), text(16, 5), text(17, 6),
               text(3000, 7), bytes(np.random.default_rng(8).integers(0, 256, 700, dtype=np.uint8))]
    for phase in range(16):
        for container in (ZLIB, GZIP):
            for s, (st, out) in zip(streams, containers(emu, container, streams, phase=phase)):
                assert st == OK
                if container == ZLIB:
                    assert out[:2] == b"\x78\x9c" and out[-4:] == struct.pack(">I", zlib.adler32(s))
                    assert zlib.decompress(out) == s
                else:
                    assert out[:10] == GZIP_HEADER == gzipfile_header(s)
                    assert out[-8:] == struct.pack("<II", zlib.crc32(s), len(s))
                    assert gzip.decompress(out) == s


def test_payload_is_the_raw_stream_and_capacity_edges(emu):
    s = text(2000, 11)
    for container, hb, tb in ((ZLIB, 2, 4), (GZIP, 10, 8)):
        (st, out), = containers(emu, container, [s])
        assert st == OK
        exact = len(out)
        raw = out[hb:-tb]
        assert zlib.decompress(raw, -15) == s
        # the exact size fits, one byte less does not, nor less than the frame itself
        res = containers(emu, container, [s, s, s, b"", b""], caps=[exact, exact - 1, hb + tb - 1, hb + tb - 1, 0])
        assert res[0] == (OK, out)
        assert [r[0] for r in res[1:]] == [DST_SMALL] * 4 and all(r[1] == b"" for r in res[1:])


@pytest.mark.parametrize("n", [0, 1, 3, 4, 15, 16, 17, P - 1, P, P + 1, 2 * P, 7 * P])
def test_bgzf_sizes(emu, n):
    data = text(n, n)
    st, f, members = bgzf(emu, data)
    assert st == OK and members == -(-n // P) + 1
    assert gzip.decompress(f) == data
    assert f.endswith(G.BGZF_EOF)
    ms = members_of(f)
    assert len(ms) == members and ms[-1] == G.BGZF_EOF
    for k, m in enumerate(ms[:-1]):
        piece = data[k * P:(k + 1) * P]
        assert len(m) - 1 <= 0xffff
        assert m[-8:] == struct.pack("<II", zlib.crc32(piece), len(piece))
        assert zlib.decompress(m[18:-8], -15) == piece
    if n == 0:
        assert f == G.BGZF_EOF


def test_bgzf_phases_and_rounds(emu):
    data = text(5 * P + 123, 99)
    st, want, members = bgzf(emu, data)
    assert st == OK and members == 7
    for phase in range(16):
        assert bgzf(emu, data, phase=phase) == (OK, want, 7)
    for r in (1, 2, 5, 6):  # rounds of r pieces: the same bytes
        assert bgzf(emu, data, round_=r, phase=r) == (OK, want, 7)


def test_bgzf_dst_too_small(emu):
    rnd = np.random.default_rng(5)
    data = bytes(rnd.integers(0, 256, 4 * P, dtype=np.uint8))  # incompressible: stored pieces
    bound = 4 * (P + 31) + 28
    st, f, members = bgzf(emu, data, cap=bound)
    assert st == OK and len(f) == bound and gzip.decompress(f) == data  # the bound is reached exactly
    for cap in (len(f) - 1, len(f) - 28, 27, 0):
        assert bgzf(emu, data, cap=cap, round_=2) == (DST_SMALL, b"", 0)
    assert bgzf(emu, b"", cap=27) == (DST_SMALL, b"", 0)
    assert bgzf(emu, b"", cap=28) == (OK, G.BGZF_EOF, 1)
