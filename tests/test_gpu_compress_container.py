"""GPU: compression to zlib, gzip and BGZF (sfb200_compress_container*, sfb200_compress_bgzf*) checked by
Python's zlib / gzip, by this library's own decoders and against the raw compressor's output — a ragged
batch of per-stream containers with their capacity edges, BGZF files from 0 bytes to 256 MiB and one of
more than 4 GiB, rounds forced by a small scratch budget, DstTooSmall without a byte touched past
dst_cap, host / device / C++ agreement and the launches per round."""
import gzip
import os
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest
import torch

from starflate_b200 import build
from tests import deflate_tools as T
from tests import gzip_file_tools as G

pytestmark = pytest.mark.gpu

RAW, ZLIB, GZIP, AUTO = 0, 1, 2, 3
OK, DST_SMALL = 0, 4
P = G.PIECE
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GZIP_HEADER = bytes.fromhex("1f8b08000000000000ff")
BGZF_HEADER = bytes.fromhex("1f8b08040000000000ff060042430200")  # up to BSIZE


def dev(ctx):
    return torch.device("cuda", ctx.device)


def to_dev(ctx, b: bytes):
    if not b:
        return torch.zeros(0, dtype=torch.uint8, device=dev(ctx))
    return torch.from_numpy(np.frombuffer(b, np.uint8).copy()).to(dev(ctx))


def i64(ctx, v):
    return torch.tensor([int(x) for x in v], dtype=torch.int64, device=dev(ctx))


def ragged_streams():
    rnd = np.random.default_rng(3)
    return [T.big_text(100_000, 1), b"a" * 70_000, bytes(rnd.integers(0, 256, 50_000, dtype=np.uint8)), b"", b"x",
            b"ab", b"abc", T.big_text(17, 2), T.big_text(65_536, 3), bytes(rnd.integers(0, 4, 3_333, dtype=np.uint8)),
            T.big_text(300_000, 4), b"\0" * 5]


def batch(ctx, container, streams, caps):
    """One compress_container_batch_device call, streams at odd offsets -> [(status, bytes)]."""
    so, at = [], 3
    for s in streams:
        so.append(at)
        at += len(s) + 5
    src = bytearray(at + 16)
    for o, s in zip(so, streams):
        src[o:o + len(s)] = s
    do, at = [], 7
    for c in caps:
        do.append(at)
        at += c + 9
    d_src = to_dev(ctx, bytes(src))
    d_dst = torch.full((at + 16,), 0xA5, dtype=torch.uint8, device=dev(ctx))
    n = len(streams)
    st = torch.full((n,), 0xEE, dtype=torch.uint8, device=dev(ctx))
    wr = torch.zeros(n, dtype=torch.int64, device=dev(ctx))
    ctx.compress_container_batch_device(container, d_src, i64(ctx, so), i64(ctx, [len(s) for s in streams]), d_dst,
                                        i64(ctx, do), i64(ctx, caps), st, wr)
    torch.cuda.synchronize()
    dst = d_dst.cpu().numpy().tobytes()
    out = []
    for i in range(n):
        w = int(wr[i])
        assert w <= caps[i]
        assert dst[do[i] - 7:do[i]] == b"\xa5" * 7  # nothing in front of the region
        out.append((int(st[i]), dst[do[i]:do[i] + w]))
    return out


def test_container_batch(ctx):
    streams = ragged_streams()
    raw = batch(ctx, RAW, streams, [ctx.compress_container_bound(RAW, len(s)) for s in streams])
    assert all(st == OK for st, _ in raw)
    for container, hb, tb in ((ZLIB, 2, 4), (GZIP, 10, 8)):
        res = batch(ctx, container, streams, [ctx.compress_container_bound(container, len(s)) for s in streams])
        for s, (st, out), (_, r) in zip(streams, res, raw):
            assert st == OK
            assert out[hb:-tb] == r  # the payload is the raw compressor's stream
            if container == ZLIB:
                assert out[:2] == b"\x78\x9c" and out[-4:] == struct.pack(">I", zlib.adler32(s))
                assert zlib.decompress(out) == s
            else:
                assert out[:10] == GZIP_HEADER and out[-8:] == struct.pack("<II", zlib.crc32(s), len(s))
                assert gzip.decompress(out) == s
        # every stream back through the container decoder under AUTO
        comp = [o for _, o in res]
        so = np.cumsum([0] + [len(c) for c in comp[:-1]])
        do = np.cumsum([0] + [len(s) for s in streams[:-1]])
        total = sum(len(s) for s in streams)
        d_dst = torch.zeros(total + 16, dtype=torch.uint8, device=dev(ctx))
        n = len(streams)
        st = torch.zeros(n, dtype=torch.uint8, device=dev(ctx))
        wr = torch.zeros(n, dtype=torch.int64, device=dev(ctx))
        ctx.decompress_container_batch_device(AUTO, to_dev(ctx, b"".join(comp)), i64(ctx, so),
                                              i64(ctx, [len(c) for c in comp]), d_dst, i64(ctx, do),
                                              i64(ctx, [len(s) for s in streams]), st, wr)
        torch.cuda.synchronize()
        assert int(st.max()) == 0 and wr.cpu().tolist() == [len(s) for s in streams]
        assert d_dst[:total].cpu().numpy().tobytes() == b"".join(streams)


def test_container_capacity_edges(ctx):
    for container, frame in ((ZLIB, 6), (GZIP, 18)):
        for s in (T.big_text(10_000, 5), b"", b"q"):
            st, out = ctx.compress_container(container, s)
            assert st == OK
            assert ctx.compress_container(container, s, len(out)) == (OK, out)
            assert ctx.compress_container(container, s, len(out) - 1) == (DST_SMALL, b"")
            assert ctx.compress_container(container, s, frame - 1) == (DST_SMALL, b"")
            res = batch(ctx, container, [s, s, s, s], [len(out), len(out) - 1, frame - 1, 0])
            assert res == [(OK, out), (DST_SMALL, b""), (DST_SMALL, b""), (DST_SMALL, b"")]
    with pytest.raises(Exception, match="BAD_ARGUMENT"):
        ctx.compress_container(AUTO, b"abc", 100)


def members_of(f: bytes):
    """Parse a BGZF file in Python -> [(member bytes)]; every header has a valid BC subfield."""
    out, p = [], 0
    while p < len(f):
        assert f[p:p + 16] == BGZF_HEADER, p
        bsize = struct.unpack_from("<H", f, p + 16)[0]
        assert bsize <= 0xffff
        out.append(f[p:p + bsize + 1])
        p += bsize + 1
    assert p == len(f)
    return out


def raw_pieces(ctx, data: bytes):
    """compress_batch_device over the pieces split on the host -> their raw-DEFLATE streams"""
    pieces = [data[i:i + P] for i in range(0, len(data), P)]
    if not pieces:
        return []
    caps = [ctx.compress_container_bound(RAW, len(p)) for p in pieces]
    d_src = to_dev(ctx, data)
    n = len(pieces)
    co = np.cumsum([0] + caps[:-1])
    d_dst = torch.zeros(sum(caps) + 16, dtype=torch.uint8, device=dev(ctx))
    st = torch.zeros(n, dtype=torch.uint8, device=dev(ctx))
    wr = torch.zeros(n, dtype=torch.int64, device=dev(ctx))
    ctx.compress_batch_device(d_src, i64(ctx, range(0, len(data), P)), i64(ctx, [len(p) for p in pieces]), d_dst,
                              i64(ctx, co), i64(ctx, caps), st, wr)
    torch.cuda.synchronize()
    assert int(st.max()) == 0
    d = d_dst.cpu().numpy().tobytes()
    return [d[o:o + w] for o, w in zip(co.tolist(), wr.cpu().tolist())]


def check_bgzf(ctx, data: bytes, f: bytes):
    n = -(-len(data) // P)
    ms = members_of(f)
    assert len(ms) == n + 1 and ms[-1] == G.BGZF_EOF
    for k, (m, r) in enumerate(zip(ms[:-1], raw_pieces(ctx, data))):
        piece = data[k * P:(k + 1) * P]
        assert m[18:-8] == r, k
        assert m[-8:] == struct.pack("<II", zlib.crc32(piece), len(piece))
    if len(data) <= 9 << 20:  # (gzip.decompress copies the rest of the file once per member)
        assert gzip.decompress(f) == data
    assert ctx.gzip_file_size(f) == (len(data), n + 1, True)
    d = torch.full((len(data) + 3,), 0xA5, dtype=torch.uint8, device=dev(ctx))
    assert ctx.decompress_gzip_file_device(to_dev(ctx, f), d) == (OK, len(data), n + 1)
    assert d[:len(data)].cpu().numpy().tobytes() == data
    if shutil.which("gzip"):
        r = subprocess.run(["gzip", "-dc"], input=f, capture_output=True, check=True)
        assert r.stdout == data


@pytest.mark.parametrize("size", [0, 1, P - 1, P, P + 1, 3 * P, "text9", "random64", "text256"])
def test_bgzf_files(ctx, size):
    if size == "text9":
        data = T.big_text(9 << 20, 9)
    elif size == "random64":
        data = np.random.default_rng(64).integers(0, 256, 64 << 20, dtype=np.uint8).tobytes()
    elif size == "text256":
        data = T.big_text(256 << 20, 11)
    else:
        data = T.big_text(size, size) if size else b""
    st, f, members = ctx.compress_bgzf(data)
    assert st == OK and members == -(-len(data) // P) + 1
    if not data:
        assert f == G.BGZF_EOF
    check_bgzf(ctx, data, f)


def test_host_device_cpp_agree_and_repeat(ctx, tmp_path):
    build.build_all()
    exe = str(tmp_path / "compress_test")
    subprocess.check_call(["g++", "-std=c++23", "-O1", "-fno-exceptions", "-w", "-pthread",
                           "-I", os.path.join(ROOT, "starflate_b200", "cpp"), "-I", os.path.join(ROOT, "include"),
                           "-o", exe, os.path.join(ROOT, "tests", "cpp", "compress_test.cpp"), "-L", build.OUT,
                           "-lstarflate", "-lstarflate_b200", f"-Wl,-rpath,{build.OUT}"])
    for data in (T.big_text(3 * P + 77, 21), b"", np.random.default_rng(2).integers(0, 256, 200_000, np.uint8).tobytes()):
        st, f, nm = ctx.compress_bgzf(data)
        assert st == OK and ctx.compress_bgzf(data) == (st, f, nm)  # two runs
        d = torch.zeros(ctx.compress_bgzf_bound(len(data)), dtype=torch.uint8, device=dev(ctx))
        st2, wr2, nm2 = ctx.compress_bgzf_device(to_dev(ctx, data), d)
        assert (st2, wr2, nm2) == (OK, len(f), nm) and d[:wr2].cpu().numpy().tobytes() == f
        inp = tmp_path / "in.bin"
        inp.write_bytes(data)
        for kind, want in (("bgzf", f), ("raw", ctx.compress_container(RAW, data)[1]),
                           ("zlib", ctx.compress_container(ZLIB, data)[1]),
                           ("gzip", ctx.compress_container(GZIP, data)[1])):
            out = tmp_path / f"out.{kind}"
            r = subprocess.run([exe, str(inp), kind, str(out)], capture_output=True, text=True)
            assert r.returncode == 0, r.stdout + r.stderr
            assert r.stdout.split()[:2] == ["0", str(len(want))], (kind, r.stdout)
            assert out.read_bytes() == want, kind


def test_bgzf_limits(ctx):
    data = T.big_text(5 * P + 1000, 31)
    st, f, nm = ctx.compress_bgzf(data)
    assert st == OK
    src = to_dev(ctx, data)
    guard = 4096
    for cap in (len(f) - 1, len(f) - 28, 100, 27, 0):
        d = torch.full((cap + guard,), 0x5A, dtype=torch.uint8, device=dev(ctx))
        assert ctx.compress_bgzf_device(src, d[:cap]) == (DST_SMALL, 0, 0)
        assert bool((d[cap:] == 0x5A).all())  # no byte past dst_cap
        assert ctx.compress_bgzf(data, cap) == (DST_SMALL, b"", 0)
    assert ctx.compress_bgzf(b"", 27) == (DST_SMALL, b"", 0)
    # incompressible data: every member stored, the bound reached exactly and enough
    rnd = np.random.default_rng(9).integers(0, 256, 7 * P, dtype=np.uint8).tobytes()
    bound = ctx.compress_bgzf_bound(len(rnd))
    assert bound == 7 * 65_311 + 28 and ctx.compress_bgzf_bound(0) == 28
    st, f, nm = ctx.compress_bgzf(rnd, bound)
    assert st == OK and nm == 8 and len(f) <= bound
    check_bgzf(ctx, rnd, f)


def test_rounds_give_the_same_bytes_and_constant_launches(ctx):
    data = T.big_text(100 * P + 5, 41)
    pieces = 101
    before = ctx.launch_info()["kernel_launches"]
    st, want, nm = ctx.compress_bgzf(data)
    assert ctx.launch_info()["kernel_launches"] - before == 5  # one round
    for mb, slots in (("1", 16), ("2", 32), ("7", 112)):
        os.environ["SFB200_BGZF_SCRATCH_MB"] = mb
        try:
            before = ctx.launch_info()["kernel_launches"]
            assert ctx.compress_bgzf(data) == (st, want, nm)
            rounds = -(-pieces // slots)
            assert ctx.launch_info()["kernel_launches"] - before == 5 * rounds
        finally:
            del os.environ["SFB200_BGZF_SCRATCH_MB"]
    check_bgzf(ctx, data, want)


def test_bgzf_over_4_gib(ctx):
    n = (4 << 30) + 123_457
    d = dev(ctx)
    g = torch.Generator(device=d)
    g.manual_seed(7)
    src = torch.randint(0, 8, (n,), dtype=torch.uint8, device=d, generator=g)  # 3 bits of entropy per byte
    bound = ctx.compress_bgzf_bound(n)
    out = torch.empty(bound, dtype=torch.uint8, device=d)
    st, wr, nm = ctx.compress_bgzf_device(src, out)
    pieces = -(-n // P)
    assert (st, nm) == (OK, pieces + 1) and wr < n // 2
    back = torch.empty(n + 64, dtype=torch.uint8, device=d)
    assert ctx.decompress_gzip_file_device(out[:wr], back) == (OK, n, pieces + 1)
    zero, ln = torch.zeros(1, dtype=torch.int64, device=d), torch.full((1,), n, dtype=torch.int64, device=d)
    s0, s1 = torch.zeros(1, dtype=torch.int64, device=d), torch.zeros(1, dtype=torch.int64, device=d)
    ctx.checksum_batch_device(src, zero, ln, s0)
    ctx.checksum_batch_device(back, zero, ln, s1)
    torch.cuda.synchronize()
    assert int(s0[0]) == int(s1[0])
    assert out[wr - 28:wr].cpu().numpy().tobytes() == G.BGZF_EOF
