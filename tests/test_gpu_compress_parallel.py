"""GPU: one buffer compressed to ONE raw-DEFLATE / zlib / gzip stream at batch speed
(sfb200_compress_parallel*), checked by Python's zlib / gzip, gzip(1) and this library's decoders — the
single-stream route side by side and one warp front to back, the container decoder, the gzip-file
decoder — against the one-stream container path for inputs of one piece, at the capacity edges, with
rounds forced by a small scratch budget, host / device / C++ agreement, and one input of more than
4 GiB."""
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
FRAME = {RAW: (0, 0), ZLIB: (2, 4), GZIP: (10, 8)}
WBITS = {RAW: -15, ZLIB: 15, GZIP: 31}
NAME = {RAW: "raw", ZLIB: "zlib", GZIP: "gzip"}


def dev(ctx):
    return torch.device("cuda", ctx.device)


def to_dev(ctx, b: bytes):
    if not b:
        return torch.zeros(0, dtype=torch.uint8, device=dev(ctx))
    return torch.from_numpy(np.frombuffer(b, np.uint8).copy()).to(dev(ctx))


def data_for(size):
    if size == "text9":
        return T.big_text(9 << 20, 9)
    if size == "random64":
        return np.random.default_rng(64).integers(0, 256, 64 << 20, dtype=np.uint8).tobytes()
    if size == "text256":
        return T.big_text(256 << 20, 11)
    return T.big_text(size, size) if size else b""


def check_stream(ctx, container, data: bytes, out: bytes):
    hb, tb = FRAME[container]
    if container == ZLIB:
        assert out[:2] == b"\x78\x9c" and out[-4:] == struct.pack(">I", zlib.adler32(data))
    elif container == GZIP:
        assert out[:10] == bytes.fromhex("1f8b08000000000000ff")
        assert out[-8:] == struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff)
    assert zlib.decompress(out, WBITS[container]) == data
    if container == GZIP:
        assert gzip.decompress(out) == data
    if container != RAW and shutil.which("gzip") and len(data) <= 64 << 20:
        # gzip(1) reads gzip and (as gzip -dc of a zlib stream does not) nothing else: wrap zlib's payload
        payload = out if container == GZIP else bytes.fromhex("1f8b08000000000000ff") + out[2:-4] + \
            struct.pack("<II", zlib.crc32(data), len(data) & 0xffffffff)
        r = subprocess.run(["gzip", "-dc"], input=payload, capture_output=True, check=True)
        assert r.stdout == data
    cap = len(data) + 64
    if container == RAW:
        st, d, wr = ctx.decompress(out, cap)  # the single-stream route: blocks side by side
        assert (st, wr) == (OK, len(data)) and d[:wr] == data
        os.environ["SFB200_BLOCKS"] = "0"  # one warp front to back
        try:
            st, d, wr = ctx.decompress(out, cap)
        finally:
            del os.environ["SFB200_BLOCKS"]
        assert (st, wr) == (OK, len(data)) and d[:wr] == data
    else:
        st, d, wr = ctx.decompress_container(container, out, cap)
        assert (st, wr) == (OK, len(data)) and d[:wr] == data
    if container == GZIP:
        st, d, wr, members = ctx.decompress_gzip_file(out, cap)
        assert (st, wr, members) == (OK, len(data), 1) and d[:wr] == data


@pytest.mark.parametrize("size", [0, 1, P - 1, P, P + 1, 3 * P, "text9", "random64", "text256"])
def test_streams(ctx, size):
    data = data_for(size)
    for container in (RAW, ZLIB, GZIP):
        st, out = ctx.compress_parallel(container, data)
        assert st == OK and len(out) <= ctx.compress_parallel_bound(container, len(data))
        check_stream(ctx, container, data, out)
        if len(data) <= P:  # one piece: the one-stream container path's bytes
            assert (st, out) == ctx.compress_container(container, data)
        elif container == GZIP and size not in ("random64", "text256"):
            st_b, bgzf, _ = ctx.compress_bgzf(data)
            assert st_b == OK and len(out) < len(bgzf)  # no per-member frames


def test_capacity(ctx):
    data = T.big_text(5 * P + 1000, 31)
    src = to_dev(ctx, data)
    guard = 4096
    for container in (RAW, ZLIB, GZIP):
        st, out = ctx.compress_parallel(container, data)
        assert st == OK
        assert ctx.compress_parallel(container, data, len(out)) == (OK, out)
        hb, tb = FRAME[container]
        for cap in sorted({len(out) - 1, max(hb + tb - 1, 0), 0}):
            d = torch.full((cap + guard,), 0x5A, dtype=torch.uint8, device=dev(ctx))
            assert ctx.compress_parallel_device(container, src, d[:cap]) == (DST_SMALL, 0)
            assert bool((d[cap:] == 0x5A).all())  # no byte past dst_cap
            assert ctx.compress_parallel(container, data, cap) == (DST_SMALL, b"")
        # incompressible data: every piece stored, the bound is enough
        rnd = np.random.default_rng(9).integers(0, 256, 7 * P, dtype=np.uint8).tobytes()
        bound = ctx.compress_parallel_bound(container, len(rnd))
        assert bound == hb + tb + 7 * P + 42
        assert ctx.compress_parallel_bound(container, 0) == hb + tb + 6
        assert ctx.compress_parallel_bound(container, P) == hb + tb + P + 6
        st, out = ctx.compress_parallel(container, rnd, bound)
        assert st == OK and len(out) <= bound
        check_stream(ctx, container, rnd, out)
    with pytest.raises(Exception, match="BAD_ARGUMENT"):
        ctx.compress_parallel(AUTO, b"abc", 100)


def test_rounds_give_the_same_bytes_and_constant_launches(ctx):
    data = T.big_text(100 * P + 5, 41)
    pieces = 101
    for container in (RAW, GZIP):
        before = ctx.launch_info()["kernel_launches"]
        st, want = ctx.compress_parallel(container, data)
        assert st == OK and ctx.launch_info()["kernel_launches"] - before == 5  # one round
        for mb, slots in (("1", 16), ("2", 32), ("7", 112)):
            os.environ["SFB200_BGZF_SCRATCH_MB"] = mb
            try:
                before = ctx.launch_info()["kernel_launches"]
                assert ctx.compress_parallel(container, data) == (st, want)
                rounds = -(-pieces // slots)
                assert ctx.launch_info()["kernel_launches"] - before == 5 * rounds
            finally:
                del os.environ["SFB200_BGZF_SCRATCH_MB"]
        check_stream(ctx, container, data, want)


def test_host_device_cpp_agree_and_repeat(ctx, tmp_path):
    build.build_all()
    exe = str(tmp_path / "compress_parallel_test")
    subprocess.check_call(["g++", "-std=c++23", "-O1", "-fno-exceptions", "-w", "-pthread",
                           "-I", os.path.join(ROOT, "starflate_b200", "cpp"), "-I", os.path.join(ROOT, "include"),
                           "-o", exe, os.path.join(ROOT, "tests", "cpp", "compress_parallel_test.cpp"), "-L", build.OUT,
                           "-lstarflate", "-lstarflate_b200", f"-Wl,-rpath,{build.OUT}"])
    rnd = np.random.default_rng(2)
    mixed = T.big_text(2 * P + 77, 21) + rnd.integers(0, 256, P + 3, np.uint8).tobytes() + T.big_text(P, 22)
    for data in (T.big_text(3 * P + 77, 21), b"", mixed):
        inp = tmp_path / "in.bin"
        inp.write_bytes(data)
        for container in (RAW, ZLIB, GZIP):
            st, f = ctx.compress_parallel(container, data)
            assert st == OK and ctx.compress_parallel(container, data) == (st, f)  # two runs
            d = torch.zeros(ctx.compress_parallel_bound(container, len(data)), dtype=torch.uint8, device=dev(ctx))
            st2, wr2 = ctx.compress_parallel_device(container, to_dev(ctx, data), d)
            assert (st2, wr2) == (OK, len(f)) and d[:wr2].cpu().numpy().tobytes() == f
            out = tmp_path / f"out.{NAME[container]}"
            r = subprocess.run([exe, str(inp), NAME[container], str(out)], capture_output=True, text=True)
            assert r.returncode == 0, r.stdout + r.stderr
            assert r.stdout.split()[:2] == ["0", str(len(f))], (container, r.stdout)
            assert out.read_bytes() == f, container
            check_stream(ctx, container, data, f)


def test_gzip_over_4_gib(ctx):
    n = (4 << 30) + 123_457
    d = dev(ctx)
    g = torch.Generator(device=d)
    g.manual_seed(7)
    src = torch.randint(0, 8, (n,), dtype=torch.uint8, device=d, generator=g)  # 3 bits of entropy per byte
    bound = ctx.compress_parallel_bound(GZIP, n)
    out = torch.empty(bound, dtype=torch.uint8, device=d)
    st, wr = ctx.compress_parallel_device(GZIP, src, out)
    assert st == OK and wr < n // 2
    f = out[:wr].cpu().numpy()
    del out
    host = src.cpu().numpy()
    del src
    assert f[-4:].tobytes() == struct.pack("<I", n & 0xffffffff)  # ISIZE = n mod 2^32
    dec = zlib.decompressobj(31)
    at, step = 0, 64 << 20
    for o in range(0, len(f), step):
        chunk = dec.decompress(f[o:o + step].tobytes())
        assert np.array_equal(np.frombuffer(chunk, np.uint8), host[at:at + len(chunk)]), at
        at += len(chunk)
    chunk = dec.flush()
    assert np.array_equal(np.frombuffer(chunk, np.uint8), host[at:at + len(chunk)])
    at += len(chunk)
    assert at == n and dec.eof and not dec.unused_data
