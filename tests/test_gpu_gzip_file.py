"""GPU: gzip files of several members (sfb200_decompress_gzip_file*, sfb200_gzip_file_size) against
Python's gzip.decompress — BGZF from 0 bytes to 256 MiB of output, `cat a.gz b.gz` with a member
large enough for the single-stream route, mixed and trap files, every error at the first, a middle
and the last member, dst cut inside a member, the host / device / C++ entry points agreeing, and the
number of launches a 10 000-member file costs."""
import gzip
import os
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

OK, BAD_HEADER, DST_SMALL, SRC_SMALL, BAD, CHECKSUM, SIZE = 0, 2, 4, 5, 8, 9, 10
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def both(ctx, f: bytes, cap: int, fill=0xA5):
    """Host and device entry points on the same file must agree -> (status, dst, written, members)."""
    st, dst, wr, nm = ctx.decompress_gzip_file(f, cap, fill=fill)
    dev = torch.device("cuda", ctx.device)
    s = torch.from_numpy(np.frombuffer(f, np.uint8).copy()).to(dev) if f else torch.zeros(0, dtype=torch.uint8, device=dev)
    d = torch.full((cap,), fill, dtype=torch.uint8, device=dev)
    st2, wr2, nm2 = ctx.decompress_gzip_file_device(s, d)
    assert (st2, wr2, nm2) == (st, wr, nm)
    assert d[:wr].cpu().numpy().tobytes() == dst[:wr]
    if st == OK:
        assert (d[wr:] == fill).all() and dst[wr:] == bytes([fill]) * (cap - wr)
    return st, dst, wr, nm


def expect_ok(ctx, f: bytes, want: bytes, members: int, slack=7):
    st, dst, wr, nm = both(ctx, f, len(want) + slack)
    assert (st, wr, nm) == (OK, len(want), members)
    assert dst[:wr] == want


def pieces_of(data: bytes, piece: int):
    return [data[i:i + piece] for i in range(0, len(data), piece)]


def test_bgzf_files(ctx):
    for size, piece in ((0, G.PIECE), (1, G.PIECE), (70_000, 4096), (3 << 20, G.PIECE), (9 << 20, 20_000)):
        data = T.big_text(size, size) if size else b""
        for eof in (True, False):
            f = G.bgzf(data, piece=piece, eof=eof)
            want = gzip.decompress(f)
            assert want == data
            n = len(pieces_of(data, piece)) + eof
            expect_ok(ctx, f, want, n)
            assert ctx.gzip_file_size(f) == (len(want), n, True)
    assert both(ctx, b"", 0)[:3:2] == (OK, 0)


def test_bgzf_256_mib(ctx):
    # (gzip.decompress copies the rest of the file once per member: the plaintext is the checker here)
    data = T.big_text(256 << 20, 11)
    f = b"".join(G.bgzf_member(p, level=1) for p in pieces_of(data, G.PIECE)) + G.BGZF_EOF
    n = len(pieces_of(data, G.PIECE)) + 1
    assert ctx.gzip_file_size(f) == (len(data), n, True)
    dev = torch.device("cuda", ctx.device)
    s = torch.from_numpy(np.frombuffer(f, np.uint8).copy()).to(dev)
    d = torch.full((len(data) + 5,), 0xA5, dtype=torch.uint8, device=dev)
    assert ctx.decompress_gzip_file_device(s, d) == (OK, len(data), n)
    assert torch.equal(d[: len(data)], torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(dev))
    assert (d[len(data):] == 0xA5).all()


def test_concatenated_plain_members(ctx):
    big = T.big_text(3 << 20, 5)  # one member above 1 MiB: the single-stream route
    parts = [b"hello ", big, b"", T.make_stream("fixed", 5000, 1)[0], T.make_stream("stored", 20000, 2)[0], b"tail"]
    f = b"".join(gzip.compress(p, compresslevel=6, mtime=0) for p in parts)
    expect_ok(ctx, f, gzip.decompress(f), len(parts))
    # alone, and with zero padding between and behind members
    expect_ok(ctx, gzip.compress(big, mtime=0), big, 1)
    f2 = gzip.compress(b"x" * 100, mtime=0) + b"\0" * 9 + gzip.compress(b"y" * 7, mtime=0) + b"\0" * 3
    expect_ok(ctx, f2, gzip.decompress(f2), 2)
    assert ctx.gzip_file_size(f2) == (0, 0, False)


def test_mixed_and_trap_files(ctx):
    a = G.bgzf(T.big_text(200_000, 1), piece=30_000, eof=False)
    b = gzip.compress(T.big_text(50_000, 2), mtime=0)
    c = G.bgzf(T.big_text(100_000, 3), piece=10_000)
    f = a + b"\0" * 5 + b + c
    expect_ok(ctx, f, gzip.decompress(f), 7 + 1 + 10 + 1)
    size, members, complete = ctx.gzip_file_size(f)
    assert (size, members, complete) == (200_000, 7, False)
    for seed in (1, 2):
        t, plain = G.trap_file(seed=seed)
        expect_ok(ctx, t, plain, 8)
        assert ctx.gzip_file_size(t) == (len(plain), 8, True)


def _members(n=6):
    ps = [T.big_text(20_000 + 3000 * k, 40 + k) for k in range(n)]
    return ps, [G.bgzf_member(p) for p in ps]


def _patch(m: bytes, at: int, val: bytes) -> bytes:
    at %= len(m)
    return m[:at] + val + m[at + len(val):]


@pytest.mark.parametrize("where", [0, 3, 5])
def test_errors_at_first_middle_last_member(ctx, where):
    ps, ms = _members()
    off = sum(len(p) for p in ps[:where])
    total = sum(len(p) for p in ps)
    p, m = ps[where], ms[where]
    crc, isz = struct.unpack("<II", m[-8:])
    cases = [
        (_patch(m, -8, struct.pack("<I", crc ^ 1)), CHECKSUM, len(p)),
        (_patch(m, -4, struct.pack("<I", isz + 3)), SIZE, len(p)),   # ISIZE larger than the output
        (_patch(m, -4, struct.pack("<I", isz - 3)), SIZE, None),     # ... smaller: the decode overruns it
        (_patch(m, 18, bytes([m[18] | 6])), BAD_HEADER, 0),          # BTYPE = 11
    ]
    for bad, want, produced in cases:
        f = b"".join(ms[:where]) + bad + b"".join(ms[where + 1:])
        st, dst, wr, nm = both(ctx, f, total + 10)
        assert st == want, (where, want, st)
        assert nm == len(ms)
        if produced is not None:
            assert wr == off + produced
        assert off <= wr <= off + len(p) and dst[:wr] == (b"".join(ps))[:wr]
        with pytest.raises(Exception):
            gzip.decompress(f)


def test_truncation_and_trailing_bytes(ctx):
    ps, ms = _members(3)
    f = b"".join(ms)
    want = b"".join(ps)
    # bytes behind the last member that are neither padding nor a member
    for tail in (b"garbage", b"\0\0\x01", b"\x1f\x8b\x08"):
        st, dst, wr, nm = both(ctx, f + tail, len(want) + 4)
        assert (st, wr, nm) == (BAD, len(want), 3) and dst[:wr] == want
    # the input ends inside the last member's payload: the raw decoder's status; inside its trailer or
    # header: BadContainer
    last = len(f) - len(ms[-1])
    st, _, wr, _ = both(ctx, f[: last + 18 + 100], len(want))
    assert st not in (OK, BAD, CHECKSUM, SIZE) and wr >= len(want) - len(ps[-1])
    for cut in (len(f) - 3, last + 10):
        st, dst, wr, nm = both(ctx, f[:cut], len(want))
        assert (st, wr) == (BAD, len(want) - len(ps[-1])) and dst[:wr] == want[:wr]
    # a file must start with a member
    assert both(ctx, b"\0" + f, len(want))[0] == BAD
    assert both(ctx, b"\0" * 40, 10)[:3:2] == (BAD, 0)


def test_dst_cut_inside_a_member(ctx):
    ps, ms = _members(4)
    want = b"".join(ps)
    for f in (b"".join(ms), b"".join(gzip.compress(p, mtime=0) for p in ps)):
        for cap in (0, 1, len(ps[0]), len(ps[0]) + 1, len(want) // 2, len(want) - 1):
            st, dst, wr, nm = both(ctx, f, cap)
            if cap == 0 or cap == len(ps[0]):  # the output ends exactly where a member starts
                assert st == DST_SMALL and wr == cap
            assert st == DST_SMALL and wr <= cap and dst[:wr] == want[:wr], (cap, st, wr)
        assert both(ctx, f, len(want))[:3:2] == (OK, len(want))


def test_launches_are_logarithmic_in_members(ctx):
    data = T.big_text(10_000 * 300, 7)
    f = G.bgzf(data, piece=300)
    before = ctx.launch_info()["kernel_launches"]
    st, _, wr, nm = ctx.decompress_gzip_file(f, len(data))
    launches = ctx.launch_info()["kernel_launches"] - before
    assert (st, wr, nm) == (OK, len(data), 10_001)
    assert launches <= 64, launches


def test_walk_fallback_gives_the_same_result(ctx):
    t, plain = G.trap_file(seed=4)
    f = t + G.bgzf(T.big_text(300_000, 8), piece=7000)
    want = gzip.decompress(f)
    os.environ["SFB200_GZIP_CHAIN"] = "walk"
    try:
        expect_ok(ctx, f, want, 8 + 43 + 1)
    finally:
        del os.environ["SFB200_GZIP_CHAIN"]
    expect_ok(ctx, f, want, 8 + 43 + 1)


def test_cpp_entry_points_agree(ctx, tmp_path):
    build.build_all()
    src = os.path.join(ROOT, "tests", "cpp", "gzip_file_test.cpp")
    exe = str(tmp_path / "gzip_file_test")
    subprocess.check_call(["g++", "-std=c++23", "-O1", "-fno-exceptions", "-w", "-pthread",
                           "-I", os.path.join(ROOT, "starflate_b200", "cpp"), "-I", os.path.join(ROOT, "include"),
                           "-o", exe, src, "-L", build.OUT, "-lstarflate", "-lstarflate_b200",
                           f"-Wl,-rpath,{build.OUT}"])
    ps, ms = _members(5)
    files = [b"".join(ms) + G.BGZF_EOF, b"".join(gzip.compress(p, mtime=0) for p in ps),
             b"".join(ms[:2]) + b"junk", _patch(b"".join(ms), -8, b"\0\0\0\0")]
    for k, f in enumerate(files):
        path = tmp_path / f"f{k}.gz"
        path.write_bytes(f)
        cap = sum(len(p) for p in ps) + 3
        r = subprocess.run([exe, str(path), str(cap)], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        st, dst, wr, nm = ctx.decompress_gzip_file(f, cap)
        size, members, complete = ctx.gzip_file_size(f)
        got = r.stdout.split()
        assert got[:4] == [str(st), str(wr), str(nm), str(size) if complete else "none"], (k, got)
        assert bytes.fromhex(got[4]) == zlib.crc32(dst[:wr]).to_bytes(4, "big")


@pytest.mark.parametrize("n_plain", [1, 30, 67, 100, 300])
def test_plain_members_before_a_bgzf_run(n_plain):
    """The member table must hold the BGZF members behind any number of plain ones (a fresh context:
    no capacity left over from earlier calls)."""
    import starflate_b200 as S
    c = S.Context(0)
    try:
        plains = [gzip.compress(b"p%d " % k * (k % 7 + 1), mtime=0) for k in range(n_plain)]
        f = b"".join(plains) + G.bgzf(T.big_text(150_000, n_plain), piece=5000)
        want = gzip.decompress(f)
        expect_ok(c, f, want, n_plain + 30 + 1)
    finally:
        c.close()


def test_plain_member_probe_on_both_routes(ctx):
    """A plain member's end is found by a decode over the rest of the file: on the single-stream route
    when dst has room for it (>= 32 KiB), on the lane route otherwise, and with the small lane geometry
    switched on (it must not take the probe)."""
    small = [gzip.compress(b"ab" * (50 + k), mtime=0) for k in range(5)]
    big = gzip.compress(T.big_text(2 << 20, 9), mtime=0)
    for f in (b"".join(small), big + b"".join(small), b"".join(small) + big):
        want = gzip.decompress(f)
        expect_ok(ctx, f, want, f.count(b"\x1f\x8b\x08\x00"))
        os.environ["SFB200_GEOMETRY"] = "small"
        try:
            expect_ok(ctx, f, want, f.count(b"\x1f\x8b\x08\x00"))
        finally:
            del os.environ["SFB200_GEOMETRY"]
