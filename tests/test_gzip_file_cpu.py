"""CPU emulation of the gzip-file kernels (starflate_b200/csrc/gzip_file.cuh, built for the host by
tests/cpu_emu/emu_gzip.cpp): the candidate scan, the chain by jump tables and the one-thread walk
must find exactly the members a plain Python walk finds — on BGZF files, on extra subfields around
'BC', on trap members full of valid-looking headers (chains that merge), and on files mixing BGZF
with plain members, zero padding and trailing garbage."""
import ctypes as C
import gzip
import os
import subprocess

import numpy as np
import pytest

from tests import gzip_file_tools as G

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_u64p = C.POINTER(C.c_uint64)


@pytest.fixture(scope="module")
def emu():
    out = os.path.join(HERE, "cpu_emu", "libemu_gzip.so")
    srcs = [os.path.join(HERE, "cpu_emu", f) for f in ("emu_gzip.cpp", "cuda_shim_warp.h")] + \
           [os.path.join(ROOT, "starflate_b200", "csrc", f) for f in ("gzip_file.cuh", "container.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-o", out, srcs[0]])
    lib = C.CDLL(out)
    lib.emu_gzip_chain.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_int, _u64p, _u64p, C.c_uint64,
                                   _u64p, _u64p, _u64p, C.c_uint64, _u64p, _u64p, _u64p]
    lib.emu_gzip_chain.restype = C.c_uint64
    return lib


def chain(lib, data: bytes, start=0, skip=False, walk=False, phase=0):
    buf = np.zeros(len(data) + 16, np.uint8)
    s = buf[phase:phase + len(data)]
    s[:] = np.frombuffer(data, np.uint8)
    cap = len(data) // 20 + 8
    cp, cn, mp, ml = (np.zeros(cap, np.uint64) for _ in range(4))
    m, head, stop, nxt = (np.zeros(1, np.uint64) for _ in range(4))
    p = lambda a: a.ctypes.data_as(_u64p)
    k = lib.emu_gzip_chain(s.ctypes.data, len(data), start, int(skip), int(walk), p(cp), p(cn), cap, p(m), p(mp), p(ml),
                           cap, p(head), p(stop), p(nxt))
    cands = list(zip(cp[:int(m[0])].tolist(), cn[:int(m[0])].tolist()))
    return cands, list(zip(mp[:k].tolist(), ml[:k].tolist())), int(head[0]), int(stop[0]), int(nxt[0])


def check(lib, data, start=0, skip=False, phases=(0, 5)):
    want_c = G.ref_candidates(data)
    want = G.ref_chain(data, start, skip)
    for walk in (False, True):
        for ph in phases:
            cands, members, head, stop, nxt = chain(lib, data, start, skip, walk, ph)
            assert cands == want_c, (walk, ph)
            assert (members, head, stop, nxt) == want, (walk, ph, len(members), len(want[0]))
    return want


@pytest.mark.parametrize("n,eof", [(1, False), (1, True), (2, True), (3, False), (100, True), (10_000, True),
                                   (10_000, False)])
def test_bgzf_member_chain(emu, n, eof):
    rnd = np.random.default_rng(n)
    data = b"".join(bytes(rnd.integers(0, 4, size=int(rnd.integers(1, 60)), dtype=np.uint8)) for _ in range(n))
    pieces = []
    at = 0
    for _ in range(n):  # n members of uneven size
        k = 1 + (at * 7919) % 57
        pieces.append(data[at:at + k])
        at += k
    f = b"".join(G.bgzf_member(p) for p in pieces) + (G.BGZF_EOF if eof else b"")
    members, head, stop, nxt = check(emu, f, phases=(3,) if n > 1000 else (0, 5))
    assert len(members) == n + eof and stop == nxt == len(f)
    assert gzip.decompress(f) == b"".join(pieces)


def test_empty_and_eof_only(emu):
    assert check(emu, G.BGZF_EOF)[0] == [(0, 28)]
    assert check(emu, b"")[0] == []


def test_extra_subfields_around_bc(emu):
    p = b"some text, some text, some more text " * 40
    ms = [G.bgzf_member(p, before=b"XY\x03\x00abc"), G.bgzf_member(p, after=b"ZZ\x00\x00"),
          G.bgzf_member(p, before=b"AB\x00\x00", after=b"CD\x05\x0012345"), G.bgzf_member(p)]
    f = b"".join(ms)
    members = check(emu, f)[0]
    assert [l for _, l in members] == [len(m) for m in ms]
    assert gzip.decompress(f) == p * 4
    # a subfield that runs past XLEN, and 'BC' with the wrong SLEN, are not BGZF headers
    bad = bytearray(ms[0])
    bad[12 + 2] = 0x40
    assert G.ref_candidate(bytes(bad), 0) is None
    assert check(emu, bytes(bad) + ms[1])[0] == []


def test_trap_members_with_headers_inside(emu):
    for seed in (1, 2, 3):
        f, plain = G.trap_file(seed=seed)
        assert gzip.decompress(f) == plain
        want_c = G.ref_candidates(f)
        members = check(emu, f)[0]
        assert len(want_c) > len(members) + 100  # the fakes are candidates, the chain passes them by
        assert len(members) == 8 and sum(l for _, l in members) == len(f)


def test_mixed_plain_members_padding_and_garbage(emu):
    a = G.bgzf(b"first part " * 3000, piece=4000, eof=False)
    b = gzip.compress(b"a plain gzip member " * 500, mtime=0)
    c = G.bgzf(b"third part " * 2000, piece=5000)
    f = a + b"\0" * 37 + b + c + b"\0" * 10
    members, head, stop, nxt = check(emu, f)
    assert stop == len(a) and nxt == len(a) + 37  # the chain stops at the plain member behind the padding
    # resumed behind the plain member, with the same tables
    rest = len(a) + 37 + len(b)
    members, head, stop, nxt = check(emu, f, start=rest, skip=True)
    assert head == rest and stop == len(f) - 10 and nxt == len(f)
    # trailing garbage ends the chain where it starts
    g = a + b"garbage!"
    members, head, stop, nxt = check(emu, g)
    assert stop == nxt == len(a)
    # a file that does not start with a member
    assert check(emu, b"\0\0" + a)[0] == []
