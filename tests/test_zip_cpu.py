"""CPU emulation of the zip-archive kernels (starflate_b200/csrc/zip_file.cuh, built for the host by
tests/cpu_emu/emu_zip.cpp).  The EOCD, candidate-scan, chain and entry kernels must list exactly what
zipfile.ZipFile(...).infolist() lists — sizes, CRC, method, flags, name bytes and the data offset
from the local header — on empty, small and large archives, a 65 535-byte comment, names that contain
PK\\1\\2, ZIP64 entries and a ZIP64 EOCD, data descriptors, prepended bytes and a torch.save file, at two
address phases; damaged archives must be rejected.  The piece and result kernels must give every
entry's CRC-32 as zlib.crc32 does, for sizes around multiples of the piece size."""
import ctypes as C
import io
import os
import struct
import subprocess
import zipfile
import zlib

import numpy as np
import pytest

from starflate_b200 import ZIP_ENTRY
from tests import zip_tools as Z

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PIECE = 1 << 20
OK, ERROR, DST_SMALL, BAD, CHECKSUM, SIZE = 0, 1, 4, 8, 9, 10


@pytest.fixture(scope="module")
def emu():
    out = os.path.join(HERE, "cpu_emu", "libemu_zip.so")
    csrc = os.path.join(ROOT, "starflate_b200", "csrc")
    srcs = [os.path.join(HERE, "cpu_emu", f) for f in ("emu_zip.cpp", "cuda_shim_warp.h")] + \
           [os.path.join(csrc, f) for f in ("zip_file.cuh", "gzip_file.cuh", "container.cuh", "stored_copy.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-o", out, srcs[0]])
    lib = C.CDLL(out)
    lib.emu_zip_list.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                 C.c_void_p]
    lib.emu_zip_list.restype = C.c_int
    lib.emu_zip_extract.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_uint, C.c_void_p]
    return lib


def listing(lib, data: bytes, phase=0, walk=False, cap=None):
    buf = np.zeros(len(data) + 16, np.uint8)
    s = buf[phase:phase + len(data)]
    s[:] = np.frombuffer(data, np.uint8)
    cap = len(data) // 46 + 1 if cap is None else cap
    rows = np.zeros(max(cap, 1), ZIP_ENTRY)
    info = np.zeros(5, np.int64)
    cnt, tot = np.zeros(1, np.uint64), np.zeros(1, np.uint64)
    st = lib.emu_zip_list(s.ctypes.data, len(data), int(walk), rows.ctypes.data, cap, info.ctypes.data, cnt.ctypes.data,
                          tot.ctypes.data)
    return st, rows[:int(cnt[0])], int(tot[0]), info


def check(lib, data: bytes, phases=(0, 5), walk=(False, True)):
    want = Z.ref_rows(data)
    for ph in phases:
        for w in walk:
            st, rows, total, _ = listing(lib, data, ph, w)
            assert st == OK, (ph, w)
            assert Z.rows_as_ref(data, rows) == want, (ph, w)
            assert (rows["status"] == 0).all()
            sizes = rows["size"].astype(np.uint64)
            assert rows["dst_off"].tolist() == (np.cumsum(sizes) - sizes).tolist() and total == int(sizes.sum())
    return want


def files(n, seed=0, size=40):
    rnd = np.random.default_rng(seed)
    return [(f"dir/f{k:06d}.txt", bytes(rnd.integers(97, 101, size=int(rnd.integers(0, size)), dtype=np.uint8)))
            for k in range(n)]


def test_empty_one_and_many_entries(emu):
    empty = Z.make_zip([])
    assert len(empty) == 22
    assert check(emu, empty) == []
    check(emu, Z.make_zip(files(1)))
    check(emu, Z.make_zip(files(10_000, 1)), phases=(0, 5), walk=(False,))
    check(emu, Z.make_zip(files(300, 2), compression=zipfile.ZIP_STORED))


def test_long_comment_and_false_records_in_names(emu):
    check(emu, Z.make_zip(files(20, 3), comment=b"c" * 65535))
    # names holding whole CD-record look-alikes: candidates the chain must pass by
    fake = "PK\x01\x02" + "\x00" * 24 + "\x05\x00\x00\x00\x00\x00" + "z" * 10
    fs = [(f"a{k}{fake}{k}", b"data %d" % k) for k in range(30)] + [("PK\x01\x02", b"")]
    data = Z.make_zip(fs)
    assert data.count(b"PK\x01\x02") > 2 * len(fs)
    check(emu, data)


def test_zip64_entries_and_eocd(emu):
    data = Z.make_zip(files(50, 5), force_zip64=True)
    assert b"PK\x06\x06" not in data  # ZIP64 extra fields only
    check(emu, data)
    big = Z.make_zip(files(70_000, 6, size=4), compression=zipfile.ZIP_STORED)
    assert b"PK\x06\x06" in big and b"PK\x06\x07" in big  # more than 65 535 entries
    check(emu, big, phases=(5,), walk=(False,))


def test_data_descriptors_prepended_bytes_and_torch_save(emu):
    dd = Z.make_zip(files(40, 7), unseekable=True)
    with zipfile.ZipFile(io.BytesIO(dd)) as z:
        assert all(i.flag_bits & 8 for i in z.infolist())
    check(emu, dd)
    pre = b"#!/bin/sh\nexit 0\n" * 37 + Z.make_zip(files(25, 8))
    check(emu, pre)
    check(emu, b"\x00" * 1000 + Z.make_zip(files(70_000, 9, size=3), compression=zipfile.ZIP_STORED), phases=(0,),
          walk=(False,))
    torch = pytest.importorskip("torch")
    f = io.BytesIO()
    torch.save({"w": torch.arange(1000, dtype=torch.float32), "b": torch.ones(3, 5), "name": "ckpt"}, f)
    data = f.getvalue()
    want = check(emu, data)
    assert all(m == 0 and fl & 8 for _, _, _, m, fl, _, _ in want)  # stored entries with data descriptors


def test_rejected_archives(emu):
    good = Z.make_zip(files(10, 10))
    e = good.rfind(b"PK\x05\x06")
    assert listing(emu, good[:-1])[0] == BAD      # truncated: the EOCD does not fit
    assert listing(emu, good[:e - 10] + good[e:])[0] == BAD  # the CD is cut short
    assert listing(emu, b"")[0] == BAD
    assert listing(emu, b"PK\x03\x04" + b"\0" * 100)[0] == BAD
    for at in (4, 6):  # disk numbers
        assert listing(emu, Z.patch(good, e + at, b"\x01\x00"))[0] == BAD
    for d in (1, -1):  # the CD's record count off by one
        n = struct.unpack("<H", good[e + 10:e + 12])[0]
        assert listing(emu, Z.patch(good, e + 10, struct.pack("<H", n + d)))[0] == BAD
    big = Z.make_zip(files(70_000, 11, size=2), compression=zipfile.ZIP_STORED)
    loc = big.rfind(b"PK\x06\x07")
    assert listing(emu, Z.patch(big, loc + 16, struct.pack("<I", 2)), walk=True)[0] == BAD  # total disks
    z64 = big.rfind(b"PK\x06\x06")
    assert listing(emu, Z.patch(big, z64 + 32, struct.pack("<Q", 70_001)), walk=True)[0] == BAD
    # a bad local signature: that row only
    lh = Z.ref_rows(good)[3][6] - 30 - len(b"dir/f000003.txt")
    assert good[lh:lh + 4] == b"PK\x03\x04"
    st, rows, _, _ = listing(emu, Z.patch(good, lh, b"PK\x03\x05"))
    assert st == OK and rows["status"].tolist() == [0, 0, 0, BAD] + [0] * 6


def extract(lib, data: bytes, rows, dst_cap, dec=None, fill=0xA5, large=1 << 62, alone=False, grid=3, in_place=None):
    """dec: {row: (status, bytes)} -- what the decoder produced for a deflated row; the emulation places
    it in the row's decoder window.  in_place: a list that receives whether each group was decoded in dst."""
    rows = rows.copy()
    d = np.full(max(dst_cap, 1) + 16, fill, np.uint8)
    ds = np.zeros(max(len(rows), 1), np.uint8)
    dw = np.zeros(max(len(rows), 1), np.uint64)
    at = np.zeros(max(len(rows), 1), np.uint64)
    parts, pos = [], 0
    for k, (st, out) in (dec or {}).items():
        ds[k], dw[k], at[k] = st, len(out), pos
        parts.append(out)
        pos += len(out)
    blob = np.frombuffer(b"".join(parts) + b"\0", np.uint8)
    ip = np.zeros(2, np.int32)
    s = np.frombuffer(data, np.uint8)
    lib.emu_zip_extract(s.ctypes.data, len(data), rows.ctypes.data, len(rows), d.ctypes.data, dst_cap, ds.ctypes.data,
                        dw.ctypes.data, blob.ctypes.data, at.ctypes.data, large, int(alone), grid, ip.ctypes.data)
    assert (d[dst_cap:] == fill).all()
    if in_place is not None:
        in_place[:] = [bool(v) for v in ip]
    return rows, d[:dst_cap].tobytes()


def test_decoder_groups_in_place_or_in_scratch(emu):
    """Deflated rows are decoded on a window of their group's own bytes: dst itself when their regions
    lie back to back, else scratch copied out by the piece kernel; the bytes and statuses are the same,
    and bytes of dst outside the rows' regions are never written."""
    rnd = np.random.default_rng(13)
    small = [bytes(rnd.integers(97, 100, size=int(rnd.integers(0, 3000)), dtype=np.uint8)) for _ in range(9)]
    big = [bytes(rnd.integers(97, 100, size=PIECE + 3000 * k, dtype=np.uint8)) for k in range(3)]
    # deflated only: both groups back to back in dst (large = 4096 puts the three big ones in group 1)
    fs = [(f"s{k}", p) for k, p in enumerate(small)] + [(f"b{k}", p) for k, p in enumerate(big)]
    for interleave in (False, True):
        if interleave:  # stored entries between them: neither group is contiguous
            fs = [x for k, p in enumerate(small + big) for x in ((f"d{k}", p), (f"x{k}", b"stored %d" % k * 50,
                                                                                 zipfile.ZIP_STORED))]
        data = Z.make_zip(fs)
        st, rows, total, _ = listing(emu, data)
        assert st == OK
        with zipfile.ZipFile(io.BytesIO(data)) as z:
            want = [z.read(i) for i in z.infolist()]
        dec = {k: (OK, want[k]) for k in range(len(fs)) if int(rows["method"][k]) == 8}
        for alone in (False, True):
            ip = [None, None]
            out, dst = extract(emu, data, rows, total, dec, large=4096, alone=alone, in_place=ip)
            assert ip == [not interleave, not interleave], (interleave, alone, ip)
            assert out["status"].tolist() == [OK] * len(fs) and dst == b"".join(want)
        # a subset with gaps between its regions: scratch, and the gaps keep their bytes
        sub = rows[[len(fs) - 1, 0, 2]].copy()
        at = 0
        for i in range(len(sub)):
            sub["dst_off"][i] = at + 5
            at += 5 + int(sub["size"][i])
        ip = [None, None]
        sdec = {j: dec[k] for j, k in enumerate((len(fs) - 1, 0, 2)) if k in dec}
        out, dst = extract(emu, data, sub, at + 5, sdec, fill=0x77, large=4096, in_place=ip)
        assert ip[0] is False and out["status"].tolist() == [OK] * 3
        exp = bytearray(b"\x77" * (at + 5))
        for j, k in enumerate((len(fs) - 1, 0, 2)):
            exp[int(sub["dst_off"][j]):int(sub["dst_off"][j]) + len(want[k])] = want[k]
        assert dst == bytes(exp)


def test_pieces_and_crc_around_piece_multiples(emu):
    rnd = np.random.default_rng(12)
    sizes = [0, 1, 17, PIECE - 1, PIECE, PIECE + 1, 2 * PIECE + 5]
    payloads = [bytes(rnd.integers(0, 256, size=n, dtype=np.uint8)) for n in sizes]
    fs = [(f"s{k}", p, zipfile.ZIP_STORED) for k, p in enumerate(payloads)] + \
         [(f"d{k}", p, zipfile.ZIP_DEFLATED) for k, p in enumerate(payloads)]
    data = Z.make_zip(fs)
    st, rows, total, _ = listing(emu, data)
    assert st == OK and total == 2 * sum(sizes)
    want = b"".join(p for _, p, _ in fs)
    dec = {k: (OK, fs[k][1]) for k in range(len(sizes), len(fs))}
    out, dst = extract(emu, data, rows, total, dec)
    assert out["status"].tolist() == [OK] * len(fs) and out["written"].tolist() == sizes * 2
    assert dst == want
    # a deflated row whose output is off by one byte: CRC; one that is a byte short: size
    bad = dict(dec)
    k = len(sizes) + 5
    bad[k] = (OK, fs[k][1][:-1] + bytes([fs[k][1][-1] ^ 1]))
    bad[k + 1] = (OK, fs[k + 1][1][:-1])
    out, _ = extract(emu, data, rows, total, bad)
    assert out["status"][k] == CHECKSUM and out["status"][k + 1] == SIZE
    # a stored row with a corrupt CRC in the table
    r2 = rows.copy()
    r2["crc32"][4] ^= 0x10
    out, _ = extract(emu, data, r2, total, dec)
    assert out["status"].tolist() == [OK] * 4 + [CHECKSUM] + [OK] * (len(fs) - 5)
    # dst cut inside stored row 5: every byte that fits is produced
    cut = sum(sizes[:5]) + 1000
    out, dst = extract(emu, data, rows[:6], cut)
    assert out["status"].tolist() == [OK] * 5 + [DST_SMALL] and int(out["written"][5]) == 1000
    assert dst == want[:cut]


def test_split_rules(emu):
    data = Z.make_zip([("a", b"x" * 100, zipfile.ZIP_STORED), ("b", b"y" * 5000, zipfile.ZIP_DEFLATED)])
    st, rows, total, _ = listing(emu, data)
    r = rows.copy()
    r["comp_size"][0] = 99                      # stored with comp_size != size
    r["method"][1] = 12                         # bzip2
    out, _ = extract(emu, data, r, total)
    assert out["status"].tolist() == [SIZE, BAD] and out["written"].tolist() == [0, 0]
    r = rows.copy()
    r["flags"][0] |= 1                          # encrypted
    r["size"][1] = 0xffffff00                   # beyond the batch precondition
    r["data_off"][1] = len(data)                # ... and (checked first) data outside the archive
    out, _ = extract(emu, data, r, total)
    assert out["status"].tolist() == [BAD, BAD]
    r = rows.copy()
    r["size"][1] = 0xffffff00
    out, _ = extract(emu, data, r, 1 << 33)
    assert out["status"].tolist() == [CHECKSUM if zlib.crc32(b"x" * 100) != int(rows["crc32"][0]) else OK, ERROR]
    # a deflated row that produced more than its size while dst had room: SizeMismatch; with dst ending
    # at its region: DstTooSmall
    out, _ = extract(emu, data, rows, total + 10, {1: (DST_SMALL, b"y" * 5000)})
    assert out["status"][1] == SIZE
    out, _ = extract(emu, data, rows, total, {1: (DST_SMALL, b"y" * 5000)})
    assert out["status"][1] == DST_SMALL
