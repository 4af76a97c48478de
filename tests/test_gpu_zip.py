"""GPU: zip archives (sfb200_zip_list*, sfb200_zip_extract*) against zipfile.read — stored and deflated
entries at every level, empty files and directories, np.savez_compressed and torch.save files,
unsupported methods and encryption, damaged entries at the first, a middle and the last row, dst cut
inside an entry, subset and reordered extraction, mixes of small and large entries, one archive above
4 GiB, the host / device / C++ entry points agreeing, and the launches a 10 000-entry archive costs."""
import io
import os
import subprocess
import zipfile
import zlib

import numpy as np
import pytest
import torch

from starflate_b200 import ZIP_ENTRY, build
from tests import deflate_tools as T
from tests import zip_tools as Z

pytestmark = pytest.mark.gpu

OK, ERROR, DST_SMALL, BAD, CHECKSUM, SIZE = 0, 1, 4, 8, 9, 10
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev_of(ctx):
    return torch.device("cuda", ctx.device)


def both(ctx, data: bytes, rows=None, dst_cap=None, fill=0xA5):
    """List (unless rows are given) and extract through the host and the device entry points, which
    must agree -> (rows after extraction, dst bytes)"""
    st, listed, names = ctx.zip_list(data)
    assert st == OK
    s = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(dev_of(ctx))
    st2, drows, total = ctx.zip_list_device(s)
    assert st2 == OK and drows.cpu().numpy().view(ZIP_ENTRY).ravel().tobytes() == listed.tobytes()
    assert total == int(listed["size"].sum())
    rows = listed if rows is None else rows
    dst_cap = total if dst_cap is None else dst_cap
    dst, out = ctx.zip_extract(data, rows, dst_cap, fill=fill)
    r = torch.from_numpy(np.ascontiguousarray(rows).view(np.uint8).reshape(-1, 64).copy()).to(dev_of(ctx))
    d = torch.full((max(dst_cap, 1),), fill, dtype=torch.uint8, device=dev_of(ctx))
    ctx.zip_extract_device(s, r, d[:dst_cap])
    assert r.cpu().numpy().view(ZIP_ENTRY).ravel().tobytes() == out.tobytes()
    assert d[:dst_cap].cpu().numpy().tobytes() == dst
    return out, dst


def expect_all(ctx, data: bytes):
    out, dst = both(ctx, data)
    with zipfile.ZipFile(io.BytesIO(data)) as z:
        want = [z.read(i) for i in z.infolist()]
    assert out["status"].tolist() == [OK] * len(want)
    assert out["written"].tolist() == [len(w) for w in want]
    assert dst == b"".join(want)
    return out, dst


def test_stored_and_every_level(ctx):
    fs = [(f"t{k}", T.big_text(1000 * k * k, k)) for k in range(12)] + [("rnd", os.urandom(70_000))]
    expect_all(ctx, Z.make_zip(fs, compression=zipfile.ZIP_STORED))
    for level in range(10):
        expect_all(ctx, Z.make_zip(fs, level=level))


def test_empty_files_directories_and_descriptors(ctx):
    f = io.BytesIO()
    with zipfile.ZipFile(f, "w", zipfile.ZIP_DEFLATED) as z:
        z.mkdir("d")
        z.writestr("d/empty", b"")
        z.writestr("d/e2", b"", compress_type=zipfile.ZIP_STORED)
        z.writestr("x", b"abc" * 1000)
    expect_all(ctx, f.getvalue())
    expect_all(ctx, Z.make_zip([(f"f{k}", T.big_text(3000 * k, k)) for k in range(20)], unseekable=True))
    expect_all(ctx, Z.make_zip([]))


def test_npz_and_torch_save(ctx):
    arrs = {"a": np.arange(100_000, dtype=np.float32), "b": np.random.default_rng(1).integers(0, 9, (300, 200)),
            "c": np.zeros(0, np.int8)}
    f = io.BytesIO()
    np.savez_compressed(f, **arrs)
    data = f.getvalue()
    out, dst = expect_all(ctx, data)
    _, _, names = ctx.zip_list(data)
    for name, r in zip(names, out):
        got = np.load(io.BytesIO(dst[int(r["dst_off"]):int(r["dst_off"]) + int(r["written"])]))
        assert np.array_equal(got, arrs[name[:-4]])
    f = io.BytesIO()
    sd = {"w": torch.randn(512, 256), "b": torch.arange(77), "n": "name"}
    torch.save(sd, f)
    expect_all(ctx, f.getvalue())


def test_unsupported_methods_and_encryption(ctx):
    fs = [("a", b"first " * 500), ("bz", b"bzip2 data " * 300, zipfile.ZIP_BZIP2), ("b", b"middle " * 400),
          ("lz", b"lzma data " * 300, zipfile.ZIP_LZMA), ("c", b"last " * 600)]
    data = Z.make_zip(fs)
    out, dst = both(ctx, data)
    assert out["status"].tolist() == [OK, BAD, OK, BAD, OK]
    assert out["method"].tolist() == [8, 12, 8, 14, 8]
    for k in (0, 2, 4):
        o = int(out["dst_off"][k])
        assert dst[o:o + len(fs[k][1])] == fs[k][1]
    # an encryption bit patched into one CD record (the listing marks it, and so does extraction)
    cd = [i for i in range(len(data)) if data.startswith(b"PK\x01\x02", i)][2]
    enc = Z.patch(data, cd + 8, bytes([data[cd + 8] | 1]))
    st, rows, _ = ctx.zip_list(enc)
    assert rows["status"].tolist() == [OK, BAD, BAD, BAD, OK] and rows["flags"][2] & 1
    dst2, out2 = ctx.zip_extract(enc, rows, int(rows["size"].sum()))
    assert out2["status"].tolist() == [OK, BAD, BAD, BAD, OK]


@pytest.mark.parametrize("where", [0, 3, 6])
def test_damage_at_first_middle_last_entry(ctx, where):
    ps = [T.big_text(20_000 + 3000 * k, 40 + k) for k in range(7)]
    data = Z.make_zip([(f"p{k}", p) for k, p in enumerate(ps)])
    _, rows, _ = ctx.zip_list(data)
    total = int(rows["size"].sum())
    r = rows.copy()
    r["crc32"][where] ^= 1
    out, dst = both(ctx, data, r)
    assert out["status"].tolist() == [CHECKSUM if k == where else OK for k in range(7)]
    assert dst == b"".join(ps)
    r = rows.copy()
    r["size"][where] += 3  # larger than the output
    out, _ = both(ctx, data, r, total + 3)
    assert out["status"][where] == SIZE and out["written"][where] == len(ps[where])
    r = rows.copy()
    r["size"][where] -= 3  # smaller: the decode overruns it
    out, _ = both(ctx, data, r)
    assert out["status"][where] == SIZE
    r = rows.copy()
    r["comp_size"][where] //= 2  # the payload is cut short
    out, _ = both(ctx, data, r)
    assert out["status"][where] not in (OK, BAD, CHECKSUM, SIZE)
    assert [s for k, s in enumerate(out["status"].tolist()) if k != where] == [OK] * 6


def test_dst_cut_inside_an_entry(ctx):
    ps = [T.big_text(30_000 + 1000 * k, k) for k in range(4)]
    for comp in (zipfile.ZIP_DEFLATED, zipfile.ZIP_STORED):
        data = Z.make_zip([(f"p{k}", p) for k, p in enumerate(ps)], compression=comp)
        want = b"".join(ps)
        for cap in (1, len(ps[0]) - 1, len(ps[0]) + 7, len(want) - 1):
            out, dst = both(ctx, data, None, cap)
            k = next(i for i in range(4) if sum(map(len, ps[:i + 1])) > cap)
            assert out["status"][k] == DST_SMALL, (comp, cap, out["status"])
            assert all(s == OK for s in out["status"][:k])
            produced = int(out["written"][k])
            assert produced <= cap - sum(map(len, ps[:k]))
            if comp == zipfile.ZIP_STORED:
                assert produced == cap - sum(map(len, ps[:k]))
            assert dst[:sum(map(len, ps[:k])) + produced] == want[:sum(map(len, ps[:k])) + produced]


def test_subset_and_reordered_extract(ctx):
    ps = [T.big_text(5000 * (k + 1), k) for k in range(8)]
    data = Z.make_zip([(f"p{k}", p) for k, p in enumerate(ps)])
    _, rows, _ = ctx.zip_list(data)
    sub = rows[[6, 1, 3]].copy()
    gap = 11
    at = 0
    for i in range(len(sub)):  # packed in the new order with guard gaps between
        sub["dst_off"][i] = at + gap
        at += gap + int(sub["size"][i])
    cap = at + gap
    out, dst = both(ctx, data, sub, cap, fill=0x5C)
    assert out["status"].tolist() == [OK] * 3
    exp = bytearray(b"\x5c" * cap)
    for r, k in zip(sub, (6, 1, 3)):
        exp[int(r["dst_off"]):int(r["dst_off"]) + len(ps[k])] = ps[k]
    assert dst == bytes(exp)


@pytest.mark.parametrize("big,count", [(300 << 20, 1), (16 << 20, 20)])
def test_small_entries_with_large_ones(ctx, big, count):
    rnd = np.random.default_rng(big + count)
    small = [bytes(rnd.integers(97, 105, size=int(rnd.integers(0, 2000)), dtype=np.uint8)) for _ in range(10_000)]
    large = [T.big_text(big, 100 + k) for k in range(count)]
    fs = [(f"s{k}", p) for k, p in enumerate(small)]
    for k, p in enumerate(large):
        fs.insert(1 + k * 37, (f"L{k}", p))
    data = Z.make_zip(fs, level=1)
    s = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(dev_of(ctx))
    st, rows, total = ctx.zip_list_device(s)
    assert st == OK and total == sum(len(p) for _, p in fs)
    d = torch.empty(total, dtype=torch.uint8, device=dev_of(ctx))
    ctx.zip_extract_device(s, rows, d)
    out = rows.cpu().numpy().view(ZIP_ENTRY).ravel()
    assert (out["status"] == OK).all()
    want = torch.from_numpy(np.frombuffer(b"".join(p for _, p in fs), np.uint8).copy()).to(dev_of(ctx))
    assert torch.equal(d, want)


def test_many_large_entries_between_stored_ones(ctx):
    """Deflated entries of >= 1 MiB numerous enough to go as one batch, and small ones, with stored
    entries between them: both decoder groups run in scratch and are copied to their regions."""
    rnd = np.random.default_rng(21)
    fs = []
    for k in range(40):
        fs.append((f"L{k}", T.big_text((1 << 20) + 777 * k, 300 + k)))
        fs.append((f"x{k}", bytes(rnd.integers(0, 256, size=5000 + k, dtype=np.uint8)), zipfile.ZIP_STORED))
        fs.append((f"s{k}", b"small %d " % k * (k + 1)))
    data = Z.make_zip(fs, level=1)
    s = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).to(dev_of(ctx))
    st, rows, total = ctx.zip_list_device(s)
    d = torch.full((total,), 0x3C, dtype=torch.uint8, device=dev_of(ctx))
    ctx.zip_extract_device(s, rows, d)
    out = rows.cpu().numpy().view(ZIP_ENTRY).ravel()
    assert st == OK and (out["status"] == OK).all()
    assert d.cpu().numpy().tobytes() == b"".join(f[1] for f in fs)


def test_archive_above_4_gib(ctx, tmp_path):
    """ZIP64 offsets and a stored entry above 4 GiB (written to disk: zipfile streams it)"""
    path = tmp_path / "big.zip"
    chunk = np.random.default_rng(3).integers(0, 256, size=64 << 20, dtype=np.uint8).tobytes()
    big_n = (4 << 30) + (100 << 20)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("head.txt", b"before " * 1000, compress_type=zipfile.ZIP_DEFLATED)
        info = zipfile.ZipInfo("tensor.bin", date_time=(2020, 1, 1, 0, 0, 0))
        with z.open(info, "w", force_zip64=True) as w:
            left = big_n
            while left:
                w.write(chunk[:min(left, len(chunk))])
                left -= min(left, len(chunk))
        z.writestr("tail.txt", b"after " * 5000, compress_type=zipfile.ZIP_DEFLATED)
    data = np.fromfile(path, np.uint8)
    s = torch.from_numpy(data).to(dev_of(ctx))
    del data
    st, rows, total = ctx.zip_list_device(s)
    out = rows.cpu().numpy().view(ZIP_ENTRY).ravel()
    assert st == OK and out["size"].tolist() == [7000, big_n, 30000]
    assert out["data_off"][2] > (4 << 30)
    d = torch.empty(total, dtype=torch.uint8, device=dev_of(ctx))
    torch.cuda.synchronize(dev_of(ctx))
    free_before = torch.cuda.mem_get_info(dev_of(ctx))[0]
    ctx.zip_extract_device(s, rows, d)
    # the two small deflated entries are decoded on a window of their own 37 000 bytes: the context
    # grows by nothing in proportion to the 4 GiB stored entry beside them
    grown = free_before - torch.cuda.mem_get_info(dev_of(ctx))[0]
    assert grown < (256 << 20), grown
    out = rows.cpu().numpy().view(ZIP_ENTRY).ravel()
    assert out["status"].tolist() == [OK] * 3 and out["written"].tolist() == [7000, big_n, 30000]
    assert d[:7000].cpu().numpy().tobytes() == b"before " * 1000
    assert d[-30000:].cpu().numpy().tobytes() == b"after " * 5000
    c = torch.from_numpy(np.frombuffer(chunk, np.uint8).copy()).to(dev_of(ctx))
    for at in (0, 4 << 30):
        assert torch.equal(d[7000 + at:7000 + at + (64 << 20)][: min(64 << 20, big_n - at)], c[: min(64 << 20, big_n - at)])


def test_launches_do_not_grow_with_entries(ctx):
    data = Z.make_zip([(f"f{k}", T.big_text(300, k)) for k in range(10_000)])
    before = ctx.launch_info()["kernel_launches"]
    st, rows, _ = ctx.zip_list(data)
    dst, out = ctx.zip_extract(data, rows, int(rows["size"].sum()))
    launches = ctx.launch_info()["kernel_launches"] - before
    assert st == OK and (out["status"] == OK).all()
    assert launches <= 64, launches


def test_cpp_entry_points_agree(ctx, tmp_path):
    build.build_all()
    src = os.path.join(ROOT, "tests", "cpp", "zip_test.cpp")
    exe = str(tmp_path / "zip_test")
    subprocess.check_call(["g++", "-std=c++23", "-O1", "-fno-exceptions", "-w", "-pthread",
                           "-I", os.path.join(ROOT, "starflate_b200", "cpp"), "-I", os.path.join(ROOT, "include"),
                           "-o", exe, src, "-L", build.OUT, "-lstarflate", "-lstarflate_b200",
                           f"-Wl,-rpath,{build.OUT}"])
    ps = [T.big_text(10_000 + 999 * k, k) for k in range(5)]
    good = Z.make_zip([(f"p{k}", p) for k, p in enumerate(ps)])
    files = [good, Z.make_zip([("a", b"x" * 10), ("b", b"y" * 10, zipfile.ZIP_BZIP2)]), good[:-3]]
    for k, f in enumerate(files):
        path = tmp_path / f"f{k}.zip"
        path.write_bytes(f)
        r = subprocess.run([exe, str(path)], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        st, rows, _ = ctx.zip_list(f)
        got = r.stdout.split()
        if st != OK:
            assert got == [str(st), "0"]
            continue
        dst, out = ctx.zip_extract(f, rows, int(rows["size"].sum()))
        assert got[:2] == [str(st), str(len(rows))]
        want = [f"{int(o['status'])}:{zlib.crc32(dst[int(o['dst_off']):int(o['dst_off']) + int(o['written'])]):08x}"
                for o in out]
        assert got[2:] == want
