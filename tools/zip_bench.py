"""zip archives at batch speed: zip_list_device + zip_extract_device against the batch paths they are
built on, in one process, every arm warmed, arms alternated, >= --min-ms timed per arm:

  Z1  C2's 65 536 level-6 streams rewrapped as one zip (payload and CRC taken from each gzip member,
      nothing recompressed): (A) decompress_container_batch_device(GZIP) over the same members,
      (B) list + extract, (L) list alone.  B's output must equal A's (compared on the device).
  Z2  1 048 576 entries of 4 KiB (C3's page mix): the same arms.
  Z3  Z1 + one 1 GiB text entry, Z1 + 64 entries of 16 MiB (one call each wins) and Z1 + 256 entries
      of 1 MiB (one batch wins): (B) against (A) + the large entries decoded alone (n = 1 each), summed.
  Z4  stored entries of 8 GiB in all, one of them 6 GiB (a checkpoint): (B) against a device-to-device
      copy_ of the same bytes.
  sweep (the large-entry threshold of capi.cu, kZipLarge): Z1 + 4 entries of 256 KiB .. 64 MiB, raw
      DEFLATE batch calls only: (in) all entries in one batch, (apart) Z1 in one batch and the 4 entries
      one call each.

Prints one JSON line with the GPU's name and power limit read in the same run.

  python tools/zip_bench.py [--streams 65536] [--skip z2,z4,sweep]
"""
from __future__ import annotations

import argparse
import json
import os
import struct
import sys
import time
import zlib

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from gzip_file_bench import gpu_info  # noqa: E402


def build_zip(entries) -> tuple[bytes, np.ndarray, np.ndarray]:
    """entries: [(method, payload bytes, crc32, size)] -> (archive, payload offsets, payload lengths);
    ZIP64 records where they are needed, as zipfile writes them."""
    parts, cd, offs, lens = [], [], [], []
    at = 0
    for k, (method, pay, crc, size) in enumerate(entries):
        name = b"e%07d" % k
        z64 = size >= 0xffffffff or len(pay) >= 0xffffffff or at >= 0xffffffff
        lh = struct.pack("<4sHHHHHIII HH", b"PK\x03\x04", 45 if z64 else 20, 0, method, 0, 0x21, crc,
                         0xffffffff if z64 else len(pay), 0xffffffff if z64 else size, len(name),
                         20 if z64 else 0) + name
        if z64:
            lh += struct.pack("<HHQQ", 1, 16, size, len(pay))
        parts += [lh, pay]
        offs.append(at + len(lh))
        lens.append(len(pay))
        extra = struct.pack("<HHQQQ", 1, 24, size, len(pay), at) if z64 else b""
        cd.append(struct.pack("<4sHHHHHHIIIHHHHHII", b"PK\x01\x02", 45 if z64 else 20, 45 if z64 else 20, 0, method, 0,
                              0x21, crc, 0xffffffff if z64 else len(pay), 0xffffffff if z64 else size, len(name),
                              len(extra), 0, 0, 0, 0, 0xffffffff if z64 else at) + name + extra)
        at += len(lh) + len(pay)
    cdb = b"".join(cd)
    n = len(entries)
    tail = b""
    if n >= 0xffff or at >= 0xffffffff or len(cdb) >= 0xffffffff:
        z = at + len(cdb)
        tail = struct.pack("<4sQHHIIQQQQ", b"PK\x06\x06", 44, 45, 45, 0, 0, n, n, len(cdb), at) + \
            struct.pack("<4sIQI", b"PK\x06\x07", 0, z, 1)
        eocd = struct.pack("<4sHHHHIIH", b"PK\x05\x06", 0, 0, 0xffff, 0xffff, 0xffffffff, 0xffffffff, 0)
    else:
        eocd = struct.pack("<4sHHHHIIH", b"PK\x05\x06", 0, 0, n, n, len(cdb), at, 0)
    return b"".join(parts) + cdb + tail + eocd, np.array(offs, np.uint64), np.array(lens, np.uint64)


def members_as_entries(w):
    """the gzip members of a bench workload -> [(8, raw payload, crc, size)] (the bench's 10-byte headers)"""
    src = w["src"].tobytes()
    out = []
    for o, n in zip(w["src_off"].tolist(), w["src_len"].tolist()):
        m = src[o:o + n]
        assert m[:4] == b"\x1f\x8b\x08\x00"
        crc, isize = struct.unpack("<II", m[-8:])
        out.append((8, m[10:-8], crc, isize))
    return out


def deflate(data: bytes, level=6) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return c.compress(data) + c.flush()


def timed(arms: dict, min_ms: float, dev) -> dict:
    import torch
    for fn in arms.values():
        fn()
    torch.cuda.synchronize(dev)
    times = {k: [] for k in arms}
    while min(sum(v) for v in times.values()) < min_ms:
        for k, fn in arms.items():
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            times[k].append(1e3 * (time.perf_counter() - t0))
    return {k: round(float(np.median(v)), 3) for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=65536)
    ap.add_argument("--min-ms", type=float, default=120.0)
    ap.add_argument("--skip", default="", help="comma-separated: z2, z3, z4, sweep")
    args = ap.parse_args()
    skip = set(filter(None, args.skip.split(",")))
    import torch

    import bench
    import starflate_b200 as S
    from tests import deflate_tools as T
    assert torch.cuda.is_available(), "needs a CUDA device"
    info = gpu_info()
    dev = torch.device("cuda", 0)
    ctx = S.Context(0)
    as_i64 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).to(dev)
    to_dev = lambda b: torch.from_numpy(np.frombuffer(b, np.uint8).copy()).to(dev)
    out = {"tool": "zip_bench", **info}

    def zip_arms(data: bytes, tag: str):
        s = to_dev(data)
        st, _, total = ctx.zip_list_device(s)
        assert st == 0
        dst = torch.empty(total, dtype=torch.uint8, device=dev)
        res = {}

        def arm_b():
            st, r, _ = ctx.zip_list_device(s)
            ctx.zip_extract_device(s, r, dst)
            res["rows"] = r

        def arm_l():
            ctx.zip_list_device(s)

        def check():
            r = res["rows"].cpu().numpy().view(S.ZIP_ENTRY).ravel()
            assert (r["status"] == 0).all(), f"{tag}: statuses {np.unique(r['status'])}"
        return arm_b, arm_l, dst, check, total, s

    def batch_arm(w, container):
        d_src = torch.from_numpy(w["src"]).to(dev)
        o, l, do, dc = (as_i64(w[k]) for k in ("src_off", "src_len", "dst_off", "dst_cap"))
        n = len(w["src_off"])
        dst = torch.empty(int(w["total_out"]), dtype=torch.uint8, device=dev)
        stt = torch.zeros(n, dtype=torch.uint8, device=dev)
        wr = torch.zeros(n, dtype=torch.int64, device=dev)

        def arm():
            ctx.decompress_container_batch_device(container, d_src, o, l, dst, do, dc, stt, wr)
        return arm, dst, stt

    # ---- Z1 ----------------------------------------------------------------------------------------
    w1 = bench.make_workload("c2", args.streams, args.streams, 0, container="gzip")
    e1 = members_as_entries(w1)
    z1, _, _ = build_zip(e1)
    arm_a, dst_a, st_a = batch_arm(w1, ctx.GZIP)
    arm_b, arm_l, dst_b, check_b, total, _ = zip_arms(z1, "Z1")
    med = timed({"A": arm_a, "B": arm_b, "L": arm_l}, args.min_ms, dev)
    check_b()
    assert int(st_a.max()) == 0
    out["Z1"] = {"entries": len(e1), "archive_bytes": len(z1), "output_bytes": total, "ms": med,
                 "B_over_A": round(med["B"] / med["A"], 4), "outputs_equal": bool(torch.equal(dst_a, dst_b)),
                 "gb_s_out_B": round(total / med["B"] / 1e6, 1)}
    assert out["Z1"]["outputs_equal"]
    del dst_a, dst_b
    # ---- Z2 ----------------------------------------------------------------------------------------
    if "z2" not in skip:
        w2 = bench.make_workload("c3", 1 << 20, 1 << 20, 0, container="gzip")
        z2, _, _ = build_zip(members_as_entries(w2))
        arm_a2, dst_a2, _ = batch_arm(w2, ctx.GZIP)
        arm_b2, arm_l2, dst_b2, check_b2, total2, _ = zip_arms(z2, "Z2")
        med = timed({"A": arm_a2, "B": arm_b2, "L": arm_l2}, args.min_ms, dev)
        check_b2()
        out["Z2"] = {"entries": 1 << 20, "output_bytes": total2, "ms": med, "B_over_A": round(med["B"] / med["A"], 4),
                     "outputs_equal": bool(torch.equal(dst_a2, dst_b2))}
        del dst_a2, dst_b2, w2, z2

    def alone_arm(payloads):
        """each raw-DEFLATE payload decoded alone with n = 1"""
        items = []
        for pay, size in payloads:
            items.append((to_dev(pay), as_i64([0]), as_i64([len(pay)]), torch.empty(size, dtype=torch.uint8, device=dev),
                          as_i64([0]), as_i64([size]), torch.zeros(1, dtype=torch.uint8, device=dev)))

        def arm():
            for s, o, l, d, do, dc, stt in items:
                ctx.decompress_batch_device(s, o, l, d, do, dc, stt)
        return arm

    # ---- Z3 ----------------------------------------------------------------------------------------
    if "z3" not in skip:
        out["Z3"] = {}
        for tag, size, count in (("one_1GiB", 1 << 30, 1), ("64x16MiB", 16 << 20, 64), ("256x1MiB", 1 << 20, 256)):
            big = [T.big_text(size, 500 + k) for k in range(count)] if count > 1 else [T.big_text(size, 500)]
            pays = [deflate(b, 6) for b in big]
            ents = list(e1)
            for k, (b, p) in enumerate(zip(big, pays)):
                ents.insert(1 + k * 997, (8, p, zlib.crc32(b), len(b)))
            z3, _, _ = build_zip(ents)
            arm_b3, _, _, check_b3, _, _ = zip_arms(z3, "Z3")
            arm_alone = alone_arm([(p, len(b)) for b, p in zip(big, pays)])
            med = timed({"A": arm_a, "alone": arm_alone, "B": arm_b3}, args.min_ms, dev)
            check_b3()
            out["Z3"][tag] = {"ms": med, "B_over_sum": round(med["B"] / (med["A"] + med["alone"]), 4)}
            del z3, big, pays
    # ---- Z4 ----------------------------------------------------------------------------------------
    if "z4" not in skip:
        chunk = np.random.default_rng(4).integers(0, 256, size=64 << 20, dtype=np.uint8).tobytes()
        sizes = [6 << 30] + [64 << 20] * 32
        ents = []
        for sz in sizes:
            pay = (chunk * (sz // len(chunk) + 1))[:sz]
            ents.append((0, pay, zlib.crc32(pay), sz))
        z4, offs, lens = build_zip(ents)
        del ents
        arm_b4, _, dst4, check_b4, total4, s4 = zip_arms(z4, "Z4")
        del z4
        src_view = [s4[int(o):int(o) + int(n)] for o, n in zip(offs, lens)]
        dst_c = torch.empty(total4, dtype=torch.uint8, device=dev)

        def arm_copy():
            at = 0
            for v in src_view:
                dst_c[at:at + v.numel()].copy_(v)
                at += v.numel()
        med = timed({"copy": arm_copy, "B": arm_b4}, args.min_ms, dev)
        check_b4()
        out["Z4"] = {"output_bytes": total4, "ms": med, "B_over_copy": round(med["B"] / med["copy"], 4),
                     "outputs_equal": bool(torch.equal(dst4, dst_c))}
        del dst4, dst_c, s4, src_view
    # ---- the threshold sweep -----------------------------------------------------------------------
    if "sweep" not in skip:
        out["sweep"] = {}
        d_src1 = torch.from_numpy(w1["src"]).to(dev)
        # raw payloads of Z1 inside the gzip members: 10-byte headers, 8-byte trailers
        o1 = as_i64(w1["src_off"].astype(np.uint64) + 10)
        l1 = as_i64(w1["src_len"].astype(np.uint64) - 18)
        for size in (256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20):
            big = [T.big_text(size, 900 + k) for k in range(4)]
            pays = [deflate(b, 6) for b in big]
            blob = b"".join(pays)
            base = len(w1["src"])
            src_all = torch.cat([d_src1, to_dev(blob)])
            po = np.cumsum([0] + [len(p) for p in pays[:-1]]).astype(np.uint64) + base
            n1 = len(w1["src_off"])
            off_all = torch.cat([o1, as_i64(po)])
            len_all = torch.cat([l1, as_i64([len(p) for p in pays])])
            doff_all = torch.cat([as_i64(w1["dst_off"]), as_i64(int(w1["total_out"]) + size * np.arange(4))])
            dcap_all = torch.cat([as_i64(w1["dst_cap"]), as_i64([size] * 4)])
            dst_all = torch.empty(int(w1["total_out"]) + 4 * size, dtype=torch.uint8, device=dev)
            st_all = torch.zeros(n1 + 4, dtype=torch.uint8, device=dev)
            arm_alone = alone_arm([(p, size) for p in pays])

            def arm_in():
                ctx.decompress_batch_device(src_all, off_all, len_all, dst_all, doff_all, dcap_all, st_all)

            def arm_apart():
                ctx.decompress_batch_device(src_all, off_all[:n1], len_all[:n1], dst_all, doff_all[:n1], dcap_all[:n1],
                                            st_all[:n1])
                arm_alone()
            med = timed({"in": arm_in, "apart": arm_apart}, args.min_ms, dev)
            assert int(st_all.max()) == 0
            out["sweep"][f"{size >> 10}KiB"] = {"ms": med, "apart_over_in": round(med["apart"] / med["in"], 4)}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
