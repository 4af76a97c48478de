"""One buffer compressed to ONE gzip / raw-DEFLATE stream at batch speed: C2's plaintexts (65 536 x 64 KiB,
decoded from the bench's streams and checked against the generator's checksums) laid out as ONE 4 GiB
buffer, compressed in one process, warmed and alternated, >= --min-ms timed per arm:

  (A)     compress_bgzf_device: the same 65 280-byte pieces as a BGZF file, the yardstick
  (B)     compress_parallel_device GZIP: the pieces joined into one stream, bit by bit
  (B_raw) compress_parallel_device RAW

then the ratios of B, BGZF and zlib level 6 (one stream) on a sample; the decode leg: a --decode-mib prefix
compressed by B as RAW and by zlib level 6 as one raw stream, both decoded by decompress_batch_device as
one stream (the single-stream route), timed, outputs checked; and one --single-mib buffer through the
one-warp compressor (compress_batch_device) and through compress_parallel_device, each timed once.
Prints one JSON line with the GPU's name and power limit read in the same run.

  python tools/parallel_compress_bench.py [--streams 65536] [--unique 2048] [--decode-mib 256] [--profile]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

PIECE = 0xff00


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "nvidia_smi_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=65536)
    ap.add_argument("--unique", type=int, default=2048)
    ap.add_argument("--min-ms", type=float, default=1500.0, help="timed milliseconds per arm, at least")
    ap.add_argument("--sample-mib", type=int, default=64, help="plaintext compressed by zlib level 6 for the ratio")
    ap.add_argument("--decode-mib", type=int, default=256, help="prefix of the decode leg (0: skip)")
    ap.add_argument("--single-mib", type=int, default=16, help="buffer of the one-warp comparison (0: skip)")
    ap.add_argument("--profile", action="store_true", help="after the timed arms, one more (B) under torch.profiler: "
                    "device time per kernel name in the JSON line")
    args = ap.parse_args()
    import zlib

    import torch

    import bench
    import starflate_b200 as S
    from tests import gzip_file_tools as G
    assert torch.cuda.is_available(), "needs a CUDA device"
    info = gpu_info()
    dev = torch.device("cuda", 0)
    w = bench.make_workload("c2", args.streams, min(args.unique, args.streams), 0)
    n = w["n"]
    as_i64 = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.uint64).view(np.int64)).to(dev)
    ctx = S.Context(0)
    # the plaintexts: the decoder's output, one contiguous buffer
    total = int(w["total_out"])
    plain = torch.zeros(total, dtype=torch.uint8, device=dev)
    d_do, d_dc = as_i64(w["dst_off"]), as_i64(w["dst_cap"])
    st = torch.zeros(n, dtype=torch.uint8, device=dev)
    wr = torch.zeros(n, dtype=torch.int64, device=dev)
    ctx.decompress_batch_device(torch.from_numpy(w["src"]).to(dev), as_i64(w["src_off"]), as_i64(w["src_len"]), plain,
                                d_do, d_dc, st, wr)
    sums = torch.zeros(n, dtype=torch.int64, device=dev)
    ctx.checksum_batch_device(plain, d_do, wr, sums)
    torch.cuda.synchronize(dev)
    assert int(st.max()) == 0 and np.array_equal(sums.cpu().numpy().view(np.uint64), w["sum"]), "decode of C2 is wrong"
    del w, st, wr, sums
    pieces = (total + PIECE - 1) // PIECE
    RAW, GZIP = 0, 2
    out_a = torch.zeros(ctx.compress_bgzf_bound(total), dtype=torch.uint8, device=dev)
    out_b = torch.zeros(ctx.compress_parallel_bound(GZIP, total), dtype=torch.uint8, device=dev)
    res = {}

    def arm_a():
        res["A"] = ctx.compress_bgzf_device(plain, out_a)

    def arm_b():
        res["B"] = ctx.compress_parallel_device(GZIP, plain, out_b)

    def arm_b_raw():
        res["B_raw"] = ctx.compress_parallel_device(RAW, plain, out_b)

    arms = {"A": arm_a, "B": arm_b, "B_raw": arm_b_raw}
    times = {k: [] for k in arms}
    for fn in arms.values():  # warm every shape
        fn()
    torch.cuda.synchronize(dev)
    while min(sum(v) for v in times.values()) < args.min_ms:
        for k, fn in arms.items():  # alternated
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            times[k].append(1e3 * (time.perf_counter() - t0))
    a_st, a_wr, a_nm = res["A"]
    assert (a_st, a_nm) == (0, pieces + 1), res["A"]
    assert res["B"][0] == 0 and res["B_raw"][0] == 0, (res["B"], res["B_raw"])
    arm_b()  # (out_b holds the gzip stream again)
    torch.cuda.synchronize(dev)
    b_wr = res["B"][1]
    # B's gzip trailer against the CRC-32 of the input computed on the host from a copy
    host_plain = plain.cpu().numpy()
    crc = 0
    for o in range(0, total, 256 << 20):
        crc = zlib.crc32(host_plain[o:o + (256 << 20)], crc)
    trailer = out_b[b_wr - 8:b_wr].cpu().numpy().tobytes()
    trailer_ok = trailer == np.array([crc, total & 0xffffffff], "<u4").tobytes()
    assert trailer_ok, "B's trailer is not the input's CRC-32 / ISIZE"
    # ratios on a sample of whole pieces from the start
    sample = min(total, (args.sample_mib << 20) // PIECE * PIECE)
    s_bytes = host_plain[:sample].tobytes()
    z6 = len(zlib.compress(s_bytes, 6))
    z6_bgzf = len(G.bgzf(s_bytes, piece=PIECE))
    ours = ctx.compress_parallel(GZIP, s_bytes)[1]
    ours_bgzf = ctx.compress_bgzf(s_bytes)[1]
    out = {
        "tool": "parallel_compress_bench", **info, "input_bytes": total, "pieces": pieces,
        "desc": f"C2 plaintexts ({n} x 64 KiB) as one buffer of {total} B",
    }
    # the decode leg: B as RAW against zlib level 6, one stream each, through the single-stream route
    if args.decode_mib:
        m = min(total, args.decode_mib << 20)
        pre = s_bytes[:m] if m <= sample else host_plain[:m].tobytes()
        st_r, ours_raw = ctx.compress_parallel(RAW, pre)
        assert st_r == 0
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        z_raw = co.compress(pre) + co.flush()
        leg = {}
        for name, comp in (("B_raw", ours_raw), ("zlib6", z_raw)):
            d_src = torch.from_numpy(np.frombuffer(comp, np.uint8).copy()).to(dev)
            d_out = torch.zeros(m + 64, dtype=torch.uint8, device=dev)
            z, ln, cap = as_i64([0]), as_i64([len(comp)]), as_i64([m])
            s1 = torch.zeros(1, dtype=torch.uint8, device=dev)
            w1 = torch.zeros(1, dtype=torch.int64, device=dev)
            ms = []
            for _ in range(6):
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                ctx.decompress_batch_device(d_src, z, ln, d_out, z, cap, s1, w1)
                torch.cuda.synchronize(dev)
                ms.append(1e3 * (time.perf_counter() - t0))
            assert int(s1[0]) == 0 and int(w1[0]) == m, (name, int(s1[0]), int(w1[0]))
            assert d_out[:m].cpu().numpy().tobytes() == pre, name
            leg[name] = {"bytes": len(comp), "ms_median_of_5": round(float(np.median(ms[1:])), 3)}
        out["decode_leg"] = {"prefix_bytes": m, **leg,
                             "B_over_zlib6": round(leg["B_raw"]["ms_median_of_5"] / leg["zlib6"]["ms_median_of_5"], 3)}
    # one buffer: the one-warp compressor against compress_parallel, each timed once
    if args.single_mib:
        one = min(total, args.single_mib << 20)
        one_o, one_l = as_i64([0]), as_i64([one])
        one_c = ctx.compress_container_bound(RAW, one)
        out_c = torch.zeros(one_c, dtype=torch.uint8, device=dev)
        st_c = torch.zeros(1, dtype=torch.uint8, device=dev)
        wr_c = torch.zeros(1, dtype=torch.int64, device=dev)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        ctx.compress_batch_device(plain, one_o, one_l, out_c, one_o, as_i64([one_c]), st_c, wr_c)
        torch.cuda.synchronize(dev)
        t_warp = 1e3 * (time.perf_counter() - t0)
        assert int(st_c[0]) == 0
        out_p = torch.zeros(ctx.compress_parallel_bound(RAW, one), dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        r = ctx.compress_parallel_device(RAW, plain[:one], out_p)
        torch.cuda.synchronize(dev)
        t_par = 1e3 * (time.perf_counter() - t0)
        assert r[0] == 0
        out["single_buffer"] = {"bytes": one, "one_warp_ms": round(t_warp, 3), "parallel_ms": round(t_par, 3),
                                "one_warp_out": int(wr_c[0]), "parallel_out": r[1]}
    prof = None
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            arm_b()
            torch.cuda.synchronize(dev)
        per = {}
        for e in p.events():
            if e.device_type.name == "CUDA":
                per[e.name[:60]] = per.get(e.name[:60], 0.0) + (getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)) / 1e3
        prof = {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:12]}
    med = {k: float(np.median(v)) for k, v in times.items()}
    out.update({
        "ms_median": {k: round(v, 3) for k, v in med.items()}, "reps": {k: len(v) for k, v in times.items()},
        "B_over_A": round(med["B"] / med["A"], 4), "B_raw_over_A": round(med["B_raw"] / med["A"], 4),
        "gb_s_in": {k: round(total / med[k] / 1e6, 2) for k in med},
        "bgzf_bytes": a_wr, "gzip_bytes": b_wr, "raw_bytes": res["B_raw"][1], "gzip_trailer_ok": trailer_ok,
        "sample_bytes": sample, "sample_ratio": {"parallel_gzip": round(sample / len(ours), 4),
                                                 "bgzf": round(sample / len(ours_bgzf), 4),
                                                 "zlib6_one_stream": round(sample / z6, 4),
                                                 "zlib6_bgzf": round(sample / z6_bgzf, 4)},
        **({"B_profile_ms": prof} if prof else {}),
    })
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
