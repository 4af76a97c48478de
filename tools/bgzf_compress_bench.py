"""One buffer compressed to BGZF at batch speed: C2's plaintexts (65 536 x 64 KiB, decoded from the
bench's streams and checked against the generator's checksums) laid out as ONE 4 GiB buffer, compressed
two ways in one process, warmed and alternated, >= --min-ms timed per arm:

  (A) compress_batch_device over the same 65 280-byte pieces split on the host: raw DEFLATE, the ceiling
  (B) compress_bgzf_device on the whole buffer: pieces, checksums, headers and placement on the device

then (B)'s output decoded by decompress_gzip_file_device (timed; device checksums must equal the
input's), the output ratio beside zlib level 6 per piece (gzip_file_tools.bgzf) on a sample, and
optionally (C) compress_batch_device of ONE --single-mib buffer, timed once after the others: the
one-warp path a caller without BGZF takes.  Prints one JSON line with the GPU's name and power limit read in the same run.

  python tools/bgzf_compress_bench.py [--streams 65536] [--unique 2048] [--single-mib 16] [--profile]
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
    ap.add_argument("--single-mib", type=int, default=16, help="size of arm C's one buffer, timed once (0: skip C)")
    ap.add_argument("--profile", action="store_true", help="after the timed arms, one more (B) under torch.profiler: "
                    "device time per kernel name in the JSON line")
    args = ap.parse_args()
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
    del w
    pieces = (total + PIECE - 1) // PIECE
    # (A) the same pieces, split on the host
    p_off = np.arange(pieces, dtype=np.uint64) * np.uint64(PIECE)
    p_len = np.minimum(np.uint64(total) - p_off, np.uint64(PIECE))
    caps = p_len + np.uint64(5) * ((p_len + np.uint64(65534)) // np.uint64(65535))
    c_off = np.zeros(pieces, np.uint64)
    c_off[1:] = np.cumsum(caps)[:-1]
    d_po, d_pl, d_co, d_cc = as_i64(p_off), as_i64(p_len), as_i64(c_off), as_i64(caps)
    out_a = torch.zeros(int(caps.sum()) + 64, dtype=torch.uint8, device=dev)
    st_a = torch.zeros(pieces, dtype=torch.uint8, device=dev)
    wr_a = torch.zeros(pieces, dtype=torch.int64, device=dev)

    def arm_a():
        ctx.compress_batch_device(plain, d_po, d_pl, out_a, d_co, d_cc, st_a, wr_a)

    out_b = torch.zeros(ctx.compress_bgzf_bound(total), dtype=torch.uint8, device=dev)
    res_b = {}

    def arm_b():
        res_b["r"] = ctx.compress_bgzf_device(plain, out_b)

    arms = {"A": arm_a, "B": arm_b}
    single = args.single_mib << 20
    if single:
        one_o, one_l = as_i64([0]), as_i64([single])
        one_c = ctx.compress_container_bound(0, single)
        out_c = torch.zeros(one_c, dtype=torch.uint8, device=dev)
        d_oc = as_i64([one_c])
        st_c = torch.zeros(1, dtype=torch.uint8, device=dev)
        wr_c = torch.zeros(1, dtype=torch.int64, device=dev)

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
    if single:  # (one warp: far too slow to alternate with the others)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        ctx.compress_batch_device(plain, one_o, one_l, out_c, one_o, d_oc, st_c, wr_c)
        torch.cuda.synchronize(dev)
        times["C"] = [1e3 * (time.perf_counter() - t0)]
        assert int(st_c[0]) == 0, "arm C failed"
    assert int(st_a.max()) == 0, "arm A failed"
    b_st, b_wr, b_nm = res_b["r"]
    assert (b_st, b_nm) == (0, pieces + 1), res_b["r"]
    # the payloads of B are A's streams: sizes add up exactly
    a_bytes = int(wr_a.sum())
    assert b_wr == a_bytes + 26 * pieces + 28, (b_wr, a_bytes)
    # decode B's output; device checksums against the input's
    back = torch.zeros(total + 64, dtype=torch.uint8, device=dev)
    f = out_b[:b_wr]
    dec = []
    for _ in range(4):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        r = ctx.decompress_gzip_file_device(f, back)
        torch.cuda.synchronize(dev)
        dec.append(1e3 * (time.perf_counter() - t0))
    assert r == (0, total, pieces + 1), r
    zero, ln = as_i64([0]), as_i64([total])
    s0, s1 = torch.zeros(1, dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
    ctx.checksum_batch_device(plain, zero, ln, s0)
    ctx.checksum_batch_device(back, zero, ln, s1)
    torch.cuda.synchronize(dev)
    round_trip = int(s0[0]) == int(s1[0])
    assert round_trip, "decode of B's output differs from the input"
    # ratio beside zlib level 6 per piece, on a sample of whole pieces from the start
    sample = min(total, (args.sample_mib << 20) // PIECE * PIECE)
    plain_sample = plain[:sample].cpu().numpy().tobytes()
    z6 = len(G.bgzf(plain_sample, piece=PIECE))
    ours_sample = ctx.compress_bgzf(plain_sample)[1]
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
    out = {
        "tool": "bgzf_compress_bench", **info, "input_bytes": total, "pieces": pieces,
        "ms_median": {k: round(v, 3) for k, v in med.items()}, "reps": {k: len(v) for k, v in times.items()},
        "B_over_A": round(med["B"] / med["A"], 4),
        "gb_s_in": {k: round((single if k == "C" else total) / med[k] / 1e6, 2) for k in med},
        "bgzf_bytes": b_wr, "ratio": round(total / b_wr, 4),
        "sample_bytes": sample, "sample_ratio": round(sample / len(ours_sample), 4), "sample_zlib6_ratio": round(sample / z6, 4),
        "decode_ms_median": round(float(np.median(dec)), 3), "decode_gb_s_out": round(total / float(np.median(dec)) / 1e6, 1),
        "round_trip_checksums_equal": round_trip,
        **({"single_buffer_bytes": single} if single else {}),
        "desc": f"C2 plaintexts ({n} x 64 KiB) as one buffer of {total} B",
        **({"B_profile_ms": prof} if prof else {}),
    }
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
