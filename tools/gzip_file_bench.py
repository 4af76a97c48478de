"""One BGZF file at batch speed: C2's plaintexts (65 536 x 64 KiB) as ONE BGZF file of 65 536 members,
decoded three ways in one process, warmed and alternated, >= 120 ms timed per arm:

  (A) decompress_container_batch_device(GZIP) over the member table split on the host — the ceiling
  (B) decompress_gzip_file_device on the file — members found on the device
  (C) gzip_file_size on the file (host buffer: includes its upload; the upload alone is timed beside it)

and, for what a plain .gz costs (its end is found by decoding it once more), one plain gzip member
of --plain-mib MiB of text:

  (P1) decompress_container_batch_device(GZIP) on it, n = 1 — the single-stream route
  (P2) decompress_gzip_file_device on it — the probe decode, then the same decode

(B)'s output must equal (A)'s, compared on the device.  Prints one JSON line with the GPU's name and
power limit read in the same run.

  python tools/gzip_file_bench.py [--streams 65536] [--unique 0]
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


def to_bgzf(w) -> tuple[bytes, np.ndarray, np.ndarray]:
    """Each gzip member of the workload gets the 'BC' extra subfield. -> (file, member offsets, lengths)"""
    src = w["src"].tobytes()
    out, offs, lens = [], [], []
    at = 0
    for o, n in zip(w["src_off"].tolist(), w["src_len"].tolist()):
        m = src[o:o + n]
        assert m[:4] == b"\x1f\x8b\x08\x00", "expected the bench's plain gzip header"
        bsize = n + 8 - 1
        assert bsize <= 0xffff, "member too large for BGZF"
        b = b"\x1f\x8b\x08\x04" + m[4:10] + b"\x06\x00BC\x02\x00" + bsize.to_bytes(2, "little") + m[10:]
        out.append(b)
        offs.append(at)
        lens.append(len(b))
        at += len(b)
    return b"".join(out), np.array(offs, np.uint64), np.array(lens, np.uint64)


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
    ap.add_argument("--unique", type=int, default=0, help="distinct seeds (0 = all streams distinct)")
    ap.add_argument("--min-ms", type=float, default=120.0, help="timed milliseconds per arm, at least")
    ap.add_argument("--plain-mib", type=int, default=256, help="size of the plain gzip member (0: skip P1 / P2)")
    ap.add_argument("--profile", action="store_true", help="after the timed arms, one more (B) under torch.profiler: "
                    "device time per kernel name in the JSON line")
    args = ap.parse_args()
    import torch

    import bench
    import starflate_b200 as S
    assert torch.cuda.is_available(), "needs a CUDA device"
    info = gpu_info()
    dev = torch.device("cuda", 0)
    w = bench.make_workload("c2", args.streams, args.unique or args.streams, 0, container="gzip")
    f, m_off, m_len = to_bgzf(w)
    ctx = S.Context(0)
    as_i64 = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).to(dev)
    d_file = torch.from_numpy(np.frombuffer(f, np.uint8).copy()).to(dev)
    d_off, d_len = as_i64(m_off), as_i64(m_len)
    d_doff, d_dcap = as_i64(w["dst_off"]), as_i64(w["dst_cap"])
    total = int(w["total_out"])
    dst_a = torch.zeros(total, dtype=torch.uint8, device=dev)
    dst_b = torch.zeros(total, dtype=torch.uint8, device=dev)
    status = torch.zeros(args.streams, dtype=torch.uint8, device=dev)
    written = torch.zeros(args.streams, dtype=torch.int64, device=dev)

    def arm_a():
        ctx.decompress_container_batch_device(ctx.GZIP, d_file, d_off, d_len, dst_a, d_doff, d_dcap, status, written)

    res_b = {}

    def arm_b():
        res_b["r"] = ctx.decompress_gzip_file_device(d_file, dst_b)

    res_c = {}

    def arm_c():
        res_c["r"] = ctx.gzip_file_size(f)

    f_host = np.frombuffer(f, np.uint8).copy()  # (pageable, like the bytes gzip_file_size uploads)

    def upload():
        torch.from_numpy(f_host).to(dev)

    arms = {"A": arm_a, "B": arm_b, "C": arm_c, "upload": upload}
    plain_total = args.plain_mib << 20
    if plain_total:
        import gzip

        from tests import deflate_tools as T
        plain = T.big_text(plain_total, 5)
        g = gzip.compress(plain, compresslevel=6, mtime=0)
        d_g = torch.from_numpy(np.frombuffer(g, np.uint8).copy()).to(dev)
        g_off, g_len = as_i64(np.array([0], np.uint64)), as_i64(np.array([len(g)], np.uint64))
        g_doff, g_dcap = as_i64(np.array([0], np.uint64)), as_i64(np.array([plain_total], np.uint64))
        dst_p1 = torch.zeros(plain_total, dtype=torch.uint8, device=dev)
        dst_p2 = torch.zeros(plain_total, dtype=torch.uint8, device=dev)
        st1 = torch.zeros(1, dtype=torch.uint8, device=dev)
        wr1 = torch.zeros(1, dtype=torch.int64, device=dev)
        res_p2 = {}

        def arm_p1():
            ctx.decompress_container_batch_device(ctx.GZIP, d_g, g_off, g_len, dst_p1, g_doff, g_dcap, st1, wr1)

        def arm_p2():
            res_p2["r"] = ctx.decompress_gzip_file_device(d_g, dst_p2)

        arms.update({"P1": arm_p1, "P2": arm_p2})
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
    assert int(status.max()) == 0 and int(written.sum()) == total, "arm A failed"
    assert res_b["r"] == (0, total, args.streams), res_b["r"]
    assert res_c["r"] == (total, args.streams, True), res_c["r"]
    same = bool(torch.equal(dst_a, dst_b))
    assert same, "B's output differs from A's"
    if plain_total:
        assert int(st1[0]) == 0 and int(wr1[0]) == plain_total, "arm P1 failed"
        assert res_p2["r"] == (0, plain_total, 1), res_p2["r"]
        assert torch.equal(dst_p1, dst_p2), "P2's output differs from P1's"
    med = {k: float(np.median(v)) for k, v in times.items()}
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
        prof = {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:16]}
    out = {
        "tool": "gzip_file_bench", **info, "members": args.streams, "file_bytes": len(f), "output_bytes": total,
        "ms_median": {k: round(v, 3) for k, v in med.items()}, "reps": {k: len(v) for k, v in times.items()},
        "B_over_A": round(med["B"] / med["A"], 4), "gb_s_out": {k: round(total / med[k] / 1e6, 1) for k in ("A", "B")},
        "C_minus_upload_ms": round(med["C"] - med["upload"], 3), "outputs_equal": same,
        **({"plain_member_bytes": plain_total, "P2_over_P1": round(med["P2"] / med["P1"], 4)} if plain_total else {}),
        "desc": w["desc"] + "; rewritten as one BGZF file", **({"B_profile_ms": prof} if prof else {}),
    }
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
