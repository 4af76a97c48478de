#!/usr/bin/env python3
"""bench.py — decompressed GB/s of batched dynamic-Huffman raw-DEFLATE decompression.

Metric (BASELINE.json): decompressed GB/s, device-timed, batched dynamic-Huffman, at 1/2/4/8
B200, next to the reference CPU path.  Workload = BASELINE.json configs[1] ("C2"): 65,536
independent 64 KiB level-6 text-like streams per GPU (weak scaling: every rank decodes its own
full batch; streams are independent, so there is no collective on the data path — the only
torch.distributed traffic is the barrier / max-over-ranks of the timing).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path
  python bench.py --impl reference ...                            the reference's CPU decompress()
  python bench.py ... --dump-outputs DIR                          also write the last timed step's outputs

One JSON line on stdout (rank 0).  See DESIGN.md §Measurement for the definition of every key.
The inputs are generated from fixed seeds, so two builds run with the same arguments decode the same
streams and their --dump-outputs files can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from

from tests import deflate_tools as T  # noqa: E402  (synthetic corpus generators)

METRIC = "decompressed GB/s (device-timed) batched dynamic-Huffman"
UNIT = "GB/s"


_HTML = None


def _html_plain(size: int, seed: int) -> bytes:
    """A `size`-byte window of real HTML: the reference's own test page (decoded from the committed
    fixture tests/golden/bases/starfleet_dynamic.deflate), read cyclically from a seeded offset."""
    global _HTML
    if _HTML is None:
        with open(os.path.join(ROOT, "tests", "golden", "bases", "starfleet_dynamic.deflate"), "rb") as f:
            _HTML = zlib.decompress(f.read(), -15)
    off = (seed * 7919) % len(_HTML)
    rep = (_HTML[off:] + _HTML * (size // len(_HTML) + 2))[:size]
    return rep


_CONTAINER = "raw"
_GOLD = np.uint64(0x9E3779B97F4A7C15)


def _weighted_sum(plain: bytes) -> int:
    """sfb200_checksum_batch_device's position-weighted sum (include/starflate_b200.h), on the host."""
    total = np.uint64(0)
    with np.errstate(over="ignore"):
        for o in range(0, len(plain), 1 << 22):  # (pieces: a 1 GiB stream would need 30 GB of temporaries)
            b = np.frombuffer(plain, dtype=np.uint8, count=min(1 << 22, len(plain) - o), offset=o).astype(np.uint64)
            j = np.arange(o + 1, o + len(b) + 1, dtype=np.uint64)
            total += ((b + np.uint64(1)) * ((_GOLD * j) | np.uint64(1))).sum(dtype=np.uint64)
    return int(total)


def _wrap(comp: bytes, plain: bytes) -> bytes:
    if _CONTAINER == "zlib":
        return b"\x78\x9c" + comp + zlib.adler32(plain).to_bytes(4, "big")
    if _CONTAINER == "gzip":
        return (b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\x03" + comp + zlib.crc32(plain).to_bytes(4, "little") +
                (len(plain) & 0xffffffff).to_bytes(4, "little"))
    return comp


def _gen_one(args):
    global _CONTAINER
    kind, size, seed, _CONTAINER = args
    if kind == "html":
        plain = _html_plain(size, seed)
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY)
        comp = co.compress(plain) + co.flush()
        return _wrap(comp, plain), zlib.crc32(plain), len(plain), _weighted_sum(plain)
    if kind == "single":
        plain = T.big_text(size, seed)
        comp = T.raw_deflate(plain, 6)
        return _wrap(comp, plain), zlib.crc32(plain), len(plain), 0  # (one large stream: its whole CRC-32 is checked)
    plain, comp = T.make_stream(kind, size, seed)
    assert T.first_block_type(comp) == {"dynamic": 2, "fixed": 1, "stored": 0}.get(kind, 2) or kind in ("repetitive", "multiblock")
    return _wrap(comp, plain), zlib.crc32(plain), len(plain), _weighted_sum(plain)


def make_workload(name: str, n_streams: int, unique: int, rank: int, container: str = "raw", first: int = 0,
                  shared_seeds: bool = False):
    """-> dict(src u8, src_off, src_len, dst_off, dst_cap (u64 numpy), total_out, desc).
    `first`, `shared_seeds`: streams [first, first + n_streams) of ONE global batch (stream g has
    seed number g mod unique whatever the rank: the shards of a strong-scaling run add up to the
    same batch at every GPU count)."""
    if name == "c2":
        kind, size = "dynamic", 65536
    elif name == "c3":
        kind, size = "mixed", 4096
    elif name in ("c3s", "c3f", "c3d"):   # diagnostics (tools/ab_bench.py): the three page types of C3, one at a time
        kind, size = {"s": "stored", "f": "fixed", "d": "dynamic"}[name[2]], 4096
    elif name == "c4":
        kind, size = "repetitive", 1 << 20
    elif name == "c1":     # one ~1 MiB text stream (the reference's own CPU-runnable case)
        kind, size = "single", 1 << 20
    elif name == "c5":     # one 1 GiB text stream: the single-stream route (block finder + pointer jumping)
        kind, size = "single", 1 << 30
    elif name == "html":   # not a BASELINE config: real-HTML statistics (rich alphabet), 64 KiB streams
        kind, size = "html", 65536
    else:
        raise ValueError(name)
    if shared_seeds:
        ids = np.unique((first + np.arange(n_streams)) % unique)   # the seeds this shard needs
    else:
        unique = min(unique, n_streams)
        ids = np.arange(unique)
    jobs = []
    for i in ids:
        k = kind if kind != "mixed" else ["stored", "fixed", "dynamic"][int(i) % 3]
        jobs.append((k, size, 1_000_003 * ((0 if shared_seeds else rank) + 1) + int(i), container))
    unique_here = len(jobs)
    workers = max(1, min(os.cpu_count() or 1, 64))
    t0 = time.time()
    with ProcessPoolExecutor(workers) as ex:
        res = list(ex.map(_gen_one, jobs, chunksize=max(1, unique_here // (workers * 4))))
    gen_s = time.time() - t0
    comp = [r[0] for r in res]
    lens = np.array([len(c) for c in comp], dtype=np.uint64)
    offs = np.zeros(unique_here, dtype=np.uint64)
    offs[1:] = np.cumsum(lens)[:-1]
    src = np.frombuffer(b"".join(comp), dtype=np.uint8)
    if shared_seeds:
        sel = np.searchsorted(ids, (first + np.arange(n_streams)) % unique)
    else:
        sel = np.arange(n_streams) % unique
    caps = np.array([r[2] for r in res], dtype=np.uint64)[sel]
    dst_off = np.zeros(n_streams, dtype=np.uint64)
    dst_off[1:] = np.cumsum(caps)[:-1]
    # every stream gets its own copy of the compressed bytes (no two streams share input lines)
    src_len = lens[sel]
    src_off = np.zeros(n_streams, dtype=np.uint64)
    src_off[1:] = np.cumsum(src_len)[:-1]
    if unique_here == n_streams and not shared_seeds:
        src_full = src
    else:
        # (gather with one index array: stream i's bytes are src[offs[u] ...], u = sel[i])
        rep = np.repeat(offs[sel].astype(np.int64) - src_off.astype(np.int64), src_len.astype(np.int64))
        src_full = src[np.arange(int(src_len.sum()), dtype=np.int64) + rep]
    return {
        "src": src_full, "src_off": src_off, "src_len": src_len, "dst_off": dst_off, "dst_cap": caps,
        "total_out": int(caps.sum()), "total_in": int(src_len.sum()), "n": n_streams,
        "crc": np.array([r[1] for r in res], dtype=np.uint64)[sel], "gen_s": gen_s,
        "sum": np.array([r[3] for r in res], dtype=np.uint64)[sel],
        "desc": f"{name}: {n_streams} x {size} B {kind} level-{'9' if name == 'c4' else '6'} streams"
                f" ({unique_here} unique seeds, zlib {zlib.ZLIB_RUNTIME_VERSION})"
                + ("" if container == "raw" else f", each in a {container} container (checksum verified on the device)"),
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.samples = []   # (host time the line arrived, line)
        self.proc = None
        self.index = index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def mark_begin(self):
        """nvidia-smi is started well before (it takes ~0.1 s to come up): only the samples between
        mark_begin() and mark_end() — the timed region — are reported."""
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [l for t, l in self.samples if self.t0 is None or (self.t0 <= t <= (self.t1 or t) + 0.03)]
        if not lines:  # a region shorter than one sampling period: the samples nearest to it
            lines = [l for t, l in self.samples][-3:]
        for s in lines:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_STREAMS = 1 << 20   # at most this many entries of status / written (12 MiB as float32 + float64) ...
DUMP_BYTES = 11 << 20    # ... and of the decompressed bytes (44 MiB as float32): under 64 MB in all


def _sample(t, k: int):
    """`t` itself when it has at most `k` elements, else `k` of them, one from each of `k` equal
    strata at an offset drawn from a fixed seed: the same positions on every run."""
    import torch
    n = t.numel()
    if n <= k:
        return t
    pos = np.arange(k, dtype=np.int64) * (n // k) + np.random.default_rng(0).integers(0, n // k, k)
    return t[torch.from_numpy(pos).to(t.device)]


def dump_outputs(out_dir: str, d_dst, total_out: int, d_status, d_written):
    """What the decode step returned to its caller, as .npy files: status.npy (float32) and
    written.npy (float64) per stream, and dst.npy (float32), the decompressed bytes of the whole
    batch end to end; each is complete or a fixed sample of DUMP_STREAMS / DUMP_BYTES entries."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("status", _sample(d_status, DUMP_STREAMS).float()),
                    ("written", _sample(d_written, DUMP_STREAMS).double()),
                    ("dst", _sample(d_dst[:total_out], DUMP_BYTES).float())):
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def cpu_baseline(w, seconds_budget: float = 15.0, threads: int | None = None):
    """The reference's own CPU decompress() (oracle/_ref, built from the unmodified reference
    sources) — or the C port if that library is absent — one stream per core over all host cores,
    on a bounded prefix of the same workload."""
    from oracle import bindings
    threads = min(threads or (os.cpu_count() or 1), w["n"])
    ref = bindings.load_reference()
    kind = "reference" if ref is not None else "port"
    impl = ref if ref is not None else bindings.load_oracle()
    # ~60 MB/s/core on text (BASELINE.md §2): bound the sample to about `seconds_budget`
    est_rate = 55e6 * threads
    avg = w["total_out"] / w["n"]
    m = int(max(threads * 4, min(w["n"], est_rate * seconds_budget / avg)))
    m = min(m, w["n"])
    out_bytes = int(w["dst_cap"][:m].sum())
    dst = np.zeros(int(w["dst_off"][m - 1] + w["dst_cap"][m - 1]) + 64, dtype=np.uint8)
    args = (w["src"], w["src_off"][:m].copy(), w["src_len"][:m].copy(), dst,
            w["dst_off"][:m].copy(), w["dst_cap"][:m].copy())
    best = None
    reps = 2 if out_bytes < (512 << 20) else 1
    for _ in range(reps):
        t0 = time.perf_counter()
        r = impl.decompress_batch(*args, threads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    status = r if kind == "reference" else r[0]
    assert not np.asarray(status).any(), "CPU baseline failed to decode the sample"
    # spot-check bytes
    for i in (0, m // 2, m - 1):
        o = int(w["dst_off"][i])
        assert zlib.crc32(dst[o:o + int(w["dst_cap"][i])].tobytes()) == int(w["crc"][i])
    return {"value": out_bytes / best / 1e9, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"first {m} of {w['n']} streams ({out_bytes / 1e6:.1f} MB out), best of {reps}, "
                      f"one stream per thread, static partition"}, best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5", "html"])
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (0 = the config's size)")
    ap.add_argument("--unique", type=int, default=0, help="distinct seeds (0 = all streams distinct)")
    ap.add_argument("--container", default="raw", choices=["raw", "zlib", "gzip"],
                    help="wrap every stream in a zlib / gzip container and verify its checksum on the device "
                         "(extension; the BASELINE metric is raw)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-shapes", action="store_true", help="only the headline workload (skip the sharded C3 batch "
                    "and the C1 / C4 / C5 lines)")
    ap.add_argument("--shard-streams", type=int, default=1048576, help="streams of the sharded (strong-scaling) batch")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps of the headline workload, write "
                    "what its last step returned (status, written, decompressed bytes as float32 / float64; a "
                    "fixed sample of the larger ones, under 64 MB in all) as DIR/<name>.npy (rank 0 under torchrun)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    default_n = {"c1": 1, "c2": 65536, "c3": 1048576, "c4": 16384, "c5": 1, "html": 65536}[args.workload]
    n_streams = args.streams or default_n
    unique = args.unique or n_streams
    if args.workload == "c3" and not args.unique:
        unique = 65536

    if args.impl == "reference":
        if rank != 0:
            return
        w = make_workload(args.workload, min(n_streams, 8192), min(unique, 8192), 0)
        vals = []
        cb = None
        for i in range(args.warmup + args.steps):
            cb, dt = cpu_baseline(w, seconds_budget=max(2.0, 120.0 / (args.warmup + args.steps)))
            if i >= args.warmup:
                vals.append(cb["value"])
        v = float(np.mean(vals)) if vals else cb["value"]
        cb["value"] = v
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": (w["total_out"] / (v * 1e9) * 1e3) if v else None, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": w["desc"], "note": "reference CPU decompress(), bounded sample per step"},
                "cpu_baseline": cb,
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path "
                         "(use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import starflate_b200 as S
    from starflate_b200 import build, sharding
    if rank == 0:
        build.build_all()
    if world > 1:
        dist.barrier()
    ctx = S.Context(local_rank)
    peak, peak_src = measured_peak_gbs()

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def traffic_of(name):
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        try:
            return json.load(open(tpath)).get(name)
        except Exception:
            return None

    def measure(name, w, steps, warmup, want_e2e, streams_total=None, min_region_ms=0.0, dump_dir=None):
        """One workload on this rank's GPU: device-timed steps (CUDA events, max over ranks), the
        correctness gate, per-pass times, optionally the end-to-end number through host buffers and
        the outputs of the last timed step (dump_dir)."""
        n = w["n"]
        to_i64 = lambda a: torch.from_numpy(a.view(np.int64))
        h_src = torch.from_numpy(w["src"]).pin_memory() if want_e2e else torch.from_numpy(w["src"])
        d_src = h_src.to(dev, non_blocking=True)
        d_src_off, d_src_len = to_i64(w["src_off"]).to(dev), to_i64(w["src_len"]).to(dev)
        d_dst_off, d_dst_cap = to_i64(w["dst_off"]).to(dev), to_i64(w["dst_cap"]).to(dev)
        d_dst = torch.zeros(w["total_out"] + 64, dtype=torch.uint8, device=dev)
        d_status = torch.zeros(n, dtype=torch.uint8, device=dev)
        d_written = torch.zeros(n, dtype=torch.int64, device=dev)

        def step():
            if args.container != "raw":
                ctx.decompress_container_batch_device({"zlib": ctx.ZLIB, "gzip": ctx.GZIP}[args.container], d_src,
                                                      d_src_off, d_src_len, d_dst, d_dst_off, d_dst_cap, d_status,
                                                      d_written)
                return
            ctx.decompress_batch_device(d_src, d_src_off, d_src_len, d_dst, d_dst_off, d_dst_cap,
                                        d_status, d_written)

        sampler = ClockSampler(local_rank)
        sampler.start()
        for _ in range(max(warmup, 0)):
            step()
        barrier()
        # correctness gate before timing anything: status, sizes, and the position-weighted checksum
        # of EVERY stream (computed on the device) against the generator's, plus the CRC-32 of a sample
        assert int(d_status.max()) == 0, "decode failed"
        assert torch.equal(d_written, d_dst_cap)
        sums = torch.zeros(n, dtype=torch.int64, device=dev)
        ctx.checksum_batch_device(d_dst, d_dst_off, d_written, sums)
        torch.cuda.synchronize(dev)
        if n > 1:
            bad = np.nonzero(sums.cpu().numpy().view(np.uint64) != w["sum"])[0]
            assert len(bad) == 0, f"{name}: {len(bad)} of {n} streams decoded to the wrong bytes (first: stream {int(bad[0])})"
        for i in np.unique(np.linspace(0, n - 1, 16).astype(np.int64)):
            o, c = int(w["dst_off"][i]), int(w["dst_cap"][i])
            assert zlib.crc32(d_dst[o:o + c].cpu().numpy().tobytes()) == int(w["crc"][i]), f"stream {i}"

        # the clock sampler must be up before the timed region starts (nvidia-smi takes ~0.1-0.5 s),
        # and a secondary shape's region is stretched to several sampling periods (more steps — the
        # headline keeps exactly the K steps it was asked for)
        t_wait = time.time()
        while sampler.proc is not None and not sampler.samples and time.time() - t_wait < 3.0:
            time.sleep(0.01)
        if min_region_ms > 0:
            ew0, ew1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ew0.record()
            step()
            ew1.record()
            torch.cuda.synchronize(dev)
            est = max(sharding.max_over_ranks(ew0.elapsed_time(ew1), dev), 0.05)
            steps = int(min(400, max(steps, np.ceil(min_region_ms / est))))
        launches0 = ctx.launch_info()["kernel_launches"]
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        sampler.mark_begin()
        t_wall0 = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        # small workloads (C1) would sit in the 126 MB L2 from one step to the next: flush it in between
        # (outside the per-step events, which are then what is summed)
        small = w["total_in"] + w["total_out"] < (512 << 20)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None
        e0.record()
        for a, b in evs:
            if small:
                flush.fill_(1)
            a.record()
            step()
            b.record()
        e1.record()
        barrier()
        t_wall = time.perf_counter() - t_wall0
        sampler.mark_end()
        kern_ms = [a.elapsed_time(b) for a, b in evs]
        total_ms = sum(kern_ms) if small else e0.elapsed_time(e1)
        launches = ctx.launch_info()["kernel_launches"] - launches0
        clocks = sampler.stop()
        total_ms = sharding.max_over_ranks(total_ms, dev)  # a sharded job is as slow as its slowest rank
        ms_per_step = total_ms / steps
        out_all = streams_total["total_out"] if streams_total else world * w["total_out"]
        value = out_all / (ms_per_step * 1e-3) / 1e9
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, d_dst, w["total_out"], d_status, d_written)

        e2e = None
        if want_e2e:
            h_dst = torch.empty(w["total_out"], dtype=torch.uint8).pin_memory()
            h_np_dst = h_dst.numpy()
            e_steps = max(1, min(steps, 3))
            ctx.decompress_batch_host(w["src"], w["src_off"], w["src_len"], h_np_dst, w["dst_off"], w["dst_cap"])
            # what the host link gives this rank while all ranks copy at once (the ceiling of e2e:
            # every decompressed byte crosses it once)
            d_probe = d_dst[: min(w["total_out"], 1 << 30)]
            h_probe = h_dst[: d_probe.numel()]
            barrier()
            t0 = time.perf_counter()
            h_probe.copy_(d_probe, non_blocking=True)
            torch.cuda.synchronize(dev)
            d2h_gbs = d_probe.numel() / (time.perf_counter() - t0) / 1e9
            barrier()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                st, wr = ctx.decompress_batch_host(h_src.numpy(), w["src_off"], w["src_len"], h_np_dst,
                                                   w["dst_off"], w["dst_cap"])
            barrier()
            dt = (time.perf_counter() - t0) / e_steps
            assert not st.any()
            o, c = int(w["dst_off"][n - 1]), int(w["dst_cap"][n - 1])
            assert zlib.crc32(h_np_dst[o:o + c].tobytes()) == int(w["crc"][n - 1])
            dt = sharding.max_over_ranks(dt, dev)
            d2h_min = -sharding.max_over_ranks(-d2h_gbs, dev)
            e2e = {"value": world * w["total_out"] / dt / 1e9, "unit": UNIT,
                   "h2d_bytes_per_step": int(w["total_in"] + 32 * n),
                   "d2h_bytes_per_step": int(w["total_out"] + 9 * n),
                   "steps": e_steps, "timer": "host wall clock around sfb200_decompress_batch_host (pinned buffers)",
                   "device_staging_bytes": ctx.staging_bytes(),
                   "host_link": {"d2h_gbs_per_rank_all_ranks_copying": d2h_min,
                                 "frac_of_link": (w["total_out"] / dt / 1e9) / d2h_min if d2h_min else None,
                                 "note": "every decompressed byte crosses PCIe device-to-host once: the measured "
                                         "pinned D2H rate (slowest rank, all ranks copying at the same time) is "
                                         "the ceiling of this number"}}
            del h_dst

        # per-pass device time (CUDA events recorded inside the C-ABI call on its stream), taken
        # on a few extra steps after the timed region so that the synchronising query stays out of it
        pass_ms = []
        for _ in range(3):
            step()
            pass_ms.append(ctx.last_pass_ms())
        clear_ms, p1_ms, p2_ms = [float(x) for x in np.mean(np.array(pass_ms), axis=0)]
        k_ms = float(np.mean(kern_ms))
        algo_bytes = w["total_in"] + w["total_out"]
        achieved = algo_bytes / (k_ms * 1e-3) / 1e9
        single = n == 1
        k1 = "find/verify candidates + huff_stream_kernel x2 + chain (pass 1)" if single else "huff_lanes_kernel (pass 1)"
        k2 = "lz_jump_* (pass 2)" if single else "lz_window_kernel (pass 2)"
        res = {
            "value": value, "ms_per_step": ms_per_step, "steps": steps,
            "workload": w["desc"], "streams_per_gpu": n, "compressed_bytes_per_gpu": w["total_in"],
            "decompressed_bytes_per_gpu": w["total_out"],
            "l2": ("L2 flushed (256 MB written) before every timed step; value = sum of the per-step events"
                   if small else "inputs+outputs far exceed the 126 MB L2; no flush needed"),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic_of(name), "peak_source": peak_src,
                         "kernel": "whole step: scratch clear + " + k1 + " + " + k2,
                         "dominant_kernel": k1 if p1_ms >= p2_ms else k2, "step_ms": k_ms,
                         "algorithmic_bytes": algo_bytes,
                         "note": "achieved = (compressed read + decompressed written) / device time of the "
                                 "WHOLE step, not of the dominant kernel alone; the two passes run back to back "
                                 "(one launch each), passes_ms = clear and batch preparation | pass 1 | pass 2",
                         "passes_ms": {"clear": clear_ms, k1.split(" (")[0]: p1_ms, k2.split(" (")[0]: p2_ms},
                         "frac_of_nominal_8TBs": achieved / 8000.0},
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e, "wall_s_timed_region": t_wall,
            "gate": f"status, written and the device checksum of all {n} streams against the generator's; CRC-32 of 16",
        }
        del d_src, d_dst, d_status, d_written, sums
        torch.cuda.empty_cache()
        return res

    # ---- the headline workload (BASELINE.json's metric is quoted on C2) ---------------------------
    w = make_workload(args.workload, n_streams, unique, rank, args.container)
    head = measure(args.workload, w, args.steps, args.warmup, not args.no_e2e and args.container == "raw",
                   dump_dir=args.dump_outputs)
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": head["workload"], "streams_per_gpu": head["streams_per_gpu"],
                   "compressed_bytes_per_gpu": head["compressed_bytes_per_gpu"],
                   "decompressed_bytes_per_gpu": head["decompressed_bytes_per_gpu"],
                   "parallelism": f"shard{world} (no collective)", "l2": head["l2"], "gate": head["gate"],
                   "launch": ctx.launch_info()},
        "roofline": head["roofline"], "clocks": head["clocks"], "gpu_launches": head["gpu_launches"],
        "e2e": head["e2e"], "wall_s_timed_region": head["wall_s_timed_region"],
    }
    if rank == 0 and world == 1 and not args.no_cpu and args.container == "raw":
        line["cpu_baseline"], _ = cpu_baseline(w, args.cpu_seconds)
    del w

    # ---- one batch sharded across the ranks (BASELINE configs[2]: 1M 4 KiB pages, mixed blocks):
    #      the same 1 048 576 streams at every GPU count, cut with the library's partition ----------
    if not args.no_shapes and args.workload == "c2" and args.container == "raw":
        total = args.shard_streams
        # (all pages hold 4096 bytes and the three kinds cycle, so equal counts are the balanced cut;
        #  ragged batches go through sfb200_partition_streams — tests/test_sharding_gloo.py)
        first = total * rank // world
        count = total * (rank + 1) // world - first
        ws = make_workload("c3", count, 65536, rank, first=first, shared_seeds=True)
        tot = {"total_out": total * 4096}
        r = measure("c3", ws, max(3, min(args.steps, 5)), 3, False, streams_total=tot, min_region_ms=120.0)
        line["sharded"] = {"workload": f"c3: {total} x 4096 B pages (stored / fixed / dynamic by turns), ONE batch cut "
                                       f"into {world} contiguous shard(s), one per GPU, no collective",
                           "scaling": "strong", "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "steps": r["steps"],
                           "streams_total": total, "streams_this_rank": count, "roofline_frac": r["roofline"]["frac"],
                           "passes_ms": r["roofline"]["passes_ms"], "clocks": r["clocks"]}
        del ws
    # ---- the other named shapes, 1 GPU (north_star: "each named shape is reported") ---------------
    # (N > 1: every rank runs its own copy — weak scaling for the batch C4, independent replicas for
    #  the single streams C1 / C5, which do not shard; value = all ranks' bytes / the slowest rank's time;
    #  roofline is one GPU's)
    if not args.no_shapes and args.workload == "c2" and args.container == "raw":
        shapes = {}
        for nm, ns, uq, st in (("c1", 1, 1, 5), ("c4", 16384, 128, 3), ("c5", 1, 1, 3)):
            wsh = make_workload(nm, ns, uq, rank)
            r = measure(nm, wsh, st, 3, False, min_region_ms=120.0)
            shapes[nm] = {k: r[k] for k in ("workload", "value", "ms_per_step", "steps", "clocks", "gpu_launches", "l2")}
            shapes[nm]["unit"] = UNIT
            shapes[nm]["n_gpus"] = world
            shapes[nm]["scaling"] = "weak" if nm == "c4" else "replicas only (one stream does not shard)"
            shapes[nm]["roofline"] = {k: r["roofline"][k] for k in ("achieved", "peak", "frac", "passes_ms", "algorithmic_bytes")}
            del wsh
        if "sharded" in line:
            shapes["c3"] = {"see": "sharded (the same workload; at 1 GPU the shard is the whole batch)", "n_gpus": world, "scaling": "strong",
                            "value": line["sharded"]["value"], "ms_per_step": line["sharded"]["ms_per_step"],
                            "unit": UNIT, "roofline": {"frac": line["sharded"]["roofline_frac"]},
                            "clocks": line["sharded"]["clocks"]}
        line["shapes"] = shapes
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
