"""TEST INFRASTRUCTURE ONLY: builds/loads the block-level kernels of tests/cpu_emu (emu_block.cpp
on blocks of host threads, see cuda_shim_block.h) and the single-stream route's pass 1 stopped
before pass 2 (emu_route.cpp).  Not a fallback: nothing in the product package can reach this."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_u8p = C.POINTER(C.c_uint8)
_u64p = C.POINTER(C.c_uint64)


def _build(name, srcs, deps) -> str:
    """g++ srcs -> tests/cpu_emu/lib<name>[_asan].so, rebuilt when a source or header is newer
    (SFB_EMU_ASAN=1: AddressSanitizer + UBSan, as tests/emu_bindings.py)"""
    asan = os.environ.get("SFB_EMU_ASAN") == "1"
    out = os.path.join(HERE, "cpu_emu", f"lib{name}{'_asan' if asan else ''}.so")
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs + deps):
        opt = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer"] if asan else ["-O2"]
        subprocess.check_call(["g++", "-std=c++20", *opt, "-fPIC", "-shared", "-pthread", "-o", out, *srcs])
    return out


def build_block() -> str:
    """libemu_block*.so: the block-level kernels — a library of its own, its warp shim differs from
    cuda_shim_warp.h."""
    emu = os.path.join(HERE, "cpu_emu")
    csrc = os.path.join(ROOT, "starflate_b200", "csrc")
    return _build("emu_block", [os.path.join(emu, "emu_block.cpp")],
                  [os.path.join(emu, "cuda_shim_block.h")] +
                  [os.path.join(csrc, f) for f in ("lz_jump.cuh", "lz_warp.cuh", "stored_copy.cuh", "deflate_lane.cuh",
                                                   "block_finder.cuh")])


def build_route() -> str:
    """libemu_route*.so: the single-stream route's pass 1 with a chain chosen by the caller."""
    emu = os.path.join(HERE, "cpu_emu")
    csrc = os.path.join(ROOT, "starflate_b200", "csrc")
    return _build("emu_route", [os.path.join(emu, "emu_route.cpp"), os.path.join(emu, "emu_lz.cpp")],
                  [os.path.join(emu, f) for f in ("emu_stream.cpp", "cuda_shim_warp.h")] +
                  [os.path.join(csrc, f) for f in ("huff_stream.cuh", "huff_lanes.cuh", "deflate_lane.cuh", "block_finder.cuh",
                                                   "container.cuh", "lz_window.cuh", "lz_warp.cuh")])


# block_finder.cuh: BlockJob
JOB_DTYPE = np.dtype([("start_bit", np.uint64), ("end_bit", np.uint64), ("out", np.uint64), ("base", np.uint64),
                      ("need", np.uint32), ("flags", np.uint32), ("next", np.uint32), ("first_rec", np.uint32)])
JOB_NONE = (1 << 64) - 1
JOB_ENDS, JOB_CLEAN, JOB_RECS, JOB_USE = 1, 2, 4, 8


class EmuBlock:
    """The block-level kernels on blocks of host threads (tests/cpu_emu/emu_block.cpp)."""

    def __init__(self):
        self.lib = C.CDLL(build_block())
        self.lib.emu_jump_resolve.argtypes = [_u8p, _u64p, _u64p, C.POINTER(C.c_uint32), C.c_uint64, C.c_uint64,
                                              C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_uint32)]
        self.lib.emu_chain.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32), C.c_int]
        self.lib.emu_prep_stored.argtypes = [_u8p, _u64p, _u64p, C.POINTER(C.c_uint32), _u8p, _u64p, _u64p, C.c_uint64,
                                             _u8p, _u64p, _u8p, C.POINTER(C.c_uint32), _u64p, C.c_uint32, C.c_int]

    @property
    def chain_parallel_fn(self) -> int:
        """Address of emu_chain_parallel_args (chain_parallel_kernel, checked against chain_kernel
        on every call), for Emu.set_chain."""
        return C.cast(self.lib.emu_chain_parallel_args, C.c_void_p).value

    def chain_checks(self):
        """-> (chains compared, chains that differed) by emu_chain_parallel_args so far"""
        out = np.zeros(2, np.uint64)
        self.lib.emu_chain_checks(out.ctypes.data_as(_u64p))
        return int(out[0]), int(out[1])

    def jump_resolve(self, base, dst_off, written, bits, stripe_tiles=0, warps=8, block_warps=8, reverse=False):
        """Pointer-jumping pass 2 (lz_jump.cuh) in place over `base` (a 128-byte aligned uint8 array)
        for the streams at dst_off with `written` bytes of pass-1 output each. -> rounds used"""
        assert base.ctypes.data % 128 == 0
        off = np.ascontiguousarray(dst_off, dtype=np.uint64)
        wr = np.ascontiguousarray(written, dtype=np.uint64)
        rounds = np.zeros(1, np.uint32)
        p = lambda a, t: a.ctypes.data_as(t)
        self.lib.emu_jump_resolve(p(base, _u8p), p(off, _u64p), p(wr, _u64p), p(bits, C.POINTER(C.c_uint32)),
                                  len(off), len(base), stripe_tiles, warps, block_warps, int(reverse),
                                  p(rounds, C.POINTER(C.c_uint32)))
        return int(rounds[0])

    def chain(self, jobs, dst_cap, parallel=True, count=None, job_cap=None):
        """chain_parallel_kernel (or chain_kernel) over a JOB_DTYPE array, in place -> tail job"""
        tail = np.full(1, 0xDEADBEEF, np.uint32)
        n = len(jobs)
        self.lib.emu_chain(jobs.ctypes.data, n if count is None else count, n if job_cap is None else job_cap,
                           dst_cap, tail.ctypes.data_as(C.POINTER(C.c_uint32)), int(parallel))
        return int(tail[0])

    def prep_stored(self, srcs, dst, dst_off, dst_cap, status, written, warps=16, reverse=False):
        """prep_count/prep_scatter_kernel + stored_streams_kernel over a batch: srcs[i] = (bytes,
        phase), each stream in an allocation of its own that ends at its last byte and starts `phase`
        bytes before it.  status / written are updated in place. -> (order, type_count, handled)"""
        n = len(srcs)
        slen = np.array([len(b) for b, _ in srcs], np.uint64)
        at = np.concatenate([[0], np.cumsum(slen)[:-1]]).astype(np.uint64)
        cat = np.frombuffer(b"".join(b for b, _ in srcs) + b"\0", dtype=np.uint8)
        phase = np.array([ph for _, ph in srcs], np.uint32)
        off = np.ascontiguousarray(dst_off, dtype=np.uint64)
        cap = np.ascontiguousarray(dst_cap, dtype=np.uint64)
        order = np.full(n, 0xFFFFFFFF, np.uint32)
        tc = np.zeros(4, np.uint64)
        handled = np.full(n, 0x77, np.uint8)
        u32p = C.POINTER(C.c_uint32)
        p = lambda a, t: a.ctypes.data_as(t)
        self.lib.emu_prep_stored(p(cat, _u8p), p(at, _u64p), p(slen, _u64p), p(phase, u32p), p(dst, _u8p), p(off, _u64p),
                                 p(cap, _u64p), n, p(status, _u8p), p(written, _u64p), p(handled, _u8p),
                                 p(order, u32p), p(tc, _u64p), warps, int(reverse))
        return order, tc, handled


class EmuRoute:
    """Pass 1 of the single-stream route (tests/cpu_emu/emu_route.cpp)."""

    def __init__(self):
        self.lib = C.CDLL(build_route())
        self.lib.emu_set_chain.argtypes = [C.c_void_p]
        self.lib.emu_stream_pass1.argtypes = [_u8p, C.c_uint64, _u8p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint32),
                                              _u8p, _u64p, _u64p, C.c_int64, C.POINTER(C.c_uint32)]

    def set_chain(self, fn=None):
        """The chain of block jobs: chain_kernel (None) or the function at address `fn`
        (EmuBlock.chain_parallel_fn)."""
        self.lib.emu_set_chain(fn)

    def stream_pass1(self, src: bytes, base, dst_off: int, cap: int, bits, cand=None):
        """Pass 1 of the single-stream route (block finder — or the candidate block starts `cand` —
        counting jobs, chain, writing jobs) into `base` (a 128-byte aligned uint8 array) at dst_off,
        match heads into `bits` (uint32, bit k <-> base[k]): the token layout pass 2 starts from.
        -> (status, written, jobs on the chain, tail job)"""
        assert base.ctypes.data % 128 == 0
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        c = np.asarray(list(cand or []) + [0], dtype=np.uint64)
        st = np.zeros(1, np.uint8)
        wr = np.zeros(1, np.uint64)
        stats = np.zeros(2, np.uint32)
        u32p = C.POINTER(C.c_uint32)
        p = lambda a, t: a.ctypes.data_as(t)
        self.lib.emu_stream_pass1(p(s, _u8p), len(src), p(base, _u8p), dst_off, cap, p(bits, u32p), p(st, _u8p),
                                  p(wr, _u64p), p(c, _u64p), -1 if cand is None else len(cand), p(stats, u32p))
        return int(st[0]), int(wr[0]), int(stats[0]), int(stats[1])
