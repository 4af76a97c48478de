"""starflate_b200 — B200-native raw-DEFLATE decompressor (drop-in for starflate's decompress path).

This Python module is only the thin harness-side binding of the C ABI in
include/starflate_b200.h (ctypes); the product is the CUDA library itself and the C++23
interface mirror under starflate_b200/cpp/.  There is NO CPU decode path: if the CUDA library
is not built, or no CUDA device is usable, everything here raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

__all__ = ["Context", "StarflateError", "STATUS_NAMES", "ZIP_ENTRY", "load_library", "library_path"]

STATUS_NAMES = {
    0: "Success", 1: "Error", 2: "InvalidBlockHeader", 3: "NoCompressionLenMismatch",
    4: "DstTooSmall", 5: "SrcTooSmall", 6: "InvalidLitOrLen", 7: "InvalidDistance",
}
_RC_NAMES = {0: "OK", 1: "NO_DEVICE", 2: "BAD_ARGUMENT", 3: "CUDA_ERROR", 4: "OUT_OF_MEMORY"}

# one row of a zip archive's entry table (include/starflate_b200.h: sfb200_zip_entry)
ZIP_ENTRY = np.dtype([("name_off", "<u8"), ("data_off", "<u8"), ("comp_size", "<u8"), ("size", "<u8"),
                      ("dst_off", "<u8"), ("written", "<u8"), ("crc32", "<u4"), ("method", "<u2"),
                      ("flags", "<u2"), ("name_len", "<u2"), ("status", "u1"), ("pad", "u1", (5,))])
assert ZIP_ENTRY.itemsize == 64


class StarflateError(RuntimeError):
    pass


_u8p = C.POINTER(C.c_uint8)
_u64p = C.POINTER(C.c_uint64)


class _LaunchInfo(C.Structure):
    _fields_ = [("sm_count", C.c_int), ("warps_per_cta", C.c_int), ("ctas_per_sm", C.c_int),
                ("smem_bytes_per_cta", C.c_int), ("regs_per_thread", C.c_int),
                ("small_warps_per_cta", C.c_int), ("small_ctas_per_sm", C.c_int),
                ("small_regs_per_thread", C.c_int),
                ("stream_ctas_per_sm", C.c_int), ("stream_regs_per_thread", C.c_int),
                ("lz_threads_per_cta", C.c_int), ("lz_ctas_per_sm", C.c_int),
                ("lz_regs_per_thread", C.c_int), ("kernel_launches", C.c_uint64)]


_lib = None


def library_path() -> str:
    return _build.CABI_SO


def load_library() -> C.CDLL:
    """Load the CUDA library.  Raises if it has not been built (no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise StarflateError(
            f"{path} is missing: build it with `python -m starflate_b200.build` "
            "(nvcc, sm_100a). starflate_b200 has no CPU implementation.")
    lib = C.CDLL(path)
    lib.sfb200_abi_version.restype = C.c_int
    lib.sfb200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.sfb200_destroy.argtypes = [C.c_void_p]
    lib.sfb200_destroy.restype = None
    lib.sfb200_last_error.argtypes = [C.c_void_p]
    lib.sfb200_last_error.restype = C.c_char_p
    lib.sfb200_decompress_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.sfb200_decompress_batch_host.argtypes = [C.c_void_p, _u8p, C.c_uint64, _u64p, _u64p, _u8p,
                                                 C.c_uint64, _u64p, _u64p, _u8p, _u64p, C.c_uint64]
    lib.sfb200_decompress.argtypes = [C.c_void_p, _u8p, C.c_size_t, _u8p, C.c_size_t, _u8p, _u64p]
    lib.sfb200_checksum_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_uint64, C.c_void_p]
    lib.sfb200_get_launch_info.argtypes = [C.c_void_p, C.POINTER(_LaunchInfo)]
    lib.sfb200_last_pass_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    _lib = lib
    return lib


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(t)


class Context:
    """One CUDA device (sfb200_ctx).  One per rank; batches shard with no communication."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.sfb200_create(device, C.byref(h))
        if rc != 0:
            raise StarflateError(f"sfb200_create(device={device}) failed: {_RC_NAMES.get(rc, rc)} "
                                 "(a CUDA device is required; there is no CPU path)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.sfb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.sfb200_last_error(self.h)
            raise StarflateError(f"{what}: {_RC_NAMES.get(rc, rc)} {msg.decode() if msg else ''}")

    # -- device-resident batch: arguments are torch CUDA tensors (uint8 data, int64 metadata) --
    def decompress_batch_device(self, src, src_off, src_len, dst, dst_off, dst_cap, status,
                                written=None, stream=None):
        import torch
        n = src_off.numel()
        for t in (src_off, src_len, dst_off, dst_cap):
            assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous() and t.numel() == n
        assert src.is_cuda and src.dtype == torch.uint8 and dst.is_cuda and dst.dtype == torch.uint8
        assert status.is_cuda and status.dtype == torch.uint8 and status.numel() == n
        if written is not None:
            assert written.is_cuda and written.dtype == torch.int64 and written.numel() == n
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        rc = self.lib.sfb200_decompress_batch_device(
            self.h, src.data_ptr(), src_off.data_ptr(), src_len.data_ptr(), dst.data_ptr(),
            dst.numel(), dst_off.data_ptr(), dst_cap.data_ptr(), status.data_ptr(),
            written.data_ptr() if written is not None else None, n, stream)
        self._check(rc, "sfb200_decompress_batch_device")

    RAW, ZLIB, GZIP, AUTO = 0, 1, 2, 3

    def decompress_container_batch_device(self, container, src, src_off, src_len, dst, dst_off, dst_cap, status,
                                          written=None, stream=None):
        """zlib / gzip containers (or AUTO per stream): header, DEFLATE payload, trailer checksum."""
        import torch
        n = src_off.numel()
        for t in (src_off, src_len, dst_off, dst_cap):
            assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous() and t.numel() == n
        assert src.is_cuda and src.dtype == torch.uint8 and dst.is_cuda and dst.dtype == torch.uint8
        assert status.is_cuda and status.dtype == torch.uint8 and status.numel() == n
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        f = self.lib.sfb200_decompress_container_batch_device
        f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        f.restype = C.c_int
        rc = f(self.h, container, src.data_ptr(), src_off.data_ptr(), src_len.data_ptr(), dst.data_ptr(),
               dst.numel(), dst_off.data_ptr(), dst_cap.data_ptr(), status.data_ptr(),
               written.data_ptr() if written is not None else None, n, stream)
        self._check(rc, "sfb200_decompress_container_batch_device")

    def decompress_container(self, container, src: bytes, dst_cap: int, fill: int = 0):
        """One container in host memory -> (status, dst bytes, written)."""
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.full(max(dst_cap, 1), fill, dtype=np.uint8)
        st = C.c_uint8(0)
        wr = C.c_uint64(0)
        f = self.lib.sfb200_decompress_container
        f.argtypes = [C.c_void_p, C.c_int, _u8p, C.c_size_t, _u8p, C.c_size_t, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        rc = f(self.h, container, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap, C.byref(st), C.byref(wr))
        self._check(rc, "sfb200_decompress_container")
        return st.value, d[:dst_cap].tobytes(), wr.value

    def decompress_gzip_file(self, src: bytes, dst_cap: int, fill: int = 0):
        """A gzip file of any number of members (BGZF, `cat a.gz b.gz`), host memory
        -> (status, dst bytes, written, members)."""
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.full(max(dst_cap, 1), fill, dtype=np.uint8)
        st, wr, nm = C.c_uint8(0), C.c_uint64(0), C.c_uint64(0)
        f = self.lib.sfb200_decompress_gzip_file
        f.argtypes = [C.c_void_p, _u8p, C.c_size_t, _u8p, C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64),
                      C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        rc = f(self.h, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap, C.byref(st), C.byref(wr), C.byref(nm))
        self._check(rc, "sfb200_decompress_gzip_file")
        return st.value, d[:dst_cap].tobytes(), wr.value, nm.value

    def decompress_gzip_file_device(self, src, dst, stream=None):
        """A gzip file in a uint8 CUDA tensor into another (synchronous) -> (status, written, members)."""
        import torch
        assert src.is_cuda and src.dtype == torch.uint8 and src.is_contiguous()
        assert dst.is_cuda and dst.dtype == torch.uint8 and dst.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        st, wr, nm = C.c_uint8(0), C.c_uint64(0), C.c_uint64(0)
        f = self.lib.sfb200_decompress_gzip_file_device
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p]
        f.restype = C.c_int
        rc = f(self.h, src.data_ptr(), src.numel(), dst.data_ptr(), dst.numel(), C.byref(st), C.byref(wr), C.byref(nm),
               stream)
        self._check(rc, "sfb200_decompress_gzip_file_device")
        return st.value, wr.value, nm.value

    def gzip_file_size(self, src: bytes):
        """-> (sum of ISIZE over the BGZF members the walk reaches, their number, whether they cover the file)"""
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        sz, nm, cp = C.c_uint64(0), C.c_uint64(0), C.c_int(0)
        f = self.lib.sfb200_gzip_file_size
        f.argtypes = [C.c_void_p, _u8p, C.c_size_t, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
        f.restype = C.c_int
        self._check(f(self.h, _p(s, _u8p), len(src), C.byref(sz), C.byref(nm), C.byref(cp)), "sfb200_gzip_file_size")
        return sz.value, nm.value, bool(cp.value)

    # -- zip archives: list the entry table, then extract any subset or order of its rows -----------
    @staticmethod
    def _zip_rows_guess(n_bytes: int) -> int:
        """Rows to offer the first listing call: every central-directory record takes >= 46 bytes, and
        the table is kept to 1/16 of the archive's size unless that is below 65 536 rows; an archive
        with more entries than this is listed a second time with room for all of them."""
        return min(n_bytes // 46, max(65536, n_bytes // 1024))

    def zip_list(self, data: bytes):
        """-> (status, entries, names): `entries` a ZIP_ENTRY numpy array (the rows of
        sfb200_zip_list), `names` the entries' file names decoded as zipfile decodes them (UTF-8 when
        flag bit 11 is set, else cp437).  status 8 (BadContainer): not an archive this reads."""
        s = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, np.uint8)
        f = self.lib.sfb200_zip_list
        f.argtypes = [C.c_void_p, _u8p, C.c_size_t, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        st, n, total = C.c_uint8(0), C.c_uint64(0), C.c_uint64(0)
        rows = np.zeros(max(self._zip_rows_guess(len(data)), 1), ZIP_ENTRY)
        for _ in range(2):
            self._check(f(self.h, _p(s, _u8p), len(data), rows.ctypes.data, len(rows), C.byref(st), C.byref(n),
                          C.byref(total)), "sfb200_zip_list")
            if n.value <= len(rows):
                break
            rows = np.zeros(n.value, ZIP_ENTRY)
        rows = rows[:n.value]
        names = [bytes(data[o:o + k]).decode("utf-8" if fl & 0x800 else "cp437")
                 for o, k, fl in zip(rows["name_off"].tolist(), rows["name_len"].tolist(), rows["flags"].tolist())]
        return st.value, rows, names

    def zip_extract(self, data: bytes, entries: np.ndarray, dst_cap: int, fill: int = 0):
        """Extract the rows of `entries` (a ZIP_ENTRY array, e.g. zip_list's or a subset of it) into a
        dst of dst_cap bytes -> (dst bytes, the rows with status / written filled in)."""
        s = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, np.uint8)
        rows = np.ascontiguousarray(entries, dtype=ZIP_ENTRY).copy()
        d = np.full(max(dst_cap, 1), fill, dtype=np.uint8)
        f = self.lib.sfb200_zip_extract
        f.argtypes = [C.c_void_p, _u8p, C.c_size_t, C.c_void_p, C.c_uint64, _u8p, C.c_size_t]
        f.restype = C.c_int
        self._check(f(self.h, _p(s, _u8p), len(data), rows.ctypes.data if len(rows) else None, len(rows), _p(d, _u8p),
                      dst_cap), "sfb200_zip_extract")
        return d[:dst_cap].tobytes(), rows

    def zip_list_device(self, src, stream=None):
        """An archive in a uint8 CUDA tensor -> (status, entries, total_size): `entries` a uint8 CUDA
        tensor of shape (n, 64) holding the rows (ZIP_ENTRY layout; .cpu().numpy().view(ZIP_ENTRY))."""
        import torch
        assert src.is_cuda and src.dtype == torch.uint8 and src.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        f = self.lib.sfb200_zip_list_device
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p]
        f.restype = C.c_int
        st, n, total = C.c_uint8(0), C.c_uint64(0), C.c_uint64(0)
        rows = torch.empty((max(self._zip_rows_guess(src.numel()), 1), 64), dtype=torch.uint8, device=src.device)
        for _ in range(2):
            self._check(f(self.h, src.data_ptr(), src.numel(), rows.data_ptr(), rows.shape[0], C.byref(st), C.byref(n),
                          C.byref(total), stream), "sfb200_zip_list_device")
            if n.value <= rows.shape[0]:
                break
            rows = torch.empty((n.value, 64), dtype=torch.uint8, device=src.device)
        rows = rows[:n.value]
        return st.value, rows, total.value

    def zip_extract_device(self, src, entries, dst, stream=None):
        """Extract the rows of `entries` (a uint8 CUDA tensor of shape (n, 64), e.g. zip_list_device's)
        into the uint8 CUDA tensor dst; status / written are written into the rows (synchronous)."""
        import torch
        assert src.is_cuda and src.dtype == torch.uint8 and src.is_contiguous()
        assert dst.is_cuda and dst.dtype == torch.uint8 and dst.is_contiguous()
        assert entries.is_cuda and entries.dtype == torch.uint8 and entries.is_contiguous()
        assert entries.numel() % 64 == 0
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        f = self.lib.sfb200_zip_extract_device
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]
        f.restype = C.c_int
        n = entries.numel() // 64
        self._check(f(self.h, src.data_ptr(), src.numel(), entries.data_ptr() if n else None, n, dst.data_ptr(),
                      dst.numel(), stream), "sfb200_zip_extract_device")

    def decompressed_size_batch_device(self, src, src_off, src_len, status, size, stream=None):
        """Size discovery: status[i] / size[i] of a decode into an unlimited dst; nothing is stored."""
        import torch
        n = src_off.numel()
        assert src.is_cuda and src.dtype == torch.uint8
        for t in (src_off, src_len, size):
            assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous() and t.numel() == n
        assert status.is_cuda and status.dtype == torch.uint8 and status.numel() == n
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        self.lib.sfb200_decompressed_size_batch_device.argtypes = [C.c_void_p] * 6 + [C.c_uint64, C.c_void_p]
        self.lib.sfb200_decompressed_size_batch_device.restype = C.c_int
        rc = self.lib.sfb200_decompressed_size_batch_device(self.h, src.data_ptr(), src_off.data_ptr(),
                                                            src_len.data_ptr(), status.data_ptr(),
                                                            size.data_ptr(), n, stream)
        self._check(rc, "sfb200_decompressed_size_batch_device")

    def checksum_batch_device(self, base, off, length, out, stream=None):
        import torch
        n = off.numel()
        if stream is None:
            stream = torch.cuda.current_stream(base.device).cuda_stream
        rc = self.lib.sfb200_checksum_batch_device(self.h, base.data_ptr(), off.data_ptr(),
                                                   length.data_ptr(), out.data_ptr(), n, stream)
        self._check(rc, "sfb200_checksum_batch_device")

    # -- host buffers (numpy) ---------------------------------------------------------------------
    def decompress_batch_host(self, src: np.ndarray, src_off, src_len, dst: np.ndarray, dst_off,
                              dst_cap):
        n = len(src_off)
        src_off = np.ascontiguousarray(src_off, dtype=np.uint64)
        src_len = np.ascontiguousarray(src_len, dtype=np.uint64)
        dst_off = np.ascontiguousarray(dst_off, dtype=np.uint64)
        dst_cap = np.ascontiguousarray(dst_cap, dtype=np.uint64)
        status = np.zeros(n, np.uint8)
        written = np.zeros(n, np.uint64)
        rc = self.lib.sfb200_decompress_batch_host(
            self.h, _p(src, _u8p), src.size, _p(src_off, _u64p), _p(src_len, _u64p),
            _p(dst, _u8p), dst.size, _p(dst_off, _u64p), _p(dst_cap, _u64p), _p(status, _u8p),
            _p(written, _u64p), n)
        self._check(rc, "sfb200_decompress_batch_host")
        return status, written

    @staticmethod
    def decompress_batch_host_multi(contexts, src: np.ndarray, src_off, src_len, dst: np.ndarray, dst_off, dst_cap):
        """One batch cut across several contexts (one per GPU), each decoding its contiguous shard
        on a host thread of its own (sfb200_decompress_batch_host_multi). -> (status, written)"""
        lib = load_library()
        n = len(src_off)
        src_off = np.ascontiguousarray(src_off, dtype=np.uint64)
        src_len = np.ascontiguousarray(src_len, dtype=np.uint64)
        dst_off = np.ascontiguousarray(dst_off, dtype=np.uint64)
        dst_cap = np.ascontiguousarray(dst_cap, dtype=np.uint64)
        status = np.zeros(n, np.uint8)
        written = np.zeros(n, np.uint64)
        arr = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
        f = lib.sfb200_decompress_batch_host_multi
        f.argtypes = [C.POINTER(C.c_void_p), C.c_int, _u8p, C.c_uint64, _u64p, _u64p, _u8p, C.c_uint64, _u64p,
                      _u64p, _u8p, _u64p, C.c_uint64]
        f.restype = C.c_int
        rc = f(arr, len(contexts), _p(src, _u8p), src.size, _p(src_off, _u64p), _p(src_len, _u64p), _p(dst, _u8p),
               dst.size, _p(dst_off, _u64p), _p(dst_cap, _u64p), _p(status, _u8p), _p(written, _u64p), n)
        if rc != 0:
            msgs = "; ".join((lib.sfb200_last_error(c.h) or b"").decode() for c in contexts)
            raise StarflateError(f"sfb200_decompress_batch_host_multi: {_RC_NAMES.get(rc, rc)} {msgs}")
        return status, written

    def decompress(self, src: bytes, dst_cap: int, fill: int = 0):
        """Single stream (the reference entry point's shape). -> (status, dst bytes, written)"""
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.full(max(dst_cap, 1), fill, dtype=np.uint8)
        st = C.c_uint8(0)
        wr = C.c_uint64(0)
        rc = self.lib.sfb200_decompress(self.h, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap,
                                        C.byref(st), C.byref(wr))
        self._check(rc, "sfb200_decompress")
        return st.value, d[:dst_cap].tobytes(), wr.value

    def compress_batch_device(self, src, src_off, src_len, dst, dst_off, dst_cap, status, written, stream=None):
        """Batched compression to raw DEFLATE (sfb200_compress_batch_device); torch CUDA tensors."""
        import torch
        n = src_off.numel()
        for t in (src_off, src_len, dst_off, dst_cap, written):
            assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous() and t.numel() == n
        assert src.is_cuda and src.dtype == torch.uint8 and dst.is_cuda and dst.dtype == torch.uint8
        assert status.is_cuda and status.dtype == torch.uint8 and status.numel() == n
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        f = self.lib.sfb200_compress_batch_device
        f.argtypes = [C.c_void_p] * 9 + [C.c_uint64, C.c_void_p]
        f.restype = C.c_int
        rc = f(self.h, src.data_ptr(), src_off.data_ptr(), src_len.data_ptr(), dst.data_ptr(), dst_off.data_ptr(),
               dst_cap.data_ptr(), status.data_ptr(), written.data_ptr(), n, stream)
        self._check(rc, "sfb200_compress_batch_device")

    def compress(self, src: bytes, dst_cap: int = -1):
        """One stream in host memory -> (status, raw-DEFLATE bytes)."""
        self.lib.sfb200_compress_bound.argtypes = [C.c_uint64]
        self.lib.sfb200_compress_bound.restype = C.c_uint64
        if dst_cap < 0:
            dst_cap = int(self.lib.sfb200_compress_bound(len(src)))
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.zeros(max(dst_cap, 1), dtype=np.uint8)
        st = C.c_uint8(0)
        wr = C.c_uint64(0)
        f = self.lib.sfb200_compress
        f.argtypes = [C.c_void_p, _u8p, C.c_size_t, _u8p, C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        self._check(f(self.h, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap, C.byref(st), C.byref(wr)), "sfb200_compress")
        return st.value, d[:wr.value].tobytes()

    def compress_container_bound(self, container, n: int) -> int:
        f = self.lib.sfb200_compress_container_bound
        f.argtypes = [C.c_int, C.c_uint64]
        f.restype = C.c_uint64
        return int(f(container, n))

    def compress_bgzf_bound(self, n: int) -> int:
        f = self.lib.sfb200_compress_bgzf_bound
        f.argtypes = [C.c_uint64]
        f.restype = C.c_uint64
        return int(f(n))

    def compress_container_batch_device(self, container, src, src_off, src_len, dst, dst_off, dst_cap, status, written,
                                        stream=None):
        """Batched compression to zlib / gzip (or RAW), checksums of the sources computed on the device
        (sfb200_compress_container_batch_device); torch CUDA tensors."""
        import torch
        n = src_off.numel()
        for t in (src_off, src_len, dst_off, dst_cap, written):
            assert t.is_cuda and t.dtype == torch.int64 and t.is_contiguous() and t.numel() == n
        assert src.is_cuda and src.dtype == torch.uint8 and dst.is_cuda and dst.dtype == torch.uint8
        assert status.is_cuda and status.dtype == torch.uint8 and status.numel() == n
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        f = self.lib.sfb200_compress_container_batch_device
        f.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_uint64, C.c_void_p]
        f.restype = C.c_int
        rc = f(self.h, container, src.data_ptr(), src_off.data_ptr(), src_len.data_ptr(), dst.data_ptr(),
               dst_off.data_ptr(), dst_cap.data_ptr(), status.data_ptr(), written.data_ptr(), n, stream)
        self._check(rc, "sfb200_compress_container_batch_device")

    def compress_container(self, container, src: bytes, dst_cap: int = -1):
        """One stream in host memory -> (status, zlib / gzip / raw-DEFLATE bytes)."""
        if dst_cap < 0:
            dst_cap = self.compress_container_bound(container, len(src))
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.zeros(max(dst_cap, 1), dtype=np.uint8)
        st, wr = C.c_uint8(0), C.c_uint64(0)
        f = self.lib.sfb200_compress_container
        f.argtypes = [C.c_void_p, C.c_int, _u8p, C.c_size_t, _u8p, C.c_size_t, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        self._check(f(self.h, container, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap, C.byref(st), C.byref(wr)),
                    "sfb200_compress_container")
        return st.value, d[:wr.value].tobytes()

    def compress_bgzf(self, src: bytes, dst_cap: int = -1):
        """One buffer in host memory -> (status, BGZF file bytes, members incl. the EOF marker)."""
        if dst_cap < 0:
            dst_cap = self.compress_bgzf_bound(len(src))
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.zeros(max(dst_cap, 1), dtype=np.uint8)
        st, wr, nm = C.c_uint8(0), C.c_uint64(0), C.c_uint64(0)
        f = self.lib.sfb200_compress_bgzf
        f.argtypes = [C.c_void_p, _u8p, C.c_size_t, _u8p, C.c_size_t, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64),
                      C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        rc = f(self.h, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap, C.byref(st), C.byref(wr), C.byref(nm))
        self._check(rc, "sfb200_compress_bgzf")
        return st.value, d[:wr.value].tobytes(), nm.value

    def compress_bgzf_device(self, src, dst, stream=None):
        """A uint8 CUDA tensor as a BGZF file into another (synchronous) -> (status, written, members)."""
        import torch
        assert src.is_cuda and src.dtype == torch.uint8 and src.is_contiguous()
        assert dst.is_cuda and dst.dtype == torch.uint8 and dst.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        st, wr, nm = C.c_uint8(0), C.c_uint64(0), C.c_uint64(0)
        f = self.lib.sfb200_compress_bgzf_device
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p]
        f.restype = C.c_int
        rc = f(self.h, src.data_ptr(), src.numel(), dst.data_ptr(), dst.numel(), C.byref(st), C.byref(wr), C.byref(nm),
               stream)
        self._check(rc, "sfb200_compress_bgzf_device")
        return st.value, wr.value, nm.value

    def compress_parallel_bound(self, container, n: int) -> int:
        f = self.lib.sfb200_compress_parallel_bound
        f.argtypes = [C.c_int, C.c_uint64]
        f.restype = C.c_uint64
        return int(f(container, n))

    def compress_parallel(self, container, src: bytes, dst_cap: int = -1):
        """One buffer in host memory -> (status, ONE raw-DEFLATE / zlib / gzip stream), its pieces
        compressed side by side (sfb200_compress_parallel)."""
        if dst_cap < 0:
            dst_cap = self.compress_parallel_bound(container, len(src))
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.zeros(max(dst_cap, 1), dtype=np.uint8)
        st, wr = C.c_uint8(0), C.c_uint64(0)
        f = self.lib.sfb200_compress_parallel
        f.argtypes = [C.c_void_p, C.c_int, _u8p, C.c_size_t, _u8p, C.c_size_t, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64)]
        f.restype = C.c_int
        self._check(f(self.h, container, _p(s, _u8p), len(src), _p(d, _u8p), dst_cap, C.byref(st), C.byref(wr)),
                    "sfb200_compress_parallel")
        return st.value, d[:wr.value].tobytes()

    def compress_parallel_device(self, container, src, dst, stream=None):
        """A uint8 CUDA tensor as one raw-DEFLATE / zlib / gzip stream into another (synchronous)
        -> (status, written)."""
        import torch
        assert src.is_cuda and src.dtype == torch.uint8 and src.is_contiguous()
        assert dst.is_cuda and dst.dtype == torch.uint8 and dst.is_contiguous()
        if stream is None:
            stream = torch.cuda.current_stream(src.device).cuda_stream
        st, wr = C.c_uint8(0), C.c_uint64(0)
        f = self.lib.sfb200_compress_parallel_device
        f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint8),
                      C.POINTER(C.c_uint64), C.c_void_p]
        f.restype = C.c_int
        rc = f(self.h, container, src.data_ptr(), src.numel(), dst.data_ptr(), dst.numel(), C.byref(st), C.byref(wr),
               stream)
        self._check(rc, "sfb200_compress_parallel_device")
        return st.value, wr.value

    def inflate_stream(self) -> "InflateStream":
        """Chunked input for one stream (sfb200_inflate_stream_*)."""
        return InflateStream(self)

    def staging_bytes(self) -> int:
        """Device memory held for the host-buffer entry points' staging slots."""
        self.lib.sfb200_staging_bytes.argtypes = [C.c_void_p]
        self.lib.sfb200_staging_bytes.restype = C.c_uint64
        return int(self.lib.sfb200_staging_bytes(self.h))

    def last_pass_ms(self):
        """(clear_ms, pass1_ms, pass2_ms) of the most recent device-batch call (CUDA events)."""
        out = (C.c_float * 3)()
        self._check(self.lib.sfb200_last_pass_ms(self.h, out), "sfb200_last_pass_ms")
        return float(out[0]), float(out[1]), float(out[2])

    def launch_info(self) -> dict:
        li = _LaunchInfo()
        self._check(self.lib.sfb200_get_launch_info(self.h, C.byref(li)), "sfb200_get_launch_info")
        return {k: getattr(li, k) for k, _ in _LaunchInfo._fields_}


class InflateStream:
    """One stream fed in pieces (sfb200_inflate_stream_*): block-granular progress, the bit offset of
    the next block header and the last 32 KiB of output are carried on the device."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        lib = ctx.lib
        lib.sfb200_inflate_stream_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        lib.sfb200_inflate_stream_create.restype = C.c_int
        lib.sfb200_inflate_stream_destroy.argtypes = [C.c_void_p]
        lib.sfb200_inflate_stream_destroy.restype = None
        lib.sfb200_inflate_stream_feed.argtypes = [C.c_void_p, _u8p, C.c_size_t, C.c_int, _u8p, C.c_size_t,
                                                   C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_int)]
        lib.sfb200_inflate_stream_feed.restype = C.c_int
        h = C.c_void_p()
        ctx._check(lib.sfb200_inflate_stream_create(ctx.h, C.byref(h)), "sfb200_inflate_stream_create")
        self.h = h

    def feed(self, src: bytes, last: bool, dst_cap: int):
        """-> (status, bytes produced by this call, finished)"""
        s = np.frombuffer(src, dtype=np.uint8) if len(src) else np.zeros(1, np.uint8)
        d = np.zeros(max(dst_cap, 1), dtype=np.uint8)
        wr = C.c_uint64(0)
        st = C.c_uint8(0)
        fin = C.c_int(0)
        rc = self.ctx.lib.sfb200_inflate_stream_feed(self.h, _p(s, _u8p), len(src), int(last), _p(d, _u8p), dst_cap,
                                                     C.byref(wr), C.byref(st), C.byref(fin))
        self.ctx._check(rc, "sfb200_inflate_stream_feed")
        return st.value, d[:wr.value].tobytes(), bool(fin.value)

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.sfb200_inflate_stream_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
