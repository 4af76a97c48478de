"""Test helpers for zip archives: archives made with Python's zipfile, and the rows zipfile's own
reading gives (the reference the device's listing must match)."""
import io
import struct
import zipfile

import numpy as np


class Unseekable(io.RawIOBase):
    """A write-only file object without tell()/seek(): zipfile then writes data descriptors."""

    def __init__(self):
        self.buf = bytearray()

    def writable(self):
        return True

    def write(self, b):
        self.buf += b
        return len(b)


def make_zip(files, compression=zipfile.ZIP_DEFLATED, level=None, comment=b"", force_zip64=False,
             unseekable=False):
    """files: [(name, bytes)] (or (name, bytes, compress_type)) -> archive bytes"""
    f = Unseekable() if unseekable else io.BytesIO()
    with zipfile.ZipFile(f, "w", compression=compression, compresslevel=level) as z:
        for item in files:
            name, data = item[0], item[1]
            info = zipfile.ZipInfo(name, date_time=(2020, 1, 1, 0, 0, 0))
            info.compress_type = item[2] if len(item) > 2 else compression
            with z.open(info, "w", force_zip64=force_zip64) as w:
                w.write(data)
        z.comment = comment
    return bytes(f.buf) if unseekable else f.getvalue()


def ref_rows(data: bytes):
    """-> [(compress_size, file_size, CRC, compress_type, flag_bits, name bytes, data offset)], the data
    offset computed from zipfile's header_offset and the local header there"""
    out = []
    with zipfile.ZipFile(io.BytesIO(data)) as z:
        for i in z.infolist():
            lh = i.header_offset
            n, m = struct.unpack("<HH", data[lh + 26:lh + 30])
            name = i.orig_filename.encode("utf-8" if i.flag_bits & 0x800 else "cp437")
            out.append((i.compress_size, i.file_size, i.CRC, i.compress_type, i.flag_bits, name, lh + 30 + n + m))
    return out


def rows_as_ref(data: bytes, rows: np.ndarray):
    """The device's rows in ref_rows' shape"""
    out = []
    for r in rows:
        no, nl, do = int(r["name_off"]), int(r["name_len"]), int(r["data_off"])
        name = data[no:no + nl]
        out.append((int(r["comp_size"]), int(r["size"]), int(r["crc32"]), int(r["method"]), int(r["flags"]), name,
                    do))
    return out


def patch(data: bytes, at: int, val: bytes) -> bytes:
    return data[:at] + val + data[at + len(val):]
