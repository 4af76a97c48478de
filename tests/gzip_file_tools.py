"""Writers of multi-member gzip files for the tests (BGZF, plain members, trap members) and a
reference walk of a file's BGZF members in plain Python."""
from __future__ import annotations

import struct
import zlib

# the 28-byte empty member that ends a BGZF file (SAM/BAM specification §4.1.2)
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
PIECE = 0xff00  # what bgzip puts into one member


def raw_deflate(data: bytes, level: int = 6) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    return c.compress(data) + c.flush()


def stored(data: bytes) -> bytes:
    """One final stored block: the plaintext appears verbatim, 5 bytes behind the block start."""
    assert len(data) <= 0xffff
    return b"\x01" + struct.pack("<HH", len(data), len(data) ^ 0xffff) + data


def bgzf_member(piece: bytes, level: int = 6, before: bytes = b"", after: bytes = b"", payload: bytes | None = None,
                isize: int | None = None, crc: int | None = None) -> bytes:
    """One BGZF member; `before` / `after`: whole extra subfields around 'BC'."""
    comp = raw_deflate(piece, level) if payload is None else payload
    xlen = len(before) + 6 + len(after)
    bsize = 12 + xlen + len(comp) + 8 - 1
    assert bsize <= 0xffff
    extra = before + b"BC" + struct.pack("<HH", 2, bsize) + after
    trailer = struct.pack("<II", zlib.crc32(piece) if crc is None else crc,
                          (len(piece) if isize is None else isize) & 0xffffffff)
    return b"\x1f\x8b\x08\x04" + struct.pack("<I", 0) + b"\x00\xff" + struct.pack("<H", xlen) + extra + comp + trailer


def bgzf(data: bytes, piece: int = PIECE, level: int = 6, eof: bool = True) -> bytes:
    out = [bgzf_member(data[i:i + piece], level) for i in range(0, len(data), piece)]
    return b"".join(out) + (BGZF_EOF if eof else b"")


def fake_header(bsize: int) -> bytes:
    """18 bytes that look like the start of a BGZF member of BSIZE `bsize`."""
    return b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize)


def trap_file(n_real: int = 6, fakes: int = 200, seed: int = 1) -> tuple[bytes, bytes]:
    """BGZF members with, in the middle, a stored-block member whose plaintext is copies of valid-looking
    BGZF headers: most point somewhere inside the trap, one exactly onto the next real member (chains
    merge there), some onto each other.  -> (file, its plaintext)"""
    import random
    rnd = random.Random(seed)
    parts = [bytes(rnd.randrange(256) for _ in range(300 + 50 * k)) * 3 for k in range(n_real)]
    before = b"".join(bgzf_member(p) for p in parts[: n_real // 2])
    plain_len = fakes * 18
    hdr = 12 + 6
    trap_start = len(before)
    trap_len = hdr + 5 + plain_len + 8
    target = trap_start + trap_len  # the next real member
    fk = []
    for i in range(fakes):
        f = trap_start + hdr + 5 + 18 * i  # where this fake header lies in the file
        if i == fakes // 2:
            bs = target - f - 1  # lands exactly on the real member behind the trap
        elif i % 3 == 0:
            bs = 18 * rnd.randrange(2, 8) - 1  # onto a later fake
        else:
            bs = rnd.randrange(26, 2000)
        fk.append(fake_header(bs))
    trap_plain = b"".join(fk)
    trap = bgzf_member(trap_plain, payload=stored(trap_plain))
    assert len(trap) == trap_len
    after = b"".join(bgzf_member(p) for p in parts[n_real // 2:])
    return before + trap + after + BGZF_EOF, b"".join(parts[: n_real // 2]) + trap_plain + b"".join(parts[n_real // 2:])


def ref_candidate(d: bytes, p: int):
    """BSIZE + 1 of the BGZF header at p, or None (the rules of gzip_file.cuh, restated)."""
    if len(d) - p < 12 or d[p:p + 3] != b"\x1f\x8b\x08":
        return None
    flg = d[p + 3]
    if not flg & 4 or flg & 0xe0:
        return None
    xlen = d[p + 10] | d[p + 11] << 8
    e = p + 12 + xlen
    if e > len(d):
        return None
    q = p + 12
    while q + 4 <= e:
        slen = d[q + 2] | d[q + 3] << 8
        if q + 4 + slen > e:
            return None
        if d[q:q + 2] == b"BC" and slen == 2:
            total = (d[q + 4] | d[q + 5] << 8) + 1
            return total if 12 + xlen + 8 <= total <= len(d) - p else None
        q += 4 + slen
    return None


def ref_candidates(d: bytes) -> list[tuple[int, int]]:
    out, p = [], d.find(b"\x1f\x8b")
    while p >= 0:
        t = ref_candidate(d, p)
        if t is not None:
            out.append((p, p + t))
        p = d.find(b"\x1f\x8b", p + 1)
    return out


def ref_chain(d: bytes, start: int, skip: bool = False):
    """-> (members [(pos, len)], head, stop, next) as the device walk defines them."""
    n = len(d)
    head = start
    if skip:
        while head < n and d[head] == 0:
            head += 1
    members, p = [], head
    while p < n:
        t = ref_candidate(d, p)
        if t is None:
            break
        members.append((p, t))
        p += t
    nxt = p
    if members:
        while nxt < n and d[nxt] == 0:
            nxt += 1
    return members, head, p, nxt
