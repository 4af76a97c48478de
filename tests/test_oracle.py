"""CPU: the oracle (oracle/inflate_oracle.c) against the reference's own test vectors, the
SURVEY §8(c) known answers and the committed golden fixtures; against the unmodified reference's
stored answers, and directly against the reference when oracle/_ref was built in this checkout."""
import hashlib
import zlib

import numpy as np
import pytest

from tests import deflate_tools as T
from tests import known_answers as K


@pytest.mark.parametrize("name,hx,cap,status,prefix,cls", K.KNOWN, ids=[k[0] for k in K.KNOWN])
def test_known_answers(oracle, name, hx, cap, status, prefix, cls):
    st, dst, written, ub = oracle.decompress(bytes.fromhex(hx), cap)
    assert st == status
    assert ub == (1 if cls == "U" else 0)
    if prefix is not None:
        assert dst[:written].hex() == prefix
    assert dst[written:] == bytes([0xA5]) * (cap - written)  # untouched beyond the cursor


def test_read_header_vectors(oracle):
    # /root/reference/src/test/decompress_test.cpp:62-89
    for data, bits, has, final, typ, err in K.READ_HEADER:
        out = oracle.read_header(data, bits)
        assert out[0] == has
        if has:
            assert (out[1], out[2], out[4]) == (final, typ, 3)
        else:
            assert out[3] == err and out[4] == 0


def test_copy_from_before(oracle):
    # /root/reference/src/test/decompress_test.cpp:176-181
    buf, idx, dist, n, want = K.COPY_FROM_BEFORE
    assert oracle.copy_from_before(bytearray(buf), idx, dist, n) == want
    # RFC 1951 §3.2.3 example: X,Y + <length 5, distance 2> -> X,Y,X,Y,X
    assert oracle.copy_from_before(bytearray(b"XY\0\0\0\0\0"), 2, 2, 5) == b"XYXYXYX"
    assert oracle.copy_from_before(bytearray(b"Z" + bytes(258)), 1, 1, 258) == b"Z" * 259


def test_bit_order_and_pop16(oracle):
    # huffman/test/bit_span_test.cpp:22-32 (LSB-first) and :159-178 (pop_16 little endian):
    # a stored block whose LEN/NLEN bytes are AA 55 / 55 AA
    w = T.BitWriter()
    payload = bytes(range(256)) * 170 + bytes(range(170))  # 0x55AA = 21930... use exact length
    payload = (payload * 2)[:0x55AA]
    w.stored(True, payload)
    s = w.tobytes()
    assert s[1:5] == bytes([0xAA, 0x55, 0x55, 0xAA])
    st, dst, written, ub = oracle.decompress(s, len(payload))
    assert (st, written, ub) == (0, 0x55AA, 0) and dst == payload


def test_canonical_rfc_examples(oracle):
    # huffman/test/table_from_symbol_bitsize_test.cpp:19-89 = RFC 1951 §3.2.2 examples
    codes, order = oracle.canonical_codes([2, 1, 3, 3])               # A..D
    assert [int(c) for c in codes] == [0b10, 0b0, 0b110, 0b111]
    assert list(order) == [1, 0, 2, 3]
    codes, _ = oracle.canonical_codes([3, 3, 3, 3, 3, 2, 4, 4])        # A..H
    assert [int(c) for c in codes] == [0b010, 0b011, 0b100, 0b101, 0b110, 0b00, 0b1110, 0b1111]


def test_fixed_table_all_288_codes(oracle):
    # huffman/test/table_from_symbol_bitsize_test.cpp:91-149: the RFC §3.2.6 static code
    codes, _ = oracle.canonical_codes(T.FIXED_LIT_LENS)
    for s in range(288):
        if s < 144:
            want = 0b00110000 + s
        elif s < 256:
            want = 0b110010000 + (s - 144)
        elif s < 280:
            want = s - 256
        else:
            want = 0b11000000 + (s - 280)
        assert int(codes[s]) == want, s


def test_decode_one_msb_first_codes(oracle):
    # huffman/test/decode_test.cpp:43-153: table {e:0, i:10, n:110, q:1110, EOT:11110, x:11111}
    lens = [1, 2, 3, 4, 5, 5]  # e i n q EOT x
    w = T.BitWriter()
    for c, n in [(0b110, 3), (0b0, 1), (0b11111, 5), (0b10, 2)]:
        w.code(c, n)
    data = w.tobytes()
    pos, got = 0, []
    for _ in range(4):
        used, sym = oracle.decode_one(lens, data, pos, len(w))
        assert used
        got.append(sym)
        pos += used
    assert got == [2, 0, 5, 1]
    # running out of bits mid-code is "not found", not an error elsewhere
    assert oracle.decode_one(lens, bytes([0b0111]), 0, 3)[0] == 0
    # empty table: every lookup fails (table_find_code_test.cpp:28-92 analogue)
    assert oracle.decode_one([0, 0, 0], bytes([0xFF]), 0, 8)[0] == 0
    # a code longer than anything in the table
    assert oracle.decode_one([1], bytes([0xFF]), 0, 8)[0] == 0


def test_starfleet_roundtrip(oracle, golden):
    # decompress_test.cpp:136-174: first header type, whole-file round trip
    for base, typ in (("starfleet_fixed", 1), ("starfleet_dynamic", 2)):
        comp = golden.bases[base]
        assert oracle.read_header(comp, len(comp) * 8)[2] == typ
        st, dst, written, ub = oracle.decompress(comp, K.STARFLEET_LEN)
        assert (st, written, ub) == (0, K.STARFLEET_LEN, 0)
        assert hashlib.md5(dst).hexdigest() == K.STARFLEET_MD5
        assert zlib.decompress(comp, -15) == dst


def test_golden_families(oracle, golden):
    """Every committed case (strided for the big sweeps to keep the CPU suite short)."""
    total = 0
    for name, fam in golden.families.items():
        stride = 9 if len(fam["params"]) > 3000 else 1
        for i, src, cap in golden.cases(name, stride):
            st, dst, written, ub = oracle.decompress(src, cap)
            want_st, want_wr, want_hash, cls = golden.expected(name, i)
            assert st == want_st and written == want_wr, (name, i)
            assert "%016x" % oracle.fnv1a64(dst) == want_hash, (name, i)
            assert ub == (1 if cls == "U" else 0), (name, i)
            total += 1
    assert total > 15000


def test_against_live_reference(oracle, reference, golden):
    """The oracle against the unmodified reference on the inputs where the reference is defined:
    against the reference's answers stored in tests/golden (status and the fingerprint of the whole
    dst capacity), and byte for byte against the reference itself when oracle/_ref was built."""
    n = 0
    for name in ("known_answers", "cut1_dynamic_4096", "flip_multiblock_12000",
                 "crafted_dynamic_headers", "cap_fixed_4096"):
        for i, src, cap in golden.cases(name, 3):
            want_st, _, want_hash, cls = golden.expected(name, i)
            if cls == "U":
                continue  # the reference may crash or loop on these
            ost, odst, _, _ = oracle.decompress(src, cap)
            assert (ost, "%016x" % oracle.fnv1a64(odst)) == (want_st, want_hash), (name, i)
            if reference is not None:
                st, dst = reference.decompress(src, cap)
                assert (st, dst) == (ost, odst), (name, i)
            n += 1
    assert n > 1000


def test_corpus_units_vs_zlib(oracle):
    for kind, size in [("dynamic", 65536), ("fixed", 4096), ("stored", 4096),
                       ("repetitive", 1 << 20), ("multiblock", 50000), ("dynamic", 1)]:
        plain, comp = T.make_stream(kind, size, 99)
        st, dst, written, ub = oracle.decompress(comp, len(plain) + 7)
        assert (st, written, ub) == (0, len(plain), 0)
        assert dst[:written] == plain == zlib.decompress(comp, -15)


def test_batch_driver_threads(oracle):
    streams, plains = [], []
    for i in range(37):
        p, c = T.make_stream(["dynamic", "fixed", "stored"][i % 3], 300 + 97 * i, i)
        streams.append(c)
        plains.append(p)
    b = T.Batch(streams, [len(p) for p in plains])
    dst = b.new_dst()
    st, wr, ub = oracle.decompress_batch(b.src, b.src_off, b.src_len, dst, b.dst_off, b.dst_cap, 4)
    assert not st.any() and not ub.any()
    for i, p in enumerate(plains):
        assert b.dst_slice(dst, i).tobytes() == p and int(wr[i]) == len(p)
