"""The host side of BGZF ingest, without a device: fileIO.bgzf_members on hand-built member chains (which files are BGZF from the
first byte to the last, and the member table they give), and the argument errors of phm_inflate, which come back before the device
is touched."""
import ctypes
import gzip
import struct
import zlib

import numpy as np
import pytest

import __graft_entry__ as entry
from phamers_b200 import fileIO

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_member(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, mem_level=8, before=b"", after=b"", payload=None):
    """One BGZF member holding `data`: raw DEFLATE from zlib.compressobj(level, DEFLATED, -15, mem_level, strategy) (or the given
    payload), a gzip header with FEXTRA whose extra field is `before` + the BC subfield + `after`, and the CRC32 / ISIZE trailer."""
    if payload is None:
        c = zlib.compressobj(level, zlib.DEFLATED, -15, mem_level, strategy)
        payload = c.compress(data) + c.flush()
    extra = before + b"BC" + struct.pack("<HH", 2, 0) + after
    size = 12 + len(extra) + len(payload) + 8
    extra = before + b"BC" + struct.pack("<HH", 2, size - 1) + after
    return (b"\x1f\x8b\x08\x04" + b"\0\0\0\0" + b"\0\xff" + struct.pack("<H", len(extra)) + extra + payload
            + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data) & 0xFFFFFFFF))


def bgzf(data, block=65280, eof=True, **kw):
    """`data` as a BGZF file: members of `block` input bytes (bgzip's 65 280), then the EOF block."""
    chunks = [data[i:i + block] for i in range(0, len(data), block)]
    return b"".join(bgzf_member(c, **kw) for c in chunks) + (EOF_BLOCK if eof else b"")


def test_eof_block_is_an_empty_member():
    assert gzip.decompress(EOF_BLOCK) == b""
    table = fileIO.bgzf_members(EOF_BLOCK)
    assert table.shape == (1,) and table["in_offset"][0] == 18 and table["in_bytes"][0] == 2
    assert table["isize"][0] == 0 and table["crc32"][0] == 0 and table["out_offset"][0] == 0


def test_member_table_of_a_chain():
    """Extra subfields before and after BC, an empty member, members of 0, 1 and 65 536 output bytes, and a member of exactly
    65 536 bytes (stored random bytes, BSIZE = 65 535): offsets, sizes, CRC32 and ISIZE of every member, and gzip reads the same
    file."""
    rng = np.random.default_rng(3)
    big = rng.integers(0, 256, size=65500, dtype=np.uint8).tobytes()
    parts = [(b"ACGT" * 100, {}), (b"", {}), (b"x", {"before": b"XY\x03\x00abc"}),
             (b"\n>h\nAC", {"after": b"ZZ\x00\x00"}), (b"G" * 65536, {"before": b"ab\x01\x00q", "after": b"cd\x02\x00rs"}),
             (big, {"level": 0}), (b"", {})]
    members = [bgzf_member(d, **kw) for d, kw in parts]
    raw = b"".join(members) + EOF_BLOCK
    assert gzip.decompress(raw) == b"".join(d for d, _ in parts)
    table = fileIO.bgzf_members(raw)
    assert table is not None and table.dtype == fileIO.BGZF_MEMBER and table.shape == (len(parts) + 1,)
    start, out = 0, 0
    for i, (data, _) in enumerate(parts + [(b"", {})]):
        m = members[i] if i < len(members) else EOF_BLOCK
        xlen = struct.unpack_from("<H", m, 10)[0]
        assert table["in_offset"][i] == start + 12 + xlen
        assert table["in_bytes"][i] == len(m) - 12 - xlen - 8
        assert zlib.decompress(raw[table["in_offset"][i]:table["in_offset"][i] + table["in_bytes"][i]], -15) == data
        assert table["out_offset"][i] == out and table["isize"][i] == len(data)
        assert table["crc32"][i] == zlib.crc32(data)
        start += len(m)
        out += len(data)
    assert len(members[5]) == 65536 and table["in_bytes"][5] == 65510


def test_not_bgzf():
    """Single-member gzip, multi-member gzip without BC, trailing bytes, a truncated last member, a BSIZE past the end, a BC of
    the wrong SLEN, extra subfields that overrun XLEN, FNAME set, and an ISIZE above 64 KiB all give None."""
    data = b">a\nACGT\n" * 1000
    good = bgzf(data, block=3000)
    assert fileIO.bgzf_members(good) is not None
    assert fileIO.bgzf_members(gzip.compress(data)) is None
    assert fileIO.bgzf_members(gzip.compress(data[:500]) + gzip.compress(data[500:])) is None
    assert fileIO.bgzf_members(good + b"\0") is None
    assert fileIO.bgzf_members(good + EOF_BLOCK[:20]) is None
    assert fileIO.bgzf_members(good[:-1]) is None
    assert fileIO.bgzf_members(b"") is None
    one = bytearray(bgzf_member(data[:100]))
    bsize = struct.unpack_from("<H", one, 16)[0]
    struct.pack_into("<H", one, 16, bsize + 10)                 # BSIZE points past the end
    assert fileIO.bgzf_members(bytes(one)) is None
    wrong = bytearray(bgzf_member(data[:100]))
    wrong[14] = 4                                               # SLEN 4
    assert fileIO.bgzf_members(bytes(wrong)) is None
    over = bgzf_member(data[:100], before=b"XY\x09\x00abc")     # a subfield longer than the extra field
    assert fileIO.bgzf_members(over) is None
    named = bytearray(bgzf_member(data[:100]))
    named[3] |= 8                                               # FNAME
    assert fileIO.bgzf_members(bytes(named)) is None
    big = bytearray(bgzf_member(data[:100]))
    struct.pack_into("<I", big, len(big) - 4, 65537)
    assert fileIO.bgzf_members(bytes(big)) is None


def test_read_fasta_arrays_on_host_reads_bgzf(tmp_path):
    """The host readers (read_fasta_arrays, read_fasta) read a BGZF file as gzip does."""
    data = b">a_ID_1 x\nACGT\nAC\n>b_ID_2\nGGTT\n" * 5000
    path = tmp_path / "c.fasta.gz"
    path.write_bytes(bgzf(data, block=65280))
    ids, seq, off = fileIO.read_fasta_arrays(str(path))
    want = fileIO.split_fasta_bytes(data)
    assert ids == want[0] and np.array_equal(seq, want[1]) and np.array_equal(off, want[2])


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib.load()


def _table(rows):
    t = np.zeros(len(rows), dtype=fileIO.BGZF_MEMBER)
    for i, (in_off, in_bytes, out_off, isize) in enumerate(rows):
        t[i]["in_offset"], t[i]["in_bytes"], t[i]["out_offset"], t[i]["isize"] = in_off, in_bytes, out_off, isize
    return t


def test_inflate_argument_errors_without_a_device(lib):
    """Null pointers, payloads or outputs outside the buffers, overlapping or descending outputs and sizes beyond the BGZF limit
    are PHM_E_ARG, reported before any device memory is read (the device pointers here are dummies)."""
    assert lib.phm_inflate_workspace_bytes(0) == 256
    assert lib.phm_inflate_workspace_bytes(1000) == (1000 * 32 + 255) // 256 * 256 + 256
    assert fileIO.BGZF_MEMBER.itemsize == 32
    dummy = ctypes.c_void_p(0x1000)
    ws = lib.phm_inflate_workspace_bytes(4)

    def call(table, in_bytes=1000, out_bytes=1000, d_in=dummy, d_out=dummy, status=dummy, work=dummy):
        t = np.ascontiguousarray(table)
        return lib.phm_inflate(d_in, in_bytes, t.ctypes.data_as(ctypes.c_void_p) if len(t) else None, len(t), d_out, out_bytes,
                               status, work, ws, None)

    ok = [(0, 10, 0, 100), (10, 20, 100, 200)]
    cases = [
        (dict(table=_table(ok), d_in=None), "d_in is null"),
        (dict(table=_table(ok), d_out=None), "d_out is null"),
        (dict(table=_table(ok), status=None), "null pointer"),
        (dict(table=_table(ok), work=None), "null pointer"),
        (dict(table=_table([(995, 10, 0, 100)])), "outside the 1000 input bytes"),
        (dict(table=_table([(-1, 10, 0, 100)])), "outside the 1000 input bytes"),
        (dict(table=_table([(0, 10, 950, 100)])), "outside the 1000 output bytes"),
        (dict(table=_table([(0, 10, 0, 100), (10, 20, 99, 200)])), "overlaps"),
        (dict(table=_table([(0, 10, 500, 100), (10, 20, 0, 200)])), "overlaps"),
        (dict(table=_table([(0, 65537, 0, 100)]), in_bytes=70000), "beyond the BGZF limit"),
        (dict(table=_table([(0, 10, 0, 65537)]), out_bytes=70000), "beyond the BGZF limit"),
    ]
    for kw, message in cases:
        rc = call(**kw)
        assert rc == -1 and message.encode() in lib.phm_last_error(), (kw, lib.phm_last_error())
    assert lib.phm_inflate(dummy, 10, None, 0, dummy, 10, None, None, 0, None) == 0        # nothing to decode
    rc = lib.phm_inflate(dummy, 1000, np.ascontiguousarray(_table(ok)).ctypes.data_as(ctypes.c_void_p), 2, dummy, 1000, dummy,
                         dummy, 10, None)
    assert rc == -3 and b"workspace too small" in lib.phm_last_error()
