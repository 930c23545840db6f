"""The host side of gzip ingest, without a device: fileIO.gzip_member against Python's own header parser (every flag, their
combinations, the FNAME / FCOMMENT terminators, FHCRC, the reserved bits, truncated headers, bytes that are not gzip, BGZF), and
the argument errors of phm_gunzip_index / phm_gunzip_extract, which come back before the device is touched."""
import ctypes
import gzip
import io
import itertools
import struct
import zlib

import numpy as np
import pytest

import __graft_entry__ as entry
from phamers_b200 import fileIO
from test_bgzf_cpu import bgzf

FTEXT, FHCRC, FEXTRA, FNAME, FCOMMENT = 1, 2, 4, 8, 16


def _header(flag, extra=b"XY\x02\x00ab", name=b"x.fasta", comment=b"made by hand", hcrc=b"\x12\x34"):
    h = b"\x1f\x8b\x08" + bytes([flag]) + b"\x01\x02\x03\x04\x00\x03"
    if flag & FEXTRA:
        h += struct.pack("<H", len(extra)) + extra
    if flag & FNAME:
        h += name + b"\0"
    if flag & FCOMMENT:
        h += comment + b"\0"
    if flag & FHCRC:
        h += hcrc
    return h


def _member(data, flag=0, **kw):
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    return _header(flag, **kw) + c.compress(data) + c.flush() + struct.pack("<II", zlib.crc32(data), len(data))


def _python_header_end(buf):
    """Where Python's gzip module finds the payload, or None when it rejects the header or runs out of bytes in it."""
    fp = io.BytesIO(buf)
    try:
        if gzip._read_gzip_header(fp) is None:
            return None
    except (gzip.BadGzipFile, EOFError):
        return None
    return fp.tell()


def _agrees(buf):
    end = _python_header_end(buf)
    got = fileIO.gzip_member(buf)
    if end is None or end + 8 > len(buf):
        assert got is None, buf[:40]
        return None
    assert got is not None, buf[:40]
    crc, isize = struct.unpack_from("<II", buf, len(buf) - 8)
    assert got == (end, len(buf) - 8, crc, isize)
    return got


DATA = b">a_ID_1 x\nACGTACGTTT\n>b\nGG\n" * 50


def test_every_flag_and_combination():
    """All 32 combinations of FTEXT, FHCRC, FEXTRA, FNAME, FCOMMENT: the payload starts where Python's parser says, and the
    payload between it and the trailer is the DEFLATE stream of the data."""
    for bits in itertools.product((0, 1), repeat=5):
        flag = sum(b << i for i, b in enumerate(bits))
        raw = _member(DATA, flag)
        got = _agrees(raw)
        assert got is not None
        assert zlib.decompress(raw[got[0]:got[1]], -15) == DATA
        assert got[2] == zlib.crc32(DATA) and got[3] == len(DATA)
        assert gzip.decompress(raw) == DATA


def test_terminators_extra_and_reserved_bits():
    """Empty name and comment, a name holding bytes >= 0x80, an empty extra field, a large one, and the reserved bits 5-7 (Python
    ignores them, and so does gzip_member)."""
    cases = [_member(DATA, FNAME, name=b""), _member(DATA, FCOMMENT, comment=b""), _member(DATA, FNAME | FCOMMENT, name=b"\xe9\xff"),
             _member(DATA, FEXTRA, extra=b""), _member(DATA, FEXTRA, extra=bytes(range(256)) * 40),
             _member(DATA, FHCRC, hcrc=b"\0\0")]
    for reserved in (32, 64, 128, 224):
        cases.append(_member(DATA, FNAME | reserved))
    for raw in cases:
        got = _agrees(raw)
        assert got is not None and zlib.decompress(raw[got[0]:got[1]], -15) == DATA


def test_truncated_headers_and_other_bytes():
    """Every prefix of a header with all fields (Python runs out of bytes; nothing is left for a trailer), a name without its NUL,
    a wrong magic, CM other than 8, plain text, an empty buffer and a header followed by fewer than 8 bytes."""
    full = _member(DATA, FEXTRA | FNAME | FCOMMENT | FHCRC)
    head_end = _python_header_end(full)
    for cut in range(head_end + 8):
        _agrees(full[:cut])
    assert fileIO.gzip_member(full[:head_end + 7]) is None
    assert fileIO.gzip_member(_header(FNAME)[:-1]) is None
    assert fileIO.gzip_member(b"\x1f\x8c" + full[2:]) is None
    assert fileIO.gzip_member(full[:2] + b"\x07" + full[3:]) is None
    assert fileIO.gzip_member(b">a\nACGT\n" * 10) is None
    assert fileIO.gzip_member(b"") is None
    for raw in (b"\x1f\x8c" + full[2:], full[:2] + b"\x07" + full[3:], b">a\nACGT\n" * 10):
        _agrees(raw)


def test_bgzf_and_multi_member_files_still_parse_as_their_first_header():
    """A BGZF file is also a gzip header (FEXTRA); _open_fasta_device asks bgzf_members first, so BGZF keeps its own road.  A file
    of two members gives the first header and the last trailer; the device declines it (the stream ends before the trailer)."""
    raw = bgzf(DATA * 10, block=3000)
    assert fileIO.bgzf_members(raw) is not None
    got = _agrees(raw)
    assert got is not None and got[0] == 18
    two = gzip.compress(DATA) + gzip.compress(DATA[:100])
    got = _agrees(two)
    assert got[1] == len(two) - 8 and got[3] == 100


@pytest.fixture(scope="module")
def lib():
    entry.build()
    from phamers_b200 import _lib
    return _lib.load()


def test_gunzip_argument_errors_without_a_device(lib):
    """Null pointers, negative sizes and workspaces that are too small are reported before any device memory is read (the device
    pointers here are dummies); an empty payload is corrupt data."""
    dummy = ctypes.c_void_p(0x1000)
    info = (ctypes.c_int64 * 7)()
    ws = lib.phm_gunzip_index_workspace_bytes(1 << 20)
    assert ws >= 256 and lib.phm_gunzip_index_workspace_bytes(1 << 22) > ws
    assert lib.phm_gunzip_extract_workspace_bytes(1000) >= 2000
    cases = [
        (lambda: lib.phm_gunzip_index(dummy, -1, 0, info, dummy, ws, None), -1, b"negative size"),
        (lambda: lib.phm_gunzip_index(None, 100, 0, info, dummy, ws, None), -1, b"d_payload is null"),
        (lambda: lib.phm_gunzip_index(dummy, 100, 0, None, dummy, ws, None), -1, b"null pointer"),
        (lambda: lib.phm_gunzip_index(dummy, 100, 0, info, None, ws, None), -1, b"null pointer"),
        (lambda: lib.phm_gunzip_index(dummy, 1 << 20, 0, info, dummy, 255, None), -3, b"workspace too small"),
        (lambda: lib.phm_gunzip_index(dummy, 0, 0, info, dummy, ws, None), -5, b"payload ends before the final block"),
        (lambda: lib.phm_gunzip_extract(dummy, -1, 0, dummy, ws, dummy, 10, dummy, 1 << 20, None), -1, b"negative size"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, dummy, ws, dummy, -1, dummy, 1 << 20, None), -1, b"negative size"),
        (lambda: lib.phm_gunzip_extract(None, 10, 0, dummy, ws, dummy, 10, dummy, 1 << 20, None), -1, b"d_payload is null"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, dummy, ws, None, 10, dummy, 1 << 20, None), -1, b"d_out is null"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, dummy, ws, ctypes.c_void_p(0x1001), 10, dummy, 1 << 20, None), -1,
         b"16-byte aligned"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, None, ws, dummy, 10, dummy, 1 << 20, None), -1, b"null pointer"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, dummy, ws, dummy, 10, None, 1 << 20, None), -1, b"null pointer"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, dummy, 100, dummy, 10, dummy, 1 << 20, None), -1,
         b"index workspace too small"),
        (lambda: lib.phm_gunzip_extract(dummy, 10, 0, dummy, ws, dummy, 1000, dummy, 100, None), -3, b"workspace too small"),
    ]
    for call, rc, message in cases:
        got = call()
        assert got == rc and message in lib.phm_last_error(), (rc, got, message, lib.phm_last_error())
    for bad in (0, 1023, (1 << 30) + 1):
        assert lib.phm_set_option(b"gunzip_chunk_bytes", bad) == -1
    assert lib.phm_set_option(b"gunzip_chunk_bytes", 1 << 20) == 0
    small = lib.phm_gunzip_index_workspace_bytes(1 << 22)
    assert lib.phm_set_option(b"gunzip_chunk_bytes", 4096) == 0
    assert lib.phm_gunzip_index_workspace_bytes(1 << 22) > small            # one row of chunk tables per chunk
    assert lib.phm_set_option(b"gunzip_chunk_bytes", 128 << 10) == 0


def test_host_readers_read_gzip_without_a_device(tmp_path):
    """read_fasta_arrays reads a single-member gzip file as gzip does (the host road the device road must match)."""
    path = tmp_path / "c.fasta.gz"
    path.write_bytes(_member(DATA, FNAME))
    ids, seq, off = fileIO.read_fasta_arrays(str(path))
    want = fileIO.split_fasta_bytes(DATA)
    assert ids == want[0] and np.array_equal(seq, want[1]) and np.array_equal(off, want[2])
