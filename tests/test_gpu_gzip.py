"""Single-member gzip decompression on the device (phm_gunzip_index / phm_gunzip_extract, ops.gunzip_cuda) and the gzip road
through read_fasta_arrays_cuda, against Python's zlib / gzip: streams from zlib's compressor at every level, strategy and several
memLevels, at the default chunk size and at 4 KiB chunks (so that back-references cross many chunk starts); hand-built streams that
force the chain to reject a candidate and repair it, and that reach through short pieces into the window; more than 1 GB of FASTA
and a stream whose output passes 4 GiB; corrupt files judged by zlib; and every caller on a gzip copy of the same contigs."""
import gzip
import os
import zlib

import numpy as np
import pytest
import torch

from test_gpu_bgzf import (CL_ORDER, BitWriter, _fasta_text, _same_arrays, complete, dynamic, fixed, stored)  # noqa: F401
from test_gpu_fasta_tiles import TILE, TILE_COUNTS, _file, _tiles, contents  # noqa: F401  (contents is a fixture)

pytestmark = pytest.mark.gpu

STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman_only": zlib.Z_HUFFMAN_ONLY,
              "rle": zlib.Z_RLE, "fixed": zlib.Z_FIXED}
DEFAULT_CHUNK = 128 << 10            # the library's default of option gunzip_chunk_bytes
SMALL_CHUNK = 4096


@pytest.fixture
def chunk_bytes():
    """Sets option gunzip_chunk_bytes for one test and restores the default afterwards."""
    from phamers_b200 import _lib

    def set_(n):
        _lib.set_option("gunzip_chunk_bytes", n)
    yield set_
    _lib.set_option("gunzip_chunk_bytes", DEFAULT_CHUNK)


def gz(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, mem_level=8):
    c = zlib.compressobj(level, zlib.DEFLATED, 31, mem_level, strategy)
    return c.compress(data) + c.flush()


def wrap(deflate, data):
    """A raw DEFLATE stream as a gzip file with the trailer of `data`."""
    return (b"\x1f\x8b\x08\x00\0\0\0\0\0\xff" + deflate + zlib.crc32(data).to_bytes(4, "little")
            + (len(data) & 0xFFFFFFFF).to_bytes(4, "little"))


def _gunzip(raw, stats=None):
    """gzip file bytes -> decompressed bytes through ops.gunzip_cuda (raises _lib.PhamersDataError when declined)."""
    from phamers_b200 import fileIO, ops
    member = fileIO.gzip_member(raw)
    assert member is not None
    d_in = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    return ops.gunzip_cuda(d_in, member, stats=stats).cpu().numpy().tobytes()


def _contents(rng):
    rand = rng.integers(0, 256, size=70000, dtype=np.uint8).tobytes()
    rep = rng.integers(0, 256, size=32768, dtype=np.uint8).tobytes()
    return {"fasta_small": _fasta_text(rng, 20000), "fasta_many_chunks": _fasta_text(rng, 700000), "random": rand,
            "runs": b"A" * 300000 + b"AC" * 20000 + b"G" * 70000, "distance_32768": rep + rep + rep[:9000],
            "empty": b"", "one": b"x", "two": b"\n>"}


@pytest.mark.parametrize("strategy", list(STRATEGIES))
def test_levels_and_contents_equal_gzip(strategy, chunk_bytes):
    """Levels 0-9 at one strategy with memLevels 1-9, on FASTA text (less than one chunk, and many chunks), random bytes, long runs
    (length-258 matches, overlapping distance-1 copies), repeats at distance 32 768 and outputs of 0, 1 and 2 bytes, each at the
    default chunk size and at 4 KiB chunks: the output equals gzip.decompress."""
    rng = np.random.default_rng(41)
    contents_ = _contents(rng)
    for chunk in (DEFAULT_CHUNK, SMALL_CHUNK):
        chunk_bytes(chunk)
        for level in range(10):
            for i, (name, data) in enumerate(contents_.items()):
                raw = gz(data, level, STRATEGIES[strategy], 1 + (level + i) % 9)
                assert _gunzip(raw) == gzip.decompress(raw), (chunk, level, name)


# ---------------------------------------------------------------------------------------------------------------------------
# the chain
# ---------------------------------------------------------------------------------------------------------------------------
A, C, G, T = (ord(c) for c in "ACGT")
LIT = complete([A, C, G, T] + list(range(256, 286)), 286)
DIST = complete(list(range(30)), 30)


def _expand(items, out=None):
    out = bytearray() if out is None else out
    for it in items:
        if isinstance(it, int):
            out.append(it)
        else:
            length, d = it
            for _ in range(length):
                out.append(out[-d])
    return out


def test_planted_header_is_rejected_and_repaired(chunk_bytes):
    """A complete, valid dynamic block planted inside a stored block's payload ahead of a chunk's true block start: the finder takes
    it, the chain rejects it, and the chunk is decoded again from the verified end (a repair round).  The true block after the
    stored one is fixed (never a candidate), so the repaired piece must run to a later candidate."""
    rng = np.random.default_rng(43)
    w = BitWriter()
    dynamic(w, [A, C, (20, 2), G, T, (258, 1)], LIT, DIST, 0)
    w.align()
    planted = w.bytes()
    payload = bytearray(9000)
    payload[5000:5000 + len(planted)] = planted
    items = [int(x) for x in rng.choice([A, C, G, T], size=3000)]
    items2 = [int(x) for x in rng.choice([A, C, G, T], size=6000)] + [(258, 7000), (40, 1)]
    w = BitWriter()
    stored(w, bytes(payload), 0)
    fixed(w, items, 0)
    dynamic(w, items2, LIT, DIST, 0)
    dynamic(w, [T, (100, 1)], LIT, DIST, 1)
    data = bytes(_expand([*payload, *items, *items2, T, (100, 1)]))
    raw = wrap(w.bytes(), data)
    assert gzip.decompress(raw) == data
    chunk_bytes(SMALL_CHUNK)
    stats = {}
    assert _gunzip(raw, stats) == data
    assert stats["rejected_candidates"] >= 1 and stats["repair_rounds"] >= 1, stats


@pytest.mark.parametrize("level,strategy", [(0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED)])
def test_streams_without_dynamic_blocks_decode_serially(level, strategy, chunk_bytes):
    """Level 0 (stored blocks) and Z_FIXED have no dynamic block to find: one piece covers the stream (serial bytes > 0)."""
    rng = np.random.default_rng(47)
    data = _fasta_text(rng, 200000)
    raw = gz(data, level, strategy)
    chunk_bytes(SMALL_CHUNK)
    stats = {}
    assert _gunzip(raw, stats) == data
    assert stats["serial_bytes"] > 0 and stats["chunks"] > 10, stats


def test_ordinary_fasta_has_no_rejections():
    """Level-6 FASTA over many chunks at the default chunk size: every candidate is a true block start."""
    rng = np.random.default_rng(53)
    data = _fasta_text(rng, 6000000)
    raw = gz(data, 6)
    stats = {}
    assert _gunzip(raw, stats) == data
    assert stats["chunks"] >= 8 and stats["rejected_candidates"] == 0 and stats["repair_rounds"] == 0, stats


# ---------------------------------------------------------------------------------------------------------------------------
# window resolution
# ---------------------------------------------------------------------------------------------------------------------------
def test_short_pieces_are_reached_through(chunk_bytes):
    """Pieces of less than 31 000 bytes of output (4 KiB chunks, and memLevel 1 so that zlib closes a block every 128 symbols and
    every chunk holds block starts) in text that copies from 31 000 bytes back: such a copy reaches through the whole piece before
    into the one before that."""
    rng = np.random.default_rng(59)
    base = bytearray(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=400000).tobytes())
    for p in range(31000, len(base) - 200, 997):
        base[p:p + 150] = base[p - 31000:p - 31000 + 150]
    data = bytes(base)
    chunk_bytes(SMALL_CHUNK)
    for level in (1, 6, 9):
        raw = gz(data, level, mem_level=1)
        stats = {}
        assert _gunzip(raw, stats) == data
        assert stats["pieces"] > 20 and 0 < stats["longest_later_piece_bytes"] < 31000, (level, stats)


def test_markers_copied_from_markers(chunk_bytes):
    """A period of 20 000 bytes: a piece after the first copies its first period from the window (markers) and every later period
    from its own first one, so markers are copied from markers; a later piece longer than three periods shows that this happens."""
    rng = np.random.default_rng(61)
    period = rng.choice(np.frombuffer(b"ACGT\n", dtype=np.uint8), size=20000).tobytes()
    data = period * 60 + _fasta_text(rng, 50000) + period * 5
    chunk_bytes(SMALL_CHUNK)
    for level in (1, 9):
        raw = gz(data, level)
        stats = {}
        assert _gunzip(raw, stats) == data
        assert stats["pieces"] >= 2 and stats["longest_later_piece_bytes"] > 3 * len(period), (level, stats)


def test_match_before_the_stream_in_a_later_piece(chunk_bytes, tmp_path):
    """A piece after the first whose second symbol copies from before the stream's start.  Pass A cannot see that (it does not know
    where the piece's output begins), so the index call sizes the stream; the extract call finds it in pass B and must stop there,
    before anything reads the piece's unwritten symbols.  The symbol buffer is first filled with markers by a valid twin of the same
    size (the allocator hands the same block back), so a resolution pass over stale symbols would read before the output."""
    from phamers_b200 import _lib, fileIO
    head = bytes(4500)                                           # zeros: no dynamic block header validates in them

    def stream(items):
        w = BitWriter()
        stored(w, head, 0)
        dynamic(w, items, LIT, DIST, 1)
        return w.bytes()
    twin_items = [A] + [(258, 4000)] * 156
    twin = bytes(_expand(twin_items, bytearray(head)))
    bad_items = [A, (258, 20000)] + [(258, 4000)] * 155
    good_raw = wrap(stream(twin_items), twin)
    bad_raw = wrap(stream(bad_items), twin)                      # the same size as the twin, so ISIZE agrees
    assert gzip.decompress(good_raw) == twin
    with pytest.raises(zlib.error, match="distance too far back"):
        zlib.decompress(bad_raw, 31)
    chunk_bytes(SMALL_CHUNK)
    stats = {}
    assert _gunzip(good_raw, stats) == twin and stats["pieces"] == 2, stats
    with pytest.raises(_lib.PhamersDataError, match="distance before the stream's start"):
        _gunzip(bad_raw)
    assert _gunzip(good_raw) == twin
    path = tmp_path / "far.fasta.gz"
    path.write_bytes(bad_raw)
    with pytest.raises(Exception) as want:
        with gzip.open(str(path), "rb") as fh:
            fh.read()
    with pytest.raises(type(want.value)) as got:
        fileIO.read_fasta_arrays_cuda(str(path))
    assert str(got.value) == str(want.value)


def test_distance_32768_to_the_windows_first_byte(chunk_bytes):
    """A dynamic block that starts a piece with a match at distance 32 768 (its source is the window's first byte), then more
    matches at that distance and an overlapping run."""
    rng = np.random.default_rng(67)
    head = rng.integers(0, 256, size=40000, dtype=np.uint8).tobytes()
    items = [(258, 32768), (3, 32768), A, (100, 32768), C, (258, 1)]
    w = BitWriter()
    stored(w, head, 0)
    dynamic(w, items, LIT, DIST, 1)
    data = bytes(_expand(items, bytearray(head)))
    raw = wrap(w.bytes(), data)
    assert gzip.decompress(raw) == data
    for chunk in (SMALL_CHUNK, 40000 // 8 * 8):
        chunk_bytes(chunk)
        assert _gunzip(raw) == data


# ---------------------------------------------------------------------------------------------------------------------------
# large outputs
# ---------------------------------------------------------------------------------------------------------------------------
def _compress_stream(pieces, level):
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    out, crc, n = [], 0, 0
    for p in pieces:
        out.append(c.compress(p))
        crc = zlib.crc32(p, crc)
        n += len(p)
    out.append(c.flush())
    return b"".join(out), crc, n


def test_one_gigabyte_of_fasta():
    """More than 1 GB of FASTA text (64 distinct 16 MiB pieces in a random order) at level 1: the output equals the text."""
    from phamers_b200 import fileIO, ops
    rng = np.random.default_rng(71)
    pieces = [_fasta_text(rng, 16 << 20) for _ in range(8)]
    order = rng.integers(0, 8, size=64)
    raw, crc, n = _compress_stream((pieces[i] for i in order), 1)
    assert n >= 1 << 30 and fileIO.gzip_member(raw)[2] == crc
    stats = {}
    out = ops.gunzip_cuda(torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda(), fileIO.gzip_member(raw), stats=stats)
    assert out.numel() == n
    want = torch.from_numpy(np.frombuffer(b"".join(pieces), dtype=np.uint8).copy()).cuda().reshape(8, 16 << 20)
    assert torch.equal(out.reshape(64, 16 << 20), want[torch.from_numpy(order).cuda()])


def test_output_past_4_gib_wraps_isize():
    """A run of 4.5 GiB of 'N' between two FASTA lines: ISIZE holds the size mod 2^32, and the output equals the input."""
    from phamers_b200 import fileIO, ops
    run = b"N" * (64 << 20)
    head, tail = b">chrUn long gap\nACGT\n", b"\nTTGA\n"
    raw, crc, n = _compress_stream([head] + [run] * 72 + [tail], 6)
    assert n > 1 << 32 and fileIO.gzip_member(raw)[3] == n % (1 << 32)
    out = ops.gunzip_cuda(torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda(), fileIO.gzip_member(raw))
    assert out.numel() == n
    assert out[:len(head)].cpu().numpy().tobytes() == head and out[n - len(tail):].cpu().numpy().tobytes() == tail
    assert bool((out[len(head):n - len(tail)] == ord("N")).all())


# ---------------------------------------------------------------------------------------------------------------------------
# corruption
# ---------------------------------------------------------------------------------------------------------------------------
def _zlib_gives(raw):
    """What zlib makes of a one-member gzip file: its bytes, or None when it fails, is unfinished or leaves bytes over."""
    d = zlib.decompressobj(31)
    try:
        out = d.decompress(raw)
    except zlib.error:
        return None
    return out if d.eof and not d.unused_data else None


def test_random_bit_flips_agree_with_zlib(chunk_bytes):
    """One random bit flipped after the header of a FASTA file (level 1-9, 4 KiB chunks): the device returns zlib's exact bytes or
    raises PhamersDataError, and it raises exactly when zlib refuses the file."""
    from phamers_b200 import _lib
    rng = np.random.default_rng(73)
    chunk_bytes(SMALL_CHUNK)
    refused = 0
    for trial in range(120):
        data = _fasta_text(rng, int(rng.integers(1000, 120000)))
        raw = bytearray(gz(data, int(rng.integers(1, 10)), list(STRATEGIES.values())[trial % 5]))
        bit = int(rng.integers(10 * 8, len(raw) * 8))
        raw[bit // 8] ^= 1 << (bit % 8)
        raw = bytes(raw)
        want = _zlib_gives(raw)
        try:
            got = _gunzip(raw)
        except _lib.PhamersDataError:
            got = None
        assert got == want, (trial, bit)
        refused += want is None
    assert refused > 60


def _bad_files(data):
    good = gz(data, 6)
    crc = bytearray(good)
    crc[-8] ^= 1
    isize = bytearray(good)
    isize[-1] ^= 0x10
    return {"crc": bytes(crc), "isize": bytes(isize), "truncated": good[:-20], "short_trailer": good[:-3],
            "trailing_byte": good + b"\x07", "zero_padding": good + b"\0" * 16, "second_member": good + gz(data[:5000], 1)}


def test_declined_files_take_the_host_road(tmp_path):
    """A flipped CRC or ISIZE, a truncated file, a trailing byte, zero padding and a second member all decline on the device; through
    read_fasta_arrays_cuda they return or raise what gzip.open(path).read() returns or raises."""
    from phamers_b200 import _lib, fileIO
    rng = np.random.default_rng(79)
    data = _fasta_text(rng, 300000)
    for name, raw in _bad_files(data).items():
        if fileIO.gzip_member(raw) is not None:
            with pytest.raises(_lib.PhamersDataError):
                _gunzip(raw)
        path = tmp_path / (name + ".fasta.gz")
        path.write_bytes(raw)
        try:
            with gzip.open(str(path), "rb") as fh:
                want = fh.read()
        except Exception as exc:                                       # noqa: BLE001  (whatever gzip raises)
            with pytest.raises(type(exc)) as got:
                fileIO.read_fasta_arrays_cuda(str(path))
            assert str(got.value) == str(exc), name
            continue
        plain = tmp_path / (name + ".fasta")
        plain.write_bytes(want)
        _same_arrays(fileIO.read_fasta_arrays_cuda(str(path)), fileIO.read_fasta_arrays_cuda(str(plain)))


# ---------------------------------------------------------------------------------------------------------------------------
# end to end
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def no_host_inflate(monkeypatch):
    """fileIO._open_bytes refuses .gz files: a well-formed gzip file must take the device road."""
    from phamers_b200 import fileIO
    orig = fileIO._open_bytes

    def refuse(path):
        if path.endswith(".gz"):
            raise AssertionError("host inflate of %s" % path)
        return orig(path)
    monkeypatch.setattr(fileIO, "_open_bytes", refuse)


@pytest.mark.parametrize("tiles", TILE_COUNTS)
def test_tile_sweep_files_read_the_same_compressed(contents, tiles, tmp_path, no_host_inflate):  # noqa: F811
    """read_fasta_arrays_cuda on gzip copies of the tokeniser's sweep files gives the ids, sequence bytes and offsets of the plain
    file."""
    from phamers_b200 import fileIO
    t = _tiles(tiles)
    for n in (t * TILE - 9, t * TILE):
        raw = _file(contents, t, n)
        plain, packed = tmp_path / "s.fasta", tmp_path / "s.fasta.gz"
        plain.write_bytes(raw)
        packed.write_bytes(gz(raw, 1))
        _same_arrays(fileIO.read_fasta_arrays_cuda(str(packed)), fileIO.read_fasta_arrays_cuda(str(plain)))


def test_control_bytes_and_empty_files_through_gzip(tmp_path, no_host_inflate):
    """The host tokeniser's fallback (a tab), files without records and an empty member, compressed with gzip, read as plain."""
    from phamers_b200 import fileIO
    for i, raw in enumerate([b">a_ID_1 x\tq\nAC\tGT\n>b\rGG\r", b"", b"no header\n", b">only\n", b">t " + b"w" * 300 + b"\nAC"]):
        plain, packed = tmp_path / ("c%d.fasta" % i), tmp_path / ("c%d.fasta.gz" % i)
        plain.write_bytes(raw)
        packed.write_bytes(gzip.compress(raw))
        _same_arrays(fileIO.read_fasta_arrays_cuda(str(packed)), fileIO.read_fasta_arrays_cuda(str(plain)))


@pytest.fixture(scope="module")
def contig_files(tmp_path_factory):
    from test_gpu_cli import _write_fasta
    d = tmp_path_factory.mktemp("gzip_e2e")
    (d / "plain").mkdir()
    (d / "packed").mkdir()
    _write_fasta(d / "plain" / "x.fasta", np.random.default_rng(31), 150)
    raw = (d / "plain" / "x.fasta").read_bytes()
    (d / "packed" / "x.fasta.gz").write_bytes(gzip.compress(raw))
    return str(d / "plain" / "x.fasta"), str(d / "packed" / "x.fasta.gz")


def test_callers_give_identical_arrays(contig_files, tmp_path, no_host_inflate):
    from phamers_b200 import fileIO, kmer, pipeline
    plain, packed = contig_files
    for k in (4, 5):
        a, b = kmer.count_file(plain, k), kmer.count_file(packed, k)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    for fn in (fileIO.get_fasta_ids, fileIO.get_fasta_lengths):
        a, b = fn(plain), fn(packed)
        for x, y in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
            assert np.array_equal(x, y)
    assert np.array_equal(fileIO.get_fasta_ids(packed), fileIO.read_fasta(plain)[0])
    scorer = pipeline.ContigScorer()
    for a, b in [(scorer.score_fasta(plain, length_requirement=5000), scorer.score_fasta(packed, length_requirement=5000)),
                 (scorer.score_windows_fasta(plain, 5000, 1000), scorer.score_windows_fasta(packed, 5000, 1000))]:
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    ids = fileIO.get_fasta_ids(plain)
    spans = np.array([[0, 1000], [200, 900], [10, 10]], dtype=np.int64)
    names = ids[[0, 5, 9]]
    a = scorer.score_spans_fasta(plain, names, spans, neighbors=True)
    b = scorer.score_spans_fasta(packed, names, spans, neighbors=True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)
    genomes = {}
    for kind, path in (("plain", plain), ("packed", packed)):
        d = tmp_path / kind
        d.mkdir()
        name = "genome_a.fna" + (".gz" if kind == "packed" else "")
        (d / name).write_bytes(open(path, "rb").read())
        genomes[kind] = kmer.count_directory(str(d), 4)
    assert np.array_equal(genomes["plain"][1], genomes["packed"][1])


def test_command_line_writes_the_same_rows(contig_files, tmp_path, no_host_inflate):
    """phamer -fasta x.fasta.gz -window -step -neighbors writes the data rows of the same run on x.fasta, and -spans the same
    span rows."""
    from phamers_b200 import fileIO, phamer
    plain, packed = contig_files
    ids = fileIO.get_fasta_ids(plain)
    bed = tmp_path / "spans.bed"
    bed.write_text("%s\t0\t900\tfirst\n%s\t100\t800\tsecond\n" % (ids[0], ids[3]))
    outs = {}
    for kind, path in (("plain", plain), ("packed", packed)):
        out = tmp_path / kind
        phamer.main(["-fasta", path, "-out", str(out), "-window", "5000", "-step", "1000", "-neighbors", "-l", "3000",
                     "-spans", str(bed)])
        outs[kind] = out
    for name in ("phamer_scores.csv", "phamer_windows.csv", "phamer_regions.csv", "phamer_neighbors.csv", "phamer_spans.csv"):
        rows = [[line for line in open(os.path.join(str(outs[k]), name)) if not line.startswith("#")] for k in ("plain", "packed")]
        assert rows[0] == rows[1] and len(rows[0]) > 0, name
