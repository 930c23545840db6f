"""BGZF decompression on the device (phm_inflate, ops.inflate_cuda) and the compressed-FASTA road through read_fasta_arrays_cuda,
against Python's zlib / gzip: members made by zlib at every level and strategy, hand-built DEFLATE streams for the RFC 1951 cases
zlib's compressor never emits, a file of about 1 GB, corrupt members (one per status, and random bit flips judged by zlib), and
every caller of read_fasta_arrays_cuda on a BGZF file against the same file uncompressed."""
import gzip
import os
import zlib

import numpy as np
import pytest
import torch

from test_bgzf_cpu import EOF_BLOCK, bgzf, bgzf_member
from test_gpu_fasta_tiles import TILE, TILE_COUNTS, _file, _tiles, contents  # noqa: F401  (contents is a fixture)

pytestmark = pytest.mark.gpu

STRATEGIES = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman_only": zlib.Z_HUFFMAN_ONLY,
              "rle": zlib.Z_RLE, "fixed": zlib.Z_FIXED}
OK, BTYPE, STORED_LEN, BAD_CODE, DISTANCE, OVERFLOW, TRUNCATED, TRAILING, ISIZE, CRC = range(10)


def _inflate(raw, expect_ok=True):
    """raw BGZF bytes -> (decompressed bytes or None, status int32[members]) through ops.inflate_cuda."""
    from phamers_b200 import _lib, fileIO, ops
    table = fileIO.bgzf_members(raw)
    assert table is not None
    d_in = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    status = torch.full((table.shape[0],), -1, dtype=torch.int32, device="cuda")
    try:
        out = ops.inflate_cuda(d_in, table, status=status)
    except _lib.PhamersDataError:
        assert not expect_ok
        return None, status.cpu().numpy()
    assert expect_ok
    return out.cpu().numpy().tobytes(), status.cpu().numpy()


def _fasta_text(rng, n):
    body = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n)
    body[::61] = ord("\n")
    body[::977] = ord(">")
    return body.tobytes()


# ---------------------------------------------------------------------------------------------------------------------------
# zlib's compressor: every level and strategy
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("strategy", list(STRATEGIES))
def test_levels_and_contents_equal_gzip(strategy):
    """Levels 0-9 at one strategy, on FASTA text, random bytes (stored blocks), long runs (distance-1 overlapping copies and
    length-258 matches), repeats at distance 32 768 and outputs of 0, 1, 2 and 65 536 bytes (65 280 at level 0): the output equals
    gzip.decompress of the file, every member's status is 0."""
    rng = np.random.default_rng(11)
    rand = rng.integers(0, 256, size=56000, dtype=np.uint8).tobytes()           # random bytes grow by up to 4 % at a small memLevel
    rep = rng.integers(0, 256, size=32768, dtype=np.uint8).tobytes()
    contents_ = [_fasta_text(rng, 65280), rand, b"A" * 65536, b"AC" * 20000 + b"G" * 25000, rep + rep[:24000], b"", b"x", b"\n>",
                 _fasta_text(rng, 65536)]
    members = []
    for level in range(10):
        for i, data in enumerate(contents_):
            data = data if level else data[:65280]         # stored blocks: 65 536 bytes do not fit in one member
            members.append(bgzf_member(data, level=level, strategy=STRATEGIES[strategy], mem_level=1 + (level + i) % 9))
    raw = b"".join(members) + EOF_BLOCK
    out, status = _inflate(raw)
    assert np.all(status == OK)
    assert out == gzip.decompress(raw)


# ---------------------------------------------------------------------------------------------------------------------------
# hand-built DEFLATE streams
# ---------------------------------------------------------------------------------------------------------------------------
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
             8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [i // 2 for i in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8


class BitWriter(object):
    def __init__(self):
        self.value, self.n = 0, 0

    def put(self, v, bits):                   # a field, least significant bit first
        self.value |= v << self.n
        self.n += bits

    def code(self, c, length):                # a Huffman code, most significant bit first
        self.put(int(format(c, "0%db" % length)[::-1], 2), length)

    def align(self):
        self.n = (self.n + 7) // 8 * 8

    def bytes(self):
        return self.value.to_bytes((self.n + 7) // 8, "little")


def canonical(lengths):
    count = np.bincount([x for x in lengths if x], minlength=16)
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1 if b > 1 else 0
        nxt[b] = code
    out = {}
    for s, x in enumerate(lengths):
        if x:
            out[s] = (nxt[x], x)
            nxt[x] += 1
    return out


def complete(symbols, n):
    """Code lengths over n symbols giving `symbols` (sorted) a complete code: 2^k symbols of length k, or a mix of k and k + 1."""
    lengths = [0] * n
    m = len(symbols)
    k = max(1, int(np.floor(np.log2(m))))
    n_long = 2 * (m - 2 ** k) if m > 2 ** k else 0
    for i, s in enumerate(symbols):
        lengths[s] = k + 1 if i >= m - n_long else k
    return lengths


def emit(w, items, lit, dist):
    """items: ints (literals) and (length, distance) pairs, then end of block."""
    for it in items:
        if isinstance(it, int):
            w.code(*lit[it])
            continue
        length, d = it
        i = 28 if length == 258 else max(j for j in range(28) if LEN_BASE[j] <= length)
        w.code(*lit[257 + i])
        w.put(length - LEN_BASE[i], LEN_EXTRA[i])
        j = max(j for j in range(30) if DIST_BASE[j] <= d)
        w.code(*dist[j])
        w.put(d - DIST_BASE[j], DIST_EXTRA[j])
    w.code(*lit[256])


def stored(w, data, final):
    w.put(final, 1)
    w.put(0, 2)
    w.align()
    w.put(len(data), 16)
    w.put(len(data) ^ 0xFFFF, 16)
    for b in data:
        w.put(b, 8)


def fixed(w, items, final):
    w.put(final, 1)
    w.put(1, 2)
    emit(w, items, canonical(FIXED_LIT), canonical([5] * 32))


def rle(lengths):
    out, i = [], 0
    while i < len(lengths):
        x, run = lengths[i], 1
        while i + run < len(lengths) and lengths[i + run] == x:
            run += 1
        if x == 0 and run >= 3:
            r = min(run, 138)
            out.append((18, r - 11, 7) if r >= 11 else (17, r - 3, 3))
        elif x != 0 and i > 0 and lengths[i - 1] == x and run >= 3:
            r = min(run, 6)
            out.append((16, r - 3, 2))
        else:
            r = 1
            out.append((x, 0, 0))
        i += r
    return out


def dynamic(w, items, lit_lengths, dist_lengths, final):
    seq = rle(list(lit_lengths) + list(dist_lengths))
    used = sorted({s for s, _, _ in seq} | ({0, 1} if len({s for s, _, _ in seq}) < 2 else set()))
    cl_lengths = complete(used, 19)
    hclen = max(4, max(i + 1 for i, s in enumerate(CL_ORDER) if cl_lengths[s]))
    w.put(final, 1)
    w.put(2, 2)
    w.put(len(lit_lengths) - 257, 5)
    w.put(len(dist_lengths) - 1, 5)
    w.put(hclen - 4, 4)
    for s in CL_ORDER[:hclen]:
        w.put(cl_lengths[s], 3)
    cl = canonical(cl_lengths)
    for s, extra, bits in seq:
        w.code(*cl[s])
        w.put(extra, bits)
    emit(w, items, canonical(lit_lengths), canonical(dist_lengths))
    return seq


def _expand(items):
    out = bytearray()
    for it in items:
        if isinstance(it, int):
            out.append(it)
        else:
            length, d = it
            for _ in range(length):
                out.append(out[-d])
    return bytes(out)


def hand_built_streams():
    """(name, raw DEFLATE, output) of the RFC 1951 cases zlib's compressor does not emit on its own."""
    rng = np.random.default_rng(5)
    A, C, G, T = (ord(c) for c in "ACGT")
    cases = []
    # mixed block types in one member, a stored block with LEN 0, matches reaching back into earlier blocks
    w = BitWriter()
    head = list(rng.integers(0, 256, size=700, dtype=np.uint8).tolist())
    items, dyn_items = [A, C, G, T, (10, 4), (258, 1), G], [C, G, (3, 1), (20, 731), T]
    stored(w, bytes(head), 0)
    fixed(w, items, 0)
    stored(w, b"", 0)
    lit = complete([A, C, G, T] + list(range(256, 272)), 286)
    dynamic(w, dyn_items, lit, complete(list(range(30)), 30), 0)
    fixed(w, [A, (258, 50)], 1)
    cases.append(("mixed_blocks", w.bytes(), _expand(head + items + dyn_items + [A, (258, 50)])))
    # a single distance code (one code of one bit), then a literals-only dynamic block (no distance code at all)
    w = BitWriter()
    dynamic(w, [A, (258, 1), C, (3, 1)], complete([A, C, G, T, 256, 257, 285], 286), [1], 0)
    dynamic(w, [G, T, A, C, C], complete([A, C, G, T, 256], 257), [0], 1)
    cases.append(("single_and_no_distance_code", w.bytes(), _expand([A, (258, 1), C, (3, 1), G, T, A, C, C])))
    # repeat code 16 carrying a length from the lit/len lengths into the distance lengths, then 18 carrying zeros across
    w = BitWriter()
    lit = [0] * 286
    for s in (A, C, G, T):
        lit[s] = 3
    for s in [256, 257] + list(range(280, 286)):
        lit[s] = 4
    first = [A] * 3 + [(3, 1), (258, 3), (131, 200), (227, 9)] + [(258, 1)] * 3 + [C, G]
    seq = dynamic(w, first, lit, [4] * 16 + [0] * 14, 0)
    assert (4, 0, 0) in seq and sum(3 + e for s, e, _ in seq if s == 16) >= 21      # the run of 4s spans both lists
    second = [A, (4, 1100), (3, 1025), T]
    seq = dynamic(w, second, complete([A, C, G, T, 256, 257, 258], 286), [0] * 20 + [1, 1] + [0] * 8, 1)
    assert any(s == 18 and 11 + e == 47 for s, e, _ in seq)                          # lit 259..285 and distances 0..19
    cases.append(("repeats_cross_into_distances", w.bytes(), _expand(first + second)))
    # matches at distance exactly 32 768
    w = BitWriter()
    head = list(rng.integers(0, 256, size=32768, dtype=np.uint8).tolist())
    matches = [(258, 32768), (3, 32768), (258, 1), (4, 32768)]
    stored(w, bytes(head), 0)
    fixed(w, matches, 1)
    cases.append(("distance_32768", w.bytes(), _expand(head + matches)))
    return cases


def test_hand_built_streams():
    cases = hand_built_streams()
    members = []
    for name, payload, out in cases:
        assert zlib.decompress(payload, -15) == out, name                  # the oracle accepts the stream as built
        members.append(bgzf_member(out, payload=payload))
    raw = b"".join(members)
    got, status = _inflate(raw)
    assert np.all(status == OK) and got == b"".join(out for _, _, out in cases)


# ---------------------------------------------------------------------------------------------------------------------------
# a file of about 1 GB
# ---------------------------------------------------------------------------------------------------------------------------
def test_one_gigabyte_of_members():
    """16 384 members of 65 280 bytes (1.07 GB of output; 64 distinct members in a random order): equal to the host bytes, every
    CRC32 checked on the device."""
    from phamers_b200 import fileIO, ops
    rng = np.random.default_rng(17)
    chunks = [_fasta_text(rng, 65280) for _ in range(64)]
    payloads = [bgzf_member(c, level=1 + i % 9) for i, c in enumerate(chunks)]
    order = rng.integers(0, 64, size=16384)
    raw = b"".join(payloads[i] for i in order)
    table = fileIO.bgzf_members(raw)
    assert table.shape == (16384,)
    status = torch.full((16384,), -1, dtype=torch.int32, device="cuda")
    out = ops.inflate_cuda(torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda(), table, status=status)
    assert out.numel() == 16384 * 65280 and bool((status == 0).all())
    want = torch.from_numpy(np.frombuffer(b"".join(chunks), dtype=np.uint8).copy()).cuda().reshape(64, 65280)
    assert torch.equal(out.reshape(16384, 65280), want[torch.from_numpy(order).cuda()])


# ---------------------------------------------------------------------------------------------------------------------------
# corrupt members
# ---------------------------------------------------------------------------------------------------------------------------
def _zlib_accepts(payload, data_crc, isize):
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(payload)
    except zlib.error:
        return False, None
    return d.eof and not d.unused_data and len(out) == isize and zlib.crc32(out) == data_crc, out


def test_corrupt_members_report_their_status():
    """One member per status among good members: each is reported against the right member, the error names the lowest one, and
    every other member's output is what gzip gives."""
    rng = np.random.default_rng(23)
    data = _fasta_text(rng, 5000)
    deflated = zlib.compressobj(6, zlib.DEFLATED, -15)
    deflated = deflated.compress(data) + deflated.flush()
    w = BitWriter(); w.put(7, 3)                                                       # BFINAL = 1, BTYPE = 11
    btype = w.bytes()
    w = BitWriter(); w.put(1, 3); w.align(); w.put(5, 16); w.put(0, 16)                # NLEN is not ~LEN
    stored_len = w.bytes() + b"ACGTA"
    w = BitWriter(); w.put(1, 1); w.put(2, 2); w.put(0, 10); w.put(15, 4)              # 19 code-length codes of one bit
    for _ in range(19):
        w.put(1, 3)
    oversubscribed = w.bytes() + b"\0" * 8
    w = BitWriter(); fixed(w, [(3, 1)], 1)                                             # a match before the first byte
    too_far = w.bytes()
    w = BitWriter(); w.put(1, 3); w.align(); w.put(100, 16); w.put(100 ^ 0xFFFF, 16)   # stored block of 100 with 50 present
    truncated = w.bytes() + data[:50]
    bad = {
        BTYPE: bgzf_member(b"ACGT", payload=btype),
        STORED_LEN: bgzf_member(b"ACGTA", payload=stored_len),
        BAD_CODE: bgzf_member(b"", payload=oversubscribed),
        DISTANCE: bgzf_member(b"AAA", payload=too_far),
        OVERFLOW: bgzf_member(data[:-1], payload=deflated),
        TRUNCATED: bgzf_member(data[:100], payload=truncated),
        TRAILING: bgzf_member(data, payload=deflated + b"\0"),
        ISIZE: bgzf_member(data + b"A", payload=deflated),
        CRC: bgzf_member(data[:-1] + b"C", payload=deflated),
    }
    good = [bgzf_member(_fasta_text(rng, 3000 + 100 * i)) for i in range(len(bad) + 1)]
    members, expect = [good[0]], [OK]
    for i, (code, m) in enumerate(sorted(bad.items(), reverse=True)):
        members += [m, good[i + 1]]
        expect += [code, OK]
    raw = b"".join(members)
    from phamers_b200 import _lib, fileIO, ops
    table = fileIO.bgzf_members(raw)
    for m, i in zip(members, range(len(members))):
        payload = raw[table["in_offset"][i]:table["in_offset"][i] + table["in_bytes"][i]]
        assert _zlib_accepts(payload, int(table["crc32"][i]), int(table["isize"][i]))[0] == (expect[i] == OK)
    status = torch.full((len(members),), -1, dtype=torch.int32, device="cuda")
    with pytest.raises(_lib.PhamersDataError, match="member 1: CRC32 mismatch"):
        ops.inflate_cuda(torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda(), table, status=status)
    assert status.cpu().tolist() == expect
    _check_good_outputs(raw, table, status.cpu().numpy())


def _check_good_outputs(raw, table, status):
    """Members with status 0 hold gzip's bytes: inflate again into a buffer of known content and compare member by member."""
    from phamers_b200 import _lib, ops
    d_in = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    try:
        out = ops.inflate_cuda(d_in, table).cpu().numpy()
    except _lib.PhamersDataError:
        out = None
    if out is None:                   # the output tensor of a failed call is not returned: decode the good members on their own
        good = table[status == 0].copy()
        good["out_offset"] = np.concatenate(([0], np.cumsum(good["isize"][:-1].astype(np.int64))))
        out = ops.inflate_cuda(d_in, good).cpu().numpy()
        table = good
    for m in table:
        payload = raw[m["in_offset"]:m["in_offset"] + m["in_bytes"]]
        got = out[m["out_offset"]:m["out_offset"] + m["isize"]].tobytes()
        assert got == zlib.decompress(payload, -15)


def test_random_bit_flips_agree_with_zlib():
    """One random bit flipped in the payload of every other member of 400: a member decodes (status 0) exactly when zlib decodes
    it to ISIZE bytes with the trailer's CRC32 and nothing left over, and every such member's output is zlib's."""
    from phamers_b200 import fileIO
    rng = np.random.default_rng(29)
    members = []
    for i in range(400):
        data = _fasta_text(rng, int(rng.integers(1, 6000))) if i % 3 else rng.integers(0, 256, size=900, dtype=np.uint8).tobytes()
        m = bytearray(bgzf_member(data, level=int(rng.integers(0, 10)), strategy=list(STRATEGIES.values())[i % 5]))
        if i % 2:
            bit = int(rng.integers(18 * 8, (len(m) - 8) * 8))
            m[bit // 8] ^= 1 << (bit % 8)
        members.append(bytes(m))
    raw = b"".join(members)
    table = fileIO.bgzf_members(raw)
    _, status = _inflate(raw, expect_ok=False)
    accepted = []
    for i in range(len(members)):
        payload = raw[table["in_offset"][i]:table["in_offset"][i] + table["in_bytes"][i]]
        accepted.append(_zlib_accepts(payload, int(table["crc32"][i]), int(table["isize"][i]))[0])
    assert np.array_equal(status == OK, np.array(accepted)), np.flatnonzero((status == OK) != np.array(accepted))
    assert np.all(status[0::2] == OK) and np.count_nonzero(status[1::2]) > 150
    _check_good_outputs(raw, table, status)


# ---------------------------------------------------------------------------------------------------------------------------
# end to end
# ---------------------------------------------------------------------------------------------------------------------------
def _same_arrays(a, b):
    ids_a, seq_a, off_a = a
    ids_b, seq_b, off_b = b
    off_a, off_b = off_a.cpu().numpy(), off_b.cpu().numpy()
    assert ids_a == ids_b and np.array_equal(off_a, off_b)
    assert torch.equal(seq_a[:int(off_a[-1])], seq_b[:int(off_b[-1])])


@pytest.mark.parametrize("tiles", TILE_COUNTS)
def test_tile_sweep_files_read_the_same_compressed(contents, tiles, tmp_path):  # noqa: F811
    """read_fasta_arrays_cuda on BGZF copies of the tokeniser's sweep files (ending mid-chunk and on a tile; the large ones hold a
    40 KB title) gives the ids, sequence bytes and offsets of the plain file."""
    from phamers_b200 import fileIO
    t = _tiles(tiles)
    for n in (t * TILE - 9, t * TILE):
        raw = _file(contents, t, n)
        plain, packed = tmp_path / "s.fasta", tmp_path / "s.fasta.gz"
        plain.write_bytes(raw)
        packed.write_bytes(bgzf(raw, level=1))
        _same_arrays(fileIO.read_fasta_arrays_cuda(str(packed)), fileIO.read_fasta_arrays_cuda(str(plain)))


def test_control_bytes_and_empty_files_through_bgzf(tmp_path):
    """The host tokeniser's fallback (a tab in the file) and files without records, compressed as BGZF, read as uncompressed."""
    from phamers_b200 import fileIO
    for i, raw in enumerate([b">a_ID_1 x\tq\nAC\tGT\n>b\rGG\r", b"", b"no header\n", b">only\n", b">t " + b"w" * 300 + b"\nAC"]):
        plain, packed = tmp_path / ("c%d.fasta" % i), tmp_path / ("c%d.fasta.gz" % i)
        plain.write_bytes(raw)
        packed.write_bytes(bgzf(raw))
        _same_arrays(fileIO.read_fasta_arrays_cuda(str(packed)), fileIO.read_fasta_arrays_cuda(str(plain)))


@pytest.fixture(scope="module")
def contig_files(tmp_path_factory):
    from test_gpu_cli import _write_fasta
    d = tmp_path_factory.mktemp("bgzf_e2e")
    (d / "plain").mkdir()
    (d / "packed").mkdir()
    _write_fasta(d / "plain" / "x.fasta", np.random.default_rng(31), 150)
    raw = (d / "plain" / "x.fasta").read_bytes()
    (d / "packed" / "x.fasta.gz").write_bytes(bgzf(raw))
    return str(d / "plain" / "x.fasta"), str(d / "packed" / "x.fasta.gz")


def test_callers_give_identical_arrays(contig_files, tmp_path):
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


def test_command_line_writes_the_same_rows(contig_files, tmp_path):
    """phamer -fasta x.fasta.gz -window -step -neighbors writes the data rows of the same run on x.fasta (headers embed the path)."""
    from phamers_b200 import phamer
    plain, packed = contig_files
    outs = {}
    for kind, path in (("plain", plain), ("packed", packed)):
        out = tmp_path / kind
        phamer.main(["-fasta", path, "-out", str(out), "-window", "5000", "-step", "1000", "-neighbors", "-l", "3000"])
        outs[kind] = out
    for name in ("phamer_scores.csv", "phamer_windows.csv", "phamer_regions.csv", "phamer_neighbors.csv"):
        rows = [[line for line in open(os.path.join(str(outs[k]), name)) if not line.startswith("#")] for k in ("plain", "packed")]
        assert rows[0] == rows[1] and len(rows[0]) > 0, name


def test_corrupt_bgzf_raises_what_gzip_raises(tmp_path):
    """A BGZF file with a wrong CRC32 in one member fails on the device and falls back to the host road, which raises gzip's
    error; a file with a corrupt DEFLATE stream raises zlib's."""
    from phamers_b200 import fileIO
    raw = bgzf(b">a\nACGT\n" * 20000)
    members = fileIO.bgzf_members(bytes(raw))
    end = int(members["in_offset"][1] + members["in_bytes"][1])
    bad_crc = bytearray(raw)
    bad_crc[end] ^= 0x55                                             # CRC32 of member 1
    bad_stream = bytearray(raw)
    bad_stream[int(members["in_offset"][0])] = 0x07                  # BTYPE 11 in member 0
    for i, data in enumerate((bad_crc, bad_stream)):
        path = tmp_path / ("bad%d.fasta.gz" % i)
        path.write_bytes(bytes(data))
        with pytest.raises(Exception) as want:
            with gzip.open(str(path), "rb") as fh:
                fh.read()
        with pytest.raises(type(want.value)) as got:
            fileIO.read_fasta_arrays_cuda(str(path))
        assert str(got.value) == str(want.value)
