"""The device FASTA tokeniser (phm_fasta_index / phm_fasta_extract) across the regimes of its kernels, against the oracle's
restatement of Bio.SeqIO over a text-mode handle (oracle/phamers_oracle.py::parse_fasta_text) and the host tokeniser.

The kernels work on 16 384-byte tiles of 1024 threads, 16 bytes a thread (a warp covers 512 bytes).  The tile and emit kernels
loop over the tiles with a grid of 8 x SMs CTAs; the one-CTA chain pass gives each of its 32 warps a range of
per = ceil(ceil(T / 32) / 32) * 32 tiles, which the warp walks 32 tiles at a time.  The files here are sized from those constants
so that every regime is reached: one tile, one warp with work, several warps, a warp that loops over its range, and the grid-stride
loops.  Each file carries an event on every tile boundary and on a sample of warp and chunk boundaries, and the large ones carry the
long-range states (a preamble, a title line and a sequence line longer than a tile, tiles of blank lines, a tile of empty
records); the test asserts, from the reference, that those paths were reached."""
import ctypes
import gzip
import re

import numpy as np
import pytest
import torch

from oracle import phamers_oracle as po

pytestmark = pytest.mark.gpu

TILE = 16384            # bytes of a tile (TILE_THREADS * PER_THREAD in fasta_scan.cu)
WARP_SPAN = 512         # bytes of a warp within a tile
CHUNK = 16              # bytes of a thread
CHAIN_WARPS = 32        # warps of the chain pass
SPECIAL_MIN_TILES = 31  # files of at least this many tiles start with the long-range states
BASES = np.frombuffer(b"ACGTACGTACGTACGTNacgt", dtype=np.uint8)
TILE_COUNTS = ["1", "2", "31", "32", "33", "64", "65", "1023", "1024", "1025", "8*SM", "8*SM+1", "3*1024+5"]


def _grid():
    return 8 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _tiles(name):
    sm8 = _grid()
    return {"8*SM": sm8, "8*SM+1": sm8 + 1, "3*1024+5": 3 * 1024 + 5}.get(name) or int(name)


def _chain_range(n_tiles, tile):
    """(warp, round) of the chain pass that handles `tile`: warp w owns [w * per, (w + 1) * per) and walks it 32 tiles a round."""
    per = ((n_tiles + CHAIN_WARPS - 1) // CHAIN_WARPS + 31) // 32 * 32
    return tile // per, (tile % per) // 32


# ---------------------------------------------------------------------------------------------------------------------------
# seeded files
# ---------------------------------------------------------------------------------------------------------------------------
def _lines(body, width, eol):
    """body (uint8 array without zero bytes) cut into lines of `width` bytes (0: one line), each ended by eol."""
    if body.shape[0] == 0:
        return b""
    width = width or body.shape[0]
    grid = np.concatenate((body, np.zeros((-body.shape[0]) % width, dtype=np.uint8))).reshape(-1, width)
    ends = np.broadcast_to(np.frombuffer(eol, dtype=np.uint8), (grid.shape[0], len(eol)))
    flat = np.concatenate((grid, ends), axis=1).reshape(-1)
    return flat[flat != 0].tobytes()


def _records(rng, n_bytes, first):
    """Records of length 0, 1, short and long; line widths 60, 80, 1000 and one line; LF, CRLF and lone-CR line ends; blank
    lines and blanks inside lines."""
    parts, size, r = [], 0, first
    while size < n_bytes:
        eol = (b"\n", b"\r\n", b"\r")[int(rng.choice(3, p=[0.5, 0.3, 0.2]))]
        u = rng.random()
        length = 0 if u < 0.1 else 1 if u < 0.2 else int(rng.integers(2, 300)) if u < 0.6 else int(rng.integers(1000, 120000))
        body = rng.choice(BASES, size=length)
        if length > 10 and rng.random() < 0.3:
            body[rng.integers(0, length, size=3)] = ord(" ")
        rec = b">rec%d_ID_%d len=%d%s" % (r, r, length, b"  " if rng.random() < 0.2 else b"") + eol
        rec += _lines(body, int(rng.choice([60, 80, 1000, 0])), eol)
        if rng.random() < 0.15:
            rec += (eol, b"  " + eol, b"\n\n", b"\r\n \r\n")[int(rng.integers(4))]
        parts.append(rec)
        size += len(rec)
        r += 1
    return b"".join(parts)


def _long_range(rng):
    """A preamble longer than a tile, a 40 000-byte title line, a 50 000-byte sequence line without a line break, 35 KB of blank
    lines and 34 KB of empty records ('>\\n')."""
    pre = _lines(rng.choice(np.frombuffer(b"ACGT xyz|", dtype=np.uint8), size=20000), 70, b"\n")
    title = b">long_title_ID_0 " + rng.choice(np.frombuffer(b"abc XYZ|>09", dtype=np.uint8), size=40000).tobytes() + b"\n"
    seq = rng.choice(BASES, size=50000).tobytes() + b"\n"
    blanks = b"".join((b"\n", b"\r\n", b"   \n", b"\r", b" \r\n")[i] for i in rng.integers(0, 5, size=16000))
    return pre + title + seq + blanks + b">\n" * 17000


def _plant(data, lo, rng):
    """An event on every tile boundary b = TILE * t past `lo`, at b + delta with delta cycling through -2..2, and on a sample of
    warp and chunk boundaries; the events cycle through a header '>', a '\\n' ending the bytes before the boundary, '\\r' | '\\n'
    split across it, a lone '\\r' followed by '>', a '>' inside a line, and a blank or CR that must be dropped."""
    n = data.shape[0]
    tiles = np.arange(TILE, n, TILE)
    pos = [tiles + (np.arange(tiles.shape[0]) % 5 - 2)]
    for step in (WARP_SPAN, CHUNK):
        cand = np.arange(step, n, step)
        size = min(2000, cand.shape[0])
        pos.append(rng.choice(cand, size=size, replace=False) + rng.integers(-2, 3, size=size))
    pos = np.concatenate(pos)
    pos = pos[(pos >= lo + 2) & (pos <= n - 3)]
    kind = np.arange(pos.shape[0]) % 6
    for k, prev, here, after in ((0, 10, 62, None), (1, 10, None, None), (2, 13, 10, None), (3, 13, 62, None),
                                 (4, 65, 62, 67)):
        p = pos[kind == k]
        data[p - 1] = prev
        if here is not None:
            data[p] = here
        if after is not None:
            data[p + 1] = after
    p = pos[kind == 5]
    data[p] = np.where(np.arange(p.shape[0]) % 2, 13, 32)


@pytest.fixture(scope="module")
def contents():
    """Two seeded base files, cut to length by each case: `small` (records from byte 0) for files under SPECIAL_MIN_TILES tiles,
    `large` (long-range states first) for the others."""
    rng = np.random.default_rng(20261021)
    small = np.frombuffer(_records(rng, SPECIAL_MIN_TILES * TILE, 0), dtype=np.uint8).copy()
    _plant(small, 0, rng)
    head = _long_range(rng)
    large = np.frombuffer(head + _records(rng, max(3 * 1024 + 5, _grid() + 1) * TILE, 1), dtype=np.uint8).copy()
    _plant(large, len(head), rng)
    return {"small": small, "large": large}


def _file(contents, n_tiles, n):
    base = contents["small"] if n_tiles < SPECIAL_MIN_TILES else contents["large"]
    assert base.shape[0] >= n
    return base[:n].tobytes()


# ---------------------------------------------------------------------------------------------------------------------------
# reference and device
# ---------------------------------------------------------------------------------------------------------------------------
class Reference(object):
    def __init__(self, raw):
        """The oracle's records, and the byte positions of the oracle's lines (a line ends at '\\r\\n', '\\r' or '\\n')."""
        text = raw.decode("latin-1")
        recs = list(po.parse_fasta_text(text))
        self.n = len(raw)
        self.data = np.frombuffer(raw, dtype=np.uint8)
        starts = np.array([0] + [m.end() for m in re.finditer("\r\n|\r|\n", text)], dtype=np.int64)
        self.line_starts = starts[starts < self.n]
        self.header_pos = self.line_starts[self.data[self.line_starts] == ord(">")]
        assert self.header_pos.shape[0] == len(recs)
        self.ids = [(t.split(None, 1) or [""])[0] for t, _ in recs]
        self.blob = "".join(s for _, s in recs).encode("latin-1")
        self.offsets = np.zeros(len(recs) + 1, dtype=np.int64)
        np.cumsum([len(s) for _, s in recs], out=self.offsets[1:])

    def tile_facts(self):
        """Per tile t >= 1: the state it is entered in (0 preamble, 1 header line, 2 sequence line) and the kept bytes before it;
        per tile: kept bytes, whether a byte of it starts a line (follows '\\n' or '\\r'), records starting in it.  Derived from the
        oracle's lines, and checked against the oracle's sequence bytes."""
        n, data, starts = self.n, self.data, self.line_starts
        is_h = data[starts] == ord(">")
        seen = (np.cumsum(is_h) - is_h) > 0
        state = np.where(is_h, 1, np.where(seen, 2, 0))
        in_seq = np.repeat(state == 2, np.diff(np.append(starts, n)))
        keep = in_seq & (data != 10) & (data != 13) & (data != 32)
        first = np.arange(0, n, TILE)
        kept = np.add.reduceat(keep.view(np.uint8), first, dtype=np.int64)
        assert int(kept.sum()) == len(self.blob)
        ends = (data == 10) | (data == 13)
        has_start = np.add.reduceat(np.concatenate(([True], ends[:-1])).view(np.uint8), first, dtype=np.int64) > 0
        entered = state[np.searchsorted(starts, first[1:] - 1, side="right") - 1]
        return {"entered": entered, "kept_before": np.cumsum(kept)[:-1], "kept": kept, "has_line_start": has_start,
                "records": np.bincount(self.header_pos // TILE, minlength=first.shape[0])}


def _device_raw(raw, fill=b">"):
    """raw on the device in an allocation padded to 16 bytes past the next multiple of 16, the padding filled with `fill`
    (bytes, repeated) or with the given uint8 array."""
    n = len(raw)
    size = (n + 15) // 16 * 16 + 16
    if isinstance(fill, np.ndarray):
        host = fill[:size].copy()
    else:
        host = np.frombuffer((fill * (size // len(fill) + 1))[:size], dtype=np.uint8).copy()
    host[:n] = np.frombuffer(raw, dtype=np.uint8)
    return torch.from_numpy(host).cuda()[:n]


def _scan(raw, fill=b">"):
    from phamers_b200 import ops
    seq, off, hpos, odd = ops.fasta_scan_cuda(_device_raw(raw, fill))
    off = off.cpu().numpy()
    return seq.cpu().numpy()[:int(off[-1])].tobytes(), off, hpos.cpu().numpy(), odd


def _compare(raw, ref):
    from phamers_b200 import fileIO
    blob, off, hpos, odd = _scan(raw)
    assert not odd
    assert np.array_equal(off, ref.offsets), "offsets"
    assert np.array_equal(hpos, ref.header_pos), "header positions"
    assert blob == ref.blob, "sequence bytes"
    ids, h_seq, h_off = fileIO.split_fasta_bytes(raw)
    assert ids == ref.ids and np.array_equal(h_off, ref.offsets) and h_seq.tobytes() == ref.blob, "host tokeniser"


# ---------------------------------------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tiles", TILE_COUNTS)
def test_tile_regimes_match_oracle(contents, tiles):
    """Files of T tiles, ending mid-chunk and exactly on a tile, against the oracle and the host tokeniser."""
    t = _tiles(tiles)
    for n in (t * TILE - 9, t * TILE):
        raw = _file(contents, t, n)
        ref = Reference(raw)
        _compare(raw, ref)
        facts = ref.tile_facts()
        assert facts["kept"].shape[0] == t
        if t >= SPECIAL_MIN_TILES:                      # the long-range states were reached
            assert set(facts["entered"].tolist()) == {0, 1, 2}
            assert not facts["has_line_start"].all()
            assert facts["records"].max() >= TILE // 2
            assert np.any((facts["kept"][1:] == 0) & (facts["entered"] == 2))
        if t >= 1023:                                   # the emit pass's unaligned head and funnel shift at every residue
            assert set((facts["kept_before"] % 16).tolist()) == set(range(16))


@pytest.mark.parametrize("ending", [b"\n", b"\r", b">", b"A", b"\t", b"\n>h"])
def test_padding_contents_do_not_matter(ending):
    """For every length 0..64 and each file ending, the bytes of the allocation past the end (zeros, '>', '\\n>', tab, random)
    change nothing: the results equal the zero-padded run and the oracle, every header lies inside the file, and a tab only in
    the padding leaves odd unset."""
    from phamers_b200 import fileIO
    rng = np.random.default_rng(7)
    template = b">r1 x\nACGT\r\nG G\n>r2\rAC\r>\n>r3\nTTGCA\n" * 4
    fills = [b"\0", b">", b"\n>", b"\t", rng.integers(0, 256, size=128, dtype=np.uint8)]
    for n in range(65):
        raw = (template[:max(n - len(ending), 0)] + ending)[-n:] if n else b""
        assert len(raw) == n
        want = _scan(raw, b"\0")
        control = any(c < 32 and c not in (10, 13) for c in raw)
        assert want[3] == control
        for fill in fills:
            got = _scan(raw, fill)
            assert got[0] == want[0] and np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]), (n, fill)
            assert got[3] == want[3] and np.all(got[2] < n)
        if not control:
            ref = Reference(raw)
            assert want[0] == ref.blob and np.array_equal(want[1], ref.offsets) and np.array_equal(want[2], ref.header_pos)
        ids, h_seq, h_off = fileIO.split_fasta_bytes(raw)
        assert [h_seq.tobytes()[h_off[i]:h_off[i + 1]] for i in range(len(ids))] == \
            [s.encode("latin-1") for _, s in po.parse_fasta_text(raw.decode("latin-1"))]


def test_odd_whitespace_flag_crosses_the_chain_pass(contents):
    """A single tab in tile 40 (warp 1 of the chain pass), in tile 1100 in the second round of a warp's range, or as the last byte
    of a file ending mid-chunk sets odd; the same files without it do not."""
    cases = []
    for n_tiles, tile in ((41, 40), (2100, 1100)):
        n = n_tiles * TILE - 3
        warp, rnd = _chain_range(n_tiles, tile)
        assert (n_tiles, warp, rnd) in ((41, 1, 0), (2100, 11, 1))
        clean = bytearray(_file(contents, n_tiles, n))
        tabbed = bytearray(clean)
        tabbed[tile * TILE + 777] = 9
        cases.append((bytes(clean), bytes(tabbed)))
    clean = _file(contents, 65, 65 * TILE - 5)
    cases.append((clean, clean[:-1] + b"\t"))
    for clean, tabbed in cases:
        assert not _scan(clean)[3]
        assert _scan(tabbed)[3]


CLASSIC_MAC = b">a_ID_1 desc\rACGTAC\r>b_ID_2\nAC\x1c\nGT\n"


def test_line_ends_by_hand(tmp_path):
    """Classic-Mac files, mixed line ends, '\\r\\r\\n', a CR as a tile's last byte before a '>', and the separators and tabs the
    reference strips at line ends: device, host and oracle agree."""
    from phamers_b200 import fileIO, kmer
    plain = [
        b">a\rACGT\rAC\r>b c\rGG\r", b">a\r\nAC\rGT\n>b\rT\r\nA\n\r>c\n\rC", b">a\r\r\nAC\r\r\nGT\r\r\n>b\r\r\nC",
        b"\r>a\r\r>b\r\rA\r", b">a\n" + b"A" * (TILE - 4) + b"\r>b\nCC\n", b">a\n" + b"C" * (TILE - 5) + b"\r\n>b\rG",
        CLASSIC_MAC.replace(b"\x1c", b""),
    ]
    assert plain[4][TILE - 1:TILE + 1] == b"\r>"
    for raw in plain:
        _compare(raw, Reference(raw))
    odd = [CLASSIC_MAC, b">a\rAC\t\rGT\r\n>b\r\r\nT T\x1f\r", b">a\x1e\nA\x1dC\x1f\r\n>b\tx\rG\x0b\x0c\r"]
    for i, raw in enumerate(plain + odd):
        path = tmp_path / ("f%d.fasta" % i)
        path.write_bytes(raw)
        ref = Reference(raw)
        ids, d_seq, d_off = fileIO.read_fasta_arrays_cuda(str(path))
        d_off = d_off.cpu().numpy()
        assert ids == ref.ids and np.array_equal(d_off, ref.offsets) and d_seq.cpu().numpy()[:d_off[-1]].tobytes() == ref.blob
        assert np.array_equal(kmer.count_file(str(path), 2)[1], po.count_file(str(path), 2)[1])
    path = tmp_path / "mac.fasta"
    path.write_bytes(CLASSIC_MAC)
    want = [("a_ID_1 desc", "ACGTAC"), ("b_ID_2", "ACGT")]
    assert list(po.parse_fasta_text(CLASSIC_MAC.decode("latin-1"))) == want
    ids, seq, off = fileIO.split_fasta_bytes(CLASSIC_MAC)
    assert ids == ["a_ID_1", "b_ID_2"] and [seq.tobytes()[off[i]:off[i + 1]] for i in range(2)] == [b"ACGTAC", b"ACGT"]
    _, _, hpos, odd = _scan(CLASSIC_MAC)
    assert odd and hpos.tolist() == [0, CLASSIC_MAC.index(b">b")]
    titles = [re.split(b"[\r\n]", CLASSIC_MAC[p + 1:])[0].decode() for p in hpos]
    assert titles == [t for t, _ in want]
    ids, d_seq, d_off = fileIO.read_fasta_arrays_cuda(str(path))
    d_off = d_off.cpu().numpy()
    assert ids == ["a_ID_1", "b_ID_2"] and [d_seq.cpu().numpy()[d_off[i]:d_off[i + 1]].tobytes() for i in range(2)] == \
        [b"ACGTAC", b"ACGT"]
    got_ids, counts = kmer.count_file(str(path), 4)
    want_ids, want_counts = po.count_file(str(path), 4)
    assert list(got_ids) == list(want_ids) == ["1", "2"] and np.array_equal(counts, want_counts) and counts.sum() == 3 + 1


def test_file_path_chunked_upload_gzip_and_counts(contents, tmp_path, monkeypatch):
    """read_fasta_arrays_cuda on the largest sweep file through staging buffers of 5 MiB + 7 bytes and on a gzipped mid-size
    file; kmer.count_file on the largest file equals kmer.count over the host tokeniser's sequences."""
    from phamers_b200 import fileIO, kmer
    big_tiles = 3 * 1024 + 5
    raw = _file(contents, big_tiles, big_tiles * TILE)
    ref = Reference(raw)
    path = tmp_path / "big.fasta"
    path.write_bytes(raw)
    with monkeypatch.context() as mp:
        mp.setattr(fileIO, "UPLOAD_CHUNK", 5 * 2 ** 20 + 7)
        ids, d_seq, d_off = fileIO.read_fasta_arrays_cuda(str(path))
    d_off = d_off.cpu().numpy()
    assert ids == ref.ids and np.array_equal(d_off, ref.offsets) and d_seq.cpu().numpy()[:d_off[-1]].tobytes() == ref.blob
    got_ids, counts = kmer.count_file(str(path), 4)
    h_ids, h_seq, h_off = fileIO.split_fasta_bytes(raw)
    blob = h_seq.tobytes().decode("latin-1")
    want = kmer.count([blob[h_off[i]:h_off[i + 1]] for i in range(len(h_ids))], 4)
    assert list(got_ids) == [fileIO.get_id(h) for h in h_ids] and np.array_equal(counts, want)
    raw = _file(contents, 65, 65 * TILE - 9)
    ref = Reference(raw)
    gz = tmp_path / "mid.fasta.gz"
    with gzip.open(gz, "wb") as fh:
        fh.write(raw)
    ids, d_seq, d_off = fileIO.read_fasta_arrays_cuda(str(gz))
    d_off = d_off.cpu().numpy()
    assert ids == ref.ids and np.array_equal(d_off, ref.offsets) and d_seq.cpu().numpy()[:d_off[-1]].tobytes() == ref.blob


def test_truncated_extract_through_the_c_abi(contents):
    """phm_fasta_extract with max_records = R - 3 and 0 writes offsets[0..max_records] (the last one is where the first dropped
    record starts) and header_pos[0..max_records), and nothing past them."""
    from phamers_b200 import _lib
    from phamers_b200._lib import check, ptr, stream_ptr
    lib = _lib.require_cuda()
    raw = _file(contents, 65, 65 * TILE - 9).replace(b"\r", b"\n")
    ref = Reference(raw)
    records = ref.header_pos.shape[0]
    assert records > 8000
    d_raw = _device_raw(raw, b"\0")                                      # padding has its own test
    ws_bytes = lib.phm_fasta_workspace_bytes(len(raw))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    result = torch.empty((4,), dtype=torch.int64, device="cuda")
    check(lib.phm_fasta_index(ptr(d_raw), len(raw), ptr(result), ptr(ws), ws_bytes, stream_ptr()))
    assert result[:2].tolist() == [records, len(ref.blob)]
    sentinel = -0x5A5A5A5A5A5A5A5A
    for max_records in (records - 3, 0):
        seq = torch.zeros(((len(ref.blob) + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
        offsets = torch.full((records + 1,), sentinel, dtype=torch.int64, device="cuda")
        header_pos = torch.full((records,), sentinel, dtype=torch.int64, device="cuda")
        check(lib.phm_fasta_extract(ptr(d_raw), len(raw), ptr(result), ptr(seq), ptr(offsets), ptr(header_pos),
                                    ctypes.c_int64(max_records), ptr(ws), ws_bytes, stream_ptr()))
        off, hpos = offsets.cpu().numpy(), header_pos.cpu().numpy()
        assert np.array_equal(off[:max_records + 1], ref.offsets[:max_records + 1])
        assert np.all(off[max_records + 1:] == sentinel)
        assert np.array_equal(hpos[:max_records], ref.header_pos[:max_records])
        assert np.all(hpos[max_records:] == sentinel)
        kept = int(ref.offsets[max_records])
        assert seq.cpu().numpy()[:kept].tobytes() == ref.blob[:kept]
