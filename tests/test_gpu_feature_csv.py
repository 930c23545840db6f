"""Feature CSVs on the device (ops.format_counts_csv_cuda / ops.parse_feature_csv_cuda, and save_counts / read_feature_file above
them) against the host road they replace (fileIO._save_counts_host / _read_feature_file_host): byte-identical files, equal arrays,
every line-end and blank convention, events on every alignment of the parser's 4 KB tiles, each decline reason (after which the host
road returns or raises what it always did), random files from a mixed grammar, compressed files and the command line."""
import argparse
import gzip

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from test_bgzf_cpu import bgzf

pytestmark = pytest.mark.gpu

TILE = 4096                                    # csv_lines / csv_index / csv_fill tile (PT_TILE in feature_csv.cu)
CSV_OK, CSV_BYTE, CSV_NO_COMMA, CSV_FIELD, CSV_RAGGED = range(5)
I64 = np.iinfo(np.int64)


def _launches():
    from phamers_b200 import ops
    return ops.kernel_launches()


def _values(rng, shape):
    """int64 values of every decimal length from 1 to 19, both signs, and the extremes."""
    digits = rng.integers(1, 20, size=shape)
    mag = np.minimum(np.floor(10.0 ** (digits - 1) * rng.uniform(1, 10, size=shape)), 9.2e18).astype(np.int64)
    v = np.where(rng.random(shape) < 0.3, -mag, mag)
    v[rng.random(shape) < 0.1] = 0
    flat = v.reshape(-1)
    if flat.size >= 2:
        flat[0], flat[-1] = I64.min, I64.max
    return v


def _same_file(tmp_path, counts, ids, device=True, **kw):
    from phamers_b200 import fileIO
    a, b = str(tmp_path / "device.csv"), str(tmp_path / "host.csv")
    before = _launches()
    fileIO.save_counts(counts, ids, a, **kw)
    took_device = _launches() > before
    fileIO._save_counts_host(counts, ids, b, **kw)
    got, want = open(a, "rb").read(), open(b, "rb").read()
    assert got == want, (got[:200], want[:200])
    assert took_device == device
    return got


# ---------------------------------------------------------------------------------------------------------------------------
# writer
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width", [1, 136, 256, 512, 1024, 2080, 4096, 0])
def test_writer_widths_and_values(tmp_path, width):
    rng = np.random.default_rng(width)
    rows = 40 if width >= 1024 else 300
    counts = _values(rng, (rows, width))
    ids = ["SuperContig_%d_length_%d_ID_%d" % (i, 1000 + i, i) for i in range(rows)]
    text = _same_file(tmp_path, counts, ids)
    assert text.count(b"\n") == rows + 1


def test_writer_count_like_values_and_negative_extremes(tmp_path):
    counts = np.array([[0, 1, 9, 10, 99, 100, 999, 1000], [-1, -9, -10, -99, -100, I64.min, I64.max, I64.min + 1]])
    _same_file(tmp_path, counts, ["a", "b"])
    for d in range(1, 20):                       # every power of ten and its neighbours
        p = 10 ** d
        vals = [v for v in (p - 1, p, p + 1, -(p - 1), -p, -(p + 1)) if I64.min <= v <= I64.max]
        _same_file(tmp_path, np.array([vals]), ["p%d" % d])


def test_writer_shapes_and_ids(tmp_path):
    rng = np.random.default_rng(7)
    counts = rng.integers(-5000, 5000, size=(20, 33))
    _same_file(tmp_path, counts[3], ["one-d"])                                   # a 1-D counts is one row
    _same_file(tmp_path, counts, ["r%d" % i for i in range(12)])                 # fewer ids than rows
    _same_file(tmp_path, counts[:5], ["r%d" % i for i in range(9)])              # more ids than rows
    _same_file(tmp_path, counts[:0], ["a", "b"], device=False)                   # no rows: the header only
    _same_file(tmp_path, counts, [], device=False)
    _same_file(tmp_path, counts[:6], ["", "a,b", "#x", " sp ace ", "line\nfeed", "t\tab"])
    _same_file(tmp_path, counts[:3], np.array(["x", "yy", "zzz"]))               # numpy strings
    _same_file(tmp_path, counts[:3], [1, 2.5, None])                             # str() of anything
    _same_file(tmp_path, counts[:3], ["i" * 3000, "j" * 5000, "k"])              # ids longer than a staging buffer
    _same_file(tmp_path, counts.astype(np.float64) + 0.7, ["f%d" % i for i in range(20)])    # astype(int64) truncates
    _same_file(tmp_path, counts[:2], ["café", "b"], device=False)             # non-ASCII id: the host road
    _same_file(tmp_path, counts[None, :2], ["a", "b"], device=False)              # 3-D counts: the host road


def test_writer_header_from_args(tmp_path):
    args = argparse.Namespace(fasta="x.fasta", k=4, out="o")
    _same_file(tmp_path, np.arange(12).reshape(3, 4), ["a", "b", "c"], args=args)
    _same_file(tmp_path, np.arange(12).reshape(3, 4), ["a", "b", "c"], header="line one\nline two")


@pytest.mark.parametrize("chunk", [1, 300, 5000, 70000])
def test_writer_slices(tmp_path, monkeypatch, chunk):
    """Slices of FORMAT_CHUNK bytes of text: one row each, a few rows each, and rows split at every kind of boundary."""
    from phamers_b200 import fileIO
    monkeypatch.setattr(fileIO, "FORMAT_CHUNK", chunk)
    rng = np.random.default_rng(chunk)
    counts = rng.integers(-10 ** 6, 10 ** 6, size=(257, 19))
    ids = ["id%d" % (i * 7919 % 1000) * (1 + i % 3) for i in range(257)]
    _same_file(tmp_path, counts, ids)


def test_format_call_places_rows_at_every_alignment():
    """ops.format_counts_csv_cuda on its own: rows of every length modulo 16 (so rows start on every byte of a 16-byte word), and
    rows longer than the 2 KB staging buffer."""
    from phamers_b200 import ops
    rng = np.random.default_rng(11)
    for width in (3, 150):
        counts = rng.integers(-999, 99999, size=(64, width))
        ids = ["x" * int(rng.integers(0, 40)) for _ in range(64)]
        want = b"".join(("%s,%s\n" % (i, ",".join(map(str, r)))).encode() for i, r in zip(ids, counts.tolist()))
        id_bytes = torch.tensor(list("".join(ids).encode()) or [0], dtype=torch.uint8)[:sum(map(len, ids))]
        offsets = torch.tensor(np.concatenate(([0], np.cumsum([len(i) for i in ids]))), dtype=torch.int64)
        got = ops.format_counts_csv_cuda(torch.from_numpy(counts).cuda(), id_bytes.cuda(), offsets.cuda())
        assert got.cpu().numpy().tobytes() == want


# ---------------------------------------------------------------------------------------------------------------------------
# reader
# ---------------------------------------------------------------------------------------------------------------------------
def _device_parse(data):
    """bytes -> (result block, parsed or None) through ops.parse_feature_csv_cuda on a padded device copy."""
    from phamers_b200 import ops
    n = len(data)
    buf = torch.full(((n + 15) // 16 * 16 + 16,), ord(","), dtype=torch.uint8)     # padding of commas must not be read as text
    buf[:n] = torch.frombuffer(bytearray(data), dtype=torch.uint8) if n else buf[:0]
    d = buf.cuda()
    result = torch.full((4,), -7, dtype=torch.int64, device="cuda")
    parsed = ops.parse_feature_csv_cuda(d[:n], result=result)
    return result.cpu().tolist(), parsed


def _host_outcome(path, **kw):
    from phamers_b200 import fileIO
    try:
        return "ok", fileIO._read_feature_file_host(path, **kw)
    except Exception as exc:                                        # noqa: BLE001  (the host road's outcome, whatever it is)
        return "raise", (type(exc), str(exc))


def _check_read(tmp_path, data, accept=True, name="f.csv", **kw):
    """read_feature_file on `data` equals the host road (same arrays, or the same exception); `accept` says whether the device
    must take the file."""
    from phamers_b200 import fileIO
    path = str(tmp_path / name)
    with open(path, "wb") as fh:
        fh.write(data)
    result, parsed = _device_parse(data)
    assert (parsed is not None) == accept, result
    want = _host_outcome(path, **kw)
    try:
        got = ("ok", fileIO.read_feature_file(path, **kw))
    except Exception as exc:                                        # noqa: BLE001
        got = ("raise", (type(exc), str(exc)))
    assert got[0] == want[0], (got, want)
    if got[0] == "raise":
        assert got[1] == want[1]
        assert not accept
        return result
    g, w = got[1], want[1]
    if isinstance(w, tuple):
        assert g[0].dtype == w[0].dtype and g[0].shape == w[0].shape and g[0].tolist() == w[0].tolist()
        g, w = g[1], w[1]
    assert g.dtype == w.dtype and g.shape == w.shape and np.array_equal(g, w, equal_nan=g.dtype.kind == "f")
    return result


def test_reader_on_both_writers_and_the_reference_format(tmp_path):
    from phamers_b200 import fileIO
    rng = np.random.default_rng(5)
    counts = rng.integers(0, 3000, size=(50, 256))
    ids = ["SuperContig_%d_length_%d_ID_%d" % (i, 5000 + i, i) for i in range(50)]
    for writer in (fileIO.save_counts, fileIO._save_counts_host):
        path = str(tmp_path / "w.csv")
        writer(counts, ids, path, args=argparse.Namespace(k=4))
        data = open(path, "rb").read()
        _check_read(tmp_path, data)
        got_ids, got = fileIO.read_feature_file(path)
        assert got_ids.tolist() == ids and np.array_equal(got, counts)
    _check_read(tmp_path, b"# K-mer count file\n# fasta:\tx\n12345,1,2,3\n67890,4,5,6\n")


@pytest.mark.parametrize("eol", [b"\n", b"\r\n", b"\r"])
@pytest.mark.parametrize("final", [True, False])
def test_reader_line_ends_blanks_and_comments(tmp_path, eol, final):
    lines = [b"# header", b"", b"   ", b"\t# indented comment", b"a,1,2,3", b"  b c  ,+4, -5 ,\t006\t", b"",
             b"c,7,8,9 # trailing note", b"d#e,1,1", b"#", b"e,000000000000000001,-999999999999999999,+999999999999999999",
             b" \t ", b",0,0,0", b"  ,1,1,1"]
    data = eol.join(lines) + (eol if final else b"")
    _check_read(tmp_path, data.replace(b"d#e,1,1", b"d,1,1,1"))
    for normalize, ident in ((True, None), (False, "b c  "), (True, "e"), (False, "nope")):
        _check_read(tmp_path, data.replace(b"d#e,1,1", b"d,1,1,1"), normalize=normalize, id=ident)


def test_reader_empty_inputs(tmp_path):
    for data in (b"", b"\n", b"# only a header\n", b"\r\n\r\n", b"   \t\n#x,1,2\n"):
        _check_read(tmp_path, data)


def test_reader_long_lines_and_many_short_lines(tmp_path):
    """One line longer than several tiles (a 5 000-byte id and 4 096 fields), then 2 M short lines and 1 M blank lines: tiles
    with 4 096 line starts each."""
    from phamers_b200 import fileIO
    rng = np.random.default_rng(9)
    wide = rng.integers(-10 ** 17, 10 ** 17, size=(3, 4096))
    data = b"".join(("%s,%s\n" % ("L" * 5000 if i == 1 else "w%d" % i, ",".join(map(str, r)))).encode() for i, r in enumerate(wide))
    _check_read(tmp_path, data)
    n = 2_000_000
    vals = np.arange(n, dtype=np.int64) % 1000
    data = b"\n" * 1_000_000 + b"".join(b"%d,%d\n" % (i % 10, v) for i, v in zip(range(n), vals))
    path = str(tmp_path / "short.csv")
    with open(path, "wb") as fh:
        fh.write(data)
    ids, got = fileIO.read_feature_file(path)
    assert got.shape == (n, 1) and np.array_equal(got[:, 0], vals)
    assert ids.tolist() == [str(i % 10) for i in range(n)]


def _sweep_file(pad, event):
    """A file whose `event` lands at byte `pad` of a 16-byte word and just around a tile boundary: a comment line fills the bytes
    before the data lines."""
    head = b"#" + b"c" * pad + b"\n"
    body = {"lf": b"a,1,2\nb,3,4\n", "crlf": b"a,1,2\r\nb,3,4\r\n", "cr": b"a,1,2\rb,3,4\r", "hash": b"a,1,2#x\nb,3,4 #\n",
            "comma": b"abc,10,-20\nd,30,+40\n", "blank": b"   a  ,  1  ,  2  \n\t\tb\t,3\t,4\t\n"}[event]
    return head + body


@pytest.mark.parametrize("event", ["lf", "crlf", "cr", "hash", "comma", "blank"])
def test_tile_sweep(event):
    """Every alignment of line ends, commas, '#', CRLF pairs and blanks against the tile boundary and the 16-byte words: the data
    lines start at every byte from 48 before the first tile boundary to 48 after it, and again around the 512-byte steps of a line."""
    for pad in list(range(TILE - 64, TILE + 48)) + list(range(0, 40)):
        data = _sweep_file(pad, event)
        result, parsed = _device_parse(data)
        assert parsed is not None and result[:3] == [2, 2, CSV_OK], (pad, result)
        ranges, counts = parsed
        text = data.decode()
        ids = [text[a:b] for a, b in ranges.tolist()]
        assert ids == {"blank": ["a  ", "b\t"], "comma": ["abc", "d"]}.get(event, ["a", "b"]), pad
        want = [[10, -20], [30, 40]] if event == "comma" else [[1, 2], [3, 4]]
        assert counts.cpu().tolist() == want, pad
    # a line that is longer than a tile, at every alignment of its start
    row = ",".join(str(i) for i in range(1500))
    for pad in range(0, 20):
        data = b" " * pad + ("x," + row + "\n" + "y," + row).encode()
        result, parsed = _device_parse(data)
        assert result[:3] == [2, 1500, CSV_OK]
        assert parsed[1].cpu().numpy().tolist() == [list(range(1500))] * 2


# ---------------------------------------------------------------------------------------------------------------------------
# declines
# ---------------------------------------------------------------------------------------------------------------------------
DECLINES = [
    (b"a,1\nb,\x0b2\n", CSV_BYTE, 2), (b"a,1\nb,2\x00\n", CSV_BYTE, 2), ("a,1\nb,2\ncé,3\n".encode(), CSV_BYTE, 3),
    (b"a,1\x7f\n", CSV_BYTE, 1), (b"#\x1c\na,1\n", CSV_BYTE, 1), (b"a,1\n\x0c\n", CSV_BYTE, 2),
    (b"# h\nabc\n", CSV_NO_COMMA, 2), (b"a,1\n\n  lone  # x,1\n", CSV_NO_COMMA, 3),
    (b"a,1_0\n", CSV_FIELD, 1), (b"a,1e3\n", CSV_FIELD, 1), (b"a,1,\n", CSV_FIELD, 1), (b"a,,1\n", CSV_FIELD, 1),
    (b"a,1 2\n", CSV_FIELD, 1), (b"a,+\n", CSV_FIELD, 1), (b"a,--1\n", CSV_FIELD, 1), (b"a,1.0\n", CSV_FIELD, 1),
    (b"a,1\nb,1234567890123456789\n", CSV_FIELD, 2), (b"a,9223372036854775808\n", CSV_FIELD, 1), (b"a,0x1\n", CSV_FIELD, 1),
    (b"a,1,2\nb,1,2\nc,1\n", CSV_RAGGED, 3), (b"a,1\nb,1,2\n", CSV_RAGGED, 2), (b"x\n" + b"a,1\nb,1,2\n", CSV_NO_COMMA, 1),
    (b"a,1,2\nb,1\nc,x\n", CSV_RAGGED, 2), ("a,٣\n".encode(), CSV_BYTE, 1),
]


@pytest.mark.parametrize("data,reason,line", DECLINES)
def test_declines(tmp_path, data, reason, line):
    result = _check_read(tmp_path, data, accept=False)
    assert result[2:] == [reason, line]


def test_decline_far_from_the_start(tmp_path):
    good = b"".join(b"r%d,%d,%d\n" % (i, i, -i) for i in range(5000))
    for bad, reason in ((b"z,1,2,3\n", CSV_RAGGED), (b"z,1,x\n", CSV_FIELD), (b"z 1 2\n", CSV_NO_COMMA), (b"z,1,\x01\n", CSV_BYTE)):
        result = _check_read(tmp_path, good + bad + good, accept=False)
        assert result[2:] == [reason, 5001]


# ---------------------------------------------------------------------------------------------------------------------------
# random files
# ---------------------------------------------------------------------------------------------------------------------------
_PIECES = [b",", b"#", b" ", b"\t", b"\n", b"\r", b"\r\n", b"+", b"-", b"0", b"7", b"42", b"123456789012345678", b"1234567890123456789",
           b"a", b"id_", b"_", b"e", b".", b"\x0b", b"\xc3\xa9", b"x,1,2\n", b"y, 3 ,-4\n", b"#c\n"]


@settings(max_examples=300, deadline=None, suppress_health_check=[HealthCheck.function_scoped_fixture])
@given(st.lists(st.sampled_from(_PIECES), max_size=60), st.integers(0, 20))
def test_property_device_matches_host_or_declines(tmp_path, pieces, pad):
    """Either the device result equals the host result, or the device declines and read_feature_file does what the host does; the
    device never accepts a file the host rejects."""
    data = b" " * pad + b"".join(pieces)
    path = str(tmp_path / "p.csv")
    with open(path, "wb") as fh:
        fh.write(data)
    _, parsed = _device_parse(data)
    host = _host_outcome(path)
    if parsed is not None:
        assert host[0] == "ok", (data, host)
    _check_read(tmp_path, data, accept=parsed is not None, name="p.csv")


# ---------------------------------------------------------------------------------------------------------------------------
# compressed files and the command line
# ---------------------------------------------------------------------------------------------------------------------------
def test_compressed_files_equal_their_plain_copies(tmp_path):
    from phamers_b200 import fileIO
    rng = np.random.default_rng(3)
    counts = rng.integers(0, 10 ** 6, size=(3000, 136))
    plain = str(tmp_path / "c.csv")
    fileIO.save_counts(counts, ["c%d" % i for i in range(3000)], plain)
    data = open(plain, "rb").read()
    assert len(data) > 3 * 65280                                   # several BGZF members
    want_ids, want = fileIO._read_feature_file_host(plain)
    for name, blob in (("b.csv.gz", bgzf(data)), ("g.csv.gz", gzip.compress(data))):
        path = str(tmp_path / name)
        with open(path, "wb") as fh:
            fh.write(blob)
        ids, got = fileIO.read_feature_file(path)
        assert ids.tolist() == want_ids.tolist() and np.array_equal(got, want) and got.dtype == np.int64


def test_command_line_cache_is_byte_identical(tmp_path, monkeypatch):
    """phamer -in DIR writes <fasta>_features.csv byte for byte as the host road does, and a second run that reads the cache gives
    the same phamer_scores.csv."""
    from test_gpu_cli import _write_fasta
    from phamers_b200 import fileIO, phamer
    rng = np.random.default_rng(20261022)
    runs = {}
    for road in ("device", "host"):
        indir = tmp_path / road
        indir.mkdir()
        _write_fasta(indir / "contigs.fasta", rng if road == "device" else np.random.default_rng(20261022), 120)
        if road == "host":
            monkeypatch.setattr(fileIO, "save_counts", fileIO._save_counts_host)
            monkeypatch.setattr(fileIO, "read_feature_file", fileIO._read_feature_file_host)
        phamer.main(["-in", str(indir), "-out", str(tmp_path / (road + "_1")), "-equal", "-l", "0"])
        cache = open(indir / "contigs_features.csv", "rb").read()
        phamer.main(["-in", str(indir), "-out", str(tmp_path / (road + "_2")), "-equal", "-l", "0"])
        scores = []
        for run in ("_1", "_2"):                           # the '#' header names the run's directories
            with open(tmp_path / (road + run) / "phamer_scores.csv", "rb") as fh:
                scores.append(b"".join(line for line in fh if not line.startswith(b"#")))
        runs[road] = (cache, scores[0], scores[1])
    monkeypatch.undo()
    assert runs["device"][0] == runs["host"][0]
    assert runs["device"][2] == runs["host"][2]
    assert runs["device"][1] == runs["device"][2]
