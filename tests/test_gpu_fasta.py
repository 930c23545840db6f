"""Device-side FASTA tokenisation (phm_fasta_index / phm_fasta_extract, SURVEY.md 8(f) rank 3) against the oracle's restatement
of the Bio.SeqIO parser the reference uses (oracle/phamers_oracle.py::parse_fasta_text) and against the host tokeniser."""
import gzip
import os
import re

import numpy as np
import pytest
import torch

from oracle import phamers_oracle as po

pytestmark = pytest.mark.gpu


def _scan(raw):
    """The device tokeniser on raw, uploaded into an allocation whose padding holds '>' (its contents must not matter)."""
    from phamers_b200 import ops
    n = len(raw)
    dev = torch.full(((n + 15) // 16 * 16 + 16,), ord(">"), dtype=torch.uint8, device="cuda")
    if n:
        dev[:n] = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    seq, off, hpos, odd = ops.fasta_scan_cuda(dev[:n])
    off = off.cpu().numpy()
    blob = seq.cpu().numpy().tobytes()[:int(off[-1])]
    return [blob[off[i]:off[i + 1]] for i in range(len(off) - 1)], hpos.cpu().numpy(), odd


def _check(raw):
    from phamers_b200 import fileIO
    seqs, hpos, odd = _scan(raw)
    assert not odd
    want = list(po.parse_fasta_text(raw.decode("latin-1")))
    assert [s.decode("latin-1") for s in seqs] == [s for _, s in want]
    ids, h_seq, h_off = fileIO.split_fasta_bytes(raw)                    # the host tokeniser agrees as well
    assert len(ids) == len(seqs) and int(h_off[-1]) == sum(len(s) for s in seqs)
    for i, p in enumerate(hpos):
        assert raw[p:p + 1] == b">" and (p == 0 or raw[p - 1:p] in (b"\n", b"\r"))
        title = re.compile(b"[^\r\n]*").match(raw, p + 1).group().decode("latin-1").rstrip()
        assert (title.split(None, 1) or [""])[0] == ids[i]


def test_hand_written_cases():
    cases = [
        b"", b"\n", b">", b">a", b">a\n", b">a\nACGT", b">a\nACGT\n", b"ACGT\n>a\nAC\nGT\n",
        b"junk line\nmore junk\n>r1 desc\nAC GT\r\nNN\n\n>r2\n>r3\nTT\n",            # preamble, CRLF, blanks, empty records
        b">a\nAC>GT\n>b\n A C\n",                                                     # '>' inside a line is sequence
        b"\n\n>a\n\n\nAC\n\n",                                                          # blank lines everywhere
        b">only header without newline",
        b">a\n" + b"ACGT" * 5000 + b"\n>b\n" + b"T" * 4095 + b"\n>c\n" + b"G" * 4096 + b"\n>d\n" + b"C" * 4097,   # tile edges
        b">x\n" + b"\n".join([b"ACGTACGTAC" * 6] * 300) + b"\n",
    ]
    for raw in cases:
        _check(raw)


def test_headers_and_newlines_on_tile_boundaries():
    """Every alignment of a header start, a line feed and a '>' that is not at a line start relative to the 16-byte thread
    chunks, the 512-byte span of a warp and the 16 384-byte tiles (a tile is 1024 threads of 16 bytes)."""
    shifts = list(range(0, 40))
    for edge in (512, 16384, 32768):
        shifts += list(range(edge - 24, edge + 8))
    for shift in shifts:
        body = b"A" * shift
        _check(b">h0\n" + body + b"\n>h1 t\nCC>GG\n" + b"T" * (16384 - (shift % 50)) + b"\r\n>h2\n\n")
        _check(body + b"\n>late\nACGT")


def test_random_files_match_oracle():
    rng = np.random.default_rng(11)
    for trial in range(12):
        parts = []
        if trial % 3 == 0:
            parts.append(b"preamble text\nsecond line\n")
        for r in range(int(rng.integers(1, 60))):
            parts.append(b">rec%d some description\n" % r if rng.random() < 0.8 else b">\n")
            n = int(rng.choice([0, 1, 59, 60, 61, 500, 4096, 20000]))
            seq = rng.choice(np.frombuffer(b"ACGTNacgt", dtype=np.uint8), size=n).tobytes()
            width = int(rng.choice([60, 70, 80, 1000000]))
            eol = b"\r\n" if rng.random() < 0.3 else b"\n"
            lines = [seq[i:i + width] for i in range(0, n, width)]
            if rng.random() < 0.3 and lines:
                lines[len(lines) // 2] = lines[len(lines) // 2][:5] + b" " + lines[len(lines) // 2][5:] + b"  "
            parts.append(eol.join(lines) + (eol if rng.random() < 0.9 else b""))
            if rng.random() < 0.2:
                parts.append(b"\n\n")
        raw = b"".join(parts)
        if not raw.endswith(b"\n") and b">" in raw[-3:]:
            raw += b"\n"
        _check(raw)


def test_count_file_uses_the_device_tokeniser(golden_dir, tmp_path):
    """kmer.count_file on plain, gzipped and tab-holding files (the last one falls back to the exact host tokeniser)."""
    from phamers_b200 import kmer, fileIO
    g = np.load(os.path.join(golden_dir, "fasta_golden.npz"))
    text = str(g["fasta_text"])
    plain, gz = tmp_path / "c.fasta", tmp_path / "c.fasta.gz"
    with open(plain, "w", newline="") as fh:
        fh.write(text)
    with gzip.open(gz, "wt", newline="") as fh:
        fh.write(text)
    for path in (plain, gz):
        ids, counts = kmer.count_file(str(path), 4)
        assert [str(x) for x in ids] == [str(x) for x in g["ids"]] and np.array_equal(counts, g["counts_k4"])
    headers, d_seq, d_off = fileIO.read_fasta_arrays_cuda(str(plain))
    h_headers, h_seq, h_off = fileIO.read_fasta_arrays(str(plain))
    assert headers == h_headers and np.array_equal(d_off.cpu().numpy(), h_off)
    assert np.array_equal(d_seq.cpu().numpy()[:int(h_off[-1])], h_seq)
    tricky = tmp_path / "t.fasta"
    with open(tricky, "w", newline="") as fh:
        fh.write(">a_ID_1 x\nAT\tGC\t\nGG  \r\n>b_ID_2\n\nAC GT\n")
    _, _, odd = _scan(open(tricky, "rb").read())
    assert odd
    ids, counts = kmer.count_file(str(tricky), 2)
    want = np.stack([po.count_string_np(s, 2) for s in ("AT\tGCGG", "ACGT")])
    assert list(ids) == ["1", "2"] and np.array_equal(counts, want)


def test_score_fasta_runs_on_the_device_tokeniser(golden_dir, tmp_path):
    from phamers_b200 import kmer, phamer, pipeline, references
    g = np.load(os.path.join(golden_dir, "fasta_golden.npz"))
    path = tmp_path / "c.fasta"
    with open(path, "w", newline="") as fh:
        fh.write(str(g["fasta_text"]))
    scorer = pipeline.ContigScorer()
    ids, scores = scorer.score_fasta(str(path))
    ids2, counts = kmer.count_file(str(path), 4)
    pos, neg = references.load_reference_features(equalize=True)
    with np.errstate(invalid="ignore"):
        want = phamer.score_points(kmer.normalize_counts(counts), pos, neg)
    assert list(ids) == list(ids2) and np.array_equal(scores, want, equal_nan=True)
    long_ids, long_scores = scorer.score_fasta(str(path), length_requirement=200)
    assert len(long_ids) == len(long_scores) <= len(ids)


def test_chunked_upload_of_a_file_larger_than_the_staging_buffers(tmp_path, monkeypatch):
    from phamers_b200 import fileIO
    rng = np.random.default_rng(3)
    path = tmp_path / "big.fasta"
    with open(path, "wb") as fh:
        for r in range(40):
            fh.write(b">rec_ID_%d x\n" % r)
            body = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=int(rng.integers(100, 9000))).tobytes()
            fh.write(b"\n".join(body[i:i + 70] for i in range(0, len(body), 70)) + b"\n")
    monkeypatch.setattr(fileIO, "UPLOAD_CHUNK", 4096 + 16)                 # many chunks, not a multiple of anything convenient
    headers, d_seq, d_off = fileIO.read_fasta_arrays_cuda(str(path))
    h_headers, h_seq, h_off = fileIO.read_fasta_arrays(str(path))
    assert headers == h_headers and np.array_equal(d_off.cpu().numpy(), h_off)
    assert np.array_equal(d_seq.cpu().numpy()[:int(h_off[-1])], h_seq)


def test_device_tokeniser_property_with_universal_newlines():
    """The same property on the device: random files over the bytes that matter ('>', line feeds, CR, blanks, letters; no tab, which
    the device reports instead of tokenising) against the oracle's restatement of the Bio.SeqIO parser over a text-mode handle.
    A lone CR ends a line as LF and CRLF do, so a '>' after it starts a record and the title stops at it."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=150, deadline=None)
    @given(st.text(alphabet=">\n\r ACGTNacgt|_1", min_size=0, max_size=300))
    def check(text):
        _check(text.encode("latin-1"))

    check()
