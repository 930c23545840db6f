"""Host-side formats either side of the path (FASTA tokenisation, feature CSV, score CSV, id parsing).  CPU only."""
import gzip
import io
import os

import numpy as np
import pytest

from oracle import phamers_oracle as po
from phamers_b200 import fileIO, kmer


@pytest.fixture(scope="module")
def fasta(golden_dir):
    return np.load(os.path.join(golden_dir, "fasta_golden.npz"))


def test_fasta_split_matches_reference_tokenisation(fasta, tmp_path):
    text = str(fasta["fasta_text"])
    path = tmp_path / "contigs.fasta"
    with open(path, "w", newline="") as fh:
        fh.write(text)
    want = list(po.parse_fasta_text(text))
    headers, seq, off = fileIO.read_fasta_arrays(str(path))
    blob = seq.tobytes().decode("latin-1")
    assert len(headers) == len(want)
    for i, (title, s) in enumerate(want):
        assert headers[i] == title.split(None, 1)[0]
        assert blob[off[i]:off[i + 1]] == s
    ids = fileIO.get_fasta_ids(str(path))
    assert [str(x) for x in ids] == [str(x) for x in fasta["ids"]]
    # gzip + the slow exact path (a tab inside a line is kept, trailing tab is stripped)
    tricky = ">a_ID_1 x\nAT\tGC\t\nGG  \r\n>b_ID_2\n\nAC GT\n"
    gz = tmp_path / "t.fasta.gz"
    with gzip.open(gz, "wt", newline="") as fh:
        fh.write(tricky)
    headers, seq, off = fileIO.read_fasta_arrays(str(gz))
    got = [seq.tobytes().decode()[off[i]:off[i + 1]] for i in range(len(headers))]
    assert got == [s for _, s in po.parse_fasta_text(tricky)] == ["AT\tGCGG", "ACGT"]
    with pytest.raises(IOError):
        fileIO.read_fasta_arrays(str(tmp_path / "missing.fasta"))
    # degenerate files
    for raw in (b"", b"\n", b">", b">a", b">a\n", b"ACGT", b">a\nACGT", b"x\n>a b\n\nAC\n>\n>c\nG"):
        ids, seq, off = fileIO.split_fasta_bytes(raw)
        want = list(po.parse_fasta_text(raw.decode()))
        assert ids == [(t.split(None, 1) or [""])[0] for t, _ in want]
        assert [seq.tobytes().decode()[off[i]:off[i + 1]] for i in range(len(ids))] == [s for _, s in want]
    assert fileIO.split_fasta_bytes(b"") [0] == [] and fileIO.split_fasta_bytes(b"no header\nACGT\n")[0] == []


def test_get_id_families():
    assert fileIO.get_id("SuperContig_12_length_500_ID_777-circular") == "777"
    assert fileIO.get_id("gi|123|gb|AY848686.1|") == "AY848686.1"
    assert fileIO.get_id("CP000084.1 Candidatus Pelagibacter") == "CP000084.1"


def test_feature_csv_round_trip(tmp_path):
    counts = np.arange(2 * 256).reshape(2, 256)
    path = str(tmp_path / "f.csv")
    fileIO.save_counts(counts, ["c1", "c2"], path)
    lines = open(path).read().split("\n")
    assert lines[0] == "# K-mer count file" and lines[1].startswith("c1,0,1,2,")
    ids, back = fileIO.read_feature_file(path)
    assert list(ids) == ["c1", "c2"] and np.array_equal(back, counts)
    ids2, back2 = po.read_feature_file(path)          # the reference's np.loadtxt reader parses our writer's output
    assert list(ids2) == ["c1", "c2"] and np.array_equal(back2, counts)


def test_score_csv_round_trip(tmp_path):
    path = str(tmp_path / "phamer_scores.csv")
    scores = np.array([1.026236041, -0.5, 0.0])
    fileIO.save_phamer_scores(np.array(["7", "8", "9"]), scores, path)
    text = open(path).read().split("\n")
    assert text[0] == "# PhaMers score file" and text[1] == "7, 1.026236041"
    back = fileIO.read_phamer_output(path)
    assert back == {"7": 1.026236041, "8": -0.5, "9": 0.0}


def test_host_helpers():
    assert kmer.kmers(2) == ["AA", "AT", "AG", "AC", "TA", "TT", "TG", "TC", "GA", "GT", "GG", "GC", "CA", "CT", "CG", "CC"]
    assert kmer.get_kmer_index("AAAT", "ATGC") == 1          # scripts/kmer.py:90-91
    assert kmer.sequence_to_integers("ATGCNa", "ATGC") == "0123--"
    assert kmer.extend_mers(["A", "T"], 1, "AT") == ["AA", "AT", "TA", "TT"]


def test_host_tokeniser_property():
    """Random files over the bytes that matter to the FASTA tokeniser ('>', line feeds, CR, blanks, tabs, VT, the separators 0x1C
    and 0x1F that str.rstrip() strips, letters): the host tokeniser agrees with the oracle's line-by-line restatement of the
    Bio.SeqIO parser on every one of them."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=400, deadline=None)
    @given(st.text(alphabet=">\n\r \t\x0b\x1c\x1fACGTNacgt|_1", min_size=0, max_size=200))
    def check(text):
        raw = text.encode("latin-1")
        ids, seq, off = fileIO.split_fasta_bytes(raw)
        want = list(po.parse_fasta_text(text))
        assert ids == [(t.split(None, 1) or [""])[0] for t, _ in want]
        got = [seq.tobytes().decode("latin-1")[off[i]:off[i + 1]] for i in range(len(ids))]
        assert got == [s for _, s in want]

    check()


def test_oracle_reads_lines_as_a_text_mode_file():
    """parse_fasta_text splits lines as the reference's text-mode handle does (universal newlines: CRLF, a lone CR and LF each end
    a line), so it agrees with Biopython's SimpleFastaParser run over such a handle, restated here on the handle's own lines."""
    rng = np.random.default_rng(5)
    alphabet = np.frombuffer(b">>\n\n\r\r \t\x0b\x0c\x1c\x1fACGTNacgt_1", dtype=np.uint8)
    cases = [b">a_ID_1 desc\rACGTAC\r>b_ID_2\nAC\x1c\nGT\n", b"\r\r\n>x\r\r\nA\rC\r\n\r>y", b">a\r", b">a\r\n\r\nGG \t\r"]
    cases += [rng.choice(alphabet, size=int(rng.integers(0, 120))).tobytes() for _ in range(300)]
    for raw in cases:
        title, chunks, want = None, [], []
        for line in io.TextIOWrapper(io.BytesIO(raw), encoding="latin-1", newline=None):
            if line.startswith(">"):
                if title is not None:
                    want.append((title, "".join(chunks).replace(" ", "").replace("\r", "")))
                title, chunks = line[1:].rstrip(), []
            elif title is not None:
                chunks.append(line.rstrip())
        if title is not None:
            want.append((title, "".join(chunks).replace(" ", "").replace("\r", "")))
        assert list(po.parse_fasta_text(raw.decode("latin-1"))) == want, raw


def test_lone_carriage_returns_and_separators_at_line_ends(tmp_path):
    """A lone CR ends a line (a classic-Mac file holds several records, not one), and 0x1C-0x1F at a line end are stripped as
    str.rstrip() strips them: the host tokeniser, the file readers and the oracle agree."""
    raw = b">a_ID_1 desc\rACGTAC\r>b_ID_2\nAC\x1c\nGT\n"
    want = [("a_ID_1 desc", "ACGTAC"), ("b_ID_2", "ACGT")]
    assert list(po.parse_fasta_text(raw.decode("latin-1"))) == want
    ids, seq, off = fileIO.split_fasta_bytes(raw)
    assert ids == ["a_ID_1", "b_ID_2"] and [seq.tobytes()[off[i]:off[i + 1]] for i in range(2)] == [b"ACGTAC", b"ACGT"]
    path = tmp_path / "mac.fasta"
    path.write_bytes(raw)
    ids, seqs = fileIO.read_fasta(str(path))
    ref_ids, ref_seqs = po.read_fasta(str(path))
    assert list(ids) == list(ref_ids) == ["1", "2"] and seqs == ref_seqs == ["ACGTAC", "ACGT"]
    for raw, want in ((b">a\rAC\t\rGT\r\n>b\r\r\nT T\x1f\r", [b"ACGT", b"TT"]),      # tab before a lone CR: exact path
                      (b">a\r\r\nAC\rGT\x0b\n\r>b\nA\x1dC\n", [b"ACGT", b"A\x1dC"]),   # a separator inside a line is kept
                      (b">a\rAC\rG\rT\r>b\rCC\r", [b"ACGT", b"CC"])):                    # fast path, CR only
        ids, seq, off = fileIO.split_fasta_bytes(raw)
        assert [seq.tobytes()[off[i]:off[i + 1]] for i in range(len(ids))] == want
        assert [s.encode("latin-1") for _, s in po.parse_fasta_text(raw.decode("latin-1"))] == want
