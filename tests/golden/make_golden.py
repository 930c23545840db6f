#!/usr/bin/env python
"""
Generates the committed golden vectors from the UNMODIFIED PhaMers reference
(scripts/{kmer,learning,phamer}.py imported through oracle/ref_loader.py):

    PHAMERS_REF=<PhaMers checkout>/scripts python tests/golden/make_golden.py

Outputs (all under tests/golden/):
  counting_golden.npz  adversarial + random sequences (laid end to end as seq_bytes + seq_offsets),
                       reference kmer.count_string counts for
                       k = 1..6, kmer.count dispatch shapes, kmer.normalize_counts
  fasta_golden.npz     a small multi-record FASTA text (wrapped lines, CRLF, lower case, N, IUPAC,
                       empty and shorter-than-k records) with reference kmer.count_file output
  scoring_golden.npz   query count vectors, reference phamer.score_points for knn / kmeans / combo
                       against the shipped (equalised) reference features, and the centroids the
                       reference's learning.kmeans + get_centroids produced (scikit-learn 1.9.0)
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_loader import load_reference  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SEED = 20260101


def random_contig(rng, length, gc=None, n_frac=0.0, lower_frac=0.0, iupac_frac=0.0):
    gc = rng.uniform(0.25, 0.75) if gc is None else gc
    p = np.array([(1 - gc) / 2, (1 - gc) / 2, gc / 2, gc / 2])          # A T G C
    seq = rng.choice(np.frombuffer(b"ATGC", dtype=np.uint8), size=length, p=p)
    for frac, alphabet in ((n_frac, b"N"), (lower_frac, b"atgcn"), (iupac_frac, b"RYKMSWBDHVU-*")):
        if frac <= 0 or length == 0:
            continue
        n_runs = max(1, int(length * frac / 8))
        for _ in range(n_runs):
            start = int(rng.integers(0, length))
            run = int(rng.integers(1, 16))
            seq[start:start + run] = rng.choice(np.frombuffer(alphabet, dtype=np.uint8),
                                                size=len(seq[start:start + run]))
    return seq.tobytes().decode("ascii")


def adversarial_sequences(rng):
    seqs = [
        "", "A", "AT", "ATG", "ATGC", "AAAT", "AAAAAAAA", "ATGCATGCATGC",
        "AATTGGCCNAa", "NNNNNNNNNN", "atgcatgcatgc", "ATGCNATGC", "ATGNCATG",
        "ACGT" * 50, "A" * 300, "AT" * 150, "GC" * 151, "ATGC" * 3 + "N" + "ATGC" * 3,
        "N" + "ATGCATGCAT", "ATGCATGCAT" + "N", "ATGCA-TGCAT", "ATGC*ATGC", "ATGC ATGC",
        "ATGCUATGC", "ATGC\tATGC", "ATGC0123ATGC", "RYKMSWBDHV" * 3, "ATGCX" * 40, "XATGC" * 40,
    ]
    for length in (5, 6, 7, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513,
                   1000, 1023, 1024, 1025, 4099):
        seqs.append(random_contig(rng, length))
    for length in (100, 777, 2048, 5000):
        seqs.append(random_contig(rng, length, n_frac=0.05, lower_frac=0.05, iupac_frac=0.03))
    seqs.append(random_contig(rng, 3000, gc=0.05))
    seqs.append(random_contig(rng, 3000, gc=0.95))
    return seqs


def make_counting(kmer):
    rng = np.random.default_rng(SEED)
    seqs = adversarial_sequences(rng)
    blob = "".join(seqs).encode("ascii")
    offsets = np.concatenate(([0], np.cumsum([len(s) for s in seqs]))).astype(np.int64)
    out = {"seq_bytes": np.frombuffer(blob, dtype=np.uint8), "seq_offsets": offsets}
    for k in range(1, 7):
        counts = np.stack([kmer.count_string(s, k) for s in seqs])
        assert counts.dtype == np.int64
        out["counts_k%d" % k] = counts
    # known-answer anchor from the reference docstring (kmer.py:90-91)
    assert kmer.get_kmer_index("AAAT", "ATGC") == 1
    assert kmer.count_string("AAAT", 4)[1] == 1
    # dispatch conventions (kmer.py:93-111)
    out["dispatch_list1"] = kmer.count([seqs[12]], 4)                   # 1-D
    out["dispatch_list3"] = kmer.count(seqs[8:11], 4)                   # [3, 256]
    out["dispatch_str_norm"] = kmer.count(seqs[13], 4, normalize=True)  # float64 1-D
    assert kmer.count(12345, 4) is None
    # normalize_counts (kmer.py:209-221), including an all-zero row -> NaN
    with np.errstate(invalid="ignore", divide="ignore"):
        out["normalized_k4"] = kmer.normalize_counts(out["counts_k4"])
    np.savez_compressed(os.path.join(HERE, "counting_golden.npz"), **out)
    print("counting_golden: %d sequences" % len(seqs))


def make_fasta(kmer):
    rng = np.random.default_rng(SEED + 1)
    records = []
    lengths = [0, 3, 59, 60, 61, 120, 121, 500, 1234, 5000, 7]
    for i, length in enumerate(lengths):
        seq = random_contig(rng, length, n_frac=0.03 if i % 2 else 0.0, lower_frac=0.03 if i % 3 == 0 else 0.0)
        records.append((">SuperContig_%d_length_%d_ID_%d some description" % (i, length, 1000 + i), seq))
    lines = []
    for i, (header, seq) in enumerate(records):
        eol = "\r\n" if i % 4 == 1 else "\n"
        width = (60, 70, 80, 61)[i % 4]
        lines.append(header + eol)
        for p in range(0, len(seq), width):
            tail = "  " if (i == 5 and p == 0) else ""
            lines.append(seq[p:p + width] + tail + eol)
        if i == 7:
            lines.append(eol)                       # blank line inside the file
    text = "".join(lines)
    out = {"fasta_text": np.array(text)}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "contigs.fasta")
        with open(path, "w", newline="") as fh:
            fh.write(text)
        for k in (4, 5, 6):
            ids, counts = kmer.count_file(path, k)
            out["ids"] = np.array([str(x) for x in ids])
            out["counts_k%d" % k] = counts
        _, freq = kmer.count_file(path, 4, normalize=True)
        out["freq_k4"] = freq
        missing_ids, missing_counts = kmer.count_file(os.path.join(tmp, "does_not_exist.fasta"), 4)
        assert missing_ids is None and missing_counts is None
    np.savez_compressed(os.path.join(HERE, "fasta_golden.npz"), **out)
    print("fasta_golden: %d records, %d bytes" % (len(records), len(text)))


def make_scoring(kmer, learning, phamer):
    rng = np.random.default_rng(SEED + 2)
    ref = np.load(os.path.join(ROOT, "phamers_b200", "data", "reference_features.npz"))
    pos_counts = ref["positive_counts"].astype(np.int64)
    neg_counts = ref["negative_counts"].astype(np.int64)
    n_ref = min(len(pos_counts), len(neg_counts))            # phamer.py:159-175 (--equalize_reference)
    pos_counts, neg_counts = pos_counts[:n_ref], neg_counts[:n_ref]
    positive = kmer.normalize_counts(pos_counts)
    negative = kmer.normalize_counts(neg_counts)

    queries = []
    # (a) random synthetic contigs counted by the reference itself
    for _ in range(120):
        length = int(np.clip(np.round(np.exp(rng.normal(np.log(10000), 1.0))), 1000, 100000))
        length = min(length, 20000)
        queries.append(kmer.count_string(random_contig(rng, length), 4))
    # (b) reference-like queries: multinomial resamples of shipped reference rows (near-neighbour ties)
    both = np.vstack((pos_counts, neg_counts))
    for _ in range(260):
        row = both[int(rng.integers(0, both.shape[0]))].astype(np.float64)
        draws = int(rng.choice([2000, 20000, 200000]))
        queries.append(rng.multinomial(draws, row / row.sum()))
    # (c) exact copies of reference rows (distance 0 to one neighbour)
    for j in (0, 5, n_ref - 1):
        queries.append(pos_counts[j].copy())
        queries.append(neg_counts[j].copy())
    query_counts = np.stack(queries).astype(np.int64)
    points = kmer.normalize_counts(query_counts)

    out = {"query_counts": query_counts, "n_ref": np.int64(n_ref)}
    for method in ("knn", "kmeans", "combo"):
        out["scores_" + method] = np.asarray(phamer.score_points(points, positive, negative, method=method),
                                             dtype=np.float64)
    again = np.asarray(phamer.score_points(points, positive, negative), dtype=np.float64)
    assert np.array_equal(again, out["scores_combo"])
    out["centroids_pos"] = learning.get_centroids(positive, learning.kmeans(positive, 86))
    out["centroids_neg"] = learning.get_centroids(negative, learning.kmeans(negative, 86))
    import sklearn
    out["sklearn_version"] = np.array(sklearn.__version__)
    np.savez_compressed(os.path.join(HERE, "scoring_golden.npz"), **out)
    knn = out["scores_knn"]
    print("scoring_golden: %d queries, knn +1: %d, -1: %d" % (len(knn), (knn > 0).sum(), (knn < 0).sum()))


def main():
    kmer, learning, phamer = load_reference()
    make_counting(kmer)
    make_fasta(kmer)
    make_scoring(kmer, learning, phamer)


if __name__ == "__main__":
    main()
