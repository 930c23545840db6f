"""
TEST INFRASTRUCTURE ONLY -- CPU restatement ("port") of the PhaMers hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package (phamers_b200/) never does; it fails loudly when its
CUDA library is missing instead of falling back to anything in here.

Parity status: PINNED.  Every function below is checked in tests/test_oracle.py against
(a) the unmodified reference modules imported through oracle/ref_loader.py when /root/reference
is present (build container), and (b) the committed golden vectors in tests/golden/ that
tests/golden/make_golden.py produced from those same reference modules.

Each function cites the reference lines it restates (paths relative to /root/reference).
Third-party arithmetic the reference delegates to scikit-learn (unpinned in requirements.txt:4;
1.9.0 in this image) is delegated to the same scikit-learn here, at the same call sites:
KNeighborsClassifier (scripts/learning.py:127-128) and KMeans (scripts/learning.py:138).
"""
import gzip
import re

import numpy as np

DNA = "ATGC"          # scripts/kmer.py:28 -- bin order A=0 T=1 G=2 C=3, first base most significant
KMEANS_SEED = 10      # scripts/learning.py:21
K_CLUSTERS = 86       # scripts/phamer.py:78
K_NEIGHBORS = 3       # scripts/phamer.py:79


# --------------------------------------------------------------------------------------
# Stage 1: k-mer counting
# --------------------------------------------------------------------------------------
def sequence_to_integers(sequence, symbols=DNA):
    """scripts/kmer.py:183-196.  Every character outside `symbols` becomes '-', then each symbol
    is replaced by its decimal index.  Case-sensitive."""
    for stranger in set(sequence) - set(symbols):
        sequence = sequence.replace(stranger, "-")
    for digit, symbol in enumerate(symbols):
        sequence = sequence.replace(symbol, str(digit))
    return sequence


def count_string(sequence, kmer_length, symbols=DNA, normalize=False):
    """scripts/kmer.py:32-79, branch len(symbols) < 10 (:42-50): slide a window of k digits,
    skip windows holding a '-', parse the window in base len(symbols), bump that bin.
    Sequences shorter than k give all zeros.  normalize divides by the sum only if it is > 0 (:77)."""
    digits = sequence_to_integers(sequence, symbols)
    radix = len(symbols)
    hist = np.zeros(radix ** kmer_length, dtype=(float if normalize else int))
    for start in range(len(digits) - kmer_length + 1):
        window = digits[start:start + kmer_length]
        if "-" in window:
            continue
        hist[int(window, radix)] += 1
    if normalize and hist.sum() > 0:
        hist = normalize_counts(hist)
    return hist


_LUT = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(DNA):
    _LUT[ord(_c)] = _i


def count_bytes_np(seq_bytes, kmer_length):
    """Vectorised restatement of scripts/kmer.py:42-50 for DNA on a uint8 array: same bins as
    count_string but in O(L) numpy operations (used for the larger parity cases)."""
    k = kmer_length
    nbins = 4 ** k
    codes = _LUT[np.asarray(seq_bytes, dtype=np.uint8)]
    n_win = codes.shape[0] - k + 1
    if n_win <= 0:
        return np.zeros(nbins, dtype=np.int64)
    idx = np.zeros(n_win, dtype=np.int64)
    bad = np.zeros(n_win, dtype=bool)
    for j in range(k):
        col = codes[j:j + n_win]
        bad |= col == 255
        idx = idx * 4 + (col & 3)
    return np.bincount(idx[~bad], minlength=nbins).astype(np.int64)


def count_string_np(sequence, kmer_length):
    return count_bytes_np(np.frombuffer(sequence.encode("latin-1"), dtype=np.uint8), kmer_length)


def count(data, kmer_length, symbols=DNA, normalize=False, fast=False):
    """scripts/kmer.py:82-111.  list of 1 -> 1-D; longer list -> [n, bins]; str -> 1-D; else None."""
    single = (lambda s: _count_fast(s, kmer_length, normalize)) if (fast and symbols == DNA) else \
             (lambda s: count_string(s, kmer_length, symbols=symbols, normalize=normalize))
    if isinstance(data, list):
        if len(data) == 1:
            return count(data[0], kmer_length, symbols=symbols, normalize=normalize, fast=fast)
        out = np.zeros((len(data), len(symbols) ** kmer_length), dtype=(float if normalize else int))
        for row, sequence in enumerate(data):
            out[row, :] = single(sequence)
        return out
    if isinstance(data, str):
        return single(data)
    return None


def _count_fast(sequence, kmer_length, normalize):
    hist = count_string_np(sequence, kmer_length)
    if normalize:
        hist = hist.astype(float)
        if hist.sum() > 0:
            hist = normalize_counts(hist)
    return hist


def normalize_counts(counts):
    """scripts/kmer.py:209-221.  float64 copy, each row divided by its own sum; a zero row gives
    0/0 = NaN (no guard here, unlike count_string's :77)."""
    counts = np.asarray(counts).astype(float)
    with np.errstate(invalid="ignore", divide="ignore"):
        if counts.ndim == 1:
            return counts / np.sum(counts)
        for row in range(counts.shape[0]):
            counts[row, :] /= np.sum(counts[row, :])
    return counts


# ---- FASTA tokenisation (Biopython SimpleFastaParser semantics; scripts/kmer.py:135) ----
def parse_fasta_text(text):
    """Yields (title, sequence).  Lines end as a text-mode file (universal newlines) ends them:
    at '\\r\\n', a lone '\\r' or '\\n'.  A record starts at a line starting with '>'; the sequence is
    every later line rstripped and joined with blanks and CR removed.  Inputs are ASCII: under
    UTF-8, str.rstrip() would also strip non-ASCII whitespace, which is not restated here."""
    title, chunks = None, []
    for line in re.split("\r\n|\r|\n", text):
        if line.startswith(">"):
            if title is not None:
                yield title, "".join(chunks).replace(" ", "").replace("\r", "")
            title, chunks = line[1:].rstrip(), []
        elif title is not None:
            chunks.append(line.rstrip())
    if title is not None:
        yield title, "".join(chunks).replace(" ", "").replace("\r", "")


def get_id(header):
    """scripts/id_parser.py:89-100 for '_ID_' contig headers (:18-29); other header families are
    outside the synthetic workloads and fall back to the first blank-separated token."""
    if "_ID_" in header:
        parts = header.strip().replace(">", "").split("_")
        return parts[1 + parts.index("ID")].replace("-circular", "")
    return header.split(" ")[0]


def read_fasta(path):
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "rt") as fh:
        text = fh.read()
    ids, seqs = [], []
    for title, seq in parse_fasta_text(text):
        token = title.split(None, 1)[0] if title.split() else ""
        ids.append(get_id(token))
        seqs.append(seq)
    return np.array(ids), seqs


def count_file(input_file, kmer_length, symbols=DNA, normalize=False, fast=False):
    """scripts/kmer.py:114-140.  (ids, counts[n, bins]); (None, None) when the file cannot be read."""
    try:
        ids, seqs = read_fasta(input_file)
    except IOError:
        return None, None
    out = np.zeros((len(ids), len(symbols) ** kmer_length), dtype=(float if normalize else int))
    for row, seq in enumerate(seqs):
        out[row, :] = count(seq, kmer_length, symbols=symbols, normalize=normalize, fast=fast)
    return ids, out


def count_directory(directory, kmer_length, identifier="fna", symbols=DNA, sum_file=True, fast=True):
    """scripts/kmer.py:143-180 (live behaviour, sample = 0): the files of `directory` whose basename contains `identifier`, in
    os.listdir order; with sum_file one row per file -- the id of its first record (:171) and the sum of its records' counts
    (:172) -- as float64 (:159); files that cannot be read or hold no window are dropped (:165-168).  (sum_file = False leaves
    file_id unset in the reference, :170-175, and is not restated.)"""
    import os
    selected = [os.path.join(directory, f) for f in os.listdir(directory) if identifier in os.path.basename(f)]
    ids, rows = [], []
    for path in selected:
        file_ids, file_counts = count_file(path, kmer_length, symbols=symbols, fast=fast)
        if file_ids is None or len(file_ids) == 0 or np.sum(file_counts) == 0:
            continue
        ids.append(file_ids[0])
        rows.append(np.sum(file_counts, axis=0) if file_counts.ndim == 2 else file_counts)
    return ids, (np.array(rows, dtype=float) if rows else np.zeros((0, len(symbols) ** kmer_length)))


# ---- canonical (reverse-complement) folding: north-star extension, no reference code ----
def revcomp_index(j, k):
    """Bin of the reverse complement of bin j in ATGC order (A<->T is 0<->1, G<->C is 2<->3)."""
    comp = (1, 0, 3, 2)
    out = 0
    for _ in range(k):
        out = out * 4 + comp[j & 3]
        j >>= 2
    return out


def canonical_map(k):
    """(rep[4^k], compact[4^k], n_canon): rep[j] = min(j, rc(j)); compact[j] = rank of rep[j] among
    the sorted distinct representatives.  136 / 512 / 2080 classes for k = 4 / 5 / 6."""
    n = 4 ** k
    rep = np.array([min(j, revcomp_index(j, k)) for j in range(n)], dtype=np.int64)
    uniq = np.unique(rep)
    compact = np.searchsorted(uniq, rep)
    return rep, compact, int(uniq.shape[0])


def canonical_fold(counts, k, compact=True):
    """SURVEY.md section 8(c): canon[min(j, rc(j))] += count[j]; either compacted to the sorted
    representatives or kept as a 4^k vector with the mass on the representative bins."""
    counts = np.asarray(counts)
    rep, comp, n_canon = canonical_map(k)
    two_d = counts.reshape(-1, counts.shape[-1])
    width = n_canon if compact else 4 ** k
    out = np.zeros((two_d.shape[0], width), dtype=counts.dtype)
    np.add.at(out, (slice(None), comp if compact else rep), two_d)
    return out.reshape(counts.shape[:-1] + (width,))


# --------------------------------------------------------------------------------------
# Stage 3: scoring
# --------------------------------------------------------------------------------------
def distances(vector, data):
    """scripts/learning.py:47-56: Euclidean norms of (vector - row) by direct difference."""
    vector = np.asarray(vector)
    if vector.ndim == 1:
        vector = vector[None, :]
    return np.linalg.norm(np.repeat(vector, data.shape[0], axis=0) - data, axis=1)


def closest_to(point, picks):
    """scripts/learning.py:59-66: the row of `picks` nearest to `point` (first minimum on ties)."""
    return picks[np.argmin(distances(point, picks))]


def get_centroids(data, assignment):
    """scripts/learning.py:69-81: mean of the members of every cluster id, in sorted id order,
    ignoring the noise label -1."""
    labels = sorted(set(assignment) - {-1})
    return np.array([np.mean(data[assignment == c], axis=0) for c in labels])


def kmeans_assign(data, k):
    """scripts/learning.py:131-146: KMeans(n_clusters=k, random_state=10).fit(data).labels_ with the
    installed scikit-learn's defaults."""
    from sklearn.cluster import KMeans
    return np.asarray(KMeans(n_clusters=k, random_state=KMEANS_SEED).fit(data).labels_)


def reference_centroids(positive, negative, k_clusters=K_CLUSTERS):
    """scripts/phamer.py:245-248."""
    pos = get_centroids(positive, kmeans_assign(positive, k_clusters))
    neg = get_centroids(negative, kmeans_assign(negative, k_clusters))
    return pos, neg


def knn_scores(queries, ref_data, ref_labels, k=K_NEIGHBORS):
    """scripts/learning.py:118-128: 2 * (KNeighborsClassifier(k).fit(refs, labels).predict(q) - 0.5)."""
    from sklearn.neighbors import KNeighborsClassifier
    model = KNeighborsClassifier(n_neighbors=k).fit(ref_data, ref_labels)
    return 2 * (model.predict(queries) - 0.5)


def knn_scores_exact(queries, ref_data, ref_labels, k=K_NEIGHBORS):
    """Same vote from direct-difference float64 distances (no GEMM trick), stable ties by index.
    Cross-check for knn_scores; identical whenever no two candidate distances tie within rounding."""
    out = np.zeros(queries.shape[0])
    for i in range(queries.shape[0]):
        d = np.sum((ref_data - queries[i]) ** 2, axis=1)
        nearest = np.argsort(d, kind="stable")[:k]
        out[i] = 1.0 if 2 * np.sum(ref_labels[nearest]) > k else -1.0
    return out


def proximity_metric(point, nearest_positive, nearest_negative):
    """scripts/phamer.py:198-210: tanh((e_neg - e_pos) / (e_pos + e_neg))."""
    e_neg = np.linalg.norm(point - nearest_negative)
    e_pos = np.linalg.norm(point - nearest_positive)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.tanh((e_neg - e_pos) / (e_pos + e_neg))


def kmeans_scores(points, positive, negative, k_clusters=K_CLUSTERS, centroids=None):
    """scripts/phamer.py:240-256.  `centroids` = (pos, neg) skips the (reference-only) clustering."""
    pos_c, neg_c = centroids if centroids is not None else reference_centroids(positive, negative, k_clusters)
    out = np.zeros(points.shape[0])
    for i in range(points.shape[0]):
        out[i] = proximity_metric(points[i], closest_to(points[i], pos_c), closest_to(points[i], neg_c))
    return out


def score_points(points, positive, negative, method=None, centroids=None,
                 k_clusters=K_CLUSTERS, k_neighbors=K_NEIGHBORS):
    """scripts/phamer.py:451-468 + :177-195 + :303-313.  method in {'knn','kmeans','combo'} (default
    'combo' = knn + kmeans, range +-1.7616)."""
    method = method or "combo"
    train = np.vstack((positive, negative))                                         # phamer.py:186
    labels = np.append(np.ones(positive.shape[0]), np.zeros(negative.shape[0]))    # phamer.py:187
    if method == "knn":
        return np.array(knn_scores(points, train, labels, k=k_neighbors))
    if method == "kmeans":
        return np.array(kmeans_scores(points, positive, negative, k_clusters, centroids))
    if method == "combo":
        return np.array(knn_scores(points, train, labels, k=k_neighbors)) + \
               np.array(kmeans_scores(points, positive, negative, k_clusters, centroids))
    raise KeyError(method)


def equalize_reference_data(positive, negative):
    """scripts/phamer.py:159-175: truncate both sets to the first min(nP, nN) rows."""
    n = min(positive.shape[0], negative.shape[0])
    return positive[:n], negative[:n]


# --------------------------------------------------------------------------------------
# Feature / score CSV formats (scripts/fileIO.py:134-181, 241-272)
# --------------------------------------------------------------------------------------
def read_feature_file(feature_file, normalize=False):
    """scripts/fileIO.py:134-166: '#' comment lines, then id,c0,...; ids as str, counts as int."""
    data = np.loadtxt(feature_file, delimiter=",", dtype=str)
    if data.ndim == 1:
        data = np.array([data])
    ids = np.array(list(data[:, 0]))
    features = data[:, 1:].astype(int)
    if normalize:
        features = normalize_counts(features)
    return ids, features
