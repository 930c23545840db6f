"""
The on-disk formats either side of the hot path, mirroring the reference's scripts/fileIO.py and the part of
scripts/id_parser.py the path touches:

    FASTA in        read_fasta :28, get_fasta_ids :62 (Bio.SeqIO tokenisation) + id_parser.get_id :89
    feature CSV     read_feature_file :134, save_counts :169  ('#' header lines, then id,c0,c1,...)
    score CSV       save_phamer_scores :241, read_phamer_output :256  ('# ' header, then 'id, score')
    neighbour CSV   save_phamer_neighbors, read_phamer_neighbors  ('# ' header, then per contig its nearest references and clusters)
    window CSV      save_phamer_windows, read_phamer_windows  ('# ' header, then 'id, start, end, score' per window)
    region CSV      save_phamer_regions, read_phamer_regions  ('# ' header, then 'id, start, end, windows, mean_score, max_score')
    BED in          read_bed  ('chrom start end [name ...]' per line)
    span CSV        save_phamer_spans, read_phamer_spans  ('# ' header, then 'id, start, end, name, score' and the neighbour columns)

Host-side only (bytes and text); no arithmetic happens here.
"""
import gzip
import io
import os

import numpy as np


# ----------------------------------------------------------------------------------------------------------
# ids (scripts/id_parser.py)
# ----------------------------------------------------------------------------------------------------------
def _represents_float(text):
    try:
        float(text)
        return True
    except ValueError:
        return False


def _is_genbank_id(token):
    """scripts/id_parser.py:79-86."""
    return len(token) >= 2 and not _represents_float(token) and token[-2] == "."


def get_id(header):
    """scripts/id_parser.py:89-100: '_ID_' contig headers -> the token after 'ID' (minus '-circular'); headers with
    four '|' -> field 3 (phage GenBank id); anything else -> the leading GenBank-style token."""
    if "_ID_" in header:
        parts = header.strip().replace(">", "").split("_")
        return parts[1 + parts.index("ID")].replace("-circular", "")
    if header.count("|") == 4:
        return header.split("|")[3].replace(">", "")
    token = header.split(" ")[0]
    if _is_genbank_id(token):
        return token
    fields = header.split("\t")
    if len(fields) > 1 and _is_genbank_id(fields[1].replace(">", "")):
        return fields[1].replace(">", "")
    return None


# ----------------------------------------------------------------------------------------------------------
# FASTA
# ----------------------------------------------------------------------------------------------------------
_TRAILING = b" \t\n\r\x0b\x0c\x1c\x1d\x1e\x1f"      # str.isspace over ASCII: what str.rstrip() strips at a line end


def _open_bytes(path):
    if path.endswith(".gz"):
        with gzip.open(path, "rb") as fh:
            return fh.read()
    with open(path, "rb") as fh:
        return fh.read()


def split_fasta_bytes(raw):
    """FASTA bytes -> (record ids [first blank-separated token of each title], uint8 array of all sequence bytes end
    to end, int64 offsets[n+1]).  Tokenisation follows Bio.SeqIO's FASTA parser over a text-mode handle as the reference
    uses it (scripts/kmer.py:135): a line ends at '\n', '\r' or '\r\n' (universal newlines); a record starts at a line
    beginning with '>', its sequence is every following line right-stripped and joined, with blanks removed -- so k-mers
    span line breaks but never records.  Text before the first '>' is ignored."""
    data = np.frombuffer(raw, dtype=np.uint8)
    n = data.shape[0]
    if n == 0:
        return [], np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.int64)
    newline = np.flatnonzero((data == 10) | (data == 13))          # line terminators: LF and CR
    line_start = np.concatenate(([0], newline + 1))
    line_start = line_start[line_start < n]
    header_start = line_start[data[line_start] == ord(">")]
    if header_start.shape[0] == 0:
        return [], np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.int64)
    # end of each header line (position of its '\n' or '\r', or n)
    idx = np.searchsorted(newline, header_start)
    if newline.shape[0]:
        header_end = np.where(idx < newline.shape[0], newline[np.minimum(idx, newline.shape[0] - 1)], n)
    else:
        header_end = np.full_like(header_start, n)                    # a lone header line without a line feed
    body_start = np.minimum(header_end + 1, n)
    body_end = np.concatenate((header_start[1:], [n]))

    ids = []
    for hs, he in zip(header_start, header_end):
        title = raw[hs + 1:he].decode("latin-1").rstrip()
        tokens = title.split(None, 1)
        ids.append(tokens[0] if tokens else "")

    if any(c in raw for c in (b"\t", b"\x0b", b"\x0c", b"\x1c", b"\x1d", b"\x1e", b"\x1f")):
        # rare: tab / VT / FF / 0x1C-0x1F are stripped only at line ends -- exact line-by-line path
        pieces, lengths = [], []
        for bs, be in zip(body_start, body_end):
            body = b"".join(line.rstrip(_TRAILING) for line in raw[bs:be].splitlines())
            body = body.replace(b" ", b"")
            pieces.append(body)
            lengths.append(len(body))
        seq = np.frombuffer(b"".join(pieces), dtype=np.uint8)
        offsets = np.concatenate(([0], np.cumsum(lengths))).astype(np.int64)
        return ids, seq, offsets

    keep = (data != 10) & (data != 13) & (data != 32)
    in_body = np.zeros(n + 1, dtype=np.int32)
    np.add.at(in_body, body_start, 1)
    np.add.at(in_body, body_end, -1)
    keep &= np.cumsum(in_body[:n]) > 0
    kept_before = np.concatenate(([0], np.cumsum(keep)))
    offsets = np.concatenate((kept_before[body_start], [kept_before[n]])).astype(np.int64)
    # bodies are disjoint and ordered, so offsets[i+1] == kept_before[body_end[i]]
    return ids, data[keep], offsets


UPLOAD_CHUNK = 256 << 20             # bytes per pinned staging buffer of the file upload (two buffers alternate)


def _upload(buf, n):
    """File bytes (an mmap, or the bytes of a decompressed .gz) -> CUDA uint8 tensor padded to 16 bytes.  The copy page cache ->
    pinned staging buffer of chunk i + 1 runs on the host while chunk i crosses PCIe (scripts/kmer.py:131-134 reads the whole
    file through Python objects instead)."""
    import torch
    d_raw = torch.empty(((n + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    chunk = min(UPLOAD_CHUNK, max(n, 1))
    stage = [torch.empty((chunk,), dtype=torch.uint8, pin_memory=True) for _ in range(2 if n > chunk else 1)]
    done = [None] * len(stage)
    src = np.frombuffer(buf, dtype=np.uint8, count=n)
    for i, lo in enumerate(range(0, n, chunk)):
        j = i % len(stage)
        if done[j] is not None:
            done[j].synchronize()                                     # the staging buffer's previous upload has left it
        m = min(chunk, n - lo)
        stage[j].numpy()[:m] = src[lo:lo + m]
        d_raw[lo:lo + m].copy_(stage[j][:m], non_blocking=True)
        done[j] = torch.cuda.Event()
        done[j].record()
    torch.cuda.current_stream().synchronize()                         # the staging buffers are released on return
    return d_raw


def read_fasta_arrays_cuda(fasta_file):
    """Device-side tokenisation of a FASTA file (phm_fasta_index / phm_fasta_extract): the file is memory-mapped, its bytes go
    to the GPU once through pinned staging buffers and the sequence bytes never come back; only the title lines are read on the
    host, at the positions the device reports.  Returns (titles' first tokens, CUDA uint8 tensor of all sequence bytes end to end
    [padded to 16], CUDA int64 offsets[n+1]).  Files holding a control byte other than '\n' '\r' (tab / VT / FF / 0x1C-0x1F are
    stripped by the reference at line ends only) are tokenised by the exact host path and uploaded.  Raises IOError when unreadable."""
    import mmap
    import torch
    from . import ops
    mapped = None
    if fasta_file.endswith(".gz"):
        raw = _open_bytes(fasta_file)
        n = len(raw)
    else:
        fh = open(fasta_file, "rb")
        n = os.fstat(fh.fileno()).st_size
        raw = mapped = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) if n else b""
        fh.close()
    try:
        if n == 0:
            return [], torch.zeros((16,), dtype=torch.uint8, device="cuda"), torch.zeros((1,), dtype=torch.int64, device="cuda")
        d_raw = _upload(raw, n)
        seq, offsets, header_pos, odd = ops.fasta_scan_cuda(d_raw[:n])
        if odd:
            ids, h_seq, h_off = split_fasta_bytes(bytes(raw[:n]))
            total = int(h_off[-1])
            pad = torch.zeros((max((total + 15) // 16 * 16, 16),), dtype=torch.uint8)
            pad[:total] = torch.from_numpy(np.ascontiguousarray(h_seq[:total]).copy()) if total else pad[:0]
            return ids, pad.cuda(), torch.from_numpy(np.ascontiguousarray(h_off)).cuda()
        ids = []
        for hs in header_pos.cpu().tolist():
            he = n
            for eol in (b"\n", b"\r"):                                  # the title line ends at the first '\n' or '\r'
                e = raw.find(eol, hs, he)
                he = e if e >= 0 else he
            title = bytes(raw[hs + 1:he]).decode("latin-1").rstrip()
            tokens = title.split(None, 1)
            ids.append(tokens[0] if tokens else "")
        return ids, seq, offsets
    finally:
        if mapped is not None:
            mapped.close()


def read_fasta_arrays(fasta_file):
    """(titles' first tokens, sequence bytes end to end, offsets).  Raises IOError when unreadable."""
    return split_fasta_bytes(_open_bytes(fasta_file))


def read_fasta(fasta_file):
    """scripts/fileIO.py:28-42: (ndarray of ids, list of sequence strings)."""
    headers, seq, offsets = read_fasta_arrays(fasta_file)
    blob = seq.tobytes().decode("latin-1")
    sequences = [blob[offsets[i]:offsets[i + 1]] for i in range(len(headers))]
    return np.array([get_id(h) for h in headers]), sequences


def get_fasta_ids(fasta_file):
    """scripts/fileIO.py:62-77."""
    headers, _, _ = read_fasta_arrays(fasta_file)
    return np.array([get_id(h) for h in headers])


def get_fasta_lengths(fasta_file):
    """Lengths of the parsed sequences (what phamer.screen_by_length measures, scripts/phamer.py:150-154)."""
    headers, _, offsets = read_fasta_arrays(fasta_file)
    return np.array([get_id(h) for h in headers]), np.diff(offsets)


# ----------------------------------------------------------------------------------------------------------
# feature CSV
# ----------------------------------------------------------------------------------------------------------
def generate_summary(args, line_start="", header=""):
    """scripts/basic.py:22-37: argparse namespace -> header text."""
    if args is None:
        return ""
    text = str(args).replace("Namespace(", line_start).replace(")", "")
    text = text.replace(", ", "\n" + line_start).replace("=", ":\t") + "\n"
    return line_start + header + "\n" + text


def read_feature_file(feature_file, normalize=False, id=None):
    """scripts/fileIO.py:134-166: (ids ndarray[str], counts int ndarray[n, bins]); normalize -> kmer.normalize_counts."""
    ids, rows = [], []
    opener = gzip.open if feature_file.endswith(".gz") else open
    with opener(feature_file, "rt") as fh:
        for line in fh:
            line = line.split("#", 1)[0].strip()
            if not line:
                continue
            first, rest = line.split(",", 1)
            ids.append(first)
            rows.append(np.array(rest.split(","), dtype=np.int64))
    features = np.stack(rows) if rows else np.zeros((0, 0), dtype=np.int64)
    ids = np.array(ids)
    if normalize:
        from . import kmer
        features = kmer.normalize_counts(features)
    if id:
        return features[ids == id]
    return ids, features


def save_counts(counts, ids, file_name, args=None, header="K-mer count file"):
    """scripts/fileIO.py:169-181: '# '-prefixed header lines, then id,c0,c1,... as integers."""
    if args is not None:
        header = generate_summary(args, header=header)
    counts = np.asarray(counts).astype(np.int64)
    if counts.ndim == 1:
        counts = counts[None, :]
    with open(file_name, "w") as fh:
        for line in header.split("\n"):
            fh.write("# " + line + "\n")
        for ident, row in zip(ids, counts):
            fh.write(str(ident) + "," + ",".join(map(str, row.tolist())) + "\n")


# ----------------------------------------------------------------------------------------------------------
# score CSV
# ----------------------------------------------------------------------------------------------------------
def save_phamer_scores(ids, scores, file_name, args=None):
    """scripts/fileIO.py:241-253: header 'PhaMers score file', rows 'id, score' with scores printed by
    numpy's float64 -> str conversion."""
    header = "PhaMers score file"
    if args is not None:
        header = generate_summary(args, header=header)
    ids = np.asarray(ids).astype(str)
    scores = np.asarray(scores, dtype=np.float64).astype(str)
    with open(file_name, "w") as fh:
        for line in header.split("\n"):
            fh.write("# " + line + "\n")
        for ident, score in zip(ids, scores):
            fh.write("%s, %s\n" % (ident, score))


def read_phamer_output(filename):
    """scripts/fileIO.py:256-272: {contig id: score}."""
    out = {}
    with open(filename, "r") as fh:
        for line in fh:
            if "#" in line or not line.strip():
                continue
            out[line.split(",")[0]] = float(line.split()[1])
    return out


# ----------------------------------------------------------------------------------------------------------
# neighbour CSV (phamer -neighbors): the references and clusters behind each score
# ----------------------------------------------------------------------------------------------------------
NEIGHBOR_CLASSES = {1: "phage", 0: "bacteria", -1: ""}


def save_phamer_neighbors(ids, reference_ids, reference_labels, reference_distances, clusters, cluster_distances, file_name,
                          args=None):
    """'# '-prefixed header lines (header 'PhaMers neighbour file', then the column names), then per contig, in the order of the
    score file: 'id, reference_1, class_1, distance_1, ..., reference_k, class_k, distance_k, phage_cluster,
    phage_cluster_distance, bacteria_cluster, bacteria_cluster_distance'.  reference_* are [contigs, k] arrays nearest first,
    labels 1 = phage / 0 = bacteria (-1: none), clusters / cluster_distances [contigs, 2] (phage, bacteria; cluster -1: none).
    Distances are printed by numpy's float64 -> str conversion, which round-trips."""
    header = "PhaMers neighbour file"
    if args is not None:
        header = generate_summary(args, header=header)
    ref_ids = np.asarray(reference_ids).astype(str)
    k = ref_ids.shape[1]
    classes = np.vectorize(NEIGHBOR_CLASSES.get, otypes=[str])(np.asarray(reference_labels, dtype=np.int64))
    ref_dist = np.asarray(reference_distances, dtype=np.float64).astype(str)
    clusters = np.asarray(clusters, dtype=np.int64)
    cl_dist = np.asarray(cluster_distances, dtype=np.float64).astype(str)
    columns = ["id"] + ["%s_%d" % (c, j + 1) for j in range(k) for c in ("reference", "class", "distance")]
    columns += ["phage_cluster", "phage_cluster_distance", "bacteria_cluster", "bacteria_cluster_distance"]
    with open(file_name, "w") as fh:
        for line in header.split("\n"):
            fh.write("# " + line + "\n")
        fh.write("# " + ", ".join(columns) + "\n")
        for i, ident in enumerate(np.asarray(ids).astype(str)):
            fields = [ident]
            for j in range(k):
                fields += [ref_ids[i, j], classes[i, j], ref_dist[i, j]]
            fields += [str(clusters[i, 0]), cl_dist[i, 0], str(clusters[i, 1]), cl_dist[i, 1]]
            fh.write(", ".join(fields) + "\n")


def read_phamer_neighbors(filename):
    """The file of save_phamer_neighbors -> (ids [contigs] str, reference_ids [contigs, k] str, reference_labels [contigs, k] int64,
    reference_distances [contigs, k] float64, clusters [contigs, 2] int64, cluster_distances [contigs, 2] float64)."""
    labels = {v: c for c, v in NEIGHBOR_CLASSES.items()}
    rows = []
    with open(filename, "r") as fh:
        for line in fh:
            if line.startswith("#") or not line.strip():
                continue
            rows.append(line.rstrip("\n").split(", "))
    n = len(rows)
    k = (len(rows[0]) - 5) // 3 if rows else 0
    ids = np.array([r[0] for r in rows], dtype=str)
    refs = np.array([[r[1 + 3 * j] for j in range(k)] for r in rows], dtype=str).reshape(n, k)
    ref_labels = np.array([[labels[r[2 + 3 * j]] for j in range(k)] for r in rows], dtype=np.int64).reshape(n, k)
    ref_dist = np.array([[float(r[3 + 3 * j]) for j in range(k)] for r in rows], dtype=np.float64).reshape(n, k)
    clusters = np.array([[int(r[-4]), int(r[-2])] for r in rows], dtype=np.int64).reshape(n, 2)
    cl_dist = np.array([[float(r[-3]), float(r[-1])] for r in rows], dtype=np.float64).reshape(n, 2)
    return ids, refs, ref_labels, ref_dist, clusters, cl_dist


# ----------------------------------------------------------------------------------------------------------
# window and region CSVs (phamer -window): scores along each contig and the phage-like regions they show
# ----------------------------------------------------------------------------------------------------------
def _write_rows(file_name, header, args, columns, rows):
    if args is not None:
        header = generate_summary(args, header=header)
    with open(file_name, "w") as fh:
        for line in header.split("\n"):
            fh.write("# " + line + "\n")
        fh.write("# " + ", ".join(columns) + "\n")
        for fields in rows:
            fh.write(", ".join(fields) + "\n")


def _read_rows(filename):
    with open(filename, "r") as fh:
        return [line.rstrip("\n").split(", ") for line in fh if not line.startswith("#") and line.strip()]


def save_phamer_windows(ids, spans, scores, file_name, args=None):
    """'# '-prefixed header lines (header 'PhaMers window file', then the column names), then one row per window:
    'id, start, end, score' -- the contig's id, the window's 0-based half-open coordinates in the contig, its score printed by
    numpy's float64 -> str conversion, which round-trips."""
    spans = np.asarray(spans, dtype=np.int64).reshape(-1, 2)
    scores = np.asarray(scores, dtype=np.float64).astype(str)
    rows = zip(np.asarray(ids).astype(str), spans[:, 0].astype(str), spans[:, 1].astype(str), scores)
    _write_rows(file_name, "PhaMers window file", args, ["id", "start", "end", "score"], rows)


def read_phamer_windows(filename):
    """The file of save_phamer_windows -> (ids [windows] str, spans int64[windows, 2], scores float64[windows])."""
    rows = _read_rows(filename)
    ids = np.array([r[0] for r in rows], dtype=str)
    spans = np.array([[int(r[1]), int(r[2])] for r in rows], dtype=np.int64).reshape(len(rows), 2)
    return ids, spans, np.array([float(r[3]) for r in rows], dtype=np.float64)


def save_phamer_regions(ids, spans, windows, mean_scores, max_scores, file_name, args=None):
    """'# '-prefixed header lines (header 'PhaMers region file', then the column names), then one row per region:
    'id, start, end, windows, mean_score, max_score' -- a region is a maximal run of consecutive windows of one contig that all
    score >= 0; start / end are those of its first / last window, scores are printed as in save_phamer_windows."""
    spans = np.asarray(spans, dtype=np.int64).reshape(-1, 2)
    rows = zip(np.asarray(ids).astype(str), spans[:, 0].astype(str), spans[:, 1].astype(str),
               np.asarray(windows, dtype=np.int64).astype(str), np.asarray(mean_scores, dtype=np.float64).astype(str),
               np.asarray(max_scores, dtype=np.float64).astype(str))
    _write_rows(file_name, "PhaMers region file", args, ["id", "start", "end", "windows", "mean_score", "max_score"], rows)


def read_phamer_regions(filename):
    """The file of save_phamer_regions -> (ids str, spans int64[regions, 2], windows int64, mean_scores float64, max_scores float64)."""
    rows = _read_rows(filename)
    ids = np.array([r[0] for r in rows], dtype=str)
    spans = np.array([[int(r[1]), int(r[2])] for r in rows], dtype=np.int64).reshape(len(rows), 2)
    return (ids, spans, np.array([int(r[3]) for r in rows], dtype=np.int64), np.array([float(r[4]) for r in rows], dtype=np.float64),
            np.array([float(r[5]) for r in rows], dtype=np.float64))


# ----------------------------------------------------------------------------------------------------------
# BED intervals in, span scores out (phamer -spans, -region_scores)
# ----------------------------------------------------------------------------------------------------------
def read_bed(path, with_lines=False):
    """BED intervals -> (contig names [n] str, spans int64[n, 2] (start, end: 0-based, half-open), names [n] str), and with
    with_lines=True a fourth element, where each interval came from ('<path> line <number>').  Fields are
    separated by tabs or any whitespace: 'chrom start end [name ...]'; columns past the name are ignored and a missing name is '.'.
    Blank lines and '#', 'track' and 'browser' lines are skipped.  A malformed line (fewer than three fields, coordinates that are
    not integers, start < 0 or end < start) is a ValueError naming its line number."""
    ids, spans, names, where = [], [], [], []
    with open(path, "r") as fh:
        for number, line in enumerate(fh, 1):
            fields = line.split()
            if not fields or fields[0].startswith("#") or fields[0] in ("track", "browser"):
                continue
            if len(fields) < 3:
                raise ValueError("%s line %d: a BED line needs chrom, start and end: %r" % (path, number, line.rstrip("\n")))
            try:
                start, end = int(fields[1]), int(fields[2])
            except ValueError:
                raise ValueError("%s line %d: start and end must be integers: %r" % (path, number, line.rstrip("\n"))) from None
            if start < 0 or end < start:
                raise ValueError("%s line %d: [%d, %d) is not an interval" % (path, number, start, end))
            ids.append(fields[0])
            spans.append((start, end))
            names.append(fields[3] if len(fields) > 3 else ".")
            where.append("%s line %d" % (path, number))
    out = np.array(ids, dtype=str), np.array(spans, dtype=np.int64).reshape(-1, 2), np.array(names, dtype=str)
    return out + (where,) if with_lines else out


def save_phamer_spans(ids, spans, names, scores, reference_ids, reference_labels, reference_distances, clusters, cluster_distances,
                      file_name, args=None):
    """'# '-prefixed header lines (header 'PhaMers span file', then the column names), then one row per span: 'id, start, end, name,
    score' followed by the neighbour columns of save_phamer_neighbors (reference_j, class_j, distance_j for j = 1..k, then the phage
    and bacteria cluster with their distances).  Floats are printed by numpy's float64 -> str conversion, which round-trips."""
    spans = np.asarray(spans, dtype=np.int64).reshape(-1, 2)
    ref_ids = np.asarray(reference_ids).astype(str)
    k = ref_ids.shape[1] if ref_ids.ndim == 2 else 0
    ref_ids = ref_ids.reshape(-1, k)
    classes = np.vectorize(NEIGHBOR_CLASSES.get, otypes=[str])(np.asarray(reference_labels, dtype=np.int64).reshape(-1, k))
    ref_dist = np.asarray(reference_distances, dtype=np.float64).reshape(-1, k).astype(str)
    clusters = np.asarray(clusters, dtype=np.int64).reshape(-1, 2)
    cl_dist = np.asarray(cluster_distances, dtype=np.float64).reshape(-1, 2).astype(str)
    scores = np.asarray(scores, dtype=np.float64).astype(str)
    columns = ["id", "start", "end", "name", "score"] + ["%s_%d" % (c, j + 1) for j in range(k) for c in ("reference", "class", "distance")]
    columns += ["phage_cluster", "phage_cluster_distance", "bacteria_cluster", "bacteria_cluster_distance"]
    rows = []
    for i, (ident, name) in enumerate(zip(np.asarray(ids).astype(str), np.asarray(names).astype(str))):
        fields = [ident, str(spans[i, 0]), str(spans[i, 1]), name, scores[i]]
        for j in range(k):
            fields += [ref_ids[i, j], classes[i, j], ref_dist[i, j]]
        rows.append(fields + [str(clusters[i, 0]), cl_dist[i, 0], str(clusters[i, 1]), cl_dist[i, 1]])
    _write_rows(file_name, "PhaMers span file", args, columns, rows)


def read_phamer_spans(filename):
    """The file of save_phamer_spans -> (ids str, spans int64[n, 2], names str, scores float64, reference_ids [n, k] str,
    reference_labels [n, k] int64, reference_distances [n, k] float64, clusters [n, 2] int64, cluster_distances [n, 2] float64)."""
    labels = {v: c for c, v in NEIGHBOR_CLASSES.items()}
    rows = _read_rows(filename)
    n = len(rows)
    k = (len(rows[0]) - 9) // 3 if rows else 0
    ids = np.array([r[0] for r in rows], dtype=str)
    spans = np.array([[int(r[1]), int(r[2])] for r in rows], dtype=np.int64).reshape(n, 2)
    names = np.array([r[3] for r in rows], dtype=str)
    scores = np.array([float(r[4]) for r in rows], dtype=np.float64)
    refs = np.array([[r[5 + 3 * j] for j in range(k)] for r in rows], dtype=str).reshape(n, k)
    ref_labels = np.array([[labels[r[6 + 3 * j]] for j in range(k)] for r in rows], dtype=np.int64).reshape(n, k)
    ref_dist = np.array([[float(r[7 + 3 * j]) for j in range(k)] for r in rows], dtype=np.float64).reshape(n, k)
    clusters = np.array([[int(r[-4]), int(r[-2])] for r in rows], dtype=np.int64).reshape(n, 2)
    cl_dist = np.array([[float(r[-3]), float(r[-1])] for r in rows], dtype=np.float64).reshape(n, 2)
    return ids, spans, names, scores, refs, ref_labels, ref_dist, clusters, cl_dist
