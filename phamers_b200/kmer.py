"""
Drop-in for the reference's scripts/kmer.py: same names, positional orders, defaults and return conventions, with the
counting and normalising done by the CUDA kernels behind include/phamers_b200.h.

    reference (scripts/kmer.py)                  here
    count_string  :32      per-base Python loop  one phm_kmer_count launch
    count         :82      dispatch str / list   same dispatch, ONE launch for the whole list
    count_file    :114     Bio.SeqIO + count     FASTA tokenised on the device (3 launches) + one launch
    count_directory :143   per-file sums         same
    normalize_counts :209  row / row-sum         phm_normalize_counts
    sequence_to_integers :183, get_kmer_index :199, kmers :224, extend_mers :235   plain host helpers

Bin order is the reference's: symbols 'ATGC', first base most significant; only exact symbol bytes count, anything
else voids the windows it touches.  Four-letter alphabets other than 'ATGC' (e.g. RNA 'AUGC') are mapped onto the
same kernels by a byte translation; alphabets of another size (the reference's broken protein branch, kmer.py:51-76)
are out of scope and raise.
"""
import gzip
import logging
import os
import random

import numpy as np

from . import fileIO

logger = logging.getLogger(__name__)
logger.setLevel(logging.WARNING)

DNA = "ATGC"
RNA = "AUGC"
protein = "RHKDESTNQCUGPAVILMFYW"


# ----------------------------------------------------------------------------------------------------------
# host <-> device plumbing
# ----------------------------------------------------------------------------------------------------------
def _translation(symbols):
    if len(symbols) != 4 or len(set(symbols)) != 4:
        raise NotImplementedError("phamers_b200 counts 4-symbol alphabets only (got %r); the reference's >= 10 symbol "
                                  "branch (kmer.py:51-76) is out of scope" % (symbols,))
    if symbols == DNA:
        return None
    table = bytearray(b"N" * 256)
    for src, dst in zip(symbols, DNA):
        if ord(src) > 255:
            raise NotImplementedError("non-latin-1 symbol %r" % src)
        table[ord(src)] = ord(dst)
    return bytes(table)


def _encode(sequences, symbols):
    """list[str] -> (uint8 ndarray of all bases end to end, int64 offsets[n+1])."""
    table = _translation(symbols)
    blob = "".join(sequences).encode("latin-1", "replace")
    if table is not None:
        blob = blob.translate(table)
    offsets = np.zeros(len(sequences) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in sequences], out=offsets[1:])
    if len(blob) != int(offsets[-1]):
        raise ValueError("internal error: encoded length differs from character count")
    return np.frombuffer(blob, dtype=np.uint8), offsets


def count_arrays(seq_bytes, offsets, kmer_length, normalize=False, canonical=False):
    """Counts k-mers of sequences laid end to end in a host uint8 array.  Returns int64 [n, bins] (float64 if
    normalize, all-zero rows staying zero like count_string's guard at kmer.py:77)."""
    import torch
    from . import ops, _lib
    _lib.require_cuda()
    n = len(offsets) - 1
    total = int(offsets[-1])
    padded = (total + 15) // 16 * 16
    host = torch.empty((max(padded, 16),), dtype=torch.uint8, pin_memory=True)
    host[:total] = torch.from_numpy(np.ascontiguousarray(seq_bytes[:total]).copy()) if total else host[:0]
    d_seq = host.to("cuda", non_blocking=True)
    d_off = torch.from_numpy(np.ascontiguousarray(offsets, dtype=np.int64)).to("cuda")
    counts, freq = ops.count_cuda(d_seq, d_off, kmer_length, canonical=canonical, counts=not normalize, freq=normalize)
    if normalize:
        out = freq.cpu().numpy()
        out[np.isnan(out).any(axis=1)] = 0.0                                   # kmer.py:77: no division for empty rows
        return out
    return counts.cpu().numpy().view(np.uint32).astype(np.int64) if n else np.zeros((0, counts.shape[1]), dtype=np.int64)


# ----------------------------------------------------------------------------------------------------------
# reference API
# ----------------------------------------------------------------------------------------------------------
def count_string(sequence, kmer_length, symbols=DNA, normalize=False):
    """scripts/kmer.py:32.  ndarray[len(symbols)^k], int64 (float64 when normalize)."""
    seq, off = _encode([sequence], symbols)
    return count_arrays(seq, off, kmer_length, normalize=normalize)[0]


def count(data, kmer_length, symbols=DNA, normalize=False):
    """scripts/kmer.py:82.  str or 1-element list -> 1-D; longer list -> [n, bins]; anything else -> None."""
    if isinstance(data, list):
        if len(data) == 1:
            return count(data[0], kmer_length, symbols=symbols, normalize=normalize)
        seq, off = _encode(data, symbols)
        return count_arrays(seq, off, kmer_length, normalize=normalize)
    if isinstance(data, str):
        return count_string(data, kmer_length, symbols=symbols, normalize=normalize)
    logger.info("Data was not str or list: %s\n%s ..." % (type(data), str(data)[:25]))
    return None


def count_file(input_file, kmer_length, symbols=DNA, normalize=False):
    """scripts/kmer.py:114.  (ids ndarray[str], counts ndarray[n, bins]); (None, None) if the file cannot be read.
    Zipped files are ok."""
    table = _translation(symbols)
    bins = len(symbols) ** kmer_length
    if table is None:
        # usual case: the file's bytes go to the device once, records are found there (phm_fasta_index / _extract) and the
        # sequence bytes feed the histogram kernel without ever coming back to the host
        from . import ops, _lib
        _lib.require_cuda()
        try:
            headers, d_seq, d_off = fileIO.read_fasta_arrays_cuda(input_file)
        except IOError:
            logger.warning("Could not read file: %s" % os.path.basename(input_file))
            return None, None
        ids = np.array([fileIO.get_id(h) for h in headers])
        if len(ids) == 0:
            return ids, np.zeros((0, bins), dtype=(float if normalize else int))
        counts, freq = ops.count_cuda(d_seq, d_off, kmer_length, counts=not normalize, freq=normalize)
        if normalize:
            out = freq.cpu().numpy()
            out[np.isnan(out).any(axis=1)] = 0.0                               # kmer.py:77: no division for empty rows
            return ids, out
        return ids, counts.cpu().numpy().view(np.uint32).astype(np.int64)
    try:
        headers, seq, offsets = fileIO.read_fasta_arrays(input_file)
    except IOError:
        logger.warning("Could not read file: %s" % os.path.basename(input_file))
        return None, None
    ids = np.array([fileIO.get_id(h) for h in headers])
    seq = np.frombuffer(seq.tobytes().translate(table), dtype=np.uint8)
    if len(ids) == 0:
        return ids, np.zeros((0, bins), dtype=(float if normalize else int))
    return ids, count_arrays(seq, offsets, kmer_length, normalize=normalize)


def count_directory(directory, kmer_length, identifier="fna", symbols=DNA, sum_file=True, sample=0):
    """scripts/kmer.py:143.  One row per file (the sum over its records); unreadable or empty files are skipped."""
    selected = [os.path.join(directory, f) for f in os.listdir(directory) if identifier in os.path.basename(f)]
    if sample:
        random.shuffle(selected)
    ids, rows = [], []
    for path in selected:
        file_ids, file_counts = count_file(path, kmer_length, symbols=symbols)
        if file_ids is None or len(file_ids) == 0 or np.sum(file_counts) == 0:
            logger.warning("Could not read file: %s" % os.path.basename(path))
            continue
        if sum_file and file_counts.ndim == 2:
            ids.append(file_ids[0])
            rows.append(np.sum(file_counts, axis=0))
        else:
            ids.extend(list(file_ids))
            rows.extend(list(file_counts))
        if sample and len(ids) >= sample:
            break
    counts = np.array(rows, dtype=float) if rows else np.zeros((0, len(symbols) ** kmer_length))
    return ids, counts


def sequence_to_integers(sequence, symbols):
    """scripts/kmer.py:183."""
    for stranger in set(sequence) - set(symbols):
        sequence = sequence.replace(stranger, "-")
    for digit, symbol in enumerate(symbols):
        sequence = sequence.replace(symbol, str(digit))
    return sequence


def get_kmer_index(kmer, symbols):
    """scripts/kmer.py:199.  NB the reference parses in base len(kmer) (:206), which is the bin index only when
    len(kmer) == len(symbols); this returns the true bin index (identical for the reference's own k = 4 use)."""
    return int(sequence_to_integers(kmer, symbols), len(symbols))


def normalize_counts(counts):
    """scripts/kmer.py:209.  float64 copy with every row divided by its sum (an all-zero row gives NaN, as there).  Any numeric
    array is taken, as by the reference: exact counts below 2^32 go through the integer kernel (bit-identical to numpy), anything
    else -- summed genome counts of count_directory, already-float features, negative values -- through the float64 one."""
    import torch
    from . import ops, _lib
    _lib.require_cuda()
    arr = np.asarray(counts)
    if arr.size == 0:
        return arr.astype(float)
    is_count = arr.dtype.kind in "iub" or (arr.dtype.kind == "f" and bool(np.all(np.isfinite(arr))) and bool(np.all(arr == np.floor(arr))))
    if is_count and arr.min() >= 0 and arr.max() < 2 ** 32:
        as_u32 = np.ascontiguousarray(arr.astype(np.uint32))
        return ops.normalize_cuda(torch.from_numpy(as_u32.view(np.int32)).to("cuda")).cpu().numpy()
    as_f64 = np.ascontiguousarray(arr, dtype=np.float64)
    return ops.normalize_rows_cuda(torch.from_numpy(as_f64).to("cuda")).cpu().numpy()


def canonical_fold(counts, kmer_length):
    """Folds every k-mer together with its reverse complement: [..., 4^k] -> [..., 136 / 512 / 2080 ...] for k = 4 / 5 / 6, the bins
    and order of the canonical counter (canon[min(j, rc(j))] += count[j], representatives ascending).  A sequence and its reverse
    complement have the same folded row.  int64 for integer input (exact below 2^53), float64 otherwise; the row total is kept, so
    normalize_counts of the folded counts equals the fold of the normalised ones up to rounding."""
    import torch
    from . import ops, _lib
    _lib.require_cuda()
    arr = np.asarray(counts)
    if arr.shape[-1:] != (4 ** int(kmer_length),):
        raise ValueError("rows of %d bins cannot be folded at k = %d (needs %d)" % (arr.shape[-1] if arr.ndim else 0, kmer_length,
                                                                                   4 ** int(kmer_length)))
    integer = arr.dtype.kind in "iub"
    rows = np.ascontiguousarray(arr.reshape(-1, arr.shape[-1]), dtype=np.float64)
    bins = ops.num_bins(kmer_length, canonical=True)
    if rows.shape[0] == 0:
        folded = np.zeros((0, bins))
    else:
        folded = ops.canonical_fold_cuda(torch.from_numpy(rows).to("cuda"), kmer_length).cpu().numpy()
    folded = folded.reshape(arr.shape[:-1] + (bins,))
    return folded.astype(np.int64) if integer else folded


def kmers(k, symbols=DNA):
    """scripts/kmer.py:224.  All k-mers in bin order."""
    out = [""]
    for _ in range(k):
        out = [prefix + s for prefix in out for s in symbols]
    return out


def extend_mers(mers, k, symbols):
    """scripts/kmer.py:235.  Prepends every symbol to every k-mer, k times (kept for API parity)."""
    for _ in range(k):
        mers = [s + m for s in symbols for m in mers]
    return mers


def load_counts(kmer_length, location=None, counts_file=None, identifier="fna", normalize=False, symbols=DNA):
    """scripts/kmer.py:254 with its dead calls repaired (see SURVEY.md 8(b) 'known defects'): a counts file wins,
    else a FASTA file, else a directory of FASTA files; freshly counted data is cached to counts_file."""
    ids = counts = None
    if counts_file and os.path.isfile(counts_file):
        ids, counts = fileIO.read_feature_file(counts_file, normalize=normalize)
    elif location and os.path.isfile(location):
        ids, counts = count_file(location, kmer_length, normalize=normalize, symbols=symbols)
        if counts_file and not normalize:
            fileIO.save_counts(counts, ids, counts_file)
    elif location and os.path.isdir(location):
        ids, counts = count_directory(location, kmer_length, identifier=identifier, symbols=symbols)
        if counts_file:
            fileIO.save_counts(counts, ids, counts_file)
        if normalize:
            counts = normalize_counts(counts)
    return ids, counts
