"""
The on-disk formats either side of the hot path, mirroring the reference's scripts/fileIO.py and the part of
scripts/id_parser.py the path touches:

    FASTA in        read_fasta :28, get_fasta_ids :62 (Bio.SeqIO tokenisation) + id_parser.get_id :89
    BGZF            bgzf_members  (the member chain of a blocked-gzip FASTA, decoded on the device by ops.inflate_cuda)
    gzip            gzip_member   (the header and trailer of a single-member gzip FASTA, decoded on the device by ops.gunzip_cuda)
    feature CSV     read_feature_file :134, save_counts :169  ('#' header lines, then id,c0,c1,...; formatted and parsed on the
                    device when there is one, ops.format_counts_csv_cuda / ops.parse_feature_csv_cuda)
    score CSV       save_phamer_scores :241, read_phamer_output :256  ('# ' header, then 'id, score')
    neighbour CSV   save_phamer_neighbors, read_phamer_neighbors  ('# ' header, then per contig its nearest references and clusters)
    window CSV      save_phamer_windows, read_phamer_windows  ('# ' header, then 'id, start, end, score' per window)
    region CSV      save_phamer_regions, read_phamer_regions  ('# ' header, then 'id, start, end, windows, mean_score, max_score')
    BED in          read_bed  ('chrom start end [name ...]' per line)
    span CSV        save_phamer_spans, read_phamer_spans  ('# ' header, then 'id, start, end, name, score' and the neighbour columns)

Bytes and text; no arithmetic happens here.
"""
import gzip
import io
import os
import struct

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
    """File bytes (an mmap of a plain or BGZF file, or the bytes of a .gz inflated on the host) -> CUDA uint8 tensor padded to 16
    bytes.  The copy page cache -> pinned staging buffer of chunk i + 1 runs on the host while chunk i crosses PCIe
    (scripts/kmer.py:131-134 reads the whole file through Python objects instead)."""
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


# phm_bgzf_member (include/phamers_b200.h): one row per member of a BGZF file
BGZF_MEMBER = np.dtype([("in_offset", "<i8"), ("out_offset", "<i8"), ("in_bytes", "<u4"), ("isize", "<u4"), ("crc32", "<u4"),
                        ("reserved", "<u4")])
_BGZF_MAGIC = b"\x1f\x8b\x08\x04"          # ID1 ID2 CM, FLG = FEXTRA only
_U16 = struct.Struct("<H").unpack_from


def bgzf_members(buf):
    """The member table of a BGZF file (what bgzip / htslib write): a structured array of BGZF_MEMBER, one row per member in file
    order -- the raw DEFLATE payload's offset and size in `buf`, the member's offset in the decompressed file, its ISIZE and CRC32
    --, or None when `buf` is not BGZF from its first byte to its last.  A member is BGZF when its header is ID1 ID2 CM = 31 139 8
    with FLG = FEXTRA (no name, comment or header CRC) and its extra field holds a 'BC' subfield of SLEN 2 (BSIZE = member size - 1)
    among well-formed subfields.  The chain must end exactly at the end of `buf`; the 28-byte empty EOF block is an ordinary member.
    The walk along the chain is serial (one header per 64 KiB of output); the trailers are read with numpy."""
    n = len(buf)
    starts, payload, sizes = [], [], []
    pos = 0
    while pos < n:
        if n - pos < 12 or buf[pos:pos + 4] != _BGZF_MAGIC:
            return None
        xlen = _U16(buf, pos + 10)[0]
        if pos + 12 + xlen > n:
            return None
        if xlen == 6 and buf[pos + 12:pos + 16] == b"BC\x02\x00":   # bgzip's layout: BC is the only subfield
            bsize = _U16(buf, pos + 16)[0]
        else:
            bsize, at, end = None, pos + 12, pos + 12 + xlen
            while at < end:
                if end - at < 4:
                    return None
                slen = _U16(buf, at + 2)[0]
                if at + 4 + slen > end:
                    return None
                if buf[at:at + 2] == b"BC" and slen == 2:
                    bsize = _U16(buf, at + 4)[0]
                at += 4 + slen
            if bsize is None:
                return None
        size = bsize + 1
        if size < 12 + xlen + 8 or pos + size > n:
            return None
        starts.append(pos)
        payload.append(pos + 12 + xlen)
        sizes.append(size)
        pos += size
    if not starts:
        return None
    ends = np.array(starts, dtype=np.int64) + np.array(sizes, dtype=np.int64)
    data = np.frombuffer(buf, dtype=np.uint8, count=n)
    trailer = data[(ends - 8)[:, None] + np.arange(8)].astype(np.uint32)         # CRC32, ISIZE (little-endian)
    crc = trailer[:, 0] | (trailer[:, 1] << 8) | (trailer[:, 2] << 16) | (trailer[:, 3] << 24)
    isize = trailer[:, 4] | (trailer[:, 5] << 8) | (trailer[:, 6] << 16) | (trailer[:, 7] << 24)
    if np.any(isize > 65536):
        return None
    table = np.zeros(len(starts), dtype=BGZF_MEMBER)
    table["in_offset"] = payload
    table["in_bytes"] = ends - 8 - table["in_offset"]
    table["isize"] = isize
    table["out_offset"][1:] = np.cumsum(isize[:-1], dtype=np.int64)
    table["crc32"] = crc
    return table


def gzip_member(buf):
    """(payload offset, payload end, CRC32, ISIZE) of `buf` read as one gzip member whose 8-byte trailer ends the buffer, or None
    when its header is not one Python's gzip module accepts.  The header is parsed as gzip._read_gzip_header parses it: ID1 ID2,
    CM = 8, then FEXTRA (XLEN bytes), FNAME and FCOMMENT (up to and including a NUL) and FHCRC (2 bytes, not checked) are skipped;
    the reserved flag bits are ignored.  Whether the DEFLATE stream in between ends exactly at the trailer, and the CRC32 and ISIZE
    of its output, are for the decoder to check (a multi-member file gives the first header and the last trailer here)."""
    n = len(buf)
    if n < 10 or buf[0:3] != b"\x1f\x8b\x08":
        return None
    flag, pos = buf[3], 10
    if flag & 4:                                                  # FEXTRA
        if pos + 2 > n:
            return None
        pos += 2 + _U16(buf, pos)[0]
    for bit in (8, 16):                                           # FNAME, FCOMMENT: zero-terminated
        if flag & bit:
            end = buf.find(b"\0", pos) if pos < n else -1
            if end < 0:
                return None
            pos = end + 1
    if flag & 2:                                                  # FHCRC
        pos += 2
    if pos + 8 > n:
        return None
    crc, isize = struct.unpack_from("<II", buf, n - 8)
    return pos, n - 8, crc, isize


def _open_fasta_device(fasta_file):
    """(the FASTA text on the host [mmap or bytes], or None when only the device holds it; the text on the device [CUDA uint8,
    padded to 16, or None when empty]; its size; the mmap to close or None).  A compressed file goes to the device compressed and is
    inflated there: BGZF by ops.inflate_cuda, a single gzip member by ops.gunzip_cuda.  Any other .gz, and any file the device
    declines (corrupt data, trailing bytes, more than one member, not enough device memory), is inflated on the host, so that it
    gives or raises exactly what gzip gives or raises.  Plain files are mapped."""
    import mmap
    import torch
    from . import _lib, ops
    with open(fasta_file, "rb") as fh:
        size = os.fstat(fh.fileno()).st_size
        mapped = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) if size else None
    if not fasta_file.endswith(".gz"):
        return mapped, (_upload(mapped, size) if size else None), size, mapped
    members = bgzf_members(mapped) if size else None
    member = gzip_member(mapped) if size and members is None else None
    if members is not None or member is not None:
        try:
            d_raw = _upload(mapped, size)[:size]
            d_text = ops.inflate_cuda(d_raw, members) if members is not None else ops.gunzip_cuda(d_raw, member)
            del d_raw
            mapped.close()
            return None, d_text, d_text.numel(), None
        except (_lib.PhamersDataError, torch.cuda.OutOfMemoryError):
            pass
    if mapped is not None:
        mapped.close()
    text = _open_bytes(fasta_file)
    return text, (_upload(text, len(text)) if text else None), len(text), None


def _device_titles(d_text, n, header_pos):
    """First tokens of the title lines whose '>' is at header_pos (CUDA int64) in the device text d_text[:n]: only the title bytes
    come back to the host -- a first window of each line, then the rest of the (rare) lines longer than it."""
    import torch
    window, batch = 128, 1 << 16
    starts = header_pos + 1
    ramp = torch.arange(window, dtype=torch.int64, device="cuda")
    win = np.concatenate([d_text[(starts[lo:lo + batch, None] + ramp).clamp_(max=max(n - 1, 0))].cpu().numpy()
                          for lo in range(0, starts.shape[0], batch)] or [np.zeros((0, window), dtype=np.uint8)])
    h_starts = starts.cpu().numpy()
    eol = (win == 10) | (win == 13) | ((h_starts[:, None] + np.arange(window)) >= n)
    ids = []
    for i in range(win.shape[0]):
        row = eol[i]
        if row.any():
            title = win[i, :int(row.argmax())].tobytes()
        else:
            lo, parts = int(h_starts[i]), []
            while True:                                                 # grow the read until the line ends
                hi = min(n, lo + window * (1 << len(parts)))
                piece = d_text[lo:hi].cpu().numpy()
                cut = np.flatnonzero((piece == 10) | (piece == 13))
                parts.append(piece[:cut[0]] if cut.shape[0] else piece)
                if cut.shape[0] or hi == n:
                    break
                lo = hi
            title = b"".join(p.tobytes() for p in parts)
        tokens = title.decode("latin-1").rstrip().split(None, 1)
        ids.append(tokens[0] if tokens else "")
    return ids


def read_fasta_arrays_cuda(fasta_file):
    """Device-side tokenisation of a FASTA file (phm_fasta_index / phm_fasta_extract): the file is memory-mapped, its bytes go
    to the GPU once through pinned staging buffers and the sequence bytes never come back; only the title lines are read on the
    host, at the positions the device reports.  A BGZF-compressed file (bgzf_members) or single-member gzip file (gzip_member)
    crosses PCIe compressed and is inflated on the device (ops.inflate_cuda, ops.gunzip_cuda); its title bytes are then copied
    back from the device.  Any other .gz, or one the device declines, is inflated on the host.
    Returns (titles' first tokens, CUDA uint8 tensor of all sequence bytes end to end [padded to 16], CUDA int64 offsets[n+1]).
    Files holding a control byte other than '\n' '\r' (tab / VT / FF / 0x1C-0x1F are stripped by the reference at line ends only)
    are tokenised by the exact host path and uploaded.  Raises IOError when unreadable."""
    import torch
    from . import ops
    raw, d_text, n, mapped = _open_fasta_device(fasta_file)
    try:
        if n == 0:
            return [], torch.zeros((16,), dtype=torch.uint8, device="cuda"), torch.zeros((1,), dtype=torch.int64, device="cuda")
        seq, offsets, header_pos, odd = ops.fasta_scan_cuda(d_text[:n])
        if odd:
            text = bytes(raw[:n]) if raw is not None else d_text[:n].cpu().numpy().tobytes()
            ids, h_seq, h_off = split_fasta_bytes(text)
            total = int(h_off[-1])
            pad = torch.zeros((max((total + 15) // 16 * 16, 16),), dtype=torch.uint8)
            pad[:total] = torch.from_numpy(np.ascontiguousarray(h_seq[:total]).copy()) if total else pad[:0]
            return ids, pad.cuda(), torch.from_numpy(np.ascontiguousarray(h_off)).cuda()
        if raw is None:
            return _device_titles(d_text, n, header_pos), seq, offsets
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


def _is_decodable_on_device(fasta_file):
    """True for a BGZF or single-member gzip file on a machine with a CUDA device: get_fasta_ids / get_fasta_lengths then read it
    through read_fasta_arrays_cuda instead of inflating it on the host again."""
    if not fasta_file.endswith(".gz"):
        return False
    import mmap
    import torch
    if not torch.cuda.is_available():
        return False
    with open(fasta_file, "rb") as fh:
        if os.fstat(fh.fileno()).st_size == 0:
            return False
        with mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) as raw:
            return bgzf_members(raw) is not None or gzip_member(raw) is not None


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
    """scripts/fileIO.py:62-77.  A BGZF or gzip file is read on the device when there is one (read_fasta_arrays_cuda)."""
    if _is_decodable_on_device(fasta_file):
        headers = read_fasta_arrays_cuda(fasta_file)[0]
    else:
        headers = read_fasta_arrays(fasta_file)[0]
    return np.array([get_id(h) for h in headers])


def get_fasta_lengths(fasta_file):
    """Lengths of the parsed sequences (what phamer.screen_by_length measures, scripts/phamer.py:150-154).  A BGZF or gzip file is
    read on the device when there is one (read_fasta_arrays_cuda), so the length screen does not inflate it on the host."""
    if _is_decodable_on_device(fasta_file):
        headers, _, d_off = read_fasta_arrays_cuda(fasta_file)
        offsets = d_off.cpu().numpy()
    else:
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


def _finish_features(ids, features, normalize, id):
    if normalize:
        from . import kmer
        features = kmer.normalize_counts(features)
    if id:
        return features[ids == id]
    return ids, features


def _read_feature_file_host(feature_file, normalize=False, id=None):
    """read_feature_file on the host: every file it accepts, and the only road without a device."""
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
    return _finish_features(np.array(ids), features, normalize, id)


def _span_strings(raw, d_text, n, ranges):
    """The ASCII strings at the byte ranges [start, end) of a text: sliced from the host copy when there is one, else copied back
    from the device (a BGZF file inflated there) -- a first window of every range in one copy, then each longer range on its own."""
    if raw is not None:
        return [bytes(raw[a:b]).decode("ascii") for a, b in ranges.tolist()]
    import torch
    window, batch = 64, 1 << 16
    ramp = torch.arange(window, dtype=torch.int64, device="cuda")
    d_starts = torch.from_numpy(np.ascontiguousarray(ranges[:, 0])).cuda()
    win = np.concatenate([d_text[(d_starts[lo:lo + batch, None] + ramp).clamp_(max=n - 1)].cpu().numpy()
                          for lo in range(0, ranges.shape[0], batch)] or [np.zeros((0, window), dtype=np.uint8)])
    out = []
    for i, (a, b) in enumerate(ranges.tolist()):
        piece = win[i, :b - a] if b - a <= window else d_text[a:b].cpu().numpy()
        out.append(piece.tobytes().decode("ascii"))
    return out


def _read_feature_file_device(feature_file):
    """(ids, counts) of a feature CSV parsed on the device (ops.parse_feature_csv_cuda), or None when the file is outside the device
    grammar.  The file is opened as FASTA files are (_open_fasta_device): plain files are mapped and uploaded, BGZF and gzip files
    inflated on the device, any other .gz on the host."""
    from . import ops
    raw, d_text, n, mapped = _open_fasta_device(feature_file)
    try:
        if n == 0:
            return np.array([]), np.zeros((0, 0), dtype=np.int64)
        parsed = ops.parse_feature_csv_cuda(d_text[:n])
        if parsed is None:
            return None
        ranges, d_counts = parsed
        return np.array(_span_strings(raw, d_text, n, ranges)), d_counts.cpu().numpy()
    finally:
        if mapped is not None:
            mapped.close()


def read_feature_file(feature_file, normalize=False, id=None):
    """scripts/fileIO.py:134-166: (ids ndarray[str], counts int ndarray[n, bins]); normalize -> kmer.normalize_counts.  With a CUDA
    device the file is parsed there (phm_feature_csv_index / phm_feature_csv_parse) when it keeps to the device grammar
    (include/phamers_b200.h), which gives the same arrays; any other file is parsed on the host, which returns or raises what it
    always did."""
    import torch
    parsed = _read_feature_file_device(feature_file) if torch.cuda.is_available() else None
    if parsed is None:
        return _read_feature_file_host(feature_file, normalize, id)
    return _finish_features(parsed[0], parsed[1], normalize, id)


FORMAT_CHUNK = 256 << 20             # text bytes one slice of save_counts may need on the device (counted at 21 bytes a field)


def _save_counts_host(counts, ids, file_name, args=None, header="K-mer count file"):
    """save_counts on the host: every input, and the only road without a device."""
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


def save_counts(counts, ids, file_name, args=None, header="K-mer count file"):
    """scripts/fileIO.py:169-181: '# '-prefixed header lines, then id,c0,c1,... as integers.  With a CUDA device, 1-D or 2-D counts
    and ASCII ids (str(id)), the rows are formatted on the device (ops.format_counts_csv_cuda) in slices of at most FORMAT_CHUNK bytes
    of text, each appended to the file in order: the file is byte for byte what the host writes."""
    import torch
    from . import ops
    if args is not None:
        header = generate_summary(args, header=header)
    table = np.asarray(counts).astype(np.int64)
    if table.ndim not in (1, 2) or not torch.cuda.is_available():
        return _save_counts_host(table, ids, file_name, header=header)
    if table.ndim == 1:
        table = table[None, :]
    names = [str(ident) for ident, _ in zip(ids, range(table.shape[0]))]        # zip's pairing: the shorter one wins
    if not all(name.isascii() for name in names):
        return _save_counts_host(table, names, file_name, header=header)
    encoded = [name.encode("ascii") for name in names]
    row_bound = np.fromiter(map(len, encoded), dtype=np.int64, count=len(encoded)) + 21 * max(table.shape[1], 1) + 2
    ends = np.cumsum(row_bound)
    with open(file_name, "w") as fh:
        for line in header.split("\n"):
            fh.write("# " + line + "\n")
        fh.flush()
        lo = 0
        while lo < len(names):
            # rows while their text fits FORMAT_CHUNK, and at least one
            hi = max(lo + 1, int(np.searchsorted(ends, (ends[lo - 1] if lo else 0) + FORMAT_CHUNK, side="right")))
            id_offsets = np.zeros(hi - lo + 1, dtype=np.int64)
            np.cumsum(row_bound[lo:hi] - (21 * max(table.shape[1], 1) + 2), out=id_offsets[1:])
            id_bytes = np.frombuffer(b"".join(encoded[lo:hi]) or b"\0", dtype=np.uint8)
            text = ops.format_counts_csv_cuda(torch.from_numpy(np.ascontiguousarray(table[lo:hi])).cuda(),
                                              torch.from_numpy(id_bytes.copy()).cuda()[:int(id_offsets[-1])],
                                              torch.from_numpy(id_offsets).cuda())
            fh.buffer.write(text.cpu().numpy().data)
            lo = hi


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
