#!/usr/bin/env python
"""Feature CSV writing and reading (fileIO.save_counts / read_feature_file), host road against device road, on synthetic count tables
drawn like contig counts: row i is a multinomial draw of L_i - 3 k-mers over F bins, L_i = clip(round(exp(N(ln 10 000, 1))), 1 000,
100 000) (SURVEY.md 8(d) config 2), ids SuperContig_i_length_L_ID_i.  Three shapes of the same 256 M values: 1 000 000 x 256,
250 000 x 1 024 and 62 500 x 4 096.  For each shape:
  - host road: _save_counts_host, _read_feature_file_host (one core)
  - device road: save_counts, read_feature_file wall time, and the same steps done one by one with a clock each: id strings,
    uploads, kernels (CUDA events), device-to-host copies, file write / read
  - text bytes, and kernel GB/s (text + int64 counts moved, over kernel time) against the 7.7 TB/s HBM bound
Then phamer -fasta on 200 000 synthetic contigs twice (the first run counts and writes <fasta>_features.csv, the second reads it with
-features), on both roads.  Files live in a temporary directory: every file time is a page-cache time.  Needs a CUDA device.
    python tools/bench_feature_csv.py [--quick] [--out FILE.json]"""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phamers_b200 import _lib, fileIO, ops, phamer  # noqa: E402

HBM_GBPS = 7700.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def progress(msg):
    print(msg, file=sys.stderr, flush=True)


def table(rows, width, seed):
    rng = np.random.default_rng(seed)
    lengths = np.clip(np.round(np.exp(rng.normal(np.log(10000), 1.0, size=rows))), 1000, 100000).astype(np.int64)
    p = rng.dirichlet(np.full(width, 4.0))
    counts = rng.multinomial(lengths - 3, p)
    ids = ["SuperContig_%d_length_%d_ID_%d" % (i, n, i) for i, n in enumerate(lengths)]
    return counts.astype(np.int64), ids


class Clock:
    def __init__(self):
        self.parts = {}

    def __call__(self, name, fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        self.parts[name] = self.parts.get(name, 0.0) + time.perf_counter() - t0
        return out


def writer_steps(counts, ids, path, kernel_ms):
    """save_counts' device road step by step (one slice of FORMAT_CHUNK at most, as the function slices)."""
    c = Clock()
    names = c("id_strings", lambda: [str(i) for i in ids])
    encoded = c("id_strings", lambda: [s.encode("ascii") for s in names])
    lengths = np.fromiter(map(len, encoded), dtype=np.int64, count=len(encoded))
    bound = lengths + 21 * counts.shape[1] + 2
    ends = np.cumsum(bound)
    with open(path, "w") as fh:
        fh.write("# K-mer count file\n")
        fh.flush()
        lo = 0
        while lo < len(names):
            hi = max(lo + 1, int(np.searchsorted(ends, (ends[lo - 1] if lo else 0) + fileIO.FORMAT_CHUNK, side="right")))
            off = np.zeros(hi - lo + 1, dtype=np.int64)
            np.cumsum(lengths[lo:hi], out=off[1:])
            d_counts = c("upload", lambda: torch.from_numpy(np.ascontiguousarray(counts[lo:hi])).cuda())
            d_ids = c("upload", lambda: torch.from_numpy(np.frombuffer(b"".join(encoded[lo:hi]), dtype=np.uint8).copy()).cuda())
            d_off = c("upload", lambda: torch.from_numpy(off).cuda())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            text = ops.format_counts_csv_cuda(d_counts, d_ids, d_off)
            e1.record()
            torch.cuda.synchronize()
            kernel_ms.append(e0.elapsed_time(e1))
            h = c("device_to_host", lambda: text.cpu().numpy())
            c("file_write", lambda: fh.buffer.write(h.data))
            lo = hi
        c("file_write", lambda: fh.flush())
    return c.parts


def reader_steps(path, kernel_ms):
    """read_feature_file's device road step by step (a plain file)."""
    c = Clock()
    raw, d_text, n, mapped = c("file_read_and_upload", lambda: fileIO._open_fasta_device(path))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    parsed = ops.parse_feature_csv_cuda(d_text[:n])
    e1.record()
    torch.cuda.synchronize()
    kernel_ms.append(e0.elapsed_time(e1))                         # includes the two small copies of the result block and id ranges
    ranges, d_counts = parsed
    counts = c("device_to_host", lambda: d_counts.cpu().numpy())
    ids = c("id_strings", lambda: np.array(fileIO._span_strings(raw, d_text, n, ranges)))
    mapped.close()
    return c.parts, ids, counts


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def bench_shape(rows, width, d):
    progress("table %d x %d" % (rows, width))
    counts, ids = table(rows, width, rows + width)
    host_path, dev_path = os.path.join(d, "host.csv"), os.path.join(d, "dev.csv")
    r = {"rows": rows, "fields": width}
    r["save_counts_s_host"], _ = timed(lambda: fileIO._save_counts_host(counts, ids, host_path))
    fileIO.save_counts(counts[:1000], ids[:1000], dev_path)      # warm-up: library, allocator, kernels
    r["save_counts_s_device"], _ = timed(lambda: fileIO.save_counts(counts, ids, dev_path))
    with open(host_path, "rb") as a, open(dev_path, "rb") as b:
        assert a.read() == b.read(), "device file differs from the host file"
    text_bytes = os.path.getsize(dev_path)
    r["text_bytes"] = text_bytes
    k_write = []
    r["save_counts_steps_s_device"] = writer_steps(counts, ids, dev_path, k_write)
    r["format_kernels_ms"] = sum(k_write)
    r["read_feature_file_s_host"], (h_ids, h_counts) = timed(lambda: fileIO._read_feature_file_host(host_path))
    fileIO.read_feature_file(host_path)                            # warm-up
    r["read_feature_file_s_device"], (g_ids, g_counts) = timed(lambda: fileIO.read_feature_file(host_path))
    assert g_ids.tolist() == h_ids.tolist() and np.array_equal(g_counts, h_counts) and np.array_equal(g_counts, counts)
    k_read = []
    steps, _, _ = reader_steps(host_path, k_read)
    r["read_feature_file_steps_s_device"] = steps
    r["parse_kernels_ms"] = k_read[0]
    moved = text_bytes + counts.nbytes                             # text and int64 counts, each crossing HBM once at least
    for name, ms in (("format", r["format_kernels_ms"]), ("parse", r["parse_kernels_ms"])):
        r["%s_kernels_GBps" % name] = round(moved / ms / 1e6, 1)
        r["%s_kernels_share_of_hbm" % name] = round(moved / ms / 1e6 / HBM_GBPS, 4)
    r["speedup_save_counts"] = round(r["save_counts_s_host"] / r["save_counts_s_device"], 1)
    r["speedup_read_feature_file"] = round(r["read_feature_file_s_host"] / r["read_feature_file_s_device"], 1)
    progress(json.dumps(r))
    return r


def bench_phamer(n_contigs, d):
    progress("phamer -fasta on %d contigs" % n_contigs)
    seq, off = ops.synth_contigs(20261022, 0, n_contigs)
    h_seq, h_off = seq.cpu().numpy(), off.cpu().numpy()
    parts = []
    for i in range(n_contigs):
        parts.append(b">SuperContig_%d_length_%d_ID_%d\n" % (i, h_off[i + 1] - h_off[i], i))
        parts.append(h_seq[h_off[i]:h_off[i + 1]].tobytes() + b"\n")
    out = {"contigs": n_contigs}
    host_save, host_read = fileIO._save_counts_host, fileIO._read_feature_file_host
    dev_save, dev_read = fileIO.save_counts, fileIO.read_feature_file
    scores = {}
    for road in ("device", "host"):
        sub = os.path.join(d, road)
        os.makedirs(sub)
        fasta = os.path.join(sub, "contigs.fasta")
        with open(fasta, "wb") as fh:
            fh.write(b"".join(parts))
        out["fasta_bytes"] = os.path.getsize(fasta)
        fileIO.save_counts, fileIO.read_feature_file = (dev_save, dev_read) if road == "device" else (host_save, host_read)
        try:
            features = os.path.join(sub, "contigs_features.csv")
            out["first_run_s_%s" % road], _ = timed(lambda: phamer.main(["-fasta", fasta, "-out", os.path.join(sub, "o1"), "-l", "0"]))
            out["second_run_s_%s" % road], _ = timed(lambda: phamer.main(["-fasta", fasta, "-features", features, "-out",
                                                                          os.path.join(sub, "o2"), "-l", "0"]))
        finally:
            fileIO.save_counts, fileIO.read_feature_file = dev_save, dev_read
        with open(features, "rb") as a, open(os.path.join(sub, "o2", "phamer_scores.csv"), "rb") as b:
            scores[road] = (a.read(), [line for line in b if not line.startswith(b"#")])      # the header names the directories
    assert scores["device"] == scores["host"], "the two roads wrote different files"
    return out


def save(result, out_path):
    if out_path:
        with open(out_path, "w") as fh:
            fh.write(json.dumps(result) + "\n")


def main():
    _lib.require_cuda()
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    quick = "--quick" in sys.argv
    shapes = [(1_000_000, 256), (250_000, 1024), (62_500, 4096)]
    if quick:
        shapes = [(r // 100, f) for r, f in shapes]
    result = {"card": card(), "host_cores": os.cpu_count(), "torch": torch.__version__,
              "note": "files in a temporary directory: file times are page-cache times", "shapes": []}
    with tempfile.TemporaryDirectory() as d:
        for rows, width in shapes:
            sub = os.path.join(d, "%dx%d" % (rows, width))
            os.makedirs(sub)
            result["shapes"].append(bench_shape(rows, width, sub))
            save(result, out_path)                                 # what is done so far, if a later step does not finish
            shutil.rmtree(sub)
        result["phamer_fasta"] = bench_phamer(2000 if quick else 200_000, d)
    print(json.dumps(result))
    save(result, out_path)


if __name__ == "__main__":
    main()
