#!/usr/bin/env python
"""gzip-compressed FASTA ingest: the synthetic 60-column FASTA of bench_bgzf_ingest.py written plain and as single-member gzip at
levels 1 and 6 (what gzip / pigz write), then for each level
  - gzip.open(path).read() on the host (one core, page cache warm),
  - phm_gunzip_index + phm_gunzip_extract alone (ops.gunzip_cuda; CUDA events, best of a few calls), at several chunk sizes,
    and the index call on its own (finder, pass A and the chain walk) to show where the time goes,
  - the index statistics (chunks, rejected candidates, repair rounds, serial bytes),
  - read_fasta_arrays_cuda and ContigScorer.score_fasta wall time on the gzip file and on the plain file,
with compressed and decompressed bytes, GB/s of output, and the card's name and power limit from the same run.
    python tools/bench_gzip_ingest.py [contigs] [--out FILE.json]"""
import ctypes
import gzip
import json
import os
import sys
import tempfile
import time
import zlib

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench_bgzf_ingest import card, progress, wall  # noqa: E402
from phamers_b200 import _lib, fileIO, ops, pipeline  # noqa: E402

CHUNKS = (64 << 10, 128 << 10, 256 << 10)
DEFAULT_CHUNK = 128 << 10


def synthetic_fasta(n_contigs):
    seq, off = ops.synth_contigs(20260101, 0, n_contigs)
    h_seq, h_off = seq.cpu().numpy(), off.cpu().numpy()
    parts = []
    for i in range(n_contigs):
        body = h_seq[h_off[i]:h_off[i + 1]]
        pad = (-len(body)) % 60
        lines = np.concatenate((body, np.full(pad, 32, dtype=np.uint8))).reshape(-1, 60)
        lines = np.concatenate((lines, np.full((lines.shape[0], 1), 10, dtype=np.uint8)), axis=1).reshape(-1)
        parts.append(np.frombuffer(b">SuperContig_%d_length_%d_ID_%d\n" % (i, len(body), i), dtype=np.uint8))
        parts.append(lines)
    return np.concatenate(parts).tobytes()


def gzip_file(raw, level):
    c = zlib.compressobj(level, zlib.DEFLATED, 31)
    step = 64 << 20
    return b"".join([c.compress(raw[i:i + step]) for i in range(0, len(raw), step)] + [c.flush()])


def device_ms(d_in, member, reps=3):
    """Best of `reps` CUDA-event timings of the whole ops.gunzip_cuda call and of phm_gunzip_index alone."""
    lib = _lib.require_cuda()
    begin, end, _, isize = member
    payload = d_in[begin:end]
    n = end - begin
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best, best_index, out = float("inf"), float("inf"), None
    for _ in range(reps):
        out = None
        torch.cuda.synchronize()
        e0.record()
        out = ops.gunzip_cuda(d_in, member)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
        ws = torch.empty((lib.phm_gunzip_index_workspace_bytes(n),), dtype=torch.uint8, device="cuda")
        info = (ctypes.c_int64 * 7)()
        e0.record()
        _lib.check(lib.phm_gunzip_index(_lib.ptr(payload), n, isize, info, _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        e1.record()
        torch.cuda.synchronize()
        best_index = min(best_index, e0.elapsed_time(e1))
        del ws
    return best, best_index, out


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_path in args:
        args.remove(out_path)
    n_contigs = int(args[0]) if args else 150000
    raw = synthetic_fasta(n_contigs)
    d_raw = torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda()
    progress("FASTA: %d bytes" % len(raw))
    result = {"card": card(), "contigs": n_contigs, "plain_bytes": len(raw), "levels": {}}
    scorer = pipeline.ContigScorer()
    with tempfile.TemporaryDirectory() as d:
        plain = os.path.join(d, "x.fasta")
        with open(plain, "wb") as fh:
            fh.write(raw)
        result["read_fasta_arrays_cuda_s_plain"] = round(wall(lambda: fileIO.read_fasta_arrays_cuda(plain)), 4)
        result["score_fasta_s_plain"] = round(wall(lambda: scorer.score_fasta(plain)), 4)
        want = scorer.score_fasta(plain)
        for level in (1, 6):
            progress("level %d: compressing" % level)
            t0 = time.perf_counter()
            packed = gzip_file(raw, level)
            row = {"gzip_bytes": len(packed), "ratio": round(len(raw) / len(packed), 3),
                   "compress_s_host": round(time.perf_counter() - t0, 2)}
            path = os.path.join(d, "x%d.fasta.gz" % level)
            with open(path, "wb") as fh:
                fh.write(packed)
            progress("level %d: host gzip.open(path).read()" % level)
            t0 = time.perf_counter()
            with gzip.open(path, "rb") as fh:
                assert fh.read() == raw
            host_s = time.perf_counter() - t0
            row["gzip_read_s_host"] = round(host_s, 3)
            row["gzip_read_GBps_host"] = round(len(raw) / host_s / 1e9, 3)
            member = fileIO.gzip_member(packed)
            d_in = torch.from_numpy(np.frombuffer(packed, dtype=np.uint8).copy()).cuda()
            for chunk in CHUNKS:
                progress("level %d: gunzip at %d KiB chunks" % (level, chunk >> 10))
                _lib.set_option("gunzip_chunk_bytes", chunk)
                stats = {}
                out = ops.gunzip_cuda(d_in, member, stats=stats)
                assert out.numel() == len(raw) and torch.equal(out, d_raw[:len(raw)])
                del out
                ms, index_ms, out = device_ms(d_in, member)
                del out
                row["chunk_%dk" % (chunk >> 10)] = {"gunzip_ms": round(ms, 2), "index_ms": round(index_ms, 2),
                                                    "extract_ms": round(ms - index_ms, 2),
                                                    "GBps_out": round(len(raw) / ms / 1e6, 2), "stats": stats}
            _lib.set_option("gunzip_chunk_bytes", DEFAULT_CHUNK)
            del d_in
            progress("level %d: read_fasta_arrays_cuda and score_fasta" % level)
            row["read_fasta_arrays_cuda_s"] = round(wall(lambda: fileIO.read_fasta_arrays_cuda(path)), 4)
            row["score_fasta_s"] = round(wall(lambda: scorer.score_fasta(path)), 4)
            got = scorer.score_fasta(path)
            assert np.array_equal(want[0], got[0]) and np.array_equal(want[1], got[1])
            result["levels"][str(level)] = row
            torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if out_path:
        with open(out_path, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
