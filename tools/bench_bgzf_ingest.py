#!/usr/bin/env python
"""BGZF-compressed FASTA ingest: the synthetic 60-column FASTA of bench_fasta_ingest.py written plain and as BGZF (level 6, members
of 65 280 input bytes, as bgzip writes them), then
  - gzip.decompress of the BGZF file on the host (one core),
  - phm_inflate alone (CUDA events over many launches; the output is larger than the 126 MB L2),
  - read_fasta_arrays_cuda and ContigScorer.score_fasta wall time on the BGZF file and on the plain file (page cache warm),
with compressed and decompressed bytes, GB/s of output, and the card's name and power limit from the same run.
    python tools/bench_bgzf_ingest.py [contigs] [--out FILE.json]"""
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phamers_b200 import fileIO, ops, pipeline  # noqa: E402

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf(raw, level=6, block=65280):
    parts = []
    for lo in range(0, len(raw), block):
        data = raw[lo:lo + block]
        c = zlib.compressobj(level, zlib.DEFLATED, -15)
        payload = c.compress(data) + c.flush()
        size = 18 + len(payload) + 8
        parts.append(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + (size - 1).to_bytes(2, "little") + payload
                     + zlib.crc32(data).to_bytes(4, "little") + len(data).to_bytes(4, "little"))
    return b"".join(parts) + EOF_BLOCK


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def progress(msg):
    print(msg, file=sys.stderr, flush=True)


def wall(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_path in args:
        args.remove(out_path)
    n_contigs = int(args[0]) if args else 40000
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
    raw = np.concatenate(parts).tobytes()
    progress("FASTA: %d bytes; writing BGZF" % len(raw))
    t0 = time.perf_counter()
    packed = bgzf(raw)
    compress_s = time.perf_counter() - t0
    progress("BGZF: %d bytes in %.1f s; gzip.decompress" % (len(packed), compress_s))
    t0 = time.perf_counter()
    assert gzip.decompress(packed) == raw
    host_s = time.perf_counter() - t0

    progress("phm_inflate")
    table = fileIO.bgzf_members(packed)
    t0 = time.perf_counter()
    fileIO.bgzf_members(packed)
    members_s = time.perf_counter() - t0
    d_in = torch.from_numpy(np.frombuffer(packed, dtype=np.uint8).copy()).cuda()
    out = ops.inflate_cuda(d_in, table)
    assert out.numel() == len(raw) and torch.equal(out, torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).cuda())
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ops.inflate_cuda(d_in, table)
    e1.record()
    torch.cuda.synchronize()
    inflate_ms = e0.elapsed_time(e1) / reps                   # each call also copies the table in and synchronises once

    progress("read_fasta_arrays_cuda and score_fasta")
    scorer = pipeline.ContigScorer()
    result = {"card": card(), "contigs": n_contigs, "members": int(table.shape[0]), "plain_bytes": len(raw),
              "bgzf_bytes": len(packed), "ratio": round(len(raw) / len(packed), 3), "bgzip_write_s_host": round(compress_s, 2),
              "gzip_decompress_s_host": round(host_s, 3), "gzip_decompress_GBps_host": round(len(raw) / host_s / 1e9, 3),
              "bgzf_members_s_host": round(members_s, 4), "phm_inflate_ms": round(inflate_ms, 3),
              "phm_inflate_GBps_out": round(len(raw) / inflate_ms / 1e6, 2)}
    with tempfile.TemporaryDirectory() as d:
        plain, gz = os.path.join(d, "x.fasta"), os.path.join(d, "x.fasta.gz")
        with open(plain, "wb") as fh:
            fh.write(raw)
        with open(gz, "wb") as fh:
            fh.write(packed)
        for name, path in (("plain", plain), ("bgzf", gz)):
            s = wall(lambda: fileIO.read_fasta_arrays_cuda(path))
            result["read_fasta_arrays_cuda_s_%s" % name] = round(s, 4)
            result["read_fasta_arrays_cuda_GBps_%s" % name] = round(len(raw) / s / 1e9, 2)
            result["score_fasta_s_%s" % name] = round(wall(lambda: scorer.score_fasta(path)), 4)
        a, b = scorer.score_fasta(plain), scorer.score_fasta(gz)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    line = json.dumps(result)
    print(line)
    if out_path:
        with open(out_path, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
