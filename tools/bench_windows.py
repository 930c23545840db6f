"""Cost of sliding-window scoring on the flagship workload.

1 M synthetic contigs (seed 20260101, the bench workload) against the shipped references, k = 4.  Variants:
  w5000_s1000            windows of 5 000 bases every 1 000 bases, plain 4-mers
  w5000_s5000            windows of 5 000 bases every 5 000 bases, plain 4-mers
  w5000_s1000_canonical  the first, canonical 4-mers
Per variant: windows, window bases against record bases (how often each base is read), the call time of
ContigScorer.score_windows_device from event timing (mean and median), the mean kmer_hist_kernel / score_tc_kernel /
score_decide_kernel times (option time_kernels, averaged over the slices of a call), windows per second, the counting time per window
base against plain count_cuda per record base over the same contigs in the same run (whether the repeated reads came from L2), and the
rows of each scoring road of the last slice (score_stats).  Prints one JSON object; the card's name and power limit are read in the
same run.

    python tools/bench_windows.py [--contigs 1000000] [--calls 5] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_neighbors import SEED, card, timed_calls   # noqa: E402

KERNELS = ("kmer_hist_kernel", "score_tc_kernel", "score_decide_kernel")
VARIANTS = (("w5000_s1000", 5000, 1000, False), ("w5000_s5000", 5000, 5000, False), ("w5000_s1000_canonical", 5000, 1000, True))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--contigs", type=int, default=1000000)
    ap.add_argument("--calls", type=int, default=5, help="timed calls per variant")
    ap.add_argument("--out", help="also write the JSON here")
    args = ap.parse_args()
    import torch
    from phamers_b200 import _lib, ops, pipeline

    torch.cuda.set_device(0)
    scorers = {False: pipeline.ContigScorer(), True: pipeline.ContigScorer(canonical=True)}
    seq, offsets = ops.synth_contigs(SEED, 0, args.contigs)
    record_bases = int(offsets[-1].item())

    def drain():
        times = {}
        for k in KERNELS:
            try:
                times[k] = ops.last_kernel_ms(k)
            except _lib.PhamersLibraryError:
                times[k] = None
        return times

    _lib.set_option("time_kernels", 1)
    counts = torch.empty((args.contigs, 256), dtype=torch.int32, device="cuda")
    plain = lambda: ops.count_cuda(seq, offsets, 4, out_counts=counts)          # noqa: E731
    timed_calls(plain, 3)
    drain()
    plain_ms = timed_calls(plain, 10)
    plain_hist = drain()["kmer_hist_kernel"]
    summary = {}
    for name, window, step, canonical in VARIANTS:
        scorer = scorers[canonical]
        call = lambda: scorer.score_windows_device(seq, offsets, window, step)   # noqa: E731
        wo, spans, _ = call()
        n_windows = int(wo[-1].item())
        window_bases = int((spans[:, 1] - spans[:, 0]).sum().item())
        timed_calls(call, 1)
        drain()
        ms, kernels = [], {k: [] for k in KERNELS}
        for _ in range(args.calls):
            ms.extend(timed_calls(call, 1))
            for k, v in drain().items():
                if v is not None:
                    kernels[k].append(v)
        slices = (n_windows + scorer.WINDOW_SLICE - 1) // scorer.WINDOW_SLICE
        st = sorted(ms)
        hist_ms = sum(kernels["kmer_hist_kernel"]) / len(kernels["kmer_hist_kernel"]) if kernels["kmer_hist_kernel"] else None
        row = {"windows": n_windows, "window_bases": window_bases, "record_bases": record_bases,
               "read_redundancy": window_bases / record_bases, "slices_per_call": slices,
               "calls": len(st), "call_ms_mean": sum(st) / len(st), "call_ms_median": st[len(st) // 2], "call_ms_min": st[0],
               "windows_per_s": n_windows / (st[len(st) // 2] / 1000.0)}
        for k, v in kernels.items():
            row[k + "_ms_per_slice"] = sum(v) / len(v) if v else None
        if hist_ms is not None and plain_hist:
            row["count_ns_per_window_base"] = hist_ms * slices * 1e6 / window_bases
            row["plain_count_ns_per_record_base"] = plain_hist * 1e6 / record_bases
        stats = ops.score_stats()
        row.update(rows_remeasured=stats["rows_remeasured"], rows_listed=stats["rows_listed"], rows_exhaustive=stats["fallback_rows"])
        summary[name] = row
    _lib.set_option("time_kernels", 0)
    st = sorted(plain_ms)
    res = {"card": card(),
           "workload": "%d synthetic contigs (seed %d, %d bases), shipped references equalised, k = 4, k_neighbors = 3; the score_stats "
                       "roads are those of the last slice of the last call" % (args.contigs, SEED, record_bases),
           "plain_count": {"call_ms_median": st[len(st) // 2], "kmer_hist_kernel_ms": plain_hist},
           "variants": summary}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
