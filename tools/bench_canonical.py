"""Cost of strand-independent (canonical 4-mer) scoring against plain scoring on the flagship workload.

1 M synthetic contigs (seed 20260101) from their bases on the device to scores against the shipped references (k = 3), each call
timed by CUDA events, after warm-up, the variants alternated within one run for about a second each:
  plain fused         count_score_cuda: the histogram kernel emits the scorer's operands (phm_count_score)
  plain two-call      count_cuda + score_cuda on the counts (phm_kmer_count + phm_score_counts, dim 256)
  canonical two-call  count_cuda(canonical) + score_cuda on the canonical counts (dim 136, tensor-core road)
  canonical exhaustive  count_cuda(canonical, freq) + score_cuda on the features with score_path "exact" (a few calls only)
Per variant: call time, mean kmer_hist_kernel / score_tc_kernel / score_decide_kernel times (option time_kernels) and the rows of
each road (score_stats).  Prints one JSON object; the card's name and power limit are read in the same run.

    python tools/bench_canonical.py [--contigs 1000000] [--seconds 1.0] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--contigs", type=int, default=1000000)
    ap.add_argument("--seconds", type=float, default=1.0, help="timed device time per variant")
    ap.add_argument("--exhaustive-calls", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON here")
    args = ap.parse_args()
    import torch
    from phamers_b200 import _lib, ops, pipeline

    torch.cuda.set_device(0)
    plain, canon = pipeline.ContigScorer(), pipeline.ContigScorer(canonical=True)
    seq, offsets = ops.synth_contigs(SEED, 0, args.contigs)
    n = args.contigs
    c256 = torch.empty((n, 256), dtype=torch.int32, device="cuda")
    c136 = torch.empty((n, 136), dtype=torch.int32, device="cuda")
    f136 = torch.empty((n, 136), dtype=torch.float64, device="cuda")
    out = tuple(torch.empty((n,), dtype=torch.float64, device="cuda") for _ in range(3))

    def score(s, counts):
        return ops.score_cuda(counts, s.refs, s.n_positive, s.cent_pos, s.cent_neg, 3, out=out)

    def exhaustive():
        ops.count_cuda(seq, offsets, 4, canonical=True, counts=False, freq=True, out_freq=f136)
        ops.set_score_path("exact")
        try:
            score(canon, f136)
        finally:
            ops.set_score_path("auto")

    variants = {
        "plain fused": lambda: ops.count_score_cuda(seq, offsets, plain.refs, plain.n_positive, plain.cent_pos, plain.cent_neg, 3,
                                                    out_counts=c256, out=out),
        "plain two-call": lambda: (ops.count_cuda(seq, offsets, 4, out_counts=c256), score(plain, c256)),
        "canonical two-call": lambda: (ops.count_cuda(seq, offsets, 4, canonical=True, out_counts=c136), score(canon, c136)),
    }
    _lib.set_option("time_kernels", 1)

    def drain():                                                    # mean time per kernel since the last drain; None: not launched
        times = {}
        for k in KERNELS:
            try:
                times[k] = ops.last_kernel_ms(k)
            except _lib.PhamersLibraryError:
                times[k] = None
        return times

    for fn in variants.values():                                    # warm-up: modules, workspaces, the L2 state of a call
        timed_calls(fn, 3)
    drain()
    one = max(sum(timed_calls(fn, 2)) / 2 for fn in variants.values())
    drain()
    rounds = max(4, int(args.seconds * 1000.0 / one / 4))           # 4 calls of each variant per round, alternating
    result = {name: {"call_ms": [], "kernels": {k: [] for k in KERNELS}} for name in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            result[name]["call_ms"].extend(timed_calls(fn, 4))
            for k, v in drain().items():
                result[name]["kernels"][k].append(v)
            result[name]["roads"] = ops.score_stats()
    exhaustive()                                                    # warm-up
    drain()
    ex_ms = timed_calls(exhaustive, args.exhaustive_calls)
    result["canonical exhaustive"] = {"call_ms": ex_ms, "kernels": {k: [v] for k, v in drain().items()}, "roads": None}
    _lib.set_option("time_kernels", 0)

    summary = {}
    for name, r in result.items():
        st = sorted(r["call_ms"])
        row = {"calls": len(st), "call_ms_mean": sum(st) / len(st), "call_ms_median": st[len(st) // 2], "call_ms_min": st[0],
               "call_ms_max": st[-1]}
        for k, v in r["kernels"].items():
            v = [x for x in v if x is not None]
            row[k + "_ms"] = sum(v) / len(v) if v else None
        if r["roads"]:
            row.update(rows_remeasured=r["roads"]["rows_remeasured"], rows_listed=r["roads"]["rows_listed"],
                       rows_exhaustive=r["roads"]["fallback_rows"])
        summary[name] = row
    res = {"card": card(),
           "workload": "%d synthetic contigs (seed %d) from bases to scores, shipped references equalised (%d rows; centroids %d + %d "
                       "plain, %d + %d canonical), k = 3" % (n, SEED, plain.refs.shape[0], plain.cent_pos.shape[0],
                                                             plain.cent_neg.shape[0], canon.cent_pos.shape[0], canon.cent_neg.shape[0]),
           "variants": summary}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
