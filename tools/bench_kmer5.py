"""Cost of scoring 5-mer count rows on the tensor cores (1024 plain and 512 canonical bins) against the exhaustive float64 road.

1 M synthetic contigs (seed 20260101) from their bases on the device to scores, counted at k = 5 plain and canonical.  References:
synthetic 5-mer rows of the shipped reference set's size (2255 + 2255 equalised rows), counted on the device from other synthetic
genomes (seed 20260202), with centroids of the library's k-means (86 per class).  Each call is timed by CUDA events after warm-up,
the two widths alternated within one run for about a second each:
  plain 1024        count_cuda(5) + score_cuda on the counts (phm_kmer_count + phm_score_counts, dim 1024, tensor-core road)
  canonical 512     count_cuda(5, canonical) + score_cuda on the counts (dim 512)
  * exhaustive      the same rows as float64 features (count_cuda freq) with score_path "exact" (a few calls only)
Per variant: call time, mean kmer_hist_kernel / score_tc_kernel / score_decide_kernel times (option time_kernels), the rows of each
road (score_stats), and the algorithmic rate 2 n (R + C_pos + C_neg) W over score_tc_kernel time and over the call.  Prints one JSON
object; the card's name, power limit and max SM clock are read in the same run.

    python tools/bench_kmer5.py [--contigs 1000000] [--seconds 1.0] [--out FILE]
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
REF_SEED = 20260202
N_REF = 2255                        # rows per class of the shipped references, equalised


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--contigs", type=int, default=1000000)
    ap.add_argument("--seconds", type=float, default=1.0, help="timed device time per variant")
    ap.add_argument("--exhaustive-calls", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON here")
    args = ap.parse_args()
    import torch
    from phamers_b200 import _lib, ops, references

    torch.cuda.set_device(0)
    n = args.contigs
    seq, offsets = ops.synth_contigs(SEED, 0, n)
    g_seq, g_off = ops.synth_contigs(REF_SEED, 0, 2 * N_REF)
    refs = {}
    for canonical, width in ((False, 1024), (True, 512)):
        counts, _ = ops.count_cuda(g_seq, g_off, 5, canonical=canonical)
        R = ops.normalize_cuda(counts)
        pos, neg = R[:N_REF].cpu().numpy(), R[N_REF:].cpu().numpy()
        cp, cn = references.reference_centroids(pos, neg, 86)
        refs[width] = (R.contiguous(), N_REF, torch.from_numpy(cp).cuda(), torch.from_numpy(cn).cuda(), canonical)
    counts = {w: torch.empty((n, w), dtype=torch.int32, device="cuda") for w in refs}
    out = tuple(torch.empty((n,), dtype=torch.float64, device="cuda") for _ in range(3))

    def road(width):
        R, n_pos, cp, cn, canonical = refs[width]
        return lambda: (ops.count_cuda(seq, offsets, 5, canonical=canonical, out_counts=counts[width]),
                        ops.score_cuda(counts[width], R, n_pos, cp, cn, 3, out=out))

    def exhaustive(width):
        R, n_pos, cp, cn, canonical = refs[width]
        feats = torch.empty((n, width), dtype=torch.float64, device="cuda")

        def call():
            ops.count_cuda(seq, offsets, 5, canonical=canonical, counts=False, freq=True, out_freq=feats)
            ops.set_score_path("exact")
            try:
                ops.score_cuda(feats, R, n_pos, cp, cn, 3, out=out)
            finally:
                ops.set_score_path("auto")
        return call

    variants = {"plain 1024": road(1024), "canonical 512": road(512)}
    widths = {"plain 1024": 1024, "canonical 512": 512}
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
    rounds = max(2, int(args.seconds * 1000.0 / one / 4))           # 4 calls of each variant per round, alternating
    result = {name: {"call_ms": [], "kernels": {k: [] for k in KERNELS}} for name in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            result[name]["call_ms"].extend(timed_calls(fn, 4))
            for k, v in drain().items():
                result[name]["kernels"][k].append(v)
            result[name]["roads"] = ops.score_stats()
    for name in list(variants):
        fn = exhaustive(widths[name])
        fn()                                                        # warm-up
        drain()
        ex_ms = timed_calls(fn, args.exhaustive_calls)
        result[name + " exhaustive"] = {"call_ms": ex_ms, "kernels": {k: [v] for k, v in drain().items()}, "roads": None}
        widths[name + " exhaustive"] = widths[name]
        torch.cuda.empty_cache()
    _lib.set_option("time_kernels", 0)

    summary = {}
    for name, r in result.items():
        st = sorted(r["call_ms"])
        R, _, cp, cn, _ = refs[widths[name]]
        flop = 2.0 * n * (R.shape[0] + cp.shape[0] + cn.shape[0]) * widths[name]
        row = {"calls": len(st), "call_ms_mean": sum(st) / len(st), "call_ms_median": st[len(st) // 2], "call_ms_min": st[0],
               "call_ms_max": st[-1], "algorithmic_tflop": flop / 1e12,
               "tflops_over_call": flop / (st[len(st) // 2] * 1e-3) / 1e12}
        for k, v in r["kernels"].items():
            v = [x for x in v if x is not None]
            row[k + "_ms"] = sum(v) / len(v) if v else None
        if row["score_tc_kernel_ms"] and r["roads"]:
            row["tflops_over_score_tc_kernel"] = flop / (row["score_tc_kernel_ms"] * 1e-3) / 1e12
        if r["roads"]:
            row.update(rows_remeasured=r["roads"]["rows_remeasured"], rows_listed=r["roads"]["rows_listed"],
                       rows_exhaustive=r["roads"]["fallback_rows"])
        summary[name] = row
    res = {"card": card(),
           "workload": "%d synthetic contigs (seed %d) from bases to scores at k = 5; references: %d + %d synthetic genomes (seed %d) "
                       "counted at k = 5, centroids 86 + 86 (library k-means); k_neighbors 3" % (n, SEED, N_REF, N_REF, REF_SEED),
           "variants": summary}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
