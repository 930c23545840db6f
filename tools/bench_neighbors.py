"""Cost of the neighbour report (phm_score_counts_neighbors) against plain scoring (phm_score_counts) on the flagship workload.

1 M synthetic contigs (seed 20260101) counted on the device, scored against the shipped references (k = 3) by score_cuda and by
score_neighbors_cuda in alternation, each call timed by CUDA events, after warm-up, for about a second per variant; per variant the
mean stage time, the mean score_decide_kernel time (option time_kernels) and the rows of each road (score_stats).  Then one run of
BASELINE configs[4]: 100 k of the contigs against 1 M synthetic references.  Prints one JSON object; the card's name and power limit
are read in the same run.

    python tools/bench_neighbors.py [--contigs 1000000] [--seconds 1.0] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 20260101


def card():
    try:
        text = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [f.strip() for f in text.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, IndexError, ValueError, subprocess.SubprocessError) as exc:
        return {"error": str(exc)}


def timed_calls(fn, reps):
    import torch
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--contigs", type=int, default=1000000)
    ap.add_argument("--seconds", type=float, default=1.0, help="timed device time per variant")
    ap.add_argument("--out", help="also write the JSON here")
    args = ap.parse_args()
    import torch
    from phamers_b200 import _lib, ops, pipeline
    from tools import workloads

    torch.cuda.set_device(0)
    scorer = pipeline.ContigScorer()
    seq, offsets = ops.synth_contigs(SEED, 0, args.contigs)
    counts, _ = ops.count_cuda(seq, offsets, 4)
    del seq
    refs, n_pos, cp, cn = scorer.refs, scorer.n_positive, scorer.cent_pos, scorer.cent_neg
    variants = {
        "scores": lambda: ops.score_cuda(counts, refs, n_pos, cp, cn, 3),
        "scores+neighbors": lambda: ops.score_neighbors_cuda(counts, refs, n_pos, cp, cn, 3),
    }
    _lib.set_option("time_kernels", 1)
    for fn in variants.values():                                    # warm-up: modules, workspaces, the L2 state of a call
        timed_calls(fn, 3)
    ops.last_kernel_ms("score_decide_kernel")
    ops.last_kernel_ms("score_tc_kernel")
    one = sum(timed_calls(variants["scores+neighbors"], 2)) / 2
    ops.last_kernel_ms("score_decide_kernel")
    ops.last_kernel_ms("score_tc_kernel")
    rounds = max(4, int(args.seconds * 1000.0 / one / 8))          # 8 calls of each variant per round, alternating
    result = {name: {"stage_ms": [], "score_decide_kernel_ms": [], "score_tc_kernel_ms": []} for name in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            ms = timed_calls(fn, 8)
            result[name]["stage_ms"].extend(ms)
            result[name]["score_decide_kernel_ms"].append(ops.last_kernel_ms("score_decide_kernel"))
            result[name]["score_tc_kernel_ms"].append(ops.last_kernel_ms("score_tc_kernel"))
            result[name]["roads"] = ops.score_stats()
    summary = {}
    for name, r in result.items():
        st = sorted(r["stage_ms"])
        summary[name] = {"calls": len(st), "stage_ms_mean": sum(st) / len(st), "stage_ms_median": st[len(st) // 2],
                         "stage_ms_min": st[0], "stage_ms_max": st[-1],
                         "score_decide_kernel_ms": sum(r["score_decide_kernel_ms"]) / len(r["score_decide_kernel_ms"]),
                         "score_tc_kernel_ms": sum(r["score_tc_kernel_ms"]) / len(r["score_tc_kernel_ms"]),
                         "rows_remeasured": r["roads"]["rows_remeasured"], "rows_listed": r["roads"]["rows_listed"],
                         "rows_exhaustive": r["roads"]["fallback_rows"]}

    # BASELINE configs[4]: 100 k contigs against 1 M synthetic references, once per variant after one warm-up call
    pos = scorer.refs[:n_pos].cpu().numpy()
    neg = scorer.refs[n_pos:].cpu().numpy()
    big, big_pos = workloads.enlarged_references(pos, neg, 1000000, seed=SEED)
    q = counts[:100000].contiguous()
    enlarged = {}
    for name, fn in (("scores", lambda: ops.score_cuda(q, big, big_pos, cp, cn, 3)),
                     ("scores+neighbors", lambda: ops.score_neighbors_cuda(q, big, big_pos, cp, cn, 3))):
        timed_calls(fn, 1)
        ops.last_kernel_ms("score_decide_kernel")
        ms = timed_calls(fn, 1)[0]
        stats = ops.score_stats()
        enlarged[name] = {"call_ms": ms, "score_decide_kernel_ms": ops.last_kernel_ms("score_decide_kernel"),
                          "rows_remeasured": stats["rows_remeasured"], "rows_listed": stats["rows_listed"],
                          "rows_exhaustive": stats["fallback_rows"]}
    _lib.set_option("time_kernels", 0)
    out = {"card": card(), "workload": "%d synthetic contigs (seed %d), counts, shipped references (%d rows, %d + %d centroids), k = 3"
           % (args.contigs, SEED, refs.shape[0], cp.shape[0], cn.shape[0]),
           "shipped": summary,
           "configs[4] enlarged": dict(enlarged, workload="100000 contigs x 1000000 synthetic references, k = 3, one timed call each")}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
