"""Cost of span scoring on the flagship workload.

1 M synthetic contigs (seed 20260101, the bench workload) against the shipped references, k = 4, plain 4-mers.  Variants:
  records   every record as one span: phm_kmer_count_spans against plain count_cuda on the same contigs in the same run, i.e. the
            cost of the span plan (validating count pass, one synchronisation, fill pass) against the record plan
  genes     gene-like spans tiling every contig (lognormal lengths around 1 kb, about 16 M spans, so many SPAN_SLICEs), counted and
            scored by ContigScorer.score_spans_device: spans per second and time per span base, comparable with the windows'
            counting cost per window base (DESIGN 4.4d)
  regions   a few thousand region-sized spans (10 - 200 kb, log-uniform, so some are counted in tiles) on genome-size records (the
            same bases cut into 4 Mb records), counted and scored
Per variant: the call time from event timing (mean, median, min), the mean kmer_hist_kernel / score_tc_kernel / score_decide_kernel
time per slice (option time_kernels) and the counting time per span base.  Prints one JSON object; the card's name and power limit
are read in the same run.

    python tools/bench_spans.py [--contigs 1000000] [--calls 5] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_neighbors import SEED, card, timed_calls   # noqa: E402

KERNELS = ("kmer_hist_kernel", "score_tc_kernel", "score_decide_kernel")


def gene_spans(offsets, rng, mean_log=np.log(1000.0), sigma=0.5):
    """Spans tiling every record: gene lengths drawn lognormal end to end over the whole sequence, cut at record boundaries."""
    total = int(offsets[-1])
    n = int(total / np.exp(mean_log + sigma * sigma / 2) * 1.05) + 16
    cuts = np.cumsum(np.maximum(1, rng.lognormal(mean_log, sigma, size=n)).astype(np.int64))
    cuts = np.unique(np.concatenate((cuts[cuts < total], offsets)))
    starts, ends = cuts[:-1], cuts[1:]
    rec = np.searchsorted(offsets, starts, side="right") - 1
    return np.stack((rec, starts - offsets[rec], ends - offsets[rec]), axis=1).astype(np.int64)


def region_spans(lengths, rng, n=4000):
    rec = rng.integers(0, len(lengths), size=n)
    size = np.exp(rng.uniform(np.log(10000), np.log(200000), size=n)).astype(np.int64)
    start = (rng.random(n) * (lengths[rec] - size)).astype(np.int64)
    return np.stack((rec, start, start + size), axis=1).astype(np.int64)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--contigs", type=int, default=1000000)
    ap.add_argument("--calls", type=int, default=5, help="timed calls per variant")
    ap.add_argument("--out", help="also write the JSON here")
    args = ap.parse_args()
    import torch
    from phamers_b200 import _lib, ops, pipeline

    torch.cuda.set_device(0)
    rng = np.random.default_rng(SEED)
    scorer = pipeline.ContigScorer()
    seq, offsets = ops.synth_contigs(SEED, 0, args.contigs)
    h_off = offsets.cpu().numpy()
    record_bases = int(h_off[-1])
    genome_off = torch.from_numpy(np.append(np.arange(0, record_bases - (4 << 20) + 1, 4 << 20), record_bases).astype(np.int64)).cuda()

    def drain():
        times = {}
        for k in KERNELS:
            try:
                times[k] = ops.last_kernel_ms(k)
            except _lib.PhamersLibraryError:
                times[k] = None
        return times

    def measure(call, slices, span_bases):
        call()
        timed_calls(call, 1)
        drain()
        ms, kernels = [], {k: [] for k in KERNELS}
        for _ in range(args.calls):
            ms.extend(timed_calls(call, 1))
            for k, v in drain().items():
                if v is not None:
                    kernels[k].append(v)
        st = sorted(ms)
        row = {"calls": len(st), "call_ms_mean": sum(st) / len(st), "call_ms_median": st[len(st) // 2], "call_ms_min": st[0],
               "slices_per_call": slices, "span_bases": span_bases}
        for k, v in kernels.items():
            row[k + "_ms_per_slice"] = sum(v) / len(v) if v else None
        if row["kmer_hist_kernel_ms_per_slice"]:
            row["count_ps_per_span_base"] = row["kmer_hist_kernel_ms_per_slice"] * slices * 1e9 / span_bases
        return row

    _lib.set_option("time_kernels", 1)
    summary = {}
    # 1. every record as one span against the record plan
    counts = torch.empty((args.contigs, 256), dtype=torch.int32, device="cuda")
    whole = torch.stack((torch.arange(args.contigs, device="cuda"), torch.zeros_like(offsets[1:]), offsets[1:] - offsets[:-1]), dim=1)
    plain = measure(lambda: ops.count_cuda(seq, offsets, 4, out_counts=counts), 1, record_bases)
    spans_row = measure(lambda: ops.count_spans_cuda(seq, offsets, whole, 4, out_counts=counts), 1, record_bases)
    summary["records"] = {"spans": args.contigs, "count_spans": spans_row, "plain_count_cuda": plain,
                          "span_over_record_call": spans_row["call_ms_median"] / plain["call_ms_median"]}
    del whole
    # 2. gene-like spans tiling every contig
    genes = gene_spans(h_off, rng)
    d_genes = torch.from_numpy(genes).cuda()
    gene_bases = int((genes[:, 2] - genes[:, 1]).sum())
    slices = (len(genes) + scorer.SPAN_SLICE - 1) // scorer.SPAN_SLICE
    row = measure(lambda: scorer.score_spans_device(seq, offsets, d_genes), slices, gene_bases)
    row.update(spans=len(genes), span_length_mean=gene_bases / len(genes), span_length_median=float(np.median(genes[:, 2] - genes[:, 1])),
               spans_per_s=len(genes) / (row["call_ms_median"] / 1000.0))
    summary["genes"] = row
    del d_genes, genes
    # 3. region-sized spans on genome-size records
    regions = region_spans(np.diff(genome_off.cpu().numpy()), rng)
    region_bases = int((regions[:, 2] - regions[:, 1]).sum())
    d_regions = torch.from_numpy(regions).cuda()
    row = measure(lambda: scorer.score_spans_device(seq, genome_off, d_regions), 1, region_bases)
    row.update(spans=len(regions), records=int(genome_off.numel() - 1), tiled_spans=int(((regions[:, 2] - regions[:, 1]) >= 131072).sum()),
               spans_per_s=len(regions) / (row["call_ms_median"] / 1000.0))
    summary["regions"] = row
    _lib.set_option("time_kernels", 0)
    res = {"card": card(),
           "workload": "%d synthetic contigs (seed %d, %d bases), shipped references equalised, k = 4, k_neighbors = 3, plain 4-mers; "
                       "kernel times are means over the launches of the timed calls (the kmer_hist_kernel bracket covers the planning "
                       "passes, the synchronisation of the span call, the histogram and the finish pass)" % (args.contigs, SEED, record_bases),
           "variants": summary}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
