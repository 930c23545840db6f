#!/usr/bin/env python
"""
bench.py -- the PhaMers hot path (k-mer count -> normalise -> score) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--contigs C] [--k 4]
                    [--workload shipped|enlarged|count] [--refs R] [--canonical] [--dump-outputs DIR]

A "step" is one pass of the whole hot path over one batch of synthetic contigs: BASELINE.json configs[1]
("synthetic metagenome 1M contigs, 1-100 kb lognormal lengths, k=4 tetranucleotide, 1xB200"), scored against the shipped
phage / bacteria reference features (2255 + 2255 rows, equalised) with the reference's default 'combo' method.
Scaling is weak: every rank holds its own 1M-contig shard of the same seeded generator (rank r = contigs
[r*C, (r+1)*C)); the only collective is the all-gather of the per-contig scores.

Other workloads (not the headline; used for DESIGN.md's tables): --workload enlarged = BASELINE configs[4], the same contigs
scored against R synthetic reference rows (default 1M: shipped rows resampled with Poisson(20000 p) counts, half labelled
phage), where the tcgen05 distance kernel dominates; --workload count = BASELINE configs[2], counting only for k = 5 / 6 with
--canonical folding.

Prints ONE JSON line (rank 0).  Keys beyond the base contract: roofline (dominant kernel), cpu_baseline (oracle port
timed on this box's host cores, rank 0, N = 1 only), kernels (per-stage device times), contigs_per_sec.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20260101
METRIC = "bases/sec k-mer counted and scored (count + normalise + combo score per step)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--contigs", type=int, default=1000000, help="contigs per GPU")
    ap.add_argument("--total-contigs", type=int, default=0,
                    help="BASELINE configs[3]: this many contigs in total, cut into one shard per GPU balanced by BASES (strong scaling)")
    ap.add_argument("--k", type=int, default=4)
    ap.add_argument("--workload", default="shipped", choices=["shipped", "enlarged", "count"])
    ap.add_argument("--refs", type=int, default=1000000, help="reference rows of --workload enlarged")
    ap.add_argument("--canonical", action="store_true", help="--workload count: fold reverse complements")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (tuning experiments)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the in-bench sanity checks (ablation builds count wrongly on purpose)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of BASELINE configs[2] and configs[4] after the main region")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample-contigs", type=int, default=2400, help="oracle-port sample on rank 0 (about 12 s of one core)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB in all): "
                         "counts, knn, kmeans, combo (counts, freq for --workload count).  An array cut to a seeded sample of its "
                         "rows has their row numbers in DIR/<name>.row_index.npy.  With several GPUs, combo holds the gathered "
                         "scores of every rank; the other arrays are rank 0's shard only.  git ignores bench_outputs/ at the top "
                         "of the tree")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of --impl b200")
    return args


def ncu_traffic():
    """DRAM bytes measured by ncu --set full for the hot kernels (profiles/traffic.json, committed with the capture it
    came from); {} when absent."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh)
    return {}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


DUMP_BYTES = 64 << 20


def dump_outputs(directory, outputs):
    """--dump-outputs: each (name, CUDA tensor) of `outputs` goes to directory/<name>.npy, float64 as float64 and everything else as
    float32 (counts stay below 2^24, so they convert exactly).  Every array gets an equal share of DUMP_BYTES; one larger than its
    share keeps a sample of its rows, drawn with SEED and sorted, whose row numbers go to <name>.row_index.npy.  The sample
    depends on the row count only, so two builds run with the same arguments dump the same rows."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    share = DUMP_BYTES // len(outputs) - 4096                            # room for the .npy headers
    for name, t in outputs:
        dtype = torch.float64 if t.dtype == torch.float64 else torch.float32
        row_bytes = int(np.prod(t.shape[1:], dtype=np.int64)) * dtype.itemsize
        if t.shape[0] * row_bytes > share:
            rows = np.sort(np.random.default_rng(SEED).choice(t.shape[0], size=share // (row_bytes + 8), replace=False))
            np.save(os.path.join(directory, name + ".row_index.npy"), rows.astype(np.float64))
            t = t[torch.from_numpy(rows).to(t.device)]
        np.save(os.path.join(directory, name + ".npy"), t.to(dtype).cpu().numpy())


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.proc = None
        self.device_index = device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    @staticmethod
    def _epoch(stamp):
        import datetime
        try:
            return datetime.datetime.strptime(stamp, "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples taken between the two host times (all samples when none fall inside)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for line in out.strip().split("\n"):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                rows.append((self._epoch(f[0]), float(f[1]), float(f[2]), float(f[3]),
                             [name for name, val in zip(names, f[5:9]) if val.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if r[0] is not None and t_begin is not None and t_begin - 0.02 <= r[0] <= t_end + 0.02]
        used = inside or rows
        reasons = sorted({name for r in used for name in r[4]})
        return {"sm_mhz": statistics.median([r[1] for r in used]) if used else None,
                "sm_max_mhz": max([r[2] for r in used]) if used else None,
                "power_w_max": max([r[3] for r in used]) if used else None,
                "samples": len(used), "samples_inside_timed_region": len(inside), "reasons": reasons}


# ----------------------------------------------------------------------------------------------------------------
# CPU arms (oracle port; the reference is pure Python and cannot travel to the GPU box)
# ----------------------------------------------------------------------------------------------------------------
def _cpu_count_worker(seqs):
    from oracle import phamers_oracle as po
    return [po.count_string(s, 4) for s in seqs]


def host_sample(n_contigs, seed=SEED):
    """Same length law as the device generator (SURVEY.md 8(d)); bases i.i.d. with a per-contig GC fraction."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lengths = np.clip(np.round(np.exp(rng.normal(np.log(10000.0), 1.0, size=n_contigs))), 1000, 100000).astype(np.int64)
    seqs = []
    for length in lengths:
        gc = rng.uniform(0.25, 0.75)
        p = [(1 - gc) / 2, (1 - gc) / 2, gc / 2, gc / 2]
        seqs.append(rng.choice(np.frombuffer(b"ATGC", dtype=np.uint8), size=int(length), p=p).tobytes().decode("ascii"))
    return seqs, int(lengths.sum())


def cpu_pass(seqs, pos, neg, pool=None, centroids=None):
    """One pass of the oracle port over `seqs`: interpreted counting loop (scripts/kmer.py:42-50), normalise, combo
    score with scikit-learn as the reference calls it.  Returns seconds."""
    import numpy as np
    from oracle import phamers_oracle as po
    t0 = time.perf_counter()
    if pool is None:
        counts = np.stack([po.count_string(s, 4) for s in seqs])
    else:
        n = pool._processes
        chunks = [seqs[i::n] for i in range(n)]
        parts = pool.map(_cpu_count_worker, chunks)
        counts = np.zeros((len(seqs), 256), dtype=np.int64)
        for i, part in enumerate(parts):
            counts[i::n] = np.stack(part) if part else counts[i::n]
    pts = po.normalize_counts(counts)
    # centroids are passed in: the reference re-runs k-means once per scoring CALL (~2 s, phamer.py:245-246); over the
    # full 1M-contig call that is negligible, so charging it to a small sample would understate the reference
    po.score_points(pts, pos, neg, centroids=centroids)
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port, kind 'port') with all host cores, on a bounded sample
    of the same workload per step."""
    if rank != 0:
        return
    import multiprocessing as mp
    import numpy as np
    from oracle import phamers_oracle as po
    ref = np.load(os.path.join(ROOT, "phamers_b200", "data", "reference_features.npz"))
    n_ref = min(len(ref["positive_counts"]), len(ref["negative_counts"]))
    pos = po.normalize_counts(ref["positive_counts"][:n_ref].astype(np.int64))
    neg = po.normalize_counts(ref["negative_counts"][:n_ref].astype(np.int64))
    cores = os.cpu_count() or 1
    n_sample = max(cores * 40, 64)
    seqs, bases = host_sample(n_sample)
    cents = po.reference_centroids(pos, neg)
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(args.warmup):
            cpu_pass(seqs[:cores], pos, neg, pool, cents)
        times = [cpu_pass(seqs, pos, neg, pool, cents) for _ in range(args.steps)]
    total = sum(times)
    value = bases * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "bases/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
        # the same workload string as the B200 arm's default line; what is timed is a bounded sample of it
        "config": {"workload": "synthetic metagenome %d contigs/GPU, 1-100 kb lognormal lengths, k=4 (BASELINE configs[1]), "
                               "scored against %d shipped reference rows + %d centroids, method combo"
                               % (args.contigs, 2 * n_ref, cents[0].shape[0] + cents[1].shape[0]),
                   "sample": "bounded: %d contigs of the same length law per step" % n_sample,
                   "sample_contigs": n_sample, "sample_bases": bases, "seed": SEED},
        "contigs_per_sec": n_sample * args.steps / total,
        "cpu_baseline": {"value": value, "unit": "bases/s", "cores": cores, "kind": "port",
                         "sample": "%d contigs / %d bases per step; oracle/phamers_oracle.py (restates scripts/kmer.py:42-50, "
                                   "phamer.py:303-313) over a %d-process pool, scikit-learn k-means + kNN per step"
                                   % (n_sample, bases, cores)},
        "e2e": {"value": value, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------
def other_configs(seq, offsets, bases, counts4, scorer, pos, neg, peaks, n_cent):
    """Short device-timed runs of the BASELINE configs the headline line does not cover, so that one driver run carries them:
    configs[2] -- counting only for k = 5, 6, plain and canonical bins (the same 1 M contigs; SURVEY 8(d) bytes: every base read
    once + one u32 histogram per contig written once) -- and configs[4] -- 100 k of the contigs scored against 1 M synthetic
    reference rows (tcgen05 contraction; flops counted once, against the BURST bf16 peak: the kernel runs for milliseconds)."""
    import torch
    from phamers_b200 import ops
    from tools import workloads
    n = offsets.numel() - 1
    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for k, canonical in ((5, False), (5, True), (6, False), (6, True)):
        bins = ops.num_bins(k, canonical)
        buf = torch.empty((n, bins), dtype=torch.int32, device="cuda")
        for _ in range(2):
            ops.count_cuda(seq, offsets, k, canonical=canonical, out_counts=buf)
        torch.cuda.synchronize()
        ops.last_kernel_ms("kmer_hist_kernel")
        reps = 3
        for _ in range(reps):
            ops.count_cuda(seq, offsets, k, canonical=canonical, out_counts=buf)
        torch.cuda.synchronize()
        ms = ops.last_kernel_ms("kmer_hist_kernel")
        nbytes = bases * 1.0 + n * bins * 4.0
        out["configs[2] k=%d%s" % (k, " canonical" if canonical else "")] = {
            "workload": "counting only, %d contigs, %d output bins (u32)" % (n, bins), "ms_per_launch": ms, "bytes_per_launch": nbytes,
            "bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": nbytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "bases_per_sec": bases / (ms * 1e-3), "launches_timed": reps}
        del buf
    # configs[4]
    n_q, n_refs = min(100000, n), 1000000
    refs_big, n_pos_big = workloads.enlarged_references(pos, neg, n_refs, seed=SEED)
    q = counts4[:n_q].contiguous()
    outs = tuple(torch.empty((n_q,), dtype=torch.float64, device="cuda") for _ in range(3))
    for _ in range(2):
        ops.score_cuda(q, refs_big, n_pos_big, scorer.cent_pos, scorer.cent_neg, 3, out=outs)
    torch.cuda.synchronize()
    ops.last_kernel_ms("score_tc_kernel")
    e0, e1 = ev(), ev()
    reps = 3
    e0.record()
    for _ in range(reps):
        ops.score_cuda(q, refs_big, n_pos_big, scorer.cent_pos, scorer.cent_neg, 3, out=outs)
    e1.record()
    torch.cuda.synchronize()
    call_ms = e0.elapsed_time(e1) / reps
    tc_ms = ops.last_kernel_ms("score_tc_kernel")
    stats = ops.score_stats()
    flops = 2.0 * n_q * (n_refs + n_cent) * 256
    out["configs[4] enlarged reference"] = {
        "workload": "%d contigs (counts) scored against %d synthetic reference rows + %d centroids, combo" % (n_q, n_refs, n_cent),
        "ms_per_call": call_ms, "score_tc_kernel_ms": tc_ms, "flops_per_launch": flops, "bound": "tensor",
        "achieved": flops / (tc_ms * 1e-3) / 1e12, "peak": peaks["bf16_tflops"], "peak_kind": "burst", "unit": "TFLOP/s",
        "frac": flops / (tc_ms * 1e-3) / 1e12 / peaks["bf16_tflops"], "frac_of_sustained": flops / (tc_ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
        "contigs_per_sec": n_q / (call_ms * 1e-3), "fallback_rows": stats["fallback_rows"], "rows_listed": stats["rows_listed"]}
    return out


def run_b200(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from phamers_b200 import _lib, ops, parallel, pipeline, references

    for opt in args.opt:
        name, value = opt.split("=")
        _lib.set_option(name, int(value))
    caps = _lib.device_caps()
    peaks = measured_peaks()

    # ---- workload (untimed) ----
    shard_sizes = None
    if args.total_contigs:
        # strong scaling (BASELINE configs[3]): the whole workload's offsets (lengths only), shards by the prefix sum of bases
        import ctypes
        lengths = torch.empty((args.total_contigs,), dtype=torch.int64, device="cuda")
        _lib.check(_lib.load().phm_synth_lengths(ctypes.c_uint64(SEED), 0, args.total_contigs, _lib.ptr(lengths), _lib.stream_ptr()))
        all_off = np.concatenate(([0], np.cumsum(lengths.cpu().numpy())))
        bounds = parallel.balanced_partition(all_off, world)
        shard_sizes = [int(bounds[r + 1] - bounds[r]) for r in range(world)]
        first, n = int(bounds[rank]), shard_sizes[rank]
        del lengths
    else:
        first, n = rank * args.contigs, args.contigs
    seq, offsets = ops.synth_contigs(SEED, first, n)
    bases = int(offsets[-1].item())
    scoring = args.workload != "count"
    if scoring and args.k != 4:
        raise SystemExit("scoring needs k = 4 (the reference features are 256 wide); use --workload count for k = %d" % args.k)
    pos, neg = references.load_reference_features(equalize=True)
    centroids = references.reference_centroids(pos, neg)               # reference-only preprocessing, cached, untimed
    scorer = pipeline.ContigScorer(pos, neg, centroids=centroids, kmer_length=4)
    n_cent = centroids[0].shape[0] + centroids[1].shape[0]
    if args.workload == "enlarged":
        # SURVEY 8(d) config 5: R rows, each a shipped row re-sampled as ~20000 4-mers (Poisson counts), positives first
        from tools import workloads
        refs_dev, n_positive = workloads.enlarged_references(pos, neg, args.refs, seed=SEED)
    else:
        refs_dev, n_positive = scorer.refs, scorer.n_positive
    n_refs = int(refs_dev.shape[0])
    _lib.set_option("time_kernels", 1)
    torch.cuda.synchronize()

    stream = torch.cuda.current_stream()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    # results are written into buffers allocated once: a production loop scores batch after batch into the same memory, and
    # allocator calls inside the timed region would only add host noise
    bins = ops.num_bins(args.k, args.canonical)
    buf_counts = torch.empty((n, bins), dtype=torch.int32, device="cuda")
    buf_freq = torch.empty((n, bins), dtype=torch.float64, device="cuda") if not scoring else None
    buf_scores = tuple(torch.empty((n,), dtype=torch.float64, device="cuda") for _ in range(3))

    def step(timed):
        e0, e1 = ev(), ev()
        e0.record(stream)
        if scoring:
            # ONE library call for the whole path (phm_count_score): the histogram kernel also emits the scorer's query
            # operands and the scorer forms count / row total where it needs an exact feature, so stage 2 (normalise) has no
            # pass of its own and the float64 feature matrix is never written
            counts, knn, km, combo = ops.count_score_cuda(seq, offsets, refs_dev, n_positive, scorer.cent_pos, scorer.cent_neg, 3,
                                                          out_counts=buf_counts, out=buf_scores)
        else:
            counts, freq = ops.count_cuda(seq, offsets, args.k, canonical=args.canonical, counts=True, freq=True,
                                          out_counts=buf_counts, out_freq=buf_freq)
            combo = buf_scores[2]
        e1.record(stream)
        if world > 1 and scoring:
            gathered = parallel.gather_scores(combo, shard_sizes or [n] * world)
        else:
            gathered = combo
        if timed:
            step.events.append((e0, e1))
        # what a caller of this path receives (the all-gathered combo scores when several GPUs score)
        outputs = ([("counts", counts), ("knn", knn), ("kmeans", km), ("combo", gathered)] if scoring
                   else [("counts", counts), ("freq", freq)])
        return counts, gathered, outputs
    step.events = []

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                                # running well before the timed region starts
    for _ in range(args.warmup):
        step(False)
    torch.cuda.synchronize()
    ops.last_kernel_ms("kmer_hist_kernel")                             # empty the event rings of the warm-up launches
    if scoring:
        ops.last_kernel_ms("score_tc_kernel")
    if world > 1:
        dist.barrier()
    launches0 = ops.kernel_launches()
    t_start, t_end = ev(), ev()
    torch.cuda.synchronize()
    wall_begin = time.time()
    t_start.record(stream)
    for _ in range(args.steps):
        counts, gathered, outputs = step(True)
    t_end.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall_end = time.time()
    clocks = sampler.stop(wall_begin, wall_end) if rank == 0 else None
    launches = ops.kernel_launches() - launches0
    elapsed_ms = t_start.elapsed_time(t_end)
    stage_ms = [e0.elapsed_time(e1) for e0, e1 in step.events]
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    tot_bases = torch.tensor([bases], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot_bases, op=dist.ReduceOp.SUM)
    elapsed_ms = float(t.item())
    all_bases = float(tot_bases.item())

    score_stats = ops.score_stats() if (scoring and ops.score_path_option != 1) else None
    tc_ms = ops.last_kernel_ms("score_tc_kernel") if (scoring and ops.score_path_option != 1) else None
    hist_ms = ops.last_kernel_ms("kmer_hist_kernel")

    # ---- sanity inside the bench: row sums of the last step's counts (clean synthetic bases) ----
    lengths = offsets[1:] - offsets[:-1]
    assert args.no_check or bool((counts.sum(dim=1, dtype=torch.int64) == lengths - (args.k - 1)).all()), "count row sums are wrong"
    if scoring and not args.no_check:
        assert bool(torch.isfinite(gathered).all()) and gathered.numel() == (sum(shard_sizes) if shard_sizes else n * world)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)

    # ---- end to end through the public API with HOST buffers (copies inside the timed region) ----
    e2e = None
    if not args.no_e2e and args.workload == "shipped":
        try:
            host_seq = torch.empty((bases,), dtype=torch.uint8, pin_memory=True)
            host_seq.copy_(seq)
            host_off = torch.empty((n + 1,), dtype=torch.int64, pin_memory=True)
            host_off.copy_(offsets)
            torch.cuda.synchronize()
            scorer.score_host(host_seq, host_off)                     # warm-up (staging allocation)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                host_scores = scorer.score_host(host_seq, host_off)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            lo = sum(shard_sizes[:rank]) if shard_sizes else rank * n
            assert np.array_equal(host_scores, gathered[lo:lo + n].cpu().numpy())
            e2e = {"value": all_bases * args.e2e_steps / dt, "unit": "bases/s",
                   "h2d_bytes_per_step": int(bases + 8 * (n + 1)), "d2h_bytes_per_step": int(8 * n),
                   "steps": args.e2e_steps, "ms_per_step": 1e3 * dt / args.e2e_steps,
                   "api": "phamers_b200.pipeline.ContigScorer.score_host (pinned host bases + offsets in, host scores out)"}
            del host_seq
        except RuntimeError as exc:                                   # e.g. pinned allocation refused
            e2e = {"value": None, "unit": "bases/s", "error": str(exc)[:200]}

    configs = None
    if world == 1 and args.workload == "shipped" and args.k == 4 and not args.no_configs:
        configs = other_configs(seq, offsets, bases, buf_counts, scorer, pos, neg, peaks, n_cent)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (algorithmic work / CUDA-event duration of that kernel, see DESIGN.md section 4) ----
    c_ms = hist_ms                                                     # the counting stage is this one kernel
    s_ms = statistics.mean(stage_ms) - hist_ms                         # everything else in the library call(s)
    # counting stage = ONE kernel launch (+ a 256-byte memset): ASCII read once + u32 counts written once (SURVEY 8(d));
    # the count-only workloads also write the float64 features
    count_bytes = bases * 1.0 + n * bins * 4.0 + (0.0 if scoring else n * bins * 8.0)
    traffic = ncu_traffic()
    bpb = traffic.get("kmer_hist_kernel_bytes_per_base", 0)
    count_roof = {"bound": "hbm", "achieved": count_bytes / (c_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                  # DRAM bytes of THIS workload extrapolated from the committed ncu capture (bytes per base of a 296 k-contig
                  # launch, profiles/traffic.json): a static figure, not a counter read during this run
                  "traffic": bpb * bases or None, "traffic_source": "static: profiles/traffic.json (ncu --set full capture) x bases",
                  "kernel": "kmer_hist_kernel", "peak_source": peaks["source"],
                  "bytes_per_launch": count_bytes, "ms_per_launch": c_ms, "frac_of_8tbs_nominal": count_bytes / (c_ms * 1e-3) / 8e12}
    count_roof["frac"] = count_roof["achieved"] / count_roof["peak"]
    score_roof = None
    if tc_ms:
        score_flops = 2.0 * n * (n_refs + n_cent) * 256
        # a kernel of a few milliseconds inside a step of ~10 ms runs at full clocks: the BURST peak is its denominator; the
        # enlarged-reference workload keeps the tensor cores busy for ~0.1 s per step and meets the power cap: sustained peak
        burst = tc_ms < 20.0
        score_roof = {"bound": "tensor", "achieved": score_flops / (tc_ms * 1e-3) / 1e12,
                      "peak": peaks["bf16_tflops"] if burst else peaks["bf16_tflops_sustained"], "peak_kind": "burst" if burst else "sustained",
                      "unit": "TFLOP/s", "traffic": None,
                      "kernel": "score_tc_kernel (tcgen05 kind::f16, one FP16 product per algorithmic product, FP32 accumulate)",
                      "peak_source": peaks["source"], "flops_per_launch": score_flops, "ms_per_launch": tc_ms,
                      "stage_ms": s_ms}
        score_roof["frac"] = score_roof["achieved"] / score_roof["peak"]
    dominant = score_roof if (score_roof and tc_ms >= c_ms) else count_roof

    # ---- CPU baseline (oracle port, rank 0, N = 1 only, bounded sample) ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline and args.workload == "shipped":
        from oracle import phamers_oracle as po
        seqs, sample_bases = host_sample(args.cpu_sample_contigs)
        dt = cpu_pass(seqs, pos, neg, None, (centroids[0], centroids[1]))
        cpu = {"value": sample_bases / dt, "unit": "bases/s", "cores": 1, "kind": "port",
               "host_cores": os.cpu_count(),
               "sample": "%d contigs / %d bases of the same length law, one pass in %.1f s: interpreted counting loop on 1 core "
                         "(as the reference runs), scikit-learn kNN + centroid loop (k-means untimed)" % (len(seqs), sample_bases, dt)}

    value = all_bases * args.steps / (elapsed_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "bases/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong" if shard_sizes else "weak", "vs_baseline": None,
        "dtype": "u8 bases -> u32 counts -> f64 features (formed in-kernel) -> f64 scores", "data": "synthetic",
        "config": {"workload": ("synthetic metagenome %d contigs/GPU, 1-100 kb lognormal lengths, k=%d (BASELINE configs[%s]), "
                                % (n, args.k, "3" if shard_sizes else {"shipped": "1", "enlarged": "4", "count": "2"}[args.workload]))
                               + ("scored against %d %s reference rows + %d centroids, method combo"
                                  % (n_refs, "shipped" if args.workload == "shipped" else "synthetic", n_cent) if scoring
                                  else "counting + normalising only%s" % (", canonical bins" if args.canonical else "")),
                   "contigs_per_gpu": n, "bases_per_gpu": bases, "seed": SEED,
                   "shards": ("%d contigs in total, shards balanced by bases (parallel.balanced_partition): %s contigs" % (args.total_contigs, shard_sizes))
                             if shard_sizes else None,
                   "l2_policy": "inputs (%.1f GB of bases per step) are far larger than the 126 MB L2" % (bases / 1e9),
                   "parallelism": "contigs sharded over %d GPU(s), references replicated, one NCCL all-gather of scores" % world,
                   "options": args.opt},
        "contigs_per_sec": (sum(shard_sizes) if shard_sizes else n * world) * args.steps / (elapsed_ms * 1e-3),
        "kernels": {"count_ms": c_ms, "score_ms": s_ms, "score_tc_kernel_ms": tc_ms, "count_roofline": count_roof,
                    "score_roofline": score_roof, "score_stats": score_stats, "configs": configs},
        "roofline": dominant, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        "device": {"sm": "%d.%d" % (caps.sm_major, caps.sm_minor), "sm_count": caps.sm_count},
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    # NCCL announces its version on STDOUT when the environment asks for NCCL_DEBUG=VERSION/INFO; stdout carries the JSON line
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "INFO", "TRACE") and "NCCL_DEBUG_FILE" not in os.environ:
        os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
