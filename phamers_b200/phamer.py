"""
Drop-in for the hot-path part of the reference's scripts/phamer.py: the `phamer_scorer` object and the
`score_points(scoring_data, positive_training_data, negative_training_data, method=None)` facade (:451-468).

Scoring methods on the device: 'knn' (:268-273), 'kmeans' (:240-256) and the default 'combo' (:303-313, knn + kmeans,
range +-1.7616 -- not [-1, 1] as the reference README says).  The other methods of the reference ('dbscan', 'svm',
'density', 'silhouette') are evaluation experiments that are not data-parallel per contig and are out of scope
(SURVEY.md section 2); asking for one raises NotImplementedError.

Differences a caller can observe, all deliberate:
  * k-means on the reference sets is cached per reference set (references.py) instead of re-run on every call.
  * a query row with NaN features (contig with no countable k-mer) scores NaN instead of making scikit-learn raise.
"""
import logging
import os

import numpy as np

from . import fileIO, kmer, references

logger = logging.getLogger(__name__)
logger.setLevel(logging.WARNING)


class phamer_scorer(object):
    """scripts/phamer.py:42-449 (hot-path attributes and methods only)."""

    def __init__(self):
        self.input_directory = None
        self.features_file = None
        self.fasta_file = None
        self.output_directory = None
        self.data_directory = None
        self.positive_features_file = None
        self.negative_features_file = None

        self.data_ids = None
        self.data_points = None
        self.positive_ids = None
        self.positive_data = None
        self.negative_ids = None
        self.negative_data = None

        self.length_requirement = 5000                       # :68
        self.scoring_method = "combo"                        # :70
        self.all_scoring_methods = ["dbscan", "kmeans", "knn", "svm", "density", "silhouette", "combo"]   # :71
        self.kmer_length = 4                                 # :77
        self.k_clusters = 86                                 # :78
        self.k_neighbors = 3                                 # :79
        # strand-independent scoring: references and contigs are folded onto canonical k-mers (a k-mer and its reverse complement
        # share a bin) before they are normalised, so a contig and its reverse complement get the same score
        self.canonical = False
        self.scores = None
        # filled by score_neighbors(): per contig the k_neighbors nearest references (ids, 1 = phage / 0 = bacteria, distances)
        # and the nearest phage / bacteria cluster (k-means label, -1 without centroids) with its distance
        self.neighbor_ids = None
        self.neighbor_labels = None
        self.neighbor_distances = None
        self.nearest_clusters = None
        self.nearest_cluster_distances = None
        # filled by score_windows(): one entry per window of the contigs kept by the length screen -- the contig's id and its position
        # in the FASTA, the window's [start, end) in the contig, its score; and by find_regions(): the phage-like regions they show
        self.screened_length = 0
        self.window_ids = None
        self.window_records = None
        self.window_spans = None
        self.window_scores = None
        self.region_ids = None
        self.region_spans = None
        self.region_windows = None
        self.region_mean_scores = None
        self.region_max_scores = None
        self.region_records = None
        # filled by score_spans() / score_regions(): per span its contig id, [start, end), name and score, and the references and
        # clusters behind the score (as the neighbor_* attributes)
        self.span_ids = None
        self.span_spans = None
        self.span_names = None
        self.span_scores = None
        self.span_neighbor_ids = None
        self.span_neighbor_labels = None
        self.span_neighbor_distances = None
        self.span_nearest_clusters = None
        self.span_nearest_cluster_distances = None

    # ---- data -------------------------------------------------------------------------------------------
    def load_reference_data(self, positive_features_file=None, negative_features_file=None):
        """:110-123.  Reference sets come from feature CSVs (the reference's FASTA fallback is dead code,
        SURVEY.md 8(b)); with no files given the shipped tables are used."""
        if positive_features_file and negative_features_file:
            self.positive_ids, pos = fileIO.read_feature_file(positive_features_file)
            self.negative_ids, neg = fileIO.read_feature_file(negative_features_file)
        else:
            self.positive_ids, pos, self.negative_ids, neg = references.load_reference_counts()
        self.positive_data, self.negative_data = kmer.normalize_counts(self._features(pos)), kmer.normalize_counts(self._features(neg))

    def _features(self, counts):
        """Count rows as scored: unchanged, or with self.canonical folded onto canonical k-mers.  In canonical mode rows that are
        already canonical width are taken as they are; any other width is a ValueError."""
        if not self.canonical:
            return counts
        counts = np.asarray(counts)
        width = counts.shape[-1] if counts.ndim else 0
        if width == 4 ** self.kmer_length:
            return kmer.canonical_fold(counts, self.kmer_length)
        from . import ops
        if width == ops.num_bins(self.kmer_length, canonical=True):
            return counts
        raise ValueError("canonical scoring at k = %d takes rows of %d (plain) or %d (canonical) k-mer counts, not %d"
                         % (self.kmer_length, 4 ** self.kmer_length, ops.num_bins(self.kmer_length, canonical=True), width))

    def load_data(self, length_requirement=None):
        """:125-142: a features CSV wins over counting the FASTA; freshly counted features are cached next to the
        FASTA as <fasta>_features.csv; then normalise and screen by length."""
        if self.features_file is not None and os.path.exists(self.features_file):
            self.data_ids, self.data_points = fileIO.read_feature_file(self.features_file)
        elif self.fasta_file is not None and os.path.exists(self.fasta_file):
            self.data_ids, self.data_points = kmer.count_file(self.fasta_file, self.kmer_length, normalize=False)
            self.features_file = "{base}_features.csv".format(base=os.path.splitext(self.fasta_file)[0])
            fileIO.save_counts(self.data_points, self.data_ids, self.features_file)
        else:
            logger.error("No input fasta file or features file. Exiting...")
            raise SystemExit()
        self.data_points = kmer.normalize_counts(self._features(self.data_points))
        if length_requirement is None:
            length_requirement = self.length_requirement
        if length_requirement and self.fasta_file is not None and os.path.exists(self.fasta_file):
            self.screen_by_length(length_requirement)

    def screen_by_length(self, length_requirement=None):
        """:144-157: keep contigs whose parsed sequence has at least `length_requirement` characters."""
        if length_requirement:
            self.length_requirement = length_requirement
        self.screened_length = self.length_requirement
        ids, lengths = fileIO.get_fasta_lengths(self.fasta_file)
        long_ids = [ids[i] for i in range(len(ids)) if lengths[i] >= self.length_requirement]
        self.data_points = self.data_points[np.isin(self.data_ids, long_ids)]
        self.data_ids = np.array(long_ids)

    def equalize_reference_data(self):
        """:159-175."""
        num_ref = min(self.positive_data.shape[0], self.negative_data.shape[0])
        self.positive_data = self.positive_data[:num_ref]
        self.negative_data = self.negative_data[:num_ref]
        if self.positive_ids is not None:
            self.positive_ids = self.positive_ids[:num_ref]
        if self.negative_ids is not None:
            self.negative_ids = self.negative_ids[:num_ref]
        self.num_positive = self.num_negative = num_ref

    # ---- scoring ----------------------------------------------------------------------------------------
    def _device_inputs(self):
        import torch
        pts = np.ascontiguousarray(self.data_points, dtype=np.float64)
        refs = self._device_references(pts.shape[1])                                   # raises first when there is no device
        return (torch.from_numpy(pts).cuda(),) + refs

    def _device_references(self, width):
        """(references, positives, positive centroids, negative centroids, k_neighbors) on the device, as score_points uses them."""
        import torch
        from . import _lib
        _lib.require_cuda()
        pos = np.ascontiguousarray(self.positive_data, dtype=np.float64)
        neg = np.ascontiguousarray(self.negative_data, dtype=np.float64)
        if self.scoring_method in ("kmeans", "combo"):
            cpos, cneg = references.reference_centroids(pos, neg, self.k_clusters)
        else:
            cpos = cneg = np.zeros((0, width))
        refs = torch.from_numpy(np.vstack((pos, neg))).cuda()                         # :186
        return (refs, pos.shape[0], torch.from_numpy(np.ascontiguousarray(cpos)).cuda(),
                torch.from_numpy(np.ascontiguousarray(cneg)).cuda(), self.k_neighbors)

    def _device_scores(self):
        from . import ops
        out = ops.score_cuda(*self._device_inputs())
        return [t.cpu().numpy() for t in out]

    def score_points(self):
        """:177-195."""
        self.num_points = self.data_points.shape[0]
        self.num_positive = self.positive_data.shape[0]
        self.num_negative = self.negative_data.shape[0]
        self.train = np.vstack((self.positive_data, self.negative_data))
        self.labels = np.append(np.ones(self.num_positive), np.zeros(self.num_negative))
        if self.scoring_method not in self.all_scoring_methods:
            raise KeyError(self.scoring_method)
        if self.scoring_method not in ("knn", "kmeans", "combo"):
            raise NotImplementedError("scoring method %r is outside the B200 hot path (knn / kmeans / combo only)"
                                      % self.scoring_method)
        knn, km, combo = self._device_scores()
        self.scores = {"knn": knn, "kmeans": km, "combo": combo}[self.scoring_method]
        return self.scores

    def score_neighbors(self):
        """score_points that also fills neighbor_ids / neighbor_labels / neighbor_distances ([contigs, k_neighbors]: the references
        that cast the kNN vote, nearest first) and nearest_clusters / nearest_cluster_distances ([contigs, 2]: the phage and the
        bacteria cluster whose centroid distances enter the kmeans score), from the same device call.  The scores are those of
        score_points.  A contig with no countable k-mer gets id "", label -1, cluster -1 and distance NaN."""
        from . import ops
        self.num_points = self.data_points.shape[0]
        self.num_positive = self.positive_data.shape[0]
        self.num_negative = self.negative_data.shape[0]
        if self.scoring_method not in self.all_scoring_methods:
            raise KeyError(self.scoring_method)
        if self.scoring_method not in ("knn", "kmeans", "combo"):
            raise NotImplementedError("scoring method %r is outside the B200 hot path (knn / kmeans / combo only)"
                                      % self.scoring_method)
        knn, km, combo, ref_i, ref_d, cen_i, cen_d = [t.cpu().numpy() for t in ops.score_neighbors_cuda(*self._device_inputs())]
        self.scores = {"knn": knn, "kmeans": km, "combo": combo}[self.scoring_method]
        self.neighbor_ids, self.neighbor_labels = self._reference_names(ref_i)
        self.neighbor_distances = ref_d
        self.nearest_clusters = cen_i
        self.nearest_cluster_distances = cen_d
        return self.scores

    def _reference_names(self, ref_index):
        """Rows of the stacked references (positives first; -1 for none) -> (their ids, labels 1 = phage / 0 = bacteria / -1 none)."""
        n_pos, n_neg = self.positive_data.shape[0], self.negative_data.shape[0]
        pos_ids = self.positive_ids if self.positive_ids is not None else np.arange(n_pos)
        neg_ids = self.negative_ids if self.negative_ids is not None else np.arange(n_neg)
        all_ids = np.concatenate((np.asarray(pos_ids).astype(str), np.asarray(neg_ids).astype(str), [""]))
        ref_index = np.asarray(ref_index, dtype=np.int64)
        return all_ids[ref_index], np.where(ref_index < 0, -1, (ref_index < n_pos).astype(np.int64))   # -1 picks the trailing ""

    def score_windows(self, window, step=None):
        """Scores overlapping windows along every contig the length screen kept (all records of the FASTA when no screen ran), with
        the scorer's references, k-mer length, k_neighbors, method and canonical mode: fills window_ids, window_records (position of
        the contig in the FASTA), window_spans ([windows, 2], 0-based half-open, in the contig) and window_scores.  A contig of length
        L has one window [0, L) when L <= window, else windows every `step` bases (default: window) plus one aligned to its end.
        Needs the FASTA file: features alone say nothing about where in a contig the phage lies."""
        from . import pipeline
        if self.fasta_file is None or not os.path.exists(self.fasta_file):
            raise ValueError("window scores need the FASTA file of the contigs; a features file alone has no positions")
        if self.scoring_method not in ("knn", "kmeans", "combo"):
            raise NotImplementedError("scoring method %r is outside the B200 hot path (knn / kmeans / combo only)" % self.scoring_method)
        pos = np.ascontiguousarray(self.positive_data, dtype=np.float64)
        neg = np.ascontiguousarray(self.negative_data, dtype=np.float64)
        scorer = pipeline.ContigScorer(pos, neg, k_clusters=self.k_clusters, k_neighbors=self.k_neighbors, kmer_length=self.kmer_length,
                                       centroids=references.reference_centroids(pos, neg, self.k_clusters), canonical=self.canonical)
        self.window_ids, self.window_records, self.window_spans, self.window_scores = scorer.score_windows_fasta(
            self.fasta_file, int(window), int(step or window), length_requirement=self.screened_length, method=self.scoring_method)
        return self.window_scores

    def score_spans(self, ids, spans, names=None, lines=None):
        """Scores any spans of the contigs of the FASTA file -- ids [n] contig names (score-file ids, or the titles' first tokens as
        BED files carry them), spans [n, 2] 0-based half-open (start, end) -- each exactly as score_neighbors scores its bases written
        as a contig of their own, with the references behind each score.  Fills span_ids, span_spans, span_names ('.' when not
        given), span_scores and span_neighbor_ids / _labels / _distances, span_nearest_clusters / _cluster_distances (as
        score_neighbors).  Spans ignore the length screen: the user named them.  lines: where each span came from, named by the
        error of a span outside its contig."""
        from . import pipeline
        self._check_span_inputs("span scores")
        self.span_ids = np.asarray(ids).astype(str)
        self.span_spans = np.asarray(spans, dtype=np.int64).reshape(-1, 2)
        self.span_names = np.asarray(names).astype(str) if names is not None else np.full((len(self.span_ids),), ".")
        return self._score_span_table(*pipeline.fasta_spans(self.fasta_file, self.span_ids, self.span_spans, lines))

    def score_regions(self):
        """score_spans for the regions find_regions found, in their order: each region scored as one sequence, with name '.'."""
        import torch
        self._check_span_inputs("region scores")
        self.span_ids = np.asarray(self.region_ids).astype(str)
        self.span_spans = np.asarray(self.region_spans, dtype=np.int64).reshape(-1, 2)
        self.span_names = np.full((len(self.span_ids),), ".")
        table = np.concatenate((np.asarray(self.region_records, dtype=np.int64).reshape(-1, 1), self.span_spans), axis=1)
        _, d_seq, d_off = fileIO.read_fasta_arrays_cuda(self.fasta_file)
        return self._score_span_table(d_seq, d_off, torch.from_numpy(np.ascontiguousarray(table)).cuda())

    def _check_span_inputs(self, what):
        if self.fasta_file is None or not os.path.exists(self.fasta_file):
            raise ValueError("%s need the FASTA file of the contigs; a features file alone has no positions" % what)
        if self.scoring_method not in ("knn", "kmeans", "combo"):
            raise NotImplementedError("scoring method %r is outside the B200 hot path (knn / kmeans / combo only)" % self.scoring_method)

    def _score_span_table(self, d_seq, d_off, table):
        """Counts the spans of a device table [n, 3] (record, start, end) as float64 feature rows and scores them with the inputs and
        entry point of score_neighbors, pipeline.ContigScorer.SPAN_SLICE spans per call."""
        import torch
        from . import ops, pipeline
        width = ops.num_bins(self.kmer_length, self.canonical)
        inputs = self._device_references(width)
        key = {"knn": 0, "kmeans": 1, "combo": 2}[self.scoring_method]
        parts = []
        for first in range(0, table.shape[0], pipeline.ContigScorer.SPAN_SLICE):
            _, feats = ops.count_spans_cuda(d_seq, d_off, table[first:first + pipeline.ContigScorer.SPAN_SLICE], self.kmer_length,
                                            canonical=self.canonical, counts=False, freq=True)
            out = ops.score_neighbors_cuda(feats, *inputs)
            parts.append([out[key]] + list(out[3:]))
        if not parts:
            parts = [[torch.empty((0, n) if n else (0,), dtype=d, device="cuda") for n, d in
                      ((0, torch.float64), (self.k_neighbors, torch.int64), (self.k_neighbors, torch.float64), (2, torch.int64),
                       (2, torch.float64))]]
        out = [torch.cat(col).cpu().numpy() for col in zip(*parts)]
        self.span_scores, ref_i, self.span_neighbor_distances, self.span_nearest_clusters, self.span_nearest_cluster_distances = out
        self.span_neighbor_ids, self.span_neighbor_labels = self._reference_names(ref_i)
        return self.span_scores

    def find_regions(self):
        """Phage-like regions from the window scores (host only): a region is a maximal run of consecutive windows of one contig whose
        scores are all >= 0 (a NaN window ends a run; a run never crosses contigs).  Fills region_ids, region_spans ([regions, 2]: start
        of the first window, end of the last), region_windows, region_mean_scores and region_max_scores."""
        scores = np.asarray(self.window_scores, dtype=np.float64)
        records = np.asarray(self.window_records, dtype=np.int64)
        spans = np.asarray(self.window_spans, dtype=np.int64).reshape(-1, 2)
        hit = scores >= 0
        opens = hit.copy()
        opens[1:] &= ~(hit[:-1] & (records[1:] == records[:-1]))
        first = np.flatnonzero(opens)
        run = np.cumsum(opens)[hit] - 1                                  # region of every window that scores >= 0
        windows = np.bincount(run, minlength=len(first)).astype(np.int64)
        last = first + windows - 1
        starts = np.concatenate(([0], np.cumsum(windows)[:-1])).astype(np.int64)
        in_runs = scores[hit]
        self.region_ids = np.asarray(self.window_ids)[first]
        self.region_records = records[first]
        self.region_spans = np.stack((spans[first, 0], spans[last, 1]), axis=1).reshape(-1, 2)
        self.region_windows = windows
        self.region_mean_scores = np.add.reduceat(in_runs, starts) / windows if len(first) else np.zeros(0)
        self.region_max_scores = np.maximum.reduceat(in_runs, starts) if len(first) else np.zeros(0)
        return self.region_spans

    def knn_score_points(self):
        return self._with_method("knn")

    def kmeans_score_points(self):
        return self._with_method("kmeans")

    def combo_score_points(self):
        return self._with_method("combo")

    def _with_method(self, method):
        saved, self.scoring_method = self.scoring_method, method
        try:
            return self.score_points()
        finally:
            self.scoring_method = saved

    # ---- files (scripts/phamer.py:405-436) -------------------------------------------------------------
    def find_data_files(self):
        """:406-415: default places of the reference feature tables inside a data directory."""
        self.positive_features_file = os.path.join(self.data_directory, "reference_features", "positive_features.csv")
        self.negative_features_file = os.path.join(self.data_directory, "reference_features", "negative_features.csv")

    def find_input_files(self):
        """:417-436: the single .fasta / .fa file of the input directory (a '*genes' file only as a last resort) and its single .csv."""
        if self.input_directory and os.path.isdir(self.input_directory):
            fasta_files = [f for f in os.listdir(self.input_directory) if f.endswith(".fasta") or f.endswith(".fa")]
            if len(fasta_files) == 1:
                self.fasta_file = os.path.join(self.input_directory, fasta_files[0])
            elif fasta_files:
                for potential_file in fasta_files:
                    if not os.path.splitext(potential_file)[0].endswith("genes"):
                        self.fasta_file = os.path.join(self.input_directory, potential_file)
                        break
                if self.fasta_file is None:
                    self.fasta_file = os.path.join(self.input_directory, fasta_files[0])
            features_files = [f for f in os.listdir(self.input_directory) if f.endswith(".csv")]
            if len(features_files) == 1:
                self.features_file = os.path.join(self.input_directory, features_files[0])

    # ---- outputs ----------------------------------------------------------------------------------------
    def get_phamer_output_filename(self):
        return os.path.join(self.output_directory, "phamer_scores.csv")              # :439-441

    def make_summary_file(self, args=None):
        """:316-323."""
        self.phamer_output_filename = self.get_phamer_output_filename()
        fileIO.save_phamer_scores(self.data_ids, self.scores, self.phamer_output_filename, args=args)

    def make_window_files(self, args=None):
        """<out>/phamer_windows.csv (one row per window) and <out>/phamer_regions.csv (one row per phage-like region)."""
        self.phamer_windows_filename = os.path.join(self.output_directory, "phamer_windows.csv")
        self.phamer_regions_filename = os.path.join(self.output_directory, "phamer_regions.csv")
        fileIO.save_phamer_windows(self.window_ids, self.window_spans, self.window_scores, self.phamer_windows_filename, args=args)
        fileIO.save_phamer_regions(self.region_ids, self.region_spans, self.region_windows, self.region_mean_scores,
                                   self.region_max_scores, self.phamer_regions_filename, args=args)

    def make_span_file(self, file_name, args=None):
        """<out>/<file_name>: one row per span of score_spans / score_regions with its score and the references behind it."""
        path = os.path.join(self.output_directory, file_name)
        fileIO.save_phamer_spans(self.span_ids, self.span_spans, self.span_names, self.span_scores, self.span_neighbor_ids,
                                 self.span_neighbor_labels, self.span_neighbor_distances, self.span_nearest_clusters,
                                 self.span_nearest_cluster_distances, path, args=args)
        return path

    def make_neighbors_file(self, args=None):
        """<out>/phamer_neighbors.csv: the rows of phamer_scores.csv with the references and clusters behind each score."""
        self.phamer_neighbors_filename = os.path.join(self.output_directory, "phamer_neighbors.csv")
        fileIO.save_phamer_neighbors(self.data_ids, self.neighbor_ids, self.neighbor_labels, self.neighbor_distances,
                                     self.nearest_clusters, self.nearest_cluster_distances, self.phamer_neighbors_filename, args=args)


def score_points(scoring_data, positive_training_data, negative_training_data, method=None):
    """scripts/phamer.py:451-468."""
    scorer = phamer_scorer()
    if method is not None:
        scorer.scoring_method = method
    scorer.data_points = scoring_data
    scorer.positive_data = positive_training_data
    scorer.negative_data = negative_training_data
    return scorer.score_points()


def decide_files(scorer, args):
    """scripts/phamer.py:470-507: explicit command-line files win over what the input / data directories hold; the output goes
    to -out, else to <input directory>/phamer_output (the reference's misspelt `input_drectory` branch is dead code)."""
    if args.kmer_length:
        scorer.kmer_length = args.kmer_length
    if args.input_directory:
        scorer.input_directory = args.input_directory
        scorer.find_input_files()
    if args.data_directory:
        scorer.data_directory = args.data_directory
        scorer.find_data_files()
    if args.output_directory:
        scorer.output_directory = args.output_directory
    else:
        base = scorer.input_directory or os.path.dirname(args.fasta_file or args.features_file or "") or "."
        scorer.output_directory = os.path.join(base, "phamer_output")
    scorer.fasta_file = args.fasta_file or scorer.fasta_file
    scorer.features_file = args.features_file or scorer.features_file
    scorer.positive_features_file = args.positive_features or scorer.positive_features_file
    scorer.negative_features_file = args.negative_features or scorer.negative_features_file


def main(argv=None):
    """The reference's command line (scripts/phamer.py:510-599) for the hot path: count the contigs of a FASTA (or read their
    feature CSV), score them against the reference features, write <out>/phamer_scores.csv (and with -neighbors
    <out>/phamer_neighbors.csv; with -window <out>/phamer_windows.csv and <out>/phamer_regions.csv, and with -region_scores also
    <out>/phamer_region_scores.csv; with -spans <out>/phamer_spans.csv).  t-SNE and plots are out of scope."""
    import argparse
    parser = argparse.ArgumentParser(description="Scores contigs based on feature similarity (B200 path)",
                                     formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    parser.add_argument("-in", "--input_directory", help="Directory containing input files")
    parser.add_argument("-fasta", "--fasta_file", help="Fasta compilation file of unknown sequences")
    parser.add_argument("-features", "--features_file", help="Input feature file")
    parser.add_argument("-data", "--data_directory", help="Directory containing all relevant data files")
    parser.add_argument("-pf", "--positive_features", help="positive feature file")
    parser.add_argument("-nf", "--negative_features", help="negative feature file")
    parser.add_argument("-out", "--output_directory", help="Directory to put output files")
    parser.add_argument("-k", "--kmer_length", type=int, default=4, help="Length of k-mers analyzed")
    parser.add_argument("-l", "--length_requirement", type=int, default=5000, help="Sequence length requirement")
    parser.add_argument("-equal", "--equalize_reference", action="store_true", help="Use same number of reference data from each")
    parser.add_argument("-m", "--method", default="combo", help="Learning algorithm name")
    parser.add_argument("-canonical", "--canonical_kmers", action="store_true",
                        help="Fold every k-mer with its reverse complement, so that a contig scores the same on either strand")
    parser.add_argument("-neighbors", "--write_neighbors", action="store_true",
                        help="Also write phamer_neighbors.csv: the nearest references and clusters behind each score")
    parser.add_argument("-window", "--window_length", type=int,
                        help="Also score windows of this many bases along each contig: phamer_windows.csv and phamer_regions.csv")
    parser.add_argument("-step", "--window_step", type=int, help="Bases between window starts (default: the window length)")
    parser.add_argument("-region_scores", "--region_scores", action="store_true",
                        help="With -window, also score each phage-like region as one sequence: phamer_region_scores.csv")
    parser.add_argument("-spans", "--span_file",
                        help="BED file of contig intervals to score, each as one sequence: phamer_spans.csv")
    parser.add_argument("-do_tsne", "--do_tsne", action="store_true", help="(out of scope)")
    parser.add_argument("-plot", "--plot_tsne", action="store_true", help="(out of scope)")
    args = parser.parse_args(argv)
    if args.do_tsne or args.plot_tsne:
        raise NotImplementedError("t-SNE and plotting are outside the B200 hot path")
    if args.window_length is not None and args.window_length < 1:
        parser.error("-window must be >= 1")
    if args.window_step is not None and (args.window_length is None or args.window_step < 1):
        parser.error("-step needs -window and must be >= 1")
    if args.region_scores and args.window_length is None:
        parser.error("-region_scores needs -window: regions are found from the window scores")
    scorer = phamer_scorer()
    decide_files(scorer, args)
    if args.window_length is not None and not (scorer.fasta_file and os.path.exists(scorer.fasta_file)):
        parser.error("-window needs the FASTA file of the contigs (-fasta, or -in with a .fasta / .fa file): "
                     "a features file alone has no positions")
    if args.span_file is not None and not (scorer.fasta_file and os.path.exists(scorer.fasta_file)):
        parser.error("-spans needs the FASTA file of the contigs (-fasta, or -in with a .fasta / .fa file): "
                     "a features file alone has no positions")
    scorer.scoring_method = args.method
    scorer.canonical = args.canonical_kmers
    scorer.load_reference_data(scorer.positive_features_file, scorer.negative_features_file)
    scorer.load_data(length_requirement=args.length_requirement)
    if args.equalize_reference:
        scorer.equalize_reference_data()
    if not os.path.isdir(scorer.output_directory):
        os.makedirs(scorer.output_directory)
    # the files that existed before span scoring do not name its options in their headers, so they stay what they were
    file_args = argparse.Namespace(**{k: v for k, v in vars(args).items() if k not in ("region_scores", "span_file")})
    if args.write_neighbors:
        scorer.scores = scorer.score_neighbors()
        scorer.make_neighbors_file(args=file_args)
    else:
        scorer.scores = scorer.score_points()
    if args.window_length is not None:
        scorer.score_windows(args.window_length, args.window_step)
        scorer.find_regions()
        scorer.make_window_files(args=file_args)
        if args.region_scores:
            scorer.score_regions()
            scorer.make_span_file("phamer_region_scores.csv", args=args)
    if args.span_file is not None:
        ids, spans, names, lines = fileIO.read_bed(args.span_file, with_lines=True)
        scorer.score_spans(ids, spans, names, lines=lines)
        scorer.make_span_file("phamer_spans.csv", args=args)
    # the score file's header does not depend on whether neighbours, windows or spans were asked for; canonical scoring is named only
    # when it is on
    score_args = argparse.Namespace(**{k: v for k, v in vars(file_args).items()
                                       if k not in ("write_neighbors", "window_length", "window_step") and (k != "canonical_kmers" or v)})
    scorer.make_summary_file(args=score_args)
    return scorer


if __name__ == "__main__":
    main()
