"""
Drop-in for the hot-path part of the reference's scripts/learning.py.

    knn            :118   brute-force k nearest neighbours + vote       -> CUDA (phm_score)
    kneighbors            the neighbours themselves (scikit-learn's NearestNeighbors.kneighbors) -> CUDA (phm_score_neighbors)
    distances      :47, closest_to :59   distances of one point to a set of points / the nearest of them -> CUDA
                          (phm_distances; inside the scorer the same search is fused into phm_score)
    get_centroids  :69, kmeans :131   reference-set preprocessing         -> host scikit-learn, see references.py

    predictor_performance :185, get_truth_table :199, get_predictor_metrics :224   ROC and truth-table metrics (host)

The other evaluation helpers of learning.py (dbscan, silhouettes, get_density) are outside the hot path.
"""
import numpy as np

from . import references

kmeans_seed = references.KMEANS_SEED


def knn(queries, ref_data, ref_labels, k=3):
    """scripts/learning.py:118-128: 2 * (KNeighborsClassifier(k).fit(refs, labels).predict(queries) - 0.5), computed on
    the GPU.  Labels must be 0 / 1; rows are reordered so that the 1-labelled references come first."""
    import torch
    from . import ops, _lib
    _lib.require_cuda()
    queries = np.ascontiguousarray(queries, dtype=np.float64)
    ref_data = np.asarray(ref_data, dtype=np.float64)
    ref_labels = np.asarray(ref_labels)
    if not np.all((ref_labels == 0) | (ref_labels == 1)):
        raise NotImplementedError("knn on the device supports the reference's 0/1 labels")
    order = np.argsort(ref_labels == 0, kind="stable")          # positives first, original order kept inside each class
    refs = np.ascontiguousarray(ref_data[order])
    n_pos = int(np.sum(ref_labels == 1))
    empty = torch.empty((0, queries.shape[1]), dtype=torch.float64, device="cuda")
    votes, _, _ = ops.score_cuda(torch.from_numpy(queries).cuda(), torch.from_numpy(refs).cuda(), n_pos, empty, empty, k)
    return votes.cpu().numpy()


def kneighbors(queries, ref_data, k=3):
    """The k nearest rows of `ref_data` to each query, as scikit-learn's NearestNeighbors(algorithm="brute").kneighbors returns
    them: (distances float64[n, k] ascending, indices int64[n, k] into ref_data), computed on the GPU (phm_score_neighbors).
    Distances are float64 direct differences (as `distances`); equal distances list the lower row first.  k is 1..15."""
    import torch
    from . import ops, _lib
    _lib.require_cuda()
    queries = np.ascontiguousarray(np.atleast_2d(queries), dtype=np.float64)
    refs = np.ascontiguousarray(ref_data, dtype=np.float64)
    empty = torch.empty((0, queries.shape[1]), dtype=torch.float64, device="cuda")
    # no labels, so no positives-first regrouping as in knn: the reported rows are already the caller's row numbers
    out = ops.score_neighbors_cuda(torch.from_numpy(queries).cuda(), torch.from_numpy(refs).cuda(), 0, empty, empty, k)
    return out[4].cpu().numpy(), out[3].cpu().numpy()


def distances(vector, data):
    """scripts/learning.py:47-56: Euclidean distance from `vector` to every row of `data` (float64 direct differences, on the
    GPU: phm_distances)."""
    import torch
    from . import ops
    point = torch.from_numpy(np.ascontiguousarray(vector, dtype=np.float64).reshape(-1)).cuda()
    rows = torch.from_numpy(np.ascontiguousarray(np.atleast_2d(np.asarray(data, dtype=np.float64)))).cuda()
    return ops.distances_cuda(point, rows).cpu().numpy()


def closest_to(point, picks):
    """scripts/learning.py:59-66: the row of `picks` nearest to `point` (the first one on ties) -- the row itself, as there."""
    picks = np.asarray(picks)
    return picks[int(np.argmin(distances(point, picks)))]


def get_centroids(data, assignment):
    """scripts/learning.py:69-81."""
    return references.get_centroids(np.asarray(data), np.asarray(assignment))


def kmeans(data, k, verbose=False, sort_by_size=False):
    """scripts/learning.py:131-146 (host scikit-learn, random_state = kmeans_seed)."""
    if sort_by_size:
        raise NotImplementedError("sort_by_size is outside the hot path")
    return references.kmeans_assign(np.asarray(data), k)


# ---- evaluation of a scored gold standard (host side: a handful of scalars per run) -----------------------------------
# Same names, arguments and return conventions as scripts/learning.py:185-245; the bodies work from ONE confusion count.
METRIC_NAMES = ("tp", "fp", "fn", "tn", "tpr", "fpr", "fnr", "tnr", "ppv", "npv", "fdr", "acc")


def _confusion(positive_scores, negative_scores, threshold):
    """(tp, fp, fn, tn) with 'score >= threshold' as the positive call (scripts/learning.py:207-210)."""
    called_pos = np.asarray(positive_scores) >= threshold
    called_neg = np.asarray(negative_scores) >= threshold
    tp, fp = int(called_pos.sum()), int(called_neg.sum())
    return tp, fp, int(called_pos.size) - tp, int(called_neg.size) - fp


def _ratio(num, den):
    return float(num) / den if den else 0


def predictor_performance(positive_scores, negative_scores):
    """scripts/learning.py:185-196: ROC of the scores against their classes -> (fpr, tpr, area under the curve), from the same
    scikit-learn routines the reference calls."""
    from sklearn import metrics
    truth = np.concatenate((np.ones(len(positive_scores), dtype=bool), np.zeros(len(negative_scores), dtype=bool)))
    fpr, tpr, _ = metrics.roc_curve(truth, np.concatenate((positive_scores, negative_scores)))
    return fpr, tpr, metrics.auc(fpr, tpr)


def get_truth_table(positive_scores, negative_scores, threshold=0):
    """scripts/learning.py:199-221: (true positive, false positive, false negative, true negative) RATES; an empty class gives
    rate 0 and its complement 1."""
    tp, fp, fn, tn = _confusion(positive_scores, negative_scores, threshold)
    tpr, fpr = _ratio(tp, tp + fn), _ratio(fp, fp + tn)
    return tpr, fpr, 1 - tpr, 1 - fpr


def get_predictor_metrics(positive_scores, negative_scores, threshold=0):
    """scripts/learning.py:224-245: pandas Series indexed tp fp fn tn tpr fpr fnr tnr ppv npv fdr acc."""
    import pandas as pd
    tp, fp, fn, tn = _confusion(positive_scores, negative_scores, threshold)
    tpr, fpr, fnr, tnr = get_truth_table(positive_scores, negative_scores, threshold=threshold)
    with np.errstate(divide="ignore", invalid="ignore"):
        ppv = np.float64(tp) / (tp + fp)                      # 0 / 0 is NaN, as the reference's float division of pandas scalars
        npv = np.float64(tn) / (tn + fn)
        acc = np.float64(tp + tn) / (tp + fp + fn + tn)
    values = (tp, fp, fn, tn, tpr, fpr, fnr, tnr, ppv, npv, 1 - ppv, acc)
    return pd.Series(dict(zip(METRIC_NAMES, values)), index=list(METRIC_NAMES), dtype=float)
