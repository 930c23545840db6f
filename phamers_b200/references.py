"""
Reference feature sets and their (host-side, cached) clustering.

The shipped phage / bacteria tables (reference data/reference_features/{positive,negative}_features.csv, raw 4-mer
counts in 'ATGC' order) travel with the package as data/reference_features.npz (tools/pack_reference_features.py).

Clustering of the reference sets is reference-only preprocessing, independent of the contigs being scored
(scripts/phamer.py:245-248 runs it twice per scoring call, ~1 s each).  By default it stays on the host with the same
scikit-learn call the reference makes (scripts/learning.py:138: KMeans(n_clusters=k, random_state=10)) so that the
centroids are the reference's centroids, and it is cached per reference set instead of being redone on every call.
`kmeans_on_device = True` moves the Lloyd iterations to the GPU (cross validation refits 40 reference subsets).
"""
import hashlib
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_NPZ = os.path.join(_HERE, "data", "reference_features.npz")
KMEANS_SEED = 10                      # scripts/learning.py:21
_centroid_cache = {}


def load_reference_counts():
    """(positive_ids, positive_counts int64[2255, 256], negative_ids, negative_counts int64[2418, 256])."""
    z = np.load(_NPZ)
    return (z["positive_ids"], z["positive_counts"].astype(np.int64),
            z["negative_ids"], z["negative_counts"].astype(np.int64))


def load_reference_features(equalize=True, canonical=False):
    """Normalised reference features as phamer.load_data builds them (scripts/phamer.py:112,119: read_feature_file(...,
    normalize=True)); equalize truncates both to min(nP, nN) rows (scripts/phamer.py:159-175).  canonical: the counts are folded
    with their reverse complements (136 bins) before they are normalised."""
    from . import kmer
    _, pos, _, neg = load_reference_counts()
    if equalize:
        n = min(len(pos), len(neg))
        pos, neg = pos[:n], neg[:n]
    if canonical:
        pos, neg = kmer.canonical_fold(pos, 4), kmer.canonical_fold(neg, 4)
    return kmer.normalize_counts(pos), kmer.normalize_counts(neg)


def _digest(arr):
    arr = np.ascontiguousarray(arr)
    return hashlib.sha1(arr.view(np.uint8)).hexdigest() + str(arr.shape)


def kmeans_assign(data, k):
    """scripts/learning.py:131-146 (host, scikit-learn, seed 10)."""
    from sklearn.cluster import KMeans
    return np.asarray(KMeans(n_clusters=k, random_state=KMEANS_SEED).fit(data).labels_)


kmeans_on_device = False              # True: Lloyd iterations on the GPU (phm_kmeans_lloyd) from scikit-learn's own k-means++ seeding


def kmeans_assign_device(data, k):
    """The same clustering with the Lloyd iterations on the device.  scikit-learn's KMeans.fit centres the data, seeds with its
    k-means++ routine from RandomState(10) and then iterates (sklearn/cluster/_kmeans.py); here the centring, the tolerance and the
    seeding are obtained from scikit-learn's own functions (so the random stream is the reference's) and only the iterations run in
    phm_kmeans_lloyd.  Labels equal scikit-learn's unless a point is equidistant from two centres to ~1e-16; a run in which a
    cluster becomes empty (scikit-learn relocates it) falls back to the host fit."""
    import torch
    import ctypes
    from sklearn.cluster import _kmeans as skk
    from sklearn.utils import check_random_state
    from sklearn.utils.extmath import row_norms
    from . import _lib, ops
    lib = _lib.require_cuda()
    x = np.array(data, dtype=np.float64, order="C", copy=True)
    n, dim = x.shape
    if k > n or dim > 1024:
        return kmeans_assign(data, k)
    tol = float(skk._tolerance(x, 1e-4))                                      # KMeans(tol=1e-4): mean feature variance * tol
    x -= x.mean(axis=0)
    centres, _ = skk._kmeans_plusplus(x, k, x_squared_norms=row_norms(x, squared=True), sample_weight=np.ones(n, dtype=x.dtype),
                                      random_state=check_random_state(KMEANS_SEED))
    d_x = torch.from_numpy(x).cuda()
    d_c = torch.from_numpy(np.ascontiguousarray(centres, dtype=np.float64)).cuda()
    d_labels = torch.empty((n,), dtype=torch.int32, device="cuda")
    ws = torch.empty((256,), dtype=torch.uint8, device="cuda")
    info = (ctypes.c_int64 * 3)()
    ops.check(lib.phm_kmeans_lloyd(ops.ptr(d_x), n, dim, ops.ptr(d_c), int(k), 300, tol, ops.ptr(d_labels), info, ops.ptr(ws), 256,
                                   ops.stream_ptr()))
    if info[2]:
        return kmeans_assign(data, k)
    return d_labels.cpu().numpy().astype(np.int32)


def get_centroids(data, assignment):
    """scripts/learning.py:69-81."""
    labels = sorted(set(assignment) - {-1})
    return np.array([np.mean(data[assignment == c], axis=0) for c in labels])


def cluster_centroids(data, k):
    key = (_digest(data), int(k))
    hit = _centroid_cache.get(key)
    if hit is None:
        hit = get_centroids(data, kmeans_assign_device(data, k) if kmeans_on_device else kmeans_assign(data, k))
        _centroid_cache[key] = hit
    return hit


def reference_centroids(positive, negative, k_clusters=86):
    """scripts/phamer.py:245-248: centroids of k-means (k = 86) on each reference set."""
    return cluster_centroids(positive, k_clusters), cluster_centroids(negative, k_clusters)


def clear_cache():
    _centroid_cache.clear()
