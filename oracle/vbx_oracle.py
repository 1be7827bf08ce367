"""TEST INFRASTRUCTURE ONLY - CPU restatement of the VBx clustering branch of the path (SURVEY.md §8 row a23).

Follows
  * diarizen/clustering/VBx.py:27-113   the VB iteration, GMM branch only (DiariZen always calls it with loopProb = 0,
                                        VBx.py:115, so the HMM forward-backward branch is unreachable on this path)
  * diarizen/clustering/VBx.py:115-127  initialisation from the AHC labels (softmax-smoothed one-hot, smoothing 7)
  * diarizen/clustering/VBx.py:146-178  the x-vector -> PLDA-space transform built from xvec_transform.npz / plda.npz
  * pyannote-audio/pyannote/audio/pipelines/clustering.py:601-700  VBxClustering.__call__

Pinned against the outputs of the reference's own VBx.py (tests/test_vbx.py: tests/golden/reference_pins.npz and
tests/golden/vbx.npz, generated from it by scripts/make_reference_golden.py and scripts/make_golden.py).  Only tests/, __graft_entry__.smoke() and bench.py's CPU
legs may import this module.
"""
from __future__ import annotations

import numpy as np


def unit_rows(x: np.ndarray) -> np.ndarray:
    return x / np.linalg.norm(x, axis=1, ord=2)[:, None]


def plda_setup(xvec_transform: dict, plda: dict):
    """VBx.py:146-178.  Returns (xvec_tf, plda_tf, psi) with psi sorted descending."""
    from scipy.linalg import eigh
    mean1, mean2, lda = xvec_transform["mean1"], xvec_transform["mean2"], xvec_transform["lda"]
    mu, tr, psi = plda["mu"], plda["tr"], plda["psi"]
    within = np.linalg.inv(tr.T.dot(tr))
    between = np.linalg.inv((tr.T / psi).dot(tr))
    ev, vec = eigh(between, within)
    psi_sorted = ev[::-1]
    basis = vec.T[::-1]
    d_in, d_out = lda.shape

    def xvec_tf(x):
        y = np.sqrt(d_in) * unit_rows(x - mean1)
        return np.sqrt(d_out) * unit_rows(lda.T.dot(y.T).T - mean2)

    def plda_tf(x0, lda_dim=d_out):
        return (x0 - mu).dot(basis.T)[:, :lda_dim]

    return xvec_tf, plda_tf, psi_sorted


def vb_gmm(X: np.ndarray, Phi: np.ndarray, gamma: np.ndarray, Fa: float, Fb: float, max_iters: int, epsilon: float = 1e-4):
    """VBx.py:73-113 with loopProb = 0.  Returns (gamma, pi, elbo_history)."""
    from scipy.special import logsumexp
    D = X.shape[1]
    S = gamma.shape[1]
    pi = np.ones(S) / S
    G = -0.5 * (np.sum(X ** 2, axis=1, keepdims=True) + D * np.log(2 * np.pi))
    rho = X * np.sqrt(Phi)
    hist = []
    for it in range(max_iters):
        invL = 1.0 / (1 + Fa / Fb * gamma.sum(axis=0, keepdims=True).T * Phi)
        alpha = Fa / Fb * invL * gamma.T.dot(rho)
        log_p = Fa * (rho.dot(alpha.T) - 0.5 * (invL + alpha ** 2).dot(Phi) + G)
        lpi = np.log(pi + 1e-8)
        log_px = logsumexp(log_p + lpi, axis=-1)
        total = np.sum(log_px, axis=0)
        gamma = np.exp(log_p + lpi - log_px[:, None])
        pi = np.sum(gamma, axis=0)
        pi = pi / pi.sum()
        elbo = total + Fb * 0.5 * np.sum(np.log(invL) - invL - alpha ** 2 + 1)
        hist.append(elbo)
        if it > 0 and elbo - hist[-2] < epsilon:
            break
    return gamma, pi, hist


def init_responsibilities(labels: np.ndarray, smoothing: float = 7.0) -> np.ndarray:
    """VBx.py:117-119."""
    from scipy.special import softmax
    q = np.zeros((len(labels), int(labels.max()) + 1))
    q[np.arange(len(labels)), labels.astype(int)] = 1.0
    return q if smoothing < 0 else softmax(q * smoothing, axis=1)


def vbx_cluster_call(embeddings: np.ndarray, binarized: np.ndarray, xvec_transform: dict, plda: dict, ahc_threshold: float,
                     Fa: float, Fb: float, lda_dim: int = 128, max_iters: int = 20, ahc_criterion: str = "distance",
                     assign_fn=None):
    """clustering.py:633-700.  `binarized` (C,T,S) hard segmentations."""
    from scipy.cluster.hierarchy import fcluster, linkage
    from scipy.optimize import linear_sum_assignment
    from scipy.spatial.distance import cdist
    from .pipeline_oracle import filter_embeddings
    train, _, _ = filter_embeddings(embeddings, binarized, min_frames_ratio=0.1)
    C, S, D = embeddings.shape
    if train.shape[0] < 2:
        return np.zeros((C, S), dtype=np.int8), np.ones((C, S, 1)), np.mean(train, axis=0, keepdims=True)
    normed = train / np.linalg.norm(train, axis=1, keepdims=True)
    Z = linkage(normed, method="centroid", metric="euclidean")
    ahc = fcluster(Z, ahc_threshold, criterion=ahc_criterion) - 1
    _, ahc = np.unique(ahc, return_inverse=True)
    xvec_tf, plda_tf, psi = plda_setup(xvec_transform, plda)
    fea = plda_tf(xvec_tf(train), lda_dim=lda_dim)
    q, sp, _ = vb_gmm(fea, psi[:lda_dim], init_responsibilities(ahc), Fa, Fb, max_iters)
    centroids = q[:, sp > 1e-7].T @ train.reshape(-1, D)
    soft = 2 - cdist(embeddings.reshape(C * S, D), centroids, metric="cosine").reshape(C, S, -1)
    sc = np.nan_to_num(soft, nan=np.nanmin(soft))
    hard = -2 * np.ones((C, S), dtype=np.int8)
    for c, cost in enumerate(sc):
        if assign_fn is not None:
            hard[c] = assign_fn(cost)
            continue
        rows, cols = linear_sum_assignment(cost, maximize=True)
        for s, k in zip(rows, cols):
            hard[c, s] = k
    _, hard = np.unique(hard, return_inverse=True)
    return hard.reshape(C, S), soft, centroids
