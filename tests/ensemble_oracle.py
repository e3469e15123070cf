"""fp64 numpy oracle of ensemble scoring (``ibm_ensemble_score``, ``EnsembleScorer``): the fair CRPS in its pair and sorted forms,
the biased (K^2) estimator it replaces, and the per-channel accumulator of a batch of K draws per window."""
import numpy as np

COP_FORCE_THRESHOLD = 10.0


def pair_sum(x):
    """sum_{i<j} |x_i - x_j| over axis 0 (pair form)."""
    x = np.asarray(x, dtype=np.float64)
    K = x.shape[0]
    return sum(np.abs(x[i] - x[j]) for i in range(K) for j in range(i + 1, K))


def pair_sum_sorted(x):
    """sum_{i<j} |x_i - x_j| = sum_k (2k - K - 1) x_(k), k 1-based over the ascending order (sorted form)."""
    x = np.sort(np.asarray(x, dtype=np.float64), axis=0)
    K = x.shape[0]
    w = (2 * np.arange(1, K + 1) - K - 1).reshape((K,) + (1,) * (x.ndim - 1))
    return (w * x).sum(axis=0)


def fair_crps(x, y):
    """(1/K) sum_k |x_k - y| - 1/(2K(K-1)) sum_{i,j} |x_i - x_j| (Ferro 2014), pair form; x (K, ...), y (...)."""
    x = np.asarray(x, dtype=np.float64)
    K = x.shape[0]
    return np.abs(x - y).mean(axis=0) - 2.0 * pair_sum(x) / (2.0 * K * (K - 1))


def fair_crps_sorted(x, y):
    x = np.asarray(x, dtype=np.float64)
    K = x.shape[0]
    return np.abs(x - y).mean(axis=0) - pair_sum_sorted(x) / (K * (K - 1))


def biased_crps(x, y):
    """The ensemble CRPS with the K^2 denominator: for a calibrated ensemble its mean is sigma/sqrt(pi) (1 + 1/K)."""
    x = np.asarray(x, dtype=np.float64)
    K = x.shape[0]
    return np.abs(x - y).mean(axis=0) - 2.0 * pair_sum_sorted(x) / (2.0 * K * K)


def contact(force3):
    """The fused loss kernel's contact test, bit for bit: fp32 (a*a + b*b) + c*c without FMA, sqrt > threshold."""
    f = np.asarray(force3, dtype=np.float32)
    n2 = (f[..., 0] * f[..., 0] + f[..., 1] * f[..., 1]) + f[..., 2] * f[..., 2]
    return np.sqrt(n2, dtype=np.float32) > np.float32(COP_FORCE_THRESHOLD)


def score(draws, labels):
    """draws (K, B, F, 30), labels (B, Fo, 30) -> (mean (B, Fo, 30) fp64, acc (5, 30) fp64, contact (B, Fo, 2) bool): acc rows
    sum crps, s^2, (m - y)^2, pair = 1/(K(K-1)) sum_{i!=j} |x_i - x_j|, count; CoP channels 0-2 / 3-5 on contact rows only."""
    x = np.asarray(draws, dtype=np.float64)
    lab = np.asarray(labels, dtype=np.float32)
    K, B, F = x.shape[:3]
    Fo = lab.shape[1]
    if Fo == 1:
        x = x[:, :, -1:]
    y = lab.astype(np.float64)
    m = x.mean(axis=0)
    s2 = ((x - m) ** 2).sum(axis=0) / (K - 1)
    ps = pair_sum(x)
    crps = np.abs(x - y).mean(axis=0) - ps / (K * (K - 1))
    pair = 2.0 * ps / (K * (K - 1))
    se = (m - y) ** 2
    con = np.stack([contact(lab[..., 6:9]), contact(lab[..., 9:12])], axis=-1)
    w = np.ones((B, Fo, 30))
    w[..., 0:3] = con[..., 0:1]
    w[..., 3:6] = con[..., 1:2]
    acc = np.stack([(v * w).sum(axis=(0, 1)) for v in (crps, s2, se, pair, np.ones_like(crps))])
    return m, acc, con
