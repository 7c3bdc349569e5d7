"""tests/calib_oracle.py -- numpy restatement of the histogram calibration of the activation scales
(csrc/calib.cu; include/slq.h section 3), test infrastructure only:

* act_histogram  slq_act_histogram of one tensor, counter for counter (exact fp32 binning rule);
* hist_scale     slq_hist_scales of one tensor (percentile or mse threshold -> scale), with the pieces the tests
                 check separately: hist_threshold, hist_scale_for_k, hist_mse_errors, hist_percentile_k.
"""
import numpy as np


def act_histogram(y, rng, bins):
    """slq_act_histogram of one tensor: uint64 [bins + 1]; counter 0 = exact zeros, counter 1 + j =
    0 < |y| with j = min(trunc(fp32(|y| * fp32(bins / rng))), bins - 1)."""
    a = np.abs(np.asarray(y, np.float32).reshape(-1))
    inv = np.float32(np.float32(bins) / np.float32(rng))
    nz = a[a != 0]
    j = np.minimum(np.floor(nz * inv), np.float32(bins - 1)).astype(np.int64)  # |y| * inv >= 0: floor == trunc
    h = np.zeros(bins + 1, np.uint64)
    h[0] = a.size - nz.size
    h[1:] = np.bincount(j, minlength=bins).astype(np.uint64)
    return h


def hist_threshold(rng, k, bins):
    """T_k = fp32(fp32(rng * k) / bins)."""
    return np.float32(np.float32(np.float32(rng) * np.float32(k)) / np.float32(bins))


def hist_scale_for_k(rng, k, bins, qmax, headroom=1.0):
    """act_scale of threshold k: fp32(fp32(T_k / qmax) * headroom)."""
    return np.float32(np.float32(hist_threshold(rng, k, bins) / np.float32(qmax)) * np.float32(headroom))


def hist_mse_errors(hist, rng, qmax):
    """float64 [bins]: entry k-1 = sum_j n_j (c_j - Q(c_j))^2 for threshold T_k, c_j = (j + 0.5) * rng / bins,
    Q(v) = D * min(rint(v / D), qmax), D = T_k / qmax (zeros, hist[0], contribute nothing)."""
    hist = np.asarray(hist, np.uint64)
    bins = hist.size - 1
    n = hist[1:].astype(np.float64)
    keep = n != 0
    c = ((np.arange(bins, dtype=np.float64) + 0.5) * np.float64(np.float32(rng)) / bins)[keep]
    n = n[keep]
    T = np.array([hist_threshold(rng, k, bins) for k in range(1, bins + 1)], np.float64)
    D = (T / np.float64(qmax))[:, None]
    e = c[None, :] - D * np.minimum(np.rint(c[None, :] / D), np.float64(qmax))
    return (n[None, :] * (e * e)).sum(1)


def hist_percentile_k(hist, percentile):
    """Smallest k with zeros + n_0 + .. + n_{k-1} >= ceil(percentile / 100 * total)."""
    hist = np.asarray(hist, np.uint64)
    bins = hist.size - 1
    target = np.ceil(float(percentile) / 100.0 * float(int(hist.sum())))
    cum = int(hist[0])
    for k in range(1, bins):
        cum += int(hist[k])
        if float(cum) >= target:
            return k
    return bins


def hist_scale(hist, rng, qmax, method, percentile=99.99, headroom=1.0):
    """slq_hist_scales of one tensor: method "percentile" or "mse"; 1.0 for a tensor without a non-zero element."""
    hist = np.asarray(hist, np.uint64)
    bins = hist.size - 1
    if not hist[1:].any():
        return np.float32(1.0)
    if method == "percentile":
        k = hist_percentile_k(hist, percentile)
    elif method == "mse":
        err = hist_mse_errors(hist, rng, qmax)
        k = int(np.flatnonzero(err == err.min())[-1]) + 1  # exact ties: the larger k
    else:
        raise ValueError(method)
    return hist_scale_for_k(rng, k, bins, qmax, headroom)
