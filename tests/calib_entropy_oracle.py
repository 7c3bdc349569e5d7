"""tests/calib_entropy_oracle.py -- numpy restatement of the entropy (KL-divergence) threshold rule of
slq_hist_scales (csrc/calib.cu hist_entropy_kernel; include/slq.h section 3), test infrastructure only:

* hist_entropy_divergences  fp64 D_k of every candidate k = 128..bins, inf where the rule says so;
* hist_entropy_k            the rule's k: the minimum of D_k, exact ties to the larger k;
* hist_entropy_scale        slq_hist_scales(SLQ_CALIB_ENTROPY) of one tensor (threshold -> scale).
The binning, T_k and the scale of a threshold are those of tests/calib_oracle.py.
"""
import numpy as np

import calib_oracle as co

ENTROPY_START_BIN = 128


def hist_entropy_divergences(hist, qmax):
    """float64 [bins - 127]: entry k - 128 = D_k, the KL divergence of the entropy rule for candidate
    k = 128..bins (zeros, hist[0], left out; N = sum n_j > 0; nq = qmax + 1 levels):
      P_j = n_j (j < k - 1), P_{k-1} = n_{k-1} + o_k with o_k = sum_{j >= k} n_j;
      group(j) = floor(j * nq / k); Q_j = m_g / c_g where n_j > 0 (m_g: counts of group g, c_g: its non-empty
      bins), else 0;
      D_k = sum_{P_j > 0} (P_j / N) ln((P_j / N) / (Q_j / (N - o_k))), inf where some P_j > 0 has Q_j = 0."""
    hist = np.asarray(hist, np.uint64)
    bins = hist.size - 1
    if bins < ENTROPY_START_BIN:
        raise ValueError("entropy needs at least %d bins, not %d" % (ENTROPY_START_BIN, bins))
    n = hist[1:].astype(np.int64)
    N = int(n.sum())
    assert N > 0
    nq = int(qmax) + 1
    M = np.concatenate([[0], np.cumsum(n)])                    # M[j] = n_0 + .. + n_{j-1}
    C = np.concatenate([[0], np.cumsum(n > 0)])                # C[j] = non-empty bins among 0 .. j-1
    out = np.empty(bins - ENTROPY_START_BIN + 1, np.float64)
    for k in range(ENTROPY_START_BIN, bins + 1):
        j = np.arange(k)
        g = j * nq // k
        lo, hi = (g * k + nq - 1) // nq, ((g + 1) * k + nq - 1) // nq   # group g = bins ceil(g k / nq) .. hi - 1
        m, c = M[hi] - M[lo], C[hi] - C[lo]
        nk = n[:k]
        Q = np.where(nk > 0, m / np.maximum(c, 1), 0.0)
        o = N - int(M[k])
        P = nk.astype(np.float64)
        P[k - 1] += o
        live = P > 0
        if (Q[live] == 0).any():
            out[k - ENTROPY_START_BIN] = np.inf
            continue
        p, q = P[live] / N, Q[live] / (N - o)
        out[k - ENTROPY_START_BIN] = float(np.sum(p * np.log(p / q)))
    return out


def hist_entropy_k(hist, qmax):
    """The entropy rule's threshold index: k minimising D_k, exact ties to the larger k."""
    d = hist_entropy_divergences(hist, qmax)
    return int(np.flatnonzero(d == d.min())[-1]) + ENTROPY_START_BIN


def hist_entropy_scale(hist, rng, qmax, headroom=1.0):
    """slq_hist_scales(SLQ_CALIB_ENTROPY) of one tensor; 1.0 for a tensor without a non-zero element."""
    hist = np.asarray(hist, np.uint64)
    if not hist[1:].any():
        return np.float32(1.0)
    return co.hist_scale_for_k(rng, hist_entropy_k(hist, qmax), hist.size - 1, qmax, headroom)
