"""Entropy (KL-divergence) calibration of the activation scales, without a GPU: the oracle's restatement of the
rule (tests/calib_entropy_oracle.py hist_entropy_divergences / hist_entropy_k, include/slq.h section 3) against a literal
transcription of pytorch-quantization's HistogramCalibrator entropy search, on random and hand-made histograms,
and the argument checks of slq_hist_scales for the new method."""
import ctypes
from collections import Counter

import numpy as np
import pytest
from scipy.stats import entropy

import slq_lib as L
import calib_oracle as co
import calib_entropy_oracle as ceo


def _pq_entropy(n, num_bits, unsigned, start_bin=128):
    """pytorch-quantization's _compute_amax_entropy (calib/histogram.py, stride 1), line for line, on the counts
    n_j of the non-zero bins.  Three departures, none of which changes a finite divergence:
      * its `bins[0] = bins[1]` (a stand-in for the zeros it keeps in bin 0) is dropped: zeros are not in n;
      * its `_normalize_distr` calls are dropped: they rebind a local and change nothing (scipy's entropy
        normalises both distributions itself);
      * scipy returns nan where every count lies at or beyond candidate i (0/0 normalising the empty candidate
        distribution); the rule calls that inf, so nan is mapped to inf before the arg-min.
    Returns (divergences for i = start_bin..len(n), the chosen i: calib_bin_edges[i] is the amax)."""
    bins = np.asarray(n, np.float64).copy()
    total_data = np.sum(bins)
    divergences = []
    nbins = 1 << (num_bits - 1 + int(unsigned))
    starting = start_bin
    stop = len(bins)
    new_density_counts = np.zeros(nbins, dtype=np.float64)
    for i in range(starting, stop + 1):
        new_density_counts.fill(0)
        space = np.linspace(0, i, num=nbins + 1)
        digitized_space = np.digitize(range(i), space) - 1
        digitized_space[bins[:i] == 0] = -1
        for idx, digitized in enumerate(digitized_space):
            if digitized != -1:
                new_density_counts[digitized] += bins[idx]
        counter = Counter(digitized_space)
        for key, val in counter.items():
            if key != -1:
                new_density_counts[key] = new_density_counts[key] / val
        new_density = np.zeros(i, dtype=np.float64)
        for idx, digitized in enumerate(digitized_space):
            if digitized != -1:
                new_density[idx] = new_density_counts[digitized]
        total_counts_new = np.sum(new_density) + np.sum(bins[i:])
        reference_density = np.array(bins[:len(digitized_space)])
        reference_density[-1] += np.sum(bins[i:])
        total_counts_old = np.sum(reference_density)
        if round(total_counts_new) != total_data or round(total_counts_old) != total_data:
            raise RuntimeError("Count mismatch")
        with np.errstate(invalid="ignore", divide="ignore"):
            ent = entropy(reference_density, new_density)
        divergences.append(np.inf if np.isnan(ent) else ent)
    divergences = np.array(divergences)
    last_argmin = len(divergences) - 1 - np.argmin(divergences[::-1])
    return divergences, int(last_argmin + starting)


def _check_against_pq(hist, qmax):
    n = np.asarray(hist, np.uint64)[1:]
    d = ceo.hist_entropy_divergences(hist, qmax)
    ref, k_ref = _pq_entropy(n, 8, qmax == 255)
    assert np.array_equal(np.isinf(d), np.isinf(ref))
    fin = np.isfinite(d)
    assert np.allclose(d[fin], ref[fin], rtol=1e-9, atol=1e-15)
    assert ceo.hist_entropy_k(hist, qmax) == k_ref
    return d, k_ref


def _hist(n, zeros=0):
    return np.concatenate([[zeros], np.asarray(n)]).astype(np.uint64)


@pytest.mark.parametrize("qmax", [255, 127])
@pytest.mark.parametrize("bins", [256, 512])
def test_entropy_matches_pytorch_quantization_on_random_histograms(bins, qmax):
    rng = np.random.default_rng(bins + qmax)
    for t in range(4):
        y = rng.standard_normal(30000) * (1 + t)
        if t % 2 == 0:
            y = np.maximum(y, 0)                                  # post-ReLU: about half zeros
        y = y.astype(np.float32)
        r = np.float32(np.abs(y).max() * (1.0, 0.9, 0.6, 0.8)[t])
        hist = co.act_histogram(y, r, bins)
        _check_against_pq(hist, qmax)


@pytest.mark.parametrize("qmax", [255, 127])
def test_entropy_single_non_empty_bin(qmax):
    for j in (0, 5, 300, 511):
        n = np.zeros(512, np.int64)
        n[j] = 1000
        d, k = _check_against_pq(_hist(n, zeros=77), qmax)
        assert k == 512                                          # D = 0 wherever the bin is inside: ties -> larger k
        first = max(j + 1, 128)
        assert np.all(d[first - 128:] == 0) and np.all(np.isinf(d[:first - 128]))


@pytest.mark.parametrize("qmax", [255, 127])
def test_entropy_all_mass_in_the_last_bin(qmax):
    n = np.zeros(256, np.int64)
    n[-1] = 12345
    d, k = _check_against_pq(_hist(n), qmax)
    assert k == 256 and d[-1] == 0 and np.all(np.isinf(d[:-1]))   # every other candidate: N == o_k


@pytest.mark.parametrize("qmax", [255, 127])
def test_entropy_empty_last_bin_with_outliers_is_inf(qmax):
    rng = np.random.default_rng(9)
    n = rng.integers(1, 100, 512)
    n[199] = 0
    n[400] = 0
    d, _ = _check_against_pq(_hist(n), qmax)
    assert np.isinf(d[200 - 128]) and np.isinf(d[401 - 128])      # n_{k-1} = 0 < o_k
    assert np.isfinite(np.delete(d, [200 - 128, 401 - 128])).all()
    assert np.isfinite(d[-1])                                       # k = bins: always finite


@pytest.mark.parametrize("qmax", [255, 127])
def test_entropy_exact_tie_goes_to_the_larger_k(qmax):
    # bins 0 and 256 / nq, unequal: group(256 / nq) = floor(256 / k), so the two are in groups of their own for
    # k <= 256 (D_k = 0) and merged beyond (D_k > 0); the first minimum is k = 128, the last k = 256
    n = np.zeros(512, np.int64)
    n[0], n[256 // (qmax + 1)] = 5, 7
    d, k = _check_against_pq(_hist(n), qmax)
    assert np.all(d[:256 - 128 + 1] == 0) and np.all(d[256 - 128 + 1:] > 0)
    assert k == 256
    assert ceo.hist_entropy_scale(_hist(n), 2.0, qmax) == co.hist_scale_for_k(2.0, 256, 512, qmax)


def test_entropy_empty_histogram_keeps_scale_one():
    assert ceo.hist_entropy_scale(np.zeros(129, np.uint64), 1.0, 255) == np.float32(1.0)
    assert ceo.hist_entropy_scale(_hist(np.zeros(2048), zeros=99), 3.0, 127) == np.float32(1.0)
    with pytest.raises(ValueError, match="128"):
        ceo.hist_entropy_divergences(_hist(np.ones(64)), 255)


def test_entropy_scale_and_headroom():
    rng = np.random.default_rng(4)
    y = np.maximum(rng.standard_normal(50000), 0).astype(np.float32)
    y[:3] = 40                                                   # far outliers: worth clipping
    r = np.float32(40)
    hist = co.act_histogram(y, r, 2048)
    k = ceo.hist_entropy_k(hist, 255)
    assert 128 <= k < 2048
    assert ceo.hist_entropy_scale(hist, r, 255, headroom=1.5) == co.hist_scale_for_k(r, k, 2048, 255, 1.5)


def test_entropy_argument_checks_without_a_gpu():
    lib = L.lib()
    buf = (ctypes.c_float * 8)()
    hist = (ctypes.c_uint64 * 8)()
    p, h = ctypes.addressof(buf), ctypes.addressof(hist)
    assert L.CALIB_ENTROPY == 3
    assert lib.slq_hist_scales(h, 1, 64, p, p, L.CALIB_ENTROPY, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert b"bins=64" in lib.slq_last_error() and b"128" in lib.slq_last_error()
    assert lib.slq_hist_scales(h, 1, 4, p, p, L.CALIB_ENTROPY, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 4096, p, p, L.CALIB_ENTROPY, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 2048, p, p, L.CALIB_ENTROPY, 99.0, 0.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 0, 2048, p, p, L.CALIB_ENTROPY, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 2048, p, p, 4, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert b"method" in lib.slq_last_error()


def test_entropy_is_a_calibration_method():
    import torch
    import resnet
    assert "entropy" in resnet.ResNet.CALIB_METHODS
    net = resnet.resnet18(num_classes=10).eval()
    with pytest.raises(TypeError, match="one-shot"):
        net.slq_calibrate(iter([torch.zeros(1, 3, 32, 32)]), method="entropy")
