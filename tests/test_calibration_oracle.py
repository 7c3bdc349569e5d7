"""Histogram calibration of the activation scales, without a GPU: the oracle's restatement of the binning and
threshold rules (tests/calib_oracle.py act_histogram / hist_scale, include/slq.h section 3) against hand-made
edge values and a brute-force evaluation of the same formulas, and the argument checks of the C ABI."""
import ctypes
import math

import numpy as np

import slq_lib as L
import calib_oracle as co


def test_histogram_edge_values():
    f = np.float32
    edge = f(0.125)  # bins = 8, range = 1: inv = 8, bin j covers [j/8, (j+1)/8)
    y = np.array([0.0, -0.0, 1.0, 2.0, edge, np.nextafter(edge, f(0)), -0.5, 1e-30, -np.nextafter(f(1), f(0))], f)
    assert y.size % 4 != 0
    h = co.act_histogram(y, 1.0, 8)
    want = np.zeros(9, np.uint64)
    want[0] = 2                      # 0 and -0
    want[1 + 7] = 3                  # range itself, above range, and just below range (j = 7)
    want[1 + 1] = 1                  # exactly on the edge of bin 1
    want[1 + 0] = 2                  # just below that edge, and a tiny value
    want[1 + 4] = 1                  # |-0.5|
    assert h.dtype == np.uint64 and np.array_equal(h, want)


def test_histogram_matches_elementwise_rule():
    rng = np.random.default_rng(3)
    y = (rng.standard_normal(1003) * 2).astype(np.float32)
    y[::7] = 0
    for r, bins in ((3.0, 16), (1.7, 2048), (0.01, 4)):
        inv = np.float32(np.float32(bins) / np.float32(r))
        want = np.zeros(bins + 1, np.uint64)
        for v in y:
            a = abs(np.float32(v))
            want[0 if a == 0 else 1 + min(math.trunc(float(np.float32(a * inv))), bins - 1)] += 1
        assert np.array_equal(co.act_histogram(y, r, bins), want)


def _brute_mse(hist, r, qmax):
    bins = len(hist) - 1
    out = []
    for k in range(1, bins + 1):
        T = float(np.float32(np.float32(np.float32(r) * np.float32(k)) / np.float32(bins)))
        D = T / qmax
        err = 0.0
        for j in range(bins):
            c = (j + 0.5) * float(np.float32(r)) / bins
            e = c - D * min(float(np.rint(c / D)), float(qmax))
            err += int(hist[1 + j]) * (e * e)
        out.append(err)
    return np.array(out)


def test_mse_rule_matches_brute_force():
    rng = np.random.default_rng(5)
    for bins, qmax, r in ((16, 255, 2.5), (32, 127, 0.3), (8, 3, 1.0)):
        hist = rng.integers(0, 50, bins + 1).astype(np.uint64)
        hist[bins - 3:] = 0
        err = co.hist_mse_errors(hist, r, qmax)
        ref = _brute_mse(hist, r, qmax)
        assert np.allclose(err, ref, rtol=1e-12, atol=0)
        k = int(np.flatnonzero(err == err.min())[-1]) + 1
        assert co.hist_scale(hist, r, qmax, "mse") == co.hist_scale_for_k(r, k, bins, qmax)


def test_mse_with_coarse_grid_clips_the_tail():
    # qmax = 3: four levels; one far outlier among many small values is worth clipping
    hist = np.zeros(65, np.uint64)
    hist[1 + 2] = 1000
    hist[1 + 63] = 1
    err = co.hist_mse_errors(hist, 1.0, 3)
    k = int(np.argmin(err)) + 1
    assert k < 64
    assert co.hist_scale(hist, 1.0, 3, "mse") < co.hist_scale_for_k(1.0, 64, 64, 3)


def test_percentile_rule():
    hist = np.array([5, 1, 0, 2, 2], np.uint64)  # 5 zeros, bins = 4, total = 10
    assert co.hist_percentile_k(hist, 50) == 1    # target 5 <= zeros + n_0
    assert co.hist_percentile_k(hist, 60) == 1
    assert co.hist_percentile_k(hist, 61) == 3    # target 7: bin 1 is empty
    assert co.hist_percentile_k(hist, 100) == 4
    assert co.hist_scale(hist, 2.0, 255, "percentile", 61) == np.float32(np.float32(1.5) / np.float32(255))
    assert co.hist_scale(hist, 2.0, 255, "percentile", 100, 1.25) == \
        np.float32(np.float32(np.float32(2.0) / np.float32(255)) * np.float32(1.25))
    # T_bins is the range itself; a tensor without a non-zero element keeps scale 1
    assert co.hist_threshold(np.float32(0.3), 2048, 2048) == np.float32(0.3)
    assert co.hist_scale(np.array([7, 0, 0], np.uint64), 1.0, 255, "mse") == np.float32(1.0)
    assert co.hist_scale(np.zeros(3, np.uint64), 1.0, 255, "percentile") == np.float32(1.0)


def test_histogram_entry_points_check_arguments_without_a_gpu():
    lib = L.lib()
    buf = (ctypes.c_float * 8)()
    hist = (ctypes.c_uint64 * 8)()
    p, h = ctypes.addressof(buf), ctypes.addressof(hist)
    assert lib.slq_act_histogram(p, 4, p, 0, 3, h, None) == L.SLQ_ERR_INVALID
    assert b"power of two" in lib.slq_last_error()
    assert lib.slq_act_histogram(p, 4, p, 0, 4096, h, None) == L.SLQ_ERR_INVALID
    assert lib.slq_act_histogram(p, 0, p, 0, 4, h, None) == L.SLQ_ERR_INVALID
    assert lib.slq_act_histogram(p + 2, 4, p, 0, 4, h, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 4, p, p, 0, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert b"method" in lib.slq_last_error()
    assert lib.slq_hist_scales(h, 1, 4, p, p, L.CALIB_PERCENTILE, 0.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 4, p, p, L.CALIB_PERCENTILE, 100.5, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 6, p, p, L.CALIB_MSE, 99.0, 1.0, p, None) == L.SLQ_ERR_INVALID
    assert lib.slq_hist_scales(h, 1, 4, p, p, L.CALIB_MSE, 99.0, 0.0, p, None) == L.SLQ_ERR_INVALID


def test_one_shot_iterator_and_unknown_method_are_refused():
    import pytest
    import torch
    import resnet
    net = resnet.resnet18(num_classes=10).eval()
    x = torch.zeros(1, 3, 32, 32)
    with pytest.raises(TypeError, match="one-shot"):
        net.slq_calibrate(iter([x]), method="percentile")
    with pytest.raises(ValueError, match="method"):
        net.slq_calibrate(x, method="kl")
