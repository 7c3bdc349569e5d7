"""Entropy (KL-divergence) calibration of the activation scales on the device (csrc/calib.cu hist_entropy_kernel,
include/slq.h section 3):

  * slq_hist_scales(SLQ_CALIB_ENTROPY) against the oracle (tests/calib_entropy_oracle.py hist_entropy_divergences) on
    synthetic, hand-made and real histograms (every tensor of ResNet-50 at batch 256, from a calibration walk):
    the kernel's k is at the oracle's minimum of D_k within fp64 rounding, and is the oracle's k wherever the
    minimum is clear of the runner-up;
  * the public API (``net.slq_calibrate(..., method="entropy")``): scales in place under a captured graph,
    repeatable, padded short batches, one-shot iterators, bounded by abs-max;
  * held-out logits parity on BASELINE.json's R50@256 and R34@128 configurations, with the bars of
    tests/test_baseline_configs_gpu.py.
"""
import numpy as np
import pytest
import torch

import slq_lib as L
import calib_oracle as co
import calib_entropy_oracle as ceo
from helpers import build_p0_model
from test_calibration_gpu import _batch, _check_heldout, _engine, _hist_cases

pytestmark = pytest.mark.gpu

START = ceo.ENTROPY_START_BIN


def _entropy_scales(h, r, q, headroom=1.0):
    """slq_hist_scales(SLQ_CALIB_ENTROPY) on device tensors h [T, bins + 1] int64, r [T] fp32, q [T] int32."""
    out = torch.full((h.shape[0],), -1.0, dtype=torch.float32, device="cuda")
    L.check(L.lib().slq_hist_scales(h.data_ptr(), h.shape[0], h.shape[1] - 1, r.data_ptr(), q.data_ptr(),
                                    L.CALIB_ENTROPY, 99.99, headroom, out.data_ptr(), L.current_stream()))
    return out.cpu().numpy()


def _device_entropy_scales(hists, rngs, qmaxs, headroom=1.0):
    h = torch.from_numpy(np.stack(hists).view(np.int64)).cuda()
    r = torch.tensor(np.asarray(rngs, np.float32), device="cuda")
    q = torch.tensor(np.asarray(qmaxs, np.int32), device="cuda")
    return _entropy_scales(h, r, q, headroom)


def _check_at_the_minimum(hists, rngs, qmaxs, got, headroom):
    """Every scale the kernel wrote is that of one candidate k whose oracle D_k is within a relative 1e-9 of the
    oracle's minimum, and is the oracle's own k wherever its runner-up is more than 1e-6 above the minimum."""
    clear = 0
    for t, (h, r, q) in enumerate(zip(hists, rngs, qmaxs)):
        bins = h.size - 1
        if not h[1:].any():
            assert got[t] == 1.0, t
            continue
        cands = [k for k in range(START, bins + 1) if co.hist_scale_for_k(r, k, bins, q, headroom) == got[t]]
        assert len(cands) == 1, (t, got[t], cands)
        k = cands[0]
        d = ceo.hist_entropy_divergences(h, q)
        dmin = d.min()
        assert np.isfinite(dmin) and d[k - START] <= dmin * (1 + 1e-9), (t, k, d[k - START], dmin)
        k_oracle = ceo.hist_entropy_k(h, q)
        runner_up = np.delete(d, k_oracle - START).min() if d.size > 1 else np.inf
        if runner_up > dmin * (1 + 1e-6):
            assert k == k_oracle, (t, k, k_oracle, dmin, runner_up)
            clear += 1
    return clear


def _constructed_cases(bins):
    """Hand-made histograms: an exact tie at D = 0 over k = 128..256 (larger k wins), one non-empty bin, all mass in
    the last bin, empty bins just below outliers (D_k = inf), an empty histogram and zeros only."""
    hists, qmaxs = [], []
    for q in (255, 127):
        n = np.zeros(bins, np.uint64)
        n[0], n[256 // (q + 1)] = 5, 7
        hists.append(n)
        qmaxs.append(q)
    one = np.zeros(bins, np.uint64)
    one[min(300, bins - 1)] = 1000
    last = np.zeros(bins, np.uint64)
    last[-1] = 12345
    gaps = np.random.default_rng(bins).integers(1, 100, bins).astype(np.uint64)
    gaps[bins // 2 - 1] = 0
    gaps[bins - 2] = 0
    hists += [one, last, gaps, np.zeros(bins, np.uint64), np.zeros(bins, np.uint64)]
    qmaxs += [255, 127, 255, 255, 127]
    zeros = [0] * (len(hists) - 1) + [9]
    hists = [np.concatenate([[z], n]).astype(np.uint64) for z, n in zip(zeros, hists)]
    return hists, [np.float32(1.5)] * len(hists), qmaxs


@pytest.mark.parametrize("bins,headroom", [(128, 1.0), (256, 1.0), (2048, 1.0), (2048, 1.5)])
def test_hist_scales_entropy_at_the_minimum(bins, headroom):
    hists, rngs, qmaxs = _hist_cases(bins)
    h2, r2, q2 = _constructed_cases(bins)
    hists, rngs, qmaxs = hists + h2, rngs + r2, qmaxs + q2
    got = _device_entropy_scales(hists, rngs, qmaxs, headroom)
    _check_at_the_minimum(hists, rngs, qmaxs, got, headroom)
    assert got[-1] == 1.0 and got[-2] == 1.0
    if bins >= 512:
        tie = [co.hist_scale_for_k(np.float32(1.5), 256, bins, q, headroom) for q in (255, 127)]
        assert list(got[len(hists) - len(h2):][:2]) == tie     # exact tie: the larger k (256), not 128


def test_hist_scales_entropy_on_resnet50_tensors():
    net = build_p0_model("resnet50", "cuda")
    x = _batch(256, 11).cuda()
    net.slq_calibrate(x)                                       # abs-max: the ranges of the histogram pass
    eng = _engine(net)
    q = eng.act_qmax()
    rng = eng.act_scales * q.to(torch.float32)
    bins = net.CALIB_BINS
    counts = torch.zeros((len(eng.act), bins + 1), dtype=torch.int64, device="cuda")
    eng.histogram(x, counts, rng, bins)
    got = _entropy_scales(counts, rng, q)
    hists = list(counts.cpu().numpy().view(np.uint64))
    clear = _check_at_the_minimum(hists, list(rng.cpu().numpy()), list(q.cpu().numpy()), got, 1.0)
    print("R50@256: %d tensors, %d with a clear minimum" % (len(hists), clear))
    # the public call takes the same two passes and the same kernel
    net.slq_calibrate(x, method="entropy")
    assert np.array_equal(eng.act_scales.cpu().numpy().view(np.uint32), got.view(np.uint32))


def test_entropy_engine_semantics():
    net = build_p0_model("resnet18", "cuda")
    a, b, c = _batch(8, 61).cuda(), _batch(8, 62).cuda(), _batch(8, 63).cuda()
    net.slq_calibrate([a, b])
    eng = _engine(net)
    s_abs = eng.act_scales.clone()
    # a graph captured under the abs-max scales
    g = eng.capture_graph(c)
    g.replay()
    before = eng.logits.clone()
    # the entropy walk measures every range under headroom-1 scales, as the abs-max calibration above did: each
    # threshold is at most that range, so each scale at most abs-max times headroom (within the fp32 roundings)
    net.slq_calibrate([a, (b, None)], headroom=1.25, method="entropy")
    assert _engine(net) is eng
    s1 = eng.act_scales.clone()
    assert not torch.equal(s1, s_abs * 1.25)
    bound = s_abs * 1.25 * (1 + 2 ** -20)
    assert bool((s1 <= bound).all()), (s1 / (s_abs * 1.25)).max()
    net.slq_calibrate([a, b], headroom=1.25, method="entropy")
    assert torch.equal(eng.act_scales, s1)                    # repeated calibration is bit-identical
    # the graph reads act_scales through its pointer: it now runs under the new scales
    g.replay()
    replayed = eng.logits.clone()
    eng.launch_all(c.data_ptr(), L.current_stream())
    assert torch.equal(replayed, eng.logits) and not torch.equal(replayed, before)


def test_entropy_padded_short_batch_equals_unpadded():
    x = _batch(8, 71).cuda()
    padded = build_p0_model("resnet18", "cuda")
    padded.slq_calibrate(x)                                   # an engine for batch 8
    padded.slq_calibrate(x[:5], method="entropy")             # 5 images, padded to 8
    assert _engine(padded).N == 8
    exact = build_p0_model("resnet18", "cuda")
    exact.slq_calibrate(x[:5], method="entropy")              # an engine for batch 5
    assert _engine(exact).N == 5
    assert torch.equal(_engine(padded).act_scales, _engine(exact).act_scales)


def test_entropy_one_shot_iterator_raises():
    net = build_p0_model("resnet18", "cuda")
    x = _batch(2, 81).cuda()
    with pytest.raises(TypeError):
        net.slq_calibrate(iter([x]), method="entropy")
    with pytest.raises(TypeError):
        net.slq_calibrate((b for b in [x]), method="entropy")


def test_resnet50_batch256_heldout_entropy():
    _check_heldout(build_p0_model("resnet50", "cuda"), 256, (11, 12, 13), "R50@256", "entropy")


def test_resnet34_batch128_heldout_entropy():
    _check_heldout(build_p0_model("resnet34", "cuda"), 128, (21, 22, 23), "R34@128", "entropy")
