"""Histogram calibration of the activation scales on the device (csrc/calib.cu, include/slq.h section 3):

  * slq_act_histogram counter for counter against the oracle (sizes, offset pointers, signed and mostly-zero
    inputs, two calls accumulating into one histogram, an R50@256-sized layer output);
  * slq_hist_scales against the oracle: percentile bit-exact; mse at the numpy minimum of its own error;
  * the engine and the public API (``net.slq_calibrate(..., method=...)``);
  * held-out logits parity of both methods on BASELINE.json's R50@256 and R34@128 configurations, with the
    bars of tests/test_baseline_configs_gpu.py.
"""
import numpy as np
import pytest
import torch

import slq_lib as L
import calib_oracle as co
import slq_oracle as so
from helpers import build_p0_model, rel_l2

pytestmark = pytest.mark.gpu

LOGITS_REL_L2_TOL = 1e-2
TOP1_AGREEMENT_MIN = 0.90


def _device_hist(parts, rng, bins, n_tensors=1, id=0):
    """parts: device fp32 tensors (any offset) added into histogram `id` one call each."""
    lib = L.lib()
    hist = torch.zeros((n_tensors, bins + 1), dtype=torch.int64, device="cuda")
    r = torch.full((n_tensors,), float(rng), dtype=torch.float32, device="cuda")
    for y in parts:
        L.check(lib.slq_act_histogram(y.data_ptr(), y.numel(), r.data_ptr(), id, bins, hist.data_ptr(), L.current_stream()))
    torch.cuda.synchronize()
    return hist.cpu().numpy().view(np.uint64)


@pytest.mark.parametrize("n", [1, 5, (1 << 20) + 3])
@pytest.mark.parametrize("offset", [0, 1, 3])
def test_act_histogram_matches_oracle(n, offset):
    g = torch.Generator(device="cuda").manual_seed(n + offset)
    base = torch.randn(n + offset, generator=g, device="cuda") * 3
    y = base[offset:]
    yh = y.cpu().numpy()
    rng = np.float32(np.abs(yh).max() * 0.8) if n > 1 else np.float32(1.0)
    for bins in (16, 2048):
        got = _device_hist([y], rng, bins)[0]
        assert np.array_equal(got, co.act_histogram(yh, rng, bins)), (n, offset, bins)
        assert int(got.sum()) == n


def test_act_histogram_mostly_zero_and_accumulating():
    g = torch.Generator(device="cuda").manual_seed(7)
    a = torch.relu(torch.randn(3_000_001, generator=g, device="cuda"))
    a[torch.rand(a.numel(), generator=g, device="cuda") < 0.99] = 0
    a[5] = -0.0
    b = torch.randn(777_777, generator=g, device="cuda")[1:]
    rng = np.float32(2.5)
    got = _device_hist([a, b], rng, 2048, n_tensors=3, id=2)
    assert not got[:2].any()
    want = co.act_histogram(a.cpu().numpy(), rng, 2048) + co.act_histogram(b.cpu().numpy(), rng, 2048)
    assert np.array_equal(got[2], want)


def test_act_histogram_r50_layer_output():
    # the largest fp32 layer output of ResNet-50 at batch 256: [256, 56, 56, 256] (822 MB)
    n = 256 * 56 * 56 * 256
    g = torch.Generator(device="cuda").manual_seed(11)
    y = torch.relu(torch.randn(n, generator=g, device="cuda") * 1.5 - 0.2)
    rng = np.float32(torch.max(y).item())
    got = _device_hist([y], rng, 2048)[0]
    assert np.array_equal(got, co.act_histogram(y.cpu().numpy(), rng, 2048))


def _device_scales(hists, rngs, qmaxs, method, percentile=99.99, headroom=1.0):
    lib = L.lib()
    h = torch.from_numpy(np.stack(hists).view(np.int64)).cuda()
    r = torch.tensor(np.asarray(rngs, np.float32), device="cuda")
    q = torch.tensor(np.asarray(qmaxs, np.int32), device="cuda")
    out = torch.full((len(hists),), -1.0, dtype=torch.float32, device="cuda")
    m = L.CALIB_PERCENTILE if method == "percentile" else L.CALIB_MSE
    L.check(lib.slq_hist_scales(h.data_ptr(), len(hists), h.shape[1] - 1, r.data_ptr(), q.data_ptr(), m, percentile,
                                headroom, out.data_ptr(), L.current_stream()))
    return out.cpu().numpy()


def _hist_cases(bins):
    rng = np.random.default_rng(bins)
    hists, rngs, qmaxs = [], [], []
    for t in range(12):
        y = np.maximum(rng.standard_normal(20000) * (1 + t), 0).astype(np.float32)
        if t % 3 == 1:
            y = (rng.standard_normal(20000) * (1 + t)).astype(np.float32)  # signed: an s8 tensor
        if t % 4 == 3:
            y[rng.random(y.size) < 0.97] = 0
        r = np.float32(np.abs(y).max() * (1.0 if t % 2 else 0.9))
        hists.append(co.act_histogram(y, r, bins))
        rngs.append(r)
        qmaxs.append(127 if t % 3 == 1 else 255)
    hists.append(np.zeros(bins + 1, np.uint64))                   # empty
    hists.append(np.array([9] + [0] * bins, np.uint64))           # zeros only
    rngs += [np.float32(1.0), np.float32(2.0)]
    qmaxs += [255, 127]
    return hists, rngs, qmaxs


@pytest.mark.parametrize("bins", [16, 2048])
@pytest.mark.parametrize("percentile,headroom", [(99.99, 1.0), (99.0, 1.25), (50.0, 1.0), (100.0, 1.0)])
def test_hist_scales_percentile_bit_exact(bins, percentile, headroom):
    hists, rngs, qmaxs = _hist_cases(bins)
    got = _device_scales(hists, rngs, qmaxs, "percentile", percentile, headroom)
    want = np.array([co.hist_scale(h, r, q, "percentile", percentile, headroom) for h, r, q in zip(hists, rngs, qmaxs)])
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert got[-1] == 1.0 and got[-2] == 1.0


@pytest.mark.parametrize("bins,headroom", [(16, 1.0), (2048, 1.0), (2048, 1.5)])
def test_hist_scales_mse_at_the_minimum(bins, headroom):
    hists, rngs, qmaxs = _hist_cases(bins)
    got = _device_scales(hists, rngs, qmaxs, "mse", headroom=headroom)
    for t, (h, r, q) in enumerate(zip(hists, rngs, qmaxs)):
        if not h[1:].any():
            assert got[t] == 1.0
            continue
        cands = [k for k in range(1, bins + 1) if co.hist_scale_for_k(r, k, bins, q, headroom) == got[t]]
        assert len(cands) == 1, (t, got[t])
        err = co.hist_mse_errors(h, r, q)
        assert err[cands[0] - 1] <= err.min() * (1 + 1e-12), (t, cands[0], err[cands[0] - 1], err.min())


def test_percentile_100_reproduces_absmax():
    lib = L.lib()
    g = torch.Generator(device="cuda").manual_seed(3)
    ys = [torch.relu(torch.randn(100_003, generator=g, device="cuda")) * (t + 1) for t in range(3)]
    ys.append(torch.randn(50_001, generator=g, device="cuda"))  # signed: qmax 127
    qmax = [255, 255, 255, 127]
    sc = torch.zeros(4, dtype=torch.float32, device="cuda")
    tmp = torch.zeros(1, dtype=torch.int32, device="cuda")
    st = L.current_stream()
    for t, y in enumerate(ys):
        L.check(lib.slq_absmax_scale(y.data_ptr(), y.numel(), sc.data_ptr(), t, qmax[t], tmp.data_ptr(), st))
    q = torch.tensor(qmax, dtype=torch.int32, device="cuda")
    rng = sc * q.to(torch.float32)
    hist = torch.zeros((4, 2049), dtype=torch.int64, device="cuda")
    for t, y in enumerate(ys):
        L.check(lib.slq_act_histogram(y.data_ptr(), y.numel(), rng.data_ptr(), t, 2048, hist.data_ptr(), st))
    out = torch.zeros(4, dtype=torch.float32, device="cuda")
    L.check(lib.slq_hist_scales(hist.data_ptr(), 4, 2048, rng.data_ptr(), q.data_ptr(), L.CALIB_PERCENTILE, 100.0, 1.0,
                                out.data_ptr(), st))
    a, b = sc.cpu().numpy().view(np.int32), out.cpu().numpy().view(np.int32)
    assert np.abs(a.astype(np.int64) - b).max() <= 1, (sc, out)


# ---- engine and public API --------------------------------------------------------------------------------------
def _batch(n, seed, hw=224):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, hw, hw, generator=g)


def _engine(net):
    return next(iter(net._slq_engines.values()))


def test_absmax_method_is_the_default_path():
    net = build_p0_model("resnet18", "cuda")
    a, b, c = _batch(8, 51).cuda(), _batch(8, 52).cuda(), _batch(8, 53).cuda()
    net.slq_calibrate([a, b])
    s0 = _engine(net).act_scales.clone()
    with torch.no_grad():
        l0 = net(c).clone()
    net.slq_calibrate([a, b], method="absmax")
    assert torch.equal(_engine(net).act_scales, s0)
    with torch.no_grad():
        assert torch.equal(net(c), l0)


@pytest.mark.parametrize("method", ["percentile", "mse"])
def test_histogram_methods_engine_semantics(method):
    net = build_p0_model("resnet18", "cuda")
    a, b, c = _batch(8, 61).cuda(), _batch(8, 62).cuda(), _batch(8, 63).cuda()
    net.slq_calibrate([a, b])
    eng = _engine(net)
    s_abs = eng.act_scales.clone()
    # a graph captured under the abs-max scales
    g = eng.capture_graph(c)
    g.replay()
    before = eng.logits.clone()
    net.slq_calibrate([a, (b, None)], method=method)
    assert _engine(net) is eng
    s1 = eng.act_scales.clone()
    assert not torch.equal(s1, s_abs)
    ulp = torch.nextafter(s_abs, torch.full_like(s_abs, float("inf")))
    assert bool((s1 <= ulp).all()), (s1 - s_abs).max()
    net.slq_calibrate([a, b], method=method)
    assert torch.equal(eng.act_scales, s1)                    # repeated calibration is bit-identical
    # the graph reads act_scales through its pointer: it now runs under the new scales
    g.replay()
    replayed = eng.logits.clone()
    eng.launch_all(c.data_ptr(), L.current_stream())
    assert torch.equal(replayed, eng.logits) and not torch.equal(replayed, before)


@pytest.mark.parametrize("method", ["percentile", "mse"])
def test_padded_short_batch_equals_unpadded(method):
    x = _batch(8, 71).cuda()
    padded = build_p0_model("resnet18", "cuda")
    padded.slq_calibrate(x)                                   # an engine for batch 8
    padded.slq_calibrate(x[:5], method=method)                # 5 images, padded to 8
    assert _engine(padded).N == 8
    exact = build_p0_model("resnet18", "cuda")
    exact.slq_calibrate(x[:5], method=method)                 # an engine for batch 5
    assert _engine(exact).N == 5
    assert torch.equal(_engine(padded).act_scales, _engine(exact).act_scales)


def test_one_shot_iterator_raises():
    net = build_p0_model("resnet18", "cuda")
    x = _batch(2, 81).cuda()
    with pytest.raises(TypeError):
        net.slq_calibrate(iter([x]), method="mse")
    with pytest.raises(TypeError):
        net.slq_calibrate((b for b in [x]), method="percentile")
    net.slq_calibrate(iter([x]))                               # abs-max reads once: fine


# ---- held-out parity --------------------------------------------------------------------------------------------
def _check_heldout(net, batch, seeds, tag, method):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net.slq_calibrate(_batch(batch, seeds[0]).cuda(), method=method)
    worst, agree, total = 0.0, 0, 0
    for s in seeds[1:]:
        x = _batch(batch, s).cuda()
        with torch.no_grad():
            got = net(x)
        ref = so.torch_forward(net, x)
        err = rel_l2(got.cpu().numpy(), ref.cpu().numpy())
        worst = max(worst, err)
        a, r = got.argmax(1), ref.argmax(1)
        agree += int((a == r).sum())
        total += batch
        flipped = (a != r).nonzero().flatten()
        if len(flipped):   # every flip a near-tie of the reference
            top2 = ref[flipped].topk(2, dim=1).values
            margin = top2[:, 0] - top2[:, 1]
            dmax = (got[flipped] - ref[flipped]).abs().max(1).values
            assert bool((margin <= 2 * dmax + 1e-6).all())
            assert (margin / ref[flipped].abs().max(1).values).max().item() < 2e-2
        print("%s %s seed %d: rel-L2 %.3e, top-1 agreement %d/%d" % (tag, method, s, err, int((a == r).sum()), batch))
    assert worst <= LOGITS_REL_L2_TOL, worst
    assert agree >= TOP1_AGREEMENT_MIN * total, (agree, total)


@pytest.mark.parametrize("method", ["percentile", "mse"])
def test_resnet50_batch256_heldout(method):
    _check_heldout(build_p0_model("resnet50", "cuda"), 256, (11, 12, 13), "R50@256", method)


@pytest.mark.parametrize("method", ["percentile", "mse"])
def test_resnet34_batch128_heldout(method):
    _check_heldout(build_p0_model("resnet34", "cuda"), 128, (21, 22, 23), "R34@128", method)
