"""tools/calib_methods.py -- what each activation-scale calibration method (``net.slq_calibrate(method=...)``) buys:

  * held-out logits parity (rel-L2 against the reference's fp32 fake-quant forward, top-1 agreement) of "absmax",
    "percentile", "mse" and "entropy" on BASELINE.json's R50 @256 and R34 @128 configurations, calibrated on
    1 batch and on 8 batches (the held-out batches are those of tests/test_baseline_configs_gpu.py);
  * calibration wall time of each method (batches already on the device; host clock around a synchronised call);
  * slq_act_histogram throughput on the largest fp32 layer output of R50 @256 ([256, 56, 56, 256], 822 MB: larger
    than L2), next to a device-to-device copy of the same tensor timed in the same run;
  * slq_hist_scales time per threshold rule (CUDA events) on the real histograms of every activation tensor of
    R50 @256, taken from one calibration walk.

The card's name and power limit are read in the same run and written beside the numbers.
usage: python tools/calib_methods.py --out profiles/calib_methods.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("semilayer-wise-mixed-precision-quantization_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))

import slq_lib as L  # noqa: E402
import slq_oracle as so  # noqa: E402
from helpers import build_p0_model, rel_l2  # noqa: E402

METHODS = ("absmax", "percentile", "mse", "entropy")
CONFIGS = [("resnet50", 256, 11, (12, 13)), ("resnet34", 128, 21, (22, 23))]


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                    text=True).splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")]
    except (OSError, subprocess.CalledProcessError) as e:
        info["power_limit"] = "unknown (%s)" % e
    return info


def batch(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, 224, 224, generator=g)


def parity(arch, n, calib_seed, heldout, n_calib):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = build_p0_model(arch, "cuda")
    xs = [batch(n, s).cuda() for s in heldout]
    refs = [so.torch_forward(net, x) for x in xs]
    cal = [batch(n, calib_seed).cuda()] + [batch(n, 1000 * calib_seed + i).cuda() for i in range(1, n_calib)]
    rows = []
    for method in METHODS:
        net.slq_calibrate(cal, method=method)  # warm: engine built, weights packed
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        net.slq_calibrate(cal, method=method)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        errs, agree = [], 0
        for x, ref in zip(xs, refs):
            with torch.no_grad():
                got = net(x)
            errs.append(rel_l2(got.cpu().numpy(), ref.cpu().numpy()))
            agree += int((got.argmax(1) == ref.argmax(1)).sum())
        scales = next(iter(net._slq_engines.values())).act_scales
        row = dict(arch=arch, batch=n, calib_batches=n_calib, method=method, calib_wall_ms=1e3 * wall,
                   heldout_rel_l2=errs, heldout_rel_l2_mean=float(np.mean(errs)),
                   top1_agreement=agree / (n * len(xs)), mean_scale=float(scales.mean()))
        print(json.dumps(row), flush=True)
        rows.append(row)
    return rows


def hist_bandwidth(iters=20):
    lib = L.lib()
    n = 256 * 56 * 56 * 256
    g = torch.Generator(device="cuda").manual_seed(0)
    y = torch.relu(torch.randn(n, generator=g, device="cuda"))  # post-ReLU: about half zeros
    rng = torch.full((1,), float(y.max()), dtype=torch.float32, device="cuda")
    hist = torch.zeros((1, 2049), dtype=torch.int64, device="cuda")
    dst = torch.empty_like(y)
    st = L.current_stream()

    def timed(fn):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e-3

    res = {}
    for rep in range(2):  # alternated, twice
        t_h = timed(lambda: L.check(lib.slq_act_histogram(y.data_ptr(), n, rng.data_ptr(), 0, 2048, hist.data_ptr(), st)))
        t_c = timed(lambda: dst.copy_(y))
        res.setdefault("act_histogram_us", []).append(t_h * 1e6)
        res.setdefault("copy_us", []).append(t_c * 1e6)
    t_h, t_c = min(res["act_histogram_us"]) * 1e-6, min(res["copy_us"]) * 1e-6
    res.update(bytes=4 * n, act_histogram_read_GBps=4 * n / t_h / 1e9, copy_read_plus_write_GBps=8 * n / t_c / 1e9,
               copy_read_GBps=4 * n / t_c / 1e9)
    print(json.dumps(res), flush=True)
    return res


def hist_scales_time(iters=20):
    lib = L.lib()
    net = build_p0_model("resnet50", "cuda")
    x = batch(256, 11).cuda()
    net.slq_calibrate(x)  # abs-max: the ranges of the histogram pass
    eng = next(iter(net._slq_engines.values()))
    q = eng.act_qmax()
    rng = eng.act_scales * q.to(torch.float32)
    bins = net.CALIB_BINS
    hist = torch.zeros((len(eng.act), bins + 1), dtype=torch.int64, device="cuda")
    eng.histogram(x, hist, rng, bins)
    out = torch.empty(len(eng.act), dtype=torch.float32, device="cuda")
    st = L.current_stream()
    rules = {"percentile": L.CALIB_PERCENTILE, "mse": L.CALIB_MSE, "entropy": L.CALIB_ENTROPY}

    def launch(rule):
        L.check(lib.slq_hist_scales(hist.data_ptr(), len(eng.act), bins, rng.data_ptr(), q.data_ptr(), rule, 99.99,
                                    1.0, out.data_ptr(), st))

    res = {"tensors": len(eng.act), "bins": bins, "iters": iters}
    for rep in range(2):  # the rules alternated, twice
        for name, rule in rules.items():
            for _ in range(3):
                launch(rule)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                launch(rule)
            e1.record()
            torch.cuda.synchronize()
            res.setdefault(name + "_us", []).append(e0.elapsed_time(e1) / iters * 1e3)
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    out = {"card": card(), "histogram": hist_bandwidth(), "hist_scales": hist_scales_time(), "parity": []}
    for arch, n, cs, held in CONFIGS:
        for n_calib in (1, 8):
            out["parity"] += parity(arch, n, cs, held, n_calib)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
