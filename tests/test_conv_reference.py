"""The torch conv reference (tests/conv_reference.py) against the numpy oracle, bit for bit, on the CPU: the exact
accumulators of conv_acc and every epilogue flavour the kernels implement.  The GPU tests at production batch
(test_conv_production_gpu.py) trust the torch reference because of this pin."""
import numpy as np
import pytest
import torch

import conv_reference as cr
import slq_oracle as so


def _naive_fma32(a, b, c):
    """float32(float64(a*b + c)): two roundings, the result fma32 must correct on midpoint ties."""
    a, b, c = (np.asarray(v, np.float32).astype(np.float64) for v in (a, b, c))
    return (a * b + c).astype(np.float32)


def _tie_cases():
    """(a, b, c) whose exact a*b + c lies within 2^-58 of a float32 midpoint: the float64 sum lands ON the
    midpoint, and rounding it to float32 (ties to even) goes the wrong way in half of the cases."""
    e = 2.0 ** -18
    base = [
        # 1 + 3*2^-24 - 3*2^-60: float64 -> 1 + 3*2^-24 (tie, even neighbour 1 + 2^-22); exact -> 1 + 2^-23
        (3 * 2.0 ** -24 * (1 + e), 1 - e, 1.0),
        # 1 + 2^-24 + 2^-60: float64 -> 1 + 2^-24 (tie, even neighbour 1); exact -> 1 + 2^-23
        (-(2.0 ** -24) * (1 + e), 1 - e, 1 + 2.0 ** -23),
        # 1 + 2^-24 - 2^-60: a tie the naive rounding already gets right (below the midpoint, even side)
        (2.0 ** -24 * (1 + e), 1 - e, 1.0),
    ]
    out = []
    for (a, b, c) in base:
        for scale in (2.0 ** -30, 1.0, 2.0 ** 20):
            for sa, sc in ((1, 1), (-1, -1)):
                out.append((sa * a * scale, b, sc * c * scale))
    return [tuple(np.float32(v) for v in t) for t in out]


def test_fma32_matches_oracle_including_double_rounding_ties():
    ties = np.array(_tie_cases(), np.float32)
    rng = np.random.default_rng(0)
    rand = np.stack([rng.standard_normal(20000), rng.standard_normal(20000) * 1e3,
                     rng.standard_normal(20000) * 1e-3], 1).astype(np.float32)
    for abc in (ties, rand):
        a, b, c = abc[:, 0], abc[:, 1], abc[:, 2]
        want = so.fma32(a, b, c)
        got = cr.fma32(*(torch.from_numpy(v.copy()) for v in (a, b, c))).numpy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    a, b, c = ties[:, 0], ties[:, 1], ties[:, 2]
    naive = _naive_fma32(a, b, c)
    got = cr.fma32(*(torch.from_numpy(v.copy()) for v in (a, b, c))).numpy()
    # the set must reach the double-rounding correction, in both directions, and also hold ties it must not touch
    fixed = got.view(np.uint32) != naive.view(np.uint32)
    assert fixed.sum() >= 4 and (~fixed).sum() >= 4
    assert ((got > naive) & fixed).any() and ((got < naive) & fixed).any()
    # and the corrected value is the correctly rounded one (exact rational arithmetic)
    from fractions import Fraction
    for i in np.nonzero(fixed)[0]:
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        err_got = abs(Fraction(float(got[i])) - exact)
        err_naive = abs(Fraction(float(naive[i])) - exact)
        assert err_got < err_naive


def _codes(cout, cin, k, w16, rng):
    hi = 65536 if w16 else 256
    c = rng.integers(0, hi, (cout, k, k, cin))
    if w16:  # limbs at their ends too
        c[0] = 65535
        c[1] = 255
    return c


CASES = [  # (N, H, cin, cout, k, stride, w16)
    (2, 7, 16, 24, 3, 1, False),
    (3, 9, 8, 16, 3, 2, False),
    (2, 8, 32, 8, 1, 1, False),
    (2, 9, 16, 12, 1, 2, False),
    (1, 6, 8, 8, 3, 1, True),
    (2, 8, 16, 8, 1, 2, True),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "n%d_h%d_c%d-%d_k%d_s%d%s" % (c[:6] + ("_w16" if c[6] else "",)))
def test_conv_acc_and_epilogues_match_oracle(case):
    N, H, cin, cout, k, stride, w16 = case
    pad = k // 2
    rng = np.random.default_rng(N * 100 + H * 10 + cin + cout)
    x = rng.integers(0, 256, (N, H, H, cin), dtype=np.uint8)
    x[0, 0] = 255
    x[-1, -1] = 0
    codes = _codes(cout, cin, k, w16, rng)
    if w16:
        lo_o, S_o, _, _ = so.conv_acc(x, codes & 255, stride, pad)
        hi_o, _, _, _ = so.conv_acc(x, codes >> 8, stride, pad)
    else:
        lo_o, S_o, _, _ = so.conv_acc(x, codes, stride, pad)
        hi_o = None
    lo, hi, S = cr.conv_acc(torch.from_numpy(x), torch.from_numpy(codes), stride, pad, w16)
    assert np.array_equal(lo.numpy(), lo_o) and np.array_equal(S.numpy(), S_o)
    if w16:
        assert np.array_equal(hi.numpy(), hi_o)
    M = lo.shape[0]
    zf = -rng.integers(0, 200, cout).astype(np.float32) * (256.0 if w16 else 1.0)
    wscale = (rng.uniform(0.5, 1.5, cout) / (cin * k * k * 40.0 * (256.0 if w16 else 1.0))).astype(np.float32)
    bias = rng.normal(0, 0.5, cout).astype(np.float32)
    s_in, s_out, s_res = np.float32(1.0), np.float32(1 / 64), np.float32(1 / 32)
    res = rng.integers(0, 256, (M, cout), dtype=np.uint8)
    tres = torch.from_numpy(res)
    for r, rs in ((None, False), (res, False), (res, True)):
        tr = tres if r is not None else None
        for relu in (True, False):
            want = so.epilogue(lo_o, S_o, zf, wscale, bias, s_in, r, s_res, relu=relu, acc_hi=hi_o, res_signed=rs)
            got = cr.epilogue(lo, S, zf, wscale, bias, s_in, "f32", hi=hi, res=tr, s_res=s_res, res_signed=rs,
                              relu=relu, rows=37).numpy()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), ("f32", r is not None, rs, relu)
        for signed_out in (False, True):
            want = so.epilogue_q(lo_o, S_o, zf, wscale, bias, s_in, s_out, r, s_res, acc_hi=hi_o, res_signed=rs,
                                 signed_out=signed_out)
            got = cr.epilogue(lo, S, zf, wscale, bias, s_in, "s8" if signed_out else "u8", s_out=s_out, hi=hi,
                              res=tr, s_res=s_res, res_signed=rs, rows=37).numpy()
            assert np.array_equal(got, want), ("q", r is not None, rs, signed_out)
            # the parameters use the range: both ends saturate
            lo_b, hi_b = (128, 127) if signed_out else (0, 255)
            assert (want == lo_b).any() and (want == hi_b).any()


def test_epilogue_constants_fold_inv_before_use():
    """chan_consts: the re-quantisation multiply is folded into each constant AFTER zw = zf * wsc is rounded."""
    rng = np.random.default_rng(5)
    ws, zf, b = (rng.standard_normal(64).astype(np.float32) for _ in range(3))
    wsc, zw, bb = cr.chan_consts(ws, zf, b, np.float32(0.37), np.float32(0.011))
    f = np.float32
    inv = f(1) / f(0.011)
    w1 = (ws * f(0.37)).astype(f)
    assert np.array_equal(wsc.numpy(), (w1 * inv).astype(f))
    assert np.array_equal(zw.numpy(), ((zf * w1).astype(f) * inv).astype(f))
    assert np.array_equal(bb.numpy(), (b * inv).astype(f))
