"""tests/conv_reference.py -- an exact reference of the quantised convolution, written in torch so that it
runs on the GPU at the production batch (256) as well as on the CPU.

It shares no code with the kernels or with their checkers (csrc/epilogue.cuh, the dp4a SIMT kernel): it restates
the arithmetic contract of include/slq.h (slq_conv_launch) from scratch, and tests/test_conv_reference.py pins
it bit for bit to the numpy oracle (oracle/slq_oracle.py conv_acc / epilogue / epilogue_q).

Accumulators.  acc[m, oc] = sum_k A[m, k] * code[oc, k] and S[m] = sum_k A[m, k] are float64 GEMMs over an
explicit im2col A (F.unfold of the NCHW input, or a strided slice for 1x1 layers) with K ordered (r, s, c) like
the GEMM-ready weights.  Every partial sum is an integer below 4608 * 255 * 255 < 2^53, so float64 is exact in
any summation order.  F.conv2d is deliberately not used: cuDNN may pick a Winograd or FFT algorithm, and those
are not exact.  Two-limb (16-bit code) layers run one GEMM per limb.

Epilogue.  The fp32 chain, every step rounded once (fma32 is a correctly rounded fused multiply-add):
  per channel : wsc = wscale * s_in ; zw = zf * wsc ; b = bias       (u8 / s8 out: each times inv = 1 / s_out)
  per element : accf = f32(acc)  [two limbs: fma(f32(hi), 256, f32(lo))]
                y = fma(accf, wsc, fma(f32(S), zw, b)) ; y = fma(f32(res), sr, y)     (sr = s_res [* inv])
  f32 out     : relu ? max(y, 0) : y        u8 / s8 out : sat(rint(y))
"""
import torch
import torch.nn.functional as F

_ELEMS = 1 << 26  # float64 elements of one im2col chunk (512 MB)


def im2col_chunks(x, k, stride, pad):
    """x: u8 NHWC [N, H, W, C] (any device).  Yields float64 A chunks [m, k*k*C], K ordered (r, s, c), in pixel
    order, a whole number of images each."""
    N, H, W, C = x.shape
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    per = max(1, _ELEMS // (Ho * Wo * k * k * C))
    for n0 in range(0, N, per):
        xs = x[n0:n0 + per]
        n = xs.shape[0]
        if k == 1 and pad == 0:
            yield xs[:, ::stride, ::stride, :].reshape(n * Ho * Wo, C).to(torch.float64)
            continue
        cols = F.unfold(xs.permute(0, 3, 1, 2).to(torch.float64), k, padding=pad, stride=stride)  # [n, C*k*k, L]
        yield cols.view(n, C, k * k, Ho * Wo).permute(0, 3, 2, 1).reshape(n * Ho * Wo, k * k * C)


def conv_acc(x, codes, stride, pad, w16=False):
    """Exact accumulators of the u8 x u8 implicit GEMM.
    x: u8 NHWC [N, H, W, C]; codes: integer [Cout, k, k, C] (OHWI, >= 0; 16-bit when w16).
    Returns int32 tensors (lo [M, Cout], hi [M, Cout] or None, S [M]) on x's device; one-limb layers return the
    whole accumulator as lo."""
    cout, k = codes.shape[0], codes.shape[1]
    B = codes.reshape(cout, -1).to(device=x.device, dtype=torch.int64)
    limbs = [B & 255, B >> 8] if w16 else [B]
    limbs = [b.to(torch.float64).t().contiguous() for b in limbs]
    outs, sums = [[] for _ in limbs], []
    for A in im2col_chunks(x, k, stride, pad):
        for o, b in zip(outs, limbs):
            o.append((A @ b).to(torch.int32))
        sums.append(A.sum(1).to(torch.int32))
    acc = [torch.cat(o) for o in outs]
    return acc[0], (acc[1] if w16 else None), torch.cat(sums)


def fma32(a, b, c):
    """Correctly rounded float32 a*b + c (what __fmaf_rn computes) on float32 tensors of broadcastable shapes.
    a*b is exact in float64; the float64 sum s is rounded once more to float32, and where s sits exactly on a
    float32 midpoint the exact TwoSum error term of s decides the direction (the double-rounding case)."""
    a, b, c = (t.to(torch.float64) for t in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)  # p + c == s + err exactly
    r = s.to(torch.float32)
    rd = r.to(torch.float64)
    other = torch.where(s > rd, torch.nextafter(r, torch.full_like(r, float("inf"))),
                        torch.nextafter(r, torch.full_like(r, float("-inf"))))
    od = other.to(torch.float64)
    tie = (s == (rd + od) / 2) & (s != rd)
    toward = torch.sign(err) == torch.sign(od - rd)
    return torch.where(tie & (err != 0) & toward, other, r)


def chan_consts(wscale, zf, bias, s_in, s_out=None):
    """Per-channel (A, Z, B) of the chain, float32, each product rounded once; s_out given: u8 / s8 output."""
    f = lambda v: torch.as_tensor(v, dtype=torch.float32).cpu()
    wsc = f(wscale) * f(s_in)
    zw = f(zf) * wsc
    b = f(bias).clone()
    if s_out is not None:
        inv = torch.tensor(1.0, dtype=torch.float32) / f(s_out)
        wsc, zw, b = wsc * inv, zw * inv, b * inv
    return wsc, zw, b


def epilogue(lo, S, zf, wscale, bias, s_in, mode, s_out=None, hi=None, res=None, s_res=None, res_signed=False,
             relu=True, rows=None):
    """The fused epilogue on exact accumulators (conv_acc), chunked over rows.
    mode: "f32" (float32 [M, Cout]), "u8" or "s8" (raw output bytes, uint8 [M, Cout]).
    res: u8 [M, Cout] residual bytes (read as int8 when res_signed) with scale s_res."""
    quant = mode != "f32"
    dev = lo.device
    wsc, zw, b = (t.to(dev) for t in chan_consts(wscale, zf, bias, s_in, s_out if quant else None))
    sr = None
    if res is not None:
        sr = torch.tensor(float(s_res), dtype=torch.float32)
        if quant:
            sr = sr * (torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(s_out), dtype=torch.float32))
        sr = sr.to(dev)
    M, cout = lo.shape
    rows = rows or max(1, (1 << 24) // cout)
    out = torch.empty((M, cout), dtype=torch.uint8 if quant else torch.float32, device=dev)
    two56 = torch.tensor(256.0, dtype=torch.float32, device=dev)
    for m0 in range(0, M, rows):
        sl = slice(m0, m0 + rows)
        accf = lo[sl].to(torch.float32)
        if hi is not None:
            accf = fma32(hi[sl].to(torch.float32), two56, accf)
        y = fma32(accf, wsc[None, :], fma32(S[sl].to(torch.float32)[:, None], zw[None, :], b[None, :]))
        if res is not None:
            r = res[sl].view(torch.int8) if res_signed else res[sl]
            y = fma32(r.to(torch.float32), sr, y)
        if not quant:
            out[sl] = torch.clamp_min(y, 0.0) if relu else y
        else:
            q = torch.nan_to_num(torch.round(y), nan=0.0)  # round half to even, like cvt.rni
            q = q.clamp(-128, 127).to(torch.int8).view(torch.uint8) if mode == "s8" else q.clamp(0, 255).to(torch.uint8)
            out[sl] = q
    return out
