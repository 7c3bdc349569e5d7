"""The stem (conv1 7x7/s2 + bn1 + ReLU + 3x3/s2 max-pool) and the calibration helpers it depends on, against a
float64 reference computed with torch's own conv2d (no code shared with the project).

Three stem kernels are covered, all driven through the C ABI:
  stem_ts_kernel     slq_stem_create picks it when W % 16 == 0 (A operand in TMEM, rows staged by TMA)
  stem_fused_kernel  the tensor-core path for every other W <= 256
  stem_conv_kernel   slq_stem_forward, the exact-fp32 CUDA-core stem (the only path for W > 256)

Error bounds are derived from the arithmetic each kernel performs, not fitted:
  * The tensor-core kernels round the image and the weights to fp16.  For W % 16 == 0 the BN scale is folded into
    the weights first, fp16(fp32(w * bn_a)), and the epilogue adds bn_b; otherwise the weights are fp16(w) and the
    epilogue computes acc * bn_a + bn_b.  Each fp16 x fp16 product is exact in fp32, so only the fp32 sum of the
    K = 192 (padded) products and the epilogue round.  The tensor core's accumulation rounding is not specified as
    round-to-nearest, so one rounding counts 2^-23 rather than 2^-24:
        delta = 192 * 2^-23 * sum|x16 * w16| * |m|  +  4 ulp(|acc * m| + |bn_b|)        (m = bn_a or 1)
    The 4 ulp cover the epilogue's fma, the fp32 roundings of bn_a / scale and bn_b / scale in the u8 path and
    the multiply by 1 / scale of the stand-alone pool kernel: at most 3 roundings of at most 1/2 ulp each.
  * The SIMT stem keeps the fp32 operands as given and sums the 147 products with sequential fmaf (IEEE
    round-to-nearest): 147 * 2^-24 * sum|x * w| * |bn_a| + 4 ulp(|acc * bn_a| + |bn_b|).
ReLU and max-pooling are 1-Lipschitz and monotone, so a bound on the conv rows carries over to the pooled output
as maxpool(delta), and a u8 byte must lie in the bracket [q(maxpool(ref - delta)), q(maxpool(ref + delta))] with
q(v) = clip(rint(v * fp32(1 / scale)), 0, 255).
"""
import contextlib
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

K_PAD = 192            # padded K of both tensor-core stem kernels (21 chunks of 8 halfs + 3 zero chunks)
UNIT_ROWS = 14         # pooled rows per work unit of the tensor-core stems
REF_CHUNK = 32         # images per float64 reference chunk (bounds its memory at the bench shape)
SENTINELS_U8 = (0x5A, 0xA5)
U_TC = 2.0 ** -23      # one fp32 rounding inside the tensor core (not specified as round-to-nearest)
U_RN = 2.0 ** -24      # one IEEE round-to-nearest fp32 rounding


def _L():
    import slq_lib as L
    return L, L.lib()


def _stream():
    import slq_lib as L
    return L.current_stream()


def sm_count():
    L, lib = _L()
    sms, major, minor = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    L.check(lib.slq_device_info(ctypes.byref(sms), ctypes.byref(major), ctypes.byref(minor)))
    return sms.value


def stem_dims(H, W):
    Hc, Wc = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    return Hc, Wc, (Hc - 1) // 2 + 1, (Wc - 1) // 2 + 1


def units_of(N, H):
    return N * math.ceil(stem_dims(H, 16)[2] / UNIT_ROWS)


def kernel_of(W):
    return "ts" if W % 16 == 0 else "fused"


def make_params(seed):
    """conv1 weights, and a BatchNorm fold a = gamma / sqrt(var + eps), b = beta - mean * a that is not the identity."""
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(64, 3, 7, 7, generator=g) * 0.05
    a = torch.rand(64, generator=g) + 0.5
    b = torch.randn(64, generator=g) * 0.2
    return w.cuda(), a.cuda(), b.cuda()


def make_image(N, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, 3, H, W, generator=g).cuda()


def norm_array():
    import imagenet
    return (ctypes.c_float * 6)(*(imagenet.MEAN + imagenet.STD))


# ------------------------------------------------------------------------------------------------------------
# launches
# ------------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def stem_handle(N, H, W, w=None):
    """slq_stem for (N, H, W) with a 256-byte aligned workspace; destroyed on the way out."""
    L, lib = _L()
    nbytes = lib.slq_stem_workspace_bytes(N, H, W)
    assert nbytes > 0
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    ws_ptr = (ws.data_ptr() + 255) // 256 * 256
    h = ctypes.c_void_p()
    L.check(lib.slq_stem_create(N, H, W, ws_ptr, ctypes.byref(h)))
    try:
        if w is not None:
            L.check(lib.slq_stem_set_weights(h, w.data_ptr(), _stream()))
        yield h
    finally:
        lib.slq_stem_destroy(h)
        del ws


def launch_f32(h, x, kind, a, b, H, W, norm=None):
    """SLQ_OUT_F32: returns (conv rows [N,Hc,Wc,64], pooled [N,Hp,Wp,64]), both NaN-filled before the launch."""
    L, lib = _L()
    N = x.shape[0]
    Hc, Wc, Hp, Wp = stem_dims(H, W)
    conv = torch.full((N, Hc, Wc, 64), float("nan"), dtype=torch.float32, device="cuda")
    pool = torch.full((N, Hp, Wp, 64), float("nan"), dtype=torch.float32, device="cuda")
    nrm = ctypes.cast(norm, ctypes.c_void_p) if norm is not None else None
    L.check(lib.slq_stem_launch_in(h, x.data_ptr(), kind, nrm, a.data_ptr(), b.data_ptr(), None, 0, pool.data_ptr(),
                                   L.OUT_F32, conv.data_ptr(), None, _stream()))
    torch.cuda.synchronize()
    return conv, pool


def launch_u8(h, x, kind, a, b, scales, H, W, norm=None, rowsum=True, sentinel=SENTINELS_U8[0]):
    """SLQ_OUT_U8: returns (pooled bytes [N,Hp,Wp,64] filled with `sentinel` before, rowsum [N*Hp*Wp] filled with -1
    before, or None when the launch gets a NULL out_rowsum)."""
    L, lib = _L()
    N = x.shape[0]
    Hc, Wc, Hp, Wp = stem_dims(H, W)
    out = torch.full((N, Hp, Wp, 64), sentinel, dtype=torch.uint8, device="cuda")
    rs = torch.full((N * Hp * Wp,), -1, dtype=torch.int32, device="cuda") if rowsum else None
    nrm = ctypes.cast(norm, ctypes.c_void_p) if norm is not None else None
    L.check(lib.slq_stem_launch_in(h, x.data_ptr(), kind, nrm, a.data_ptr(), b.data_ptr(), scales.data_ptr(), 0,
                                   out.data_ptr(), L.OUT_U8, None, L.ptr(rs), _stream()))
    torch.cuda.synchronize()
    return out, rs


def simt_forward(x, w, a, b, mode, scales=None, rowsum=True, sentinel=SENTINELS_U8[0]):
    """slq_stem_forward.  F32: (conv rows, pooled fp32); U8: (pooled bytes, rowsum or None)."""
    L, lib = _L()
    N, _, H, W = x.shape
    Hc, Wc, Hp, Wp = stem_dims(H, W)
    conv = torch.full((N, Hc, Wc, 64), float("nan"), dtype=torch.float32, device="cuda")
    if mode == L.OUT_F32:
        out = torch.full((N, Hp, Wp, 64), float("nan"), dtype=torch.float32, device="cuda")
        rs = None
    else:
        out = torch.full((N, Hp, Wp, 64), sentinel, dtype=torch.uint8, device="cuda")
        rs = torch.full((N * Hp * Wp,), -1, dtype=torch.int32, device="cuda") if rowsum else None
    L.check(lib.slq_stem_forward(x.data_ptr(), N, H, W, w.data_ptr(), a.data_ptr(), b.data_ptr(), L.ptr(scales), 0,
                                 conv.data_ptr(), out.data_ptr(), mode, L.ptr(rs), _stream()))
    torch.cuda.synchronize()
    return (conv, out) if mode == L.OUT_F32 else (out, rs)


def absmax_scale(y, scales, idx, qmax):
    L, lib = _L()
    tmp = torch.full((1,), 12345, dtype=torch.int32, device="cuda")  # the call zeroes it
    L.check(lib.slq_absmax_scale(y.data_ptr(), y.numel(), scales.data_ptr(), idx, qmax, tmp.data_ptr(), _stream()))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------------------------
def conv64(x, w):
    return F.conv2d(x.double(), w.double(), None, 2, 3)


def ulp32(v):
    """ulp of a non-negative fp32 value given in float64 (subnormal spacing below 2^-126)."""
    return torch.exp2(torch.floor(torch.log2(v.clamp_min(2.0 ** -126))) - 23)


def nhwc(t):
    return t.permute(0, 2, 3, 1)


def pool64(t):  # NCHW
    return F.max_pool2d(t, 3, 2, 1)


class StemRef:
    """What one stem kernel computes, in float64: the pre-ReLU value and the error bound delta (NCHW)."""

    def __init__(self, kernel, w, a, b):
        self.kernel, self.w, self.a, self.b = kernel, w, a, b
        col = lambda v: v.double()[None, :, None, None]
        self.bb = col(b)
        if kernel == "ts":      # stem_weights_ts_kernel + stem_ts_kernel's set-up: BN scale folded before fp16
            self.wk, self.m, self.k_err = (w * a[:, None, None, None]).half(), torch.ones_like(self.bb), K_PAD * U_TC
        elif kernel == "fused":  # stem_weights_kernel + the fused kernel's prm: fp16(w), acc * a + b
            self.wk, self.m, self.k_err = w.half(), col(a), K_PAD * U_TC
        else:                    # stem_conv_kernel: fp32 operands as given, 147 sequential fmaf
            self.wk, self.m, self.k_err = w, col(a), 147 * U_RN

    def operand(self, x):
        return x if self.kernel == "simt" else x.half()

    def __call__(self, x):
        xk = self.operand(x)
        am = conv64(xk, self.wk) * self.m
        ref = am + self.bb
        delta = self.k_err * conv64(xk.abs(), self.wk.abs()) * self.m.abs() + 4 * ulp32(am.abs() + self.bb.abs())
        return ref, delta

    def exact(self, x):
        """float64 conv of the unrounded operands (the fp32 model) and the extra room for rounding both operands of
        the tensor-core kernels to fp16: 2^-11 each, 2^-10 for a product.  The second-order terms (the fp32
        rounding of w * a, the product of the two fp16 errors: below 2^-21 of sum|x*w*a|) are covered by the
        accumulation term of delta, 192 * 2^-23 = 2^-15.4 of the same sum."""
        col = self.a.double()[None, :, None, None]
        return conv64(x, self.w) * col + self.bb, 2.0 ** -10 * conv64(x.abs(), self.w.abs()) * col.abs()


def _where(bad, got, want, tol, what, rows_per_unit):
    """A failure message that says where: count, NaNs, first positions with their work unit."""
    idx = bad.nonzero()
    lines = ["%s: %d of %d elements out of bound (%d NaN); rows %s" % (
        what, idx.shape[0], bad.numel(), int(torch.isnan(got.double()).sum()),
        sorted(set(idx[:, 1].tolist()))[:16])]
    for n, r, c, ch in idx[:6].tolist():
        lines.append("  image %d row %d col %d ch %d (unit %d of the image): got %r want %r tol %r" % (
            n, r, c, ch, r // rows_per_unit, float(got[n, r, c, ch]),
            float(want[n, r, c, ch]) if want is not None else float("nan"),
            float(tol[n, r, c, ch]) if tol is not None else 0.0))
    return "\n".join(lines)


def assert_within(got, want, tol, what, rows_per_unit):
    bad = ~((got.double() - want).abs() <= tol)  # NaN (a sentinel never overwritten) counts as out of bound
    assert not bool(bad.any()), _where(bad, got, want, tol, what, rows_per_unit)


def check_f32(ref, x32, conv, pool, exact):
    """conv rows and pooled fp32 output against the reference, chunk by chunk; the pooled output is also exactly
    the max-pool of the kernel's own conv rows."""
    for n0 in range(0, x32.shape[0], REF_CHUNK):
        xs = x32[n0:n0 + REF_CHUNK]
        cv, pl = conv[n0:n0 + REF_CHUNK], pool[n0:n0 + REF_CHUNK]
        r, d = ref(xs)
        assert_within(cv, nhwc(r.clamp_min(0)), nhwc(d), "conv rows (images %d..)" % n0, 2 * UNIT_ROWS)
        assert_within(pl, nhwc(pool64(r.clamp_min(0))), nhwc(pool64(d)), "pooled fp32 (images %d..)" % n0, UNIT_ROWS)
        own = nhwc(pool64(cv.permute(0, 3, 1, 2)))
        assert torch.equal(pl, own), "pooled fp32 is not the max-pool of the kernel's conv rows (images %d..)" % n0
        if exact:
            e, te = ref.exact(xs)
            assert_within(cv, nhwc(e.clamp_min(0)), nhwc(te + d), "conv rows vs fp32 model (images %d..)" % n0,
                          2 * UNIT_ROWS)
        del r, d


def check_u8(ref, x32, out, scale):
    """Monotone bracket: q(maxpool(ref - delta)) <= byte <= q(maxpool(ref + delta))."""
    inv = float(np.float32(1.0) / np.float32(scale))
    q = lambda v: torch.clamp(torch.round(v * inv), 0, 255)  # torch.round: half to even, like cvt.rni
    for n0 in range(0, x32.shape[0], REF_CHUNK):
        r, d = ref(x32[n0:n0 + REF_CHUNK])
        lo, hi = nhwc(q(pool64(r - d))), nhwc(q(pool64(r + d)))
        got = out[n0:n0 + REF_CHUNK].double()
        bad = (got < lo) | (got > hi)
        assert not bool(bad.any()), _where(bad, got, lo, hi - lo, "u8 bracket (want = lo, tol = hi - lo) images %d.." % n0,
                                           UNIT_ROWS)
        del r, d


def check_rowsum(out, rs):
    want = out.to(torch.int32).sum(-1).reshape(-1)
    assert torch.equal(rs, want), "out_rowsum is not the channel sum of the output bytes (%d wrong, %d never written)" % (
        int((rs != want).sum()), int((rs == -1).sum()))


# ------------------------------------------------------------------------------------------------------------
# the tensor-core stems: shapes, the persistent walk, calibration
# ------------------------------------------------------------------------------------------------------------
def run_tc_case(N, H, W, seed, exact):
    """fp32 input: F32 launch (conv rows + pooled) -> slq_absmax_scale(255) -> U8 launches, all against float64."""
    L, _ = _L()
    Hc, Wc, Hp, Wp = stem_dims(H, W)
    x = make_image(N, H, W, seed)
    w, a, b = make_params(seed + 1)
    ref = StemRef(kernel_of(W), w, a, b)
    with stem_handle(N, H, W, w) as h:
        conv, pool = launch_f32(h, x, L.IN_F32, a, b, H, W)
        check_f32(ref, x, conv, pool, exact)
        scales = torch.full((1,), -1.0, dtype=torch.float32, device="cuda")
        absmax_scale(pool, scales, 0, 255)
        want = np.float32(float(pool.max())) / np.float32(255)
        assert scales.cpu().numpy()[0].view(np.uint32) == want.view(np.uint32)
        del conv, pool
        outs = [launch_u8(h, x, L.IN_F32, a, b, scales, H, W, sentinel=s) for s in SENTINELS_U8]
        # two launches with different sentinels give the same bytes: every byte was written, and nothing a launch
        # leaves behind changes the next one
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        out, rs = outs[0]
        assert int(out.max()) == 255  # the calibrated scale maps the largest pooled value to the top byte
        check_rowsum(out, rs)
        out_norow, _ = launch_u8(h, x, L.IN_F32, a, b, scales, H, W, rowsum=False, sentinel=SENTINELS_U8[1])
        assert torch.equal(out_norow, out)
        check_u8(ref, x, out, float(scales[0]))


TS_SHAPES = [(2, 224, 224), (1, 7, 16), (3, 225, 224), (2, 61, 256), (2, 230, 32)]
FUSED_SHAPES = [(1, 7, 7), (2, 224, 200), (2, 227, 227), (3, 101, 255), (1, 33, 17)]


def _shape_id(p):
    return "%s-%dx%dx%d" % ((kernel_of(p[2]),) + tuple(p))


@pytest.mark.parametrize("N,H,W", TS_SHAPES + FUSED_SHAPES, ids=[_shape_id(p) for p in TS_SHAPES + FUSED_SHAPES])
def test_tensor_core_stem_against_float64(N, H, W):
    """Both tensor-core kernels at the shape edges: the minimum image, odd Hc (the last pooled row is closed by the
    last conv row), a short last unit (Hp % 14 != 0), Wc == 128 (a full tile) and TMA pairs that cross the bottom
    edge.  Conv rows, pooled fp32 and u8 bytes within the derived bound; the fp32 rows also against the fp32 model."""
    assert (W % 16 == 0) == (kernel_of(W) == "ts")
    run_tc_case(N, H, W, seed=N * 100003 + H * 1009 + W, exact=True)


WALK_SHAPES = [(225, 224), (101, 255), (227, 227)]


@pytest.mark.parametrize("H,W", WALK_SHAPES)
def test_tensor_core_stem_persistent_walk(H, W):
    """Every CTA walks at least three work units (one per SM are launched), of different sizes where Hp % 14 != 0:
    the mbarrier phases, rings and counters one unit hands to the next."""
    sms = sm_count()
    per_img = units_of(1, H)
    N = math.ceil(3 * sms / per_img)
    assert units_of(N, H) >= 3 * sms > sms
    run_tc_case(N, H, W, seed=H * 7 + W, exact=False)


def test_tensor_core_stem_bench_shape():
    """The benchmark's shape: N = 256 at 224x224, fp32 in, u8 out (about 7 units per CTA)."""
    assert units_of(256, 224) > 3 * sm_count()
    run_tc_case(256, 224, 224, seed=256, exact=False)


@pytest.mark.parametrize("N,H,W", [(3, 225, 224), (2, 227, 227)], ids=["ts-3x225x224", "fused-2x227x227"])
def test_fp16_and_u8_inputs_match_the_fp32_call_bit_for_bit(N, H, W):
    """SLQ_IN_F16 equals the fp32 call on the same fp16-representable image, and SLQ_IN_U8 with the ImageNet
    normalisation equals the fp32 call on imagenet.normalize_u8 of it -- every conv row, pooled value and byte.
    Rows above and below the image must become 0, not -mean / std."""
    import imagenet
    L, _ = _L()
    seed = N * 31 + H + W
    w, a, b = make_params(seed)
    x16 = make_image(N, H, W, seed).half()
    g = torch.Generator().manual_seed(seed + 1)
    x_u8 = torch.randint(0, 256, (N, 3, H, W), generator=g, dtype=torch.uint8)
    cases = [("fp16", x16, L.IN_F16, None, x16.float()),
             ("u8", x_u8.cuda(), L.IN_U8, norm_array(), imagenet.normalize_u8(x_u8).cuda())]
    scales = torch.full((1,), 0.02, dtype=torch.float32, device="cuda")
    with stem_handle(N, H, W, w) as h:
        for name, xin, kind, norm, x32 in cases:
            got = launch_f32(h, xin, kind, a, b, H, W, norm=norm)
            want = launch_f32(h, x32, L.IN_F32, a, b, H, W)
            for g_, w_, what in zip(got, want, ("conv rows", "pooled")):
                assert not bool(torch.isnan(w_).any())
                assert torch.equal(g_.view(torch.int32), w_.view(torch.int32)), "%s input: %s differ" % (name, what)
            got = launch_u8(h, xin, kind, a, b, scales, H, W, norm=norm)
            want = launch_u8(h, x32, L.IN_F32, a, b, scales, H, W, sentinel=SENTINELS_U8[1])
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), "%s input: u8 bytes differ" % name
            assert int(want[0].max()) > 0


@pytest.mark.parametrize("N,H,W", [(2, 61, 256), (3, 101, 255)], ids=["ts-2x61x256", "fused-3x101x255"])
def test_bn_and_weight_changes_are_seen_by_the_next_launch(N, H, W):
    """New bn_a / bn_b in the same buffers are honoured without slq_stem_set_weights (the ts kernel folds bn_a into
    the weights at every launch), and set_weights with new weights is honoured on the next launch."""
    L, _ = _L()
    seed = N + H + W
    x = make_image(N, H, W, seed)
    w1, a1, b1 = make_params(seed + 1)
    w2, a2, b2 = make_params(seed + 2)
    a, b = a1.clone(), b1.clone()
    with stem_handle(N, H, W, w1) as h:
        check_f32(StemRef(kernel_of(W), w1, a1, b1), x, *launch_f32(h, x, L.IN_F32, a, b, H, W), exact=False)
        a.copy_(a2)
        b.copy_(b2)
        check_f32(StemRef(kernel_of(W), w1, a2, b2), x, *launch_f32(h, x, L.IN_F32, a, b, H, W), exact=False)
        L.check(L.lib().slq_stem_set_weights(h, w2.data_ptr(), _stream()))
        check_f32(StemRef(kernel_of(W), w2, a2, b2), x, *launch_f32(h, x, L.IN_F32, a, b, H, W), exact=False)


# ------------------------------------------------------------------------------------------------------------
# the exact-fp32 CUDA-core stem
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,H,W", [(2, 64, 288), (1, 31, 301), (2, 99, 255)])
def test_simt_stem_against_float64(N, H, W):
    L, _ = _L()
    x = make_image(N, H, W, seed=N + H + W)
    w, a, b = make_params(N * H)
    ref = StemRef("simt", w, a, b)
    conv, pool = simt_forward(x, w, a, b, L.OUT_F32)
    check_f32(ref, x, conv, pool, exact=False)
    scales = torch.full((1,), -1.0, dtype=torch.float32, device="cuda")
    absmax_scale(pool, scales, 0, 255)
    out, rs = simt_forward(x, w, a, b, L.OUT_U8, scales)
    out2, _ = simt_forward(x, w, a, b, L.OUT_U8, scales, rowsum=False, sentinel=SENTINELS_U8[1])
    assert torch.equal(out, out2)
    assert int(out.max()) == 255
    check_rowsum(out, rs)
    check_u8(ref, x, out, float(scales[0]))


# ------------------------------------------------------------------------------------------------------------
# shape contract
# ------------------------------------------------------------------------------------------------------------
def _create_rc(N, H, W):
    L, lib = _L()
    ws = torch.empty(64 * K_PAD * 6 + 256, dtype=torch.uint8, device="cuda")
    h = ctypes.c_void_p()
    rc = lib.slq_stem_create(N, H, W, (ws.data_ptr() + 255) // 256 * 256, ctypes.byref(h))
    if rc == L.SLQ_OK:
        lib.slq_stem_destroy(h)
    return rc, (lib.slq_last_error() or b"").decode()


def test_stem_create_shape_contract():
    L, _ = _L()
    assert _create_rc(1, 16, 256)[0] == L.SLQ_OK
    assert _create_rc(1, 7, 7)[0] == L.SLQ_OK
    rc, msg = _create_rc(1, 16, 257)
    assert rc == L.SLQ_ERR_UNSUPPORTED and "slq_stem_forward" in msg
    for shape in [(1, 6, 16), (1, 16, 6), (0, 16, 16)]:
        assert _create_rc(*shape)[0] == L.SLQ_ERR_INVALID, shape


def test_ts_launch_rejects_an_image_that_is_not_16_byte_aligned():
    L, lib = _L()
    N, H, W = 1, 16, 16
    w, a, b = make_params(5)
    buf = torch.zeros(N * 3 * H * W + 4, dtype=torch.float32, device="cuda")
    x = buf[1:1 + N * 3 * H * W]  # 4 bytes into a valid allocation
    assert x.data_ptr() % 16 != 0
    scales = torch.ones(1, dtype=torch.float32, device="cuda")
    out = torch.full((N, *stem_dims(H, W)[2:], 64), 0x5A, dtype=torch.uint8, device="cuda")
    with stem_handle(N, H, W, w) as h:
        rc = lib.slq_stem_launch_in(h, x.data_ptr(), L.IN_F32, None, a.data_ptr(), b.data_ptr(), scales.data_ptr(), 0,
                                    out.data_ptr(), L.OUT_U8, None, None, _stream())
        assert rc == L.SLQ_ERR_INVALID and "16-byte aligned" in lib.slq_last_error().decode()
        torch.cuda.synchronize()
        assert bool((out == 0x5A).all())  # rejected before any launch


def test_engine_wider_than_256_uses_the_simt_stem_and_rejects_fp16_u8_input():
    import imagenet
    import resnet
    import slq_engine
    torch.manual_seed(0)
    net = resnet.resnet18(num_classes=1000).cuda().eval()
    net.input_norm = (imagenet.MEAN, imagenet.STD)
    eng = slq_engine.Engine(net, 1, 64, 288, torch.device("cuda"))
    assert eng.stem is None and eng.stem_kind == "simt"
    for x in (torch.randn(1, 3, 64, 288, device="cuda").half(),
              torch.randint(0, 256, (1, 3, 64, 288), dtype=torch.uint8, device="cuda")):
        with pytest.raises(ValueError):
            eng.calibrate(x)


# ------------------------------------------------------------------------------------------------------------
# calibration helpers
# ------------------------------------------------------------------------------------------------------------
def _big_n():
    """Large enough that absmax_kernel's grid (capped at 8 CTAs per SM) strides twice, with a 3-element tail."""
    return 2 * sm_count() * 8 * 256 * 4 + 3


@pytest.mark.parametrize("qmax", [255, 127])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 1023, "big"])
def test_absmax_scale_is_exact(n, qmax):
    """act_scales[id] == fp32(max|y|) / fp32(qmax) (1.0 for an all-zero tensor), with the maximum anywhere: in the
    vectorised body, in the n % 4 tail that block 0 walks after its grid-stride loop, and negative."""
    n = _big_n() if n == "big" else n
    rng = np.random.default_rng(n + qmax)
    base = (rng.standard_normal(n) * 3).astype(np.float32)
    tail = n - 1  # in the n % 4 tail whenever n % 4 != 0
    patterns = {"random": base, "zeros": np.zeros(n, np.float32)}
    for name, pos, v in (("tail", tail, 50.0), ("tail_negative", tail, -50.0), ("negative", n // 3, -75.0),
                         ("first", 0, 60.0)):
        y = base.copy()
        y[pos] = v
        patterns[name] = y
    for name, y in patterns.items():
        yd = torch.from_numpy(y).cuda()
        scales = torch.full((3,), -2.0, dtype=torch.float32, device="cuda")
        absmax_scale(yd, scales, 1, qmax)
        got = scales.cpu().numpy()
        amax = np.float32(np.abs(y).max())
        want = np.float32(1.0) if amax == 0 else amax / np.float32(qmax)
        assert got[1].view(np.uint32) == want.view(np.uint32), (name, n, qmax, got[1], want)
        assert got[0] == -2.0 and got[2] == -2.0


def _quant_ref(y, scale, signed):
    inv = np.float32(1.0) / np.float32(scale)
    q = np.rint(y.astype(np.float32) * inv)  # fp32 product, then round half to even
    if signed:
        return np.clip(q, -128, 127).astype(np.int8).view(np.uint8)
    return np.clip(q, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("signed", [0, 1], ids=["u8", "s8"])
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 26, 1023, "big"])
def test_quantize_act_is_exact(n, signed):
    """out = clamp(rint(y * fp32(1 / scale))) with round-half-even, saturation at both ends (u8: [0, 255],
    s8: [-128, 127], the range of every s8 producer), in the vectorised body and the n % 4 tail."""
    import slq_oracle as so
    L, lib = _L()
    n = _big_n() if n == "big" else n
    special = np.array([2.5, 3.5, -2.5, -3.5, 0.5, -0.5, 1.5, 254.5, 255.5, 126.5, 127.5, -127.5, -128.5, -200.0,
                        300.0, -0.4, -3.0, 0.0, 127.0, -128.0, 255.0, 1e30, -1e30], np.float32)
    rng = np.random.default_rng(n * 2 + signed)
    inputs = [(1.0, np.resize(special, n)), (1.0, np.resize(special[::-1], n)),
              (0.037, (rng.standard_normal(n) * 4).astype(np.float32))]
    for scale, y in inputs:
        yd = torch.from_numpy(y).cuda()
        sc = torch.tensor([7.0, scale], dtype=torch.float32, device="cuda")
        out = torch.full((n,), 0x77, dtype=torch.uint8, device="cuda")
        L.check(lib.slq_quantize_act(yd.data_ptr(), n, sc.data_ptr(), 1, signed, out.data_ptr(), _stream()))
        torch.cuda.synchronize()
        got = out.cpu().numpy()
        want = _quant_ref(y, scale, signed)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, [(int(i), float(y[i]), int(got[i]), int(want[i])) for i in bad[:8]]
        # the numpy oracle's requantisers use the same contract
        oracle = so.requant_s8(y, scale) if signed else so.requant_u8(y, scale)
        assert np.array_equal(oracle, want)


def test_quantize_act_s8_saturates_to_minus_128():
    """Pins the s8 range: cvt.rni.sat.s8 saturates to -128, not -127 (include/slq.h, slq_oracle.requant_s8)."""
    L, lib = _L()
    y = torch.tensor([-127.4, -127.5, -127.6, -128.0, -128.6, -1000.0, 127.6, 1000.0], device="cuda")
    sc = torch.ones(1, dtype=torch.float32, device="cuda")
    out = torch.zeros(y.numel(), dtype=torch.uint8, device="cuda")
    L.check(lib.slq_quantize_act(y.data_ptr(), y.numel(), sc.data_ptr(), 0, 1, out.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert out.cpu().numpy().view(np.int8).tolist() == [-127, -128, -128, -128, -128, -128, 127, 127]
