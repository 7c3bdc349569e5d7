"""tests/helpers.py -- shared builders for the parity tests (CUDA path vs oracle)."""
import ctypes
import os

import numpy as np
import torch

import slq_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
PKG = os.path.join(ROOT, "semilayer-wise-mixed-precision-quantization_b200")

# the 19 unique quantised conv shapes of ResNet-50 (SURVEY.md Appendix B): Cin, Cout, k, stride, Hin
R50_SHAPES = [
    (64, 64, 1, 1, 56), (64, 64, 3, 1, 56), (64, 256, 1, 1, 56), (256, 64, 1, 1, 56),
    (256, 128, 1, 1, 56), (128, 128, 3, 2, 56), (128, 512, 1, 1, 28), (512, 128, 1, 1, 28),
    (128, 128, 3, 1, 28), (512, 256, 1, 1, 28), (256, 256, 3, 2, 28), (256, 1024, 1, 1, 14),
    (1024, 256, 1, 1, 14), (256, 256, 3, 1, 14), (1024, 512, 1, 1, 14), (512, 512, 3, 2, 14),
    (512, 2048, 1, 1, 7), (2048, 512, 1, 1, 7), (512, 512, 3, 1, 7),
]
# ResNet-18/34 quantised shapes (all 3x3) and the 1x1 stride-2 downsample convs
R18_SHAPES = [
    (64, 64, 3, 1, 56), (64, 128, 3, 2, 56), (128, 128, 3, 1, 28), (128, 256, 3, 2, 28),
    (256, 256, 3, 1, 14), (256, 512, 3, 2, 14), (512, 512, 3, 1, 7),
]
DOWNSAMPLE_SHAPES = [(64, 256, 1, 1, 56), (256, 512, 1, 2, 56), (512, 1024, 1, 2, 28), (1024, 2048, 1, 2, 14),
                     (64, 128, 1, 2, 56)]


def p0_table(arch):
    return np.load(os.path.join(PKG, "data", "p0_bits.npz"))[arch]


def make_weights(cout, cin, k, bits, seed):
    """fp32 OIHW weights whose row oc is fake-quantised to bits[oc] bits (32 = left in fp32),
    produced with the ORACLE quantizer.  Returns (w fp32 [cout,cin,k,k], per-row (bit, codes, z, s))."""
    rng = np.random.default_rng(seed)
    K = cin * k * k
    w = (rng.standard_normal((cout, K)) * np.sqrt(2.0 / (cout * k * k))).astype(np.float32)
    for oc in range(cout):
        if bits[oc] <= 8:
            q, _, _, _, _ = so.quantize_row(w[oc], int(bits[oc]))
            w[oc] = q
    meta = [so.encode_row(w[oc]) for oc in range(cout)]
    return w.reshape(cout, cin, k, k), meta


def expected_gemm_weights(meta, cout, cin, k, w16):
    """numpy restatement of slq_build_gemm_weights (include/slq.h)."""
    K = cin * k * k
    bn_ch = 64 if w16 else (128 if cout > 64 else 64)
    n_tiles = (cout + bn_ch - 1) // bn_ch
    rows = n_tiles * (128 if w16 else bn_ch)
    wg = np.zeros((rows, K), np.uint8)
    for oc in range(cout):
        codes = meta[oc][1].reshape(cin, k, k).transpose(1, 2, 0).reshape(-1)  # (c,r,s) -> (r,s,c)
        if w16:
            base = (oc // 64) * 128 + (oc % 64)
            wg[base] = codes & 255
            wg[base + 64] = codes >> 8
        else:
            wg[oc] = codes
    return wg


def codes_ohwi(meta, cout, cin, k):
    return np.stack([m[1].reshape(cin, k, k).transpose(1, 2, 0) for m in meta]).astype(np.int64)


class ConvCase:
    """One conv layer on the device, built through the C ABI exactly like slq_engine does."""

    def __init__(self, N, H, cin, cout, k, stride, bits, seed=0, impl=None, a_mode=0, device="cuda", packed_b=False,
                 x=None):
        """bits: per output channel, any of 2/4/6/8 (quantised rows) or 32 (an fp32 row: 16-bit codes, two limbs).
        x: the input as a u8 NHWC [N, H, H, cin] device tensor (made on the device; self.x, the host copy the
        numpy oracle reads, is then None); None draws it from `seed` on the host."""
        import slq_engine
        import slq_lib as L
        self.L = L
        lib = L.lib()
        impl = L.IMPL_UMMA if impl is None else impl
        self.N, self.H, self.cin, self.cout, self.k, self.stride = N, H, cin, cout, k, stride
        self.pad = k // 2
        self.w, self.meta = make_weights(cout, cin, k, bits, seed)
        self.w16 = 1 if max(m[0] for m in self.meta) > 8 else 0
        if x is None:
            rng = np.random.default_rng(seed + 1)
            self.x = rng.integers(0, 256, (N, H, H, cin), dtype=np.uint8)
            self.xd = torch.from_numpy(self.x).to(device)
        else:
            assert x.dtype == torch.uint8 and tuple(x.shape) == (N, H, H, cin) and x.is_contiguous()
            self.x, self.xd = None, x
        # per-pixel channel sums of the input (what the producing layer's epilogue accumulates)
        self.rowsum = self.xd.sum(-1, dtype=torch.int32).reshape(-1)
        wd = torch.from_numpy(self.w.reshape(cout, -1)).to(device)
        (bit, z, s, bits_host, _exact), = slq_engine.classify_weights([wd])
        self.bits_dev, self.z_dev, self.s_dev, self.bits_host = bit, z, s, bits_host
        self.packed = slq_engine.encode_weight(wd, bit, z, s, bits_host)
        self.desc = L.ConvDesc(N, H, H, cin, cout, k, k, stride, self.pad, self.w16, impl, a_mode)
        rows = lib.slq_gemm_weight_rows(ctypes.byref(self.desc))
        self.wg = torch.empty((rows, k * k * cin), dtype=torch.uint8, device=device)
        L.check(lib.slq_build_gemm_weights(ctypes.byref(self.desc), self.packed.blob.data_ptr(),
                                           self.packed.offsets.data_ptr(), self.packed.bits.data_ptr(),
                                           self.wg.data_ptr(), L.current_stream()))
        h = ctypes.c_void_p()
        L.check(lib.slq_conv_create(ctypes.byref(self.desc), self.xd.data_ptr(), self.wg.data_ptr(), ctypes.byref(h)))
        self.handle = h
        self.packed_gemm = None
        if packed_b:  # B operand as the packed store, unpacked in shared memory (resident-weight layers)
            self.packed_gemm = slq_engine.build_packed_gemm(self.desc, self.packed, self.bits_host, device)
            if self.packed_gemm is not None:
                pg = self.packed_gemm
                L.check(lib.slq_conv_set_packed_weights(h, pg.blob.data_ptr(), pg.tile_base.data_ptr(),
                                                        pg.seg_bytes.data_ptr(), pg.row_offsets.data_ptr()))
        self.Ho = (H + 2 * self.pad - k) // stride + 1
        self.M = N * self.Ho * self.Ho
        self.device = device

    def close(self):
        if self.handle is not None:
            self.L.lib().slq_conv_destroy(self.handle)
            self.handle = None

    # ---- oracle side ----
    def oracle_acc(self):
        codes = codes_ohwi(self.meta, self.cout, self.cin, self.k)
        if self.w16:
            lo, S, _, _ = so.conv_acc(self.x, codes & 255, self.stride, self.pad)
            hi, _, _, _ = so.conv_acc(self.x, codes >> 8, self.stride, self.pad)
            return lo, hi, S
        acc, S, _, _ = so.conv_acc(self.x, codes, self.stride, self.pad)
        return acc, None, S

    # ---- device side ----
    def _in_rowsum(self, in_rowsum, in_planes):
        """The launch's rowsum fields: in_rowsum is a [planes, plane_stride] int32 device tensor whose first
        in_planes planes (default: all) sum to the input's per-pixel channel sums; None = the one exact plane."""
        rs = self.rowsum.view(1, -1) if in_rowsum is None else in_rowsum
        assert rs.dim() == 2 and rs.dtype == torch.int32 and rs.is_contiguous()
        return rs, rs.shape[0] if in_planes is None else in_planes, rs.shape[1]

    def launch_acc(self, in_rowsum=None, in_planes=None):
        """SLQ_OUT_ACC launch; returns the device tensors (out [M, Cout or 2*Cout] int32, S [M] int32) unsynchronised."""
        L = self.L
        rs, planes, stride = self._in_rowsum(in_rowsum, in_planes)
        ncol = self.cout * (2 if self.w16 else 1)
        out = torch.full((self.M, ncol), -7, dtype=torch.int32, device=self.device)
        S = torch.full((self.M,), -7, dtype=torch.int32, device=self.device)
        e = L.Epilogue(None, None, None, None, 0, 0, -1, None, 0, out.data_ptr(), S.data_ptr(), L.OUT_ACC, 0,
                       rs.data_ptr(), None, planes, stride)
        L.check(L.lib().slq_conv_launch(self.handle, ctypes.byref(e), L.current_stream()))
        return out, S

    def run_acc(self):
        out, S = self.launch_acc()
        torch.cuda.synchronize()
        return out.cpu().numpy(), S.cpu().numpy()

    def launch_epi(self, mode, wscale, zf, bias, scales, in_id, out_id, res=None, res_id=-1, res_signed=0, relu=1,
                   in_rowsum=None, in_planes=None, out=None):
        """One epilogue launch; the vectors and res may be numpy arrays or device tensors.  out: the output
        buffer (default: a fresh one filled with a sentinel).  Returns the device output unsynchronised and
        sets self.out_rowsum (U8 launches: [slq_conv_rowsum_planes, M], filled with -3 before the launch)."""
        L = self.L
        dev = self.device
        t = lambda a: a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        ws, zz, bb, sc = t(wscale), t(zf), t(bias), t(scales)
        rs = t(res) if res is not None else None
        if out is None and mode == L.OUT_F32:
            out = torch.full((self.M, self.cout), float("nan"), dtype=torch.float32, device=dev)
        elif out is None:
            out = torch.full((self.M, self.cout), 77, dtype=torch.uint8, device=dev)
        planes = L.lib().slq_conv_rowsum_planes(self.handle, 1 if res is not None else 0)
        self.out_rowsum = (torch.full((max(planes, 1), self.M), -3, dtype=torch.int32, device=dev)
                           if mode == L.OUT_U8 else None)
        irs, in_planes, in_stride = self._in_rowsum(in_rowsum, in_planes)
        e = L.Epilogue(ws.data_ptr(), zz.data_ptr(), bb.data_ptr(), sc.data_ptr(), in_id, out_id, res_id,
                       L.ptr(rs), res_signed, out.data_ptr(), None, mode, relu, irs.data_ptr(),
                       L.ptr(self.out_rowsum), in_planes, in_stride)
        L.check(L.lib().slq_conv_launch(self.handle, ctypes.byref(e), L.current_stream()))
        return out

    def run_epi(self, mode, wscale, zf, bias, scales, in_id, out_id, res=None, res_id=-1, res_signed=0, relu=1):
        out = self.launch_epi(mode, wscale, zf, bias, scales, in_id, out_id, res, res_id, res_signed, relu)
        torch.cuda.synchronize()
        got = out.cpu().numpy()
        if self.out_rowsum is not None and self.desc.impl == self.L.IMPL_UMMA:
            # the side tensor the next layer's epilogue gathers its window sums from
            # (one plane per n-tile of the launch; their sum is the channel sum of the pixel)
            want = got.astype(np.int64).sum(1)
            assert np.array_equal(self.out_rowsum.cpu().numpy().astype(np.int64).sum(0), want), "out_rowsum"
        return got


def oracle_epilogue_case(case, wscale, zf, bias, scales, in_id, out_id, res, res_id, res_signed, relu, mode):
    import slq_lib as L
    lo, hi, S = case.oracle_acc()
    s_res = scales[res_id] if res is not None else None
    if mode == L.OUT_F32:
        return so.epilogue(lo, S, zf, wscale, bias, scales[in_id], res, s_res, relu=bool(relu), acc_hi=hi,
                           res_signed=bool(res_signed))
    return so.epilogue_q(lo, S, zf, wscale, bias, scales[in_id], scales[out_id], res, s_res, acc_hi=hi,
                         res_signed=bool(res_signed), signed_out=(mode == L.OUT_S8))


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def build_p0_model(arch, device, seed=0):
    """Seeded random-init model with the P0 8/4-bit assignment applied through the product's own
    quantizer (functions.quantize_rows, one launch per conv)."""
    import functions
    import resnet
    torch.manual_seed(seed)
    net = getattr(resnet, arch)(num_classes=1000).to(device).eval()
    table = p0_table(arch)
    cpb = 3 if arch == "resnet50" else 2
    blocks = [b for s in (net.layer1, net.layer2, net.layer3, net.layer4) for b in s]
    for lnum in np.unique(table[:, 0]):
        sel = table[table[:, 0] == lnum]
        conv = getattr(blocks[(lnum - 1) // cpb], "conv%d" % ((lnum - 1) % cpb + 1))
        functions.quantize_rows(conv.weight.data, sel[:, 1], sel[:, 2], write_back=True, want_codes=False,
                                div_mode=0)
    return net
