"""The tcgen05 conv kernel (conv_umma_kernel, through the C ABI) bit for bit against the exact torch reference of
tests/conv_reference.py, at the batch bench.py runs (256) and at batch sizes picked to hit the edges of the tile
walk.  Accumulators, window sums, u8 / s8 / fp32 outputs and the rowsum side tensor must all be identical.

Inputs are made on the device from seeded generators: uniform u8 images, post-ReLU-like images (about half
zeros), one all-zero image and one all-255 image (the largest window sums).  Weight rows are drawn from
{2, 4, 6, 8} bits (the search's progressive chain); one layer is all 2-bit, the downsample convs keep fp32 rows
(16-bit codes, two limbs), and resident-weight layers run both from the u8 GEMM-ready matrix and from the packed
store (slq_conv_set_packed_weights: 2- and 4-bit rows as nibbles, unpacked in shared memory).

Modes per shape are the launches the engine issues for it: u8 without residual, u8 with a u8 residual
(Bottleneck conv3, BasicBlock conv2), u8 with an s8 residual (the unfused stage-4 tail, BasicBlock downsample
blocks), s8 two-limb downsample, fp32 with and without residual (the calibration pass), and the raw accumulators.

Tile walk (conv_umma.cu: plan_grid, TileWalk).  With m_tiles = ceil(N*Ho*Wo / 128):
  resident weights : per_n = min(max(SMs // n_tiles, 1), m_tiles), grid = per_n * n_tiles; CTA b keeps n-tile
                     b % n_tiles and walks m-tiles b // n_tiles + i * per_n
  streamed weights : grid = min(m_tiles * n_tiles, SMs); CTA b walks tiles b + i * grid (m-major)
Neither walk launches a CTA without a tile; a CTA with a single tile leaves its second epilogue team (and the
second MMA warp) with none.  The accumulators form a ring of 3 (2 for 256-channel tiles) and the per-tile barrier
sets a ring of 6, so per-CTA counts that cross 3 and 6 wrap both.  test_tile_walk_edges picks N from the SM count
of the device; at 148 SMs it runs:

  layer         shape (Cin-Cout k s H)    tiling (launch)                       edge      N     m_tiles grid tiles/CTA excess
  resident64    64-64 3x3 s1 @56 u8       resident B, 64-ch, 1 n-tile, packed   under        6   147    147   1         0
                                                                                one_over     7   172    148   1-2      24
                                                                                cross3      19   466    148   3-4     318
                                                                                cross6      37   907    148   6-7     759
                                                                                ragged      13   319    148   2-3     171
  resident128   128-512 1x1 s1 @28 +u8res resident B, 128-ch, 4 n-tiles, packed under        5    31    124   1         0
                                                                                one_over     7    43    148   1-2      24
                                                                                cross3      19   117    148   3-4     320
                                                                                cross6      37   227    148   6-7     760
                                                                                ragged      13    80    148   2-3     172
  streamed      128-128 3x3 s1 @28 u8     streamed B, 128-ch, shared staging    under       24   147    147   1         0
                                                                                one_over    25   154    148   1-2       6
                                                                                cross3      73   448    148   3-4     300
                                                                                cross6     145   889    148   6-7     741
                                                                                ragged      49   301    148   2-3     153
  streamed_res  256-256 3x3 s1 @14 +u8res streamed B, 128-ch, 2 n-tiles, shared under       47    72    144   1         0
                                                                                one_over    49    76    148   1-2       4
                                                                                cross3     145   223    148   3-4     298
                                                                                cross6     290   445    148   6-7     742
                                                                                ragged      97   149    148   2-3     150
  wide3x3       256-256 3x3 s1 @14 u8     wide (256-ch), 1 n-tile, gathered S    under       96   147    147   1         0
                                                                                one_over    97   149    148   1-2       1
                                                                                cross3     290   445    148   3-4     297
                                                                                cross6     580   889    148   6-7     741
                                                                                ragged     195   299    148   2-3     151
  wide1x1       2048-512 1x1 s1 @7 u8     wide (256-ch), 2 n-tiles, gathered S  under      190    73    146   1         0
                                                                                one_over   194    75    148   1-2       2
                                                                                cross3     580   223    148   3-4     298
                                                                                cross6    1160   445    148   6-7     742
                                                                                ragged     387   149    148   2-3     150
(excess = m_tiles * n_tiles - grid: the tiles past the first wave.  `one_over` takes the N with the least excess:
exactly one tile where m_tiles * n_tiles can equal grid + 1.  `ragged`: N odd, M % 128 != 0, up to 3 tiles a CTA.)
"""
import ctypes

import numpy as np
import pytest
import torch

import conv_reference as cr
from helpers import ConvCase, DOWNSAMPLE_SHAPES, R18_SHAPES, R50_SHAPES, codes_ohwi

pytestmark = pytest.mark.gpu

N_PROD = 256  # bench.py's batch


# ---------------------------------------------------------------------------------------------------------------
# inputs and parameters
# ---------------------------------------------------------------------------------------------------------------
def make_x(N, H, C, seed):
    """u8 NHWC on the device: image 0 all zeros, image 1 all 255 (when N > 2), then uniform and post-ReLU-like
    (about half zeros) images in turn."""
    g = torch.Generator("cuda").manual_seed(seed)
    x = torch.randint(0, 256, (N, H, H, C), generator=g, device="cuda", dtype=torch.uint8)
    relu_like = torch.rand((N, H, H, C), generator=g, device="cuda") < 0.5
    relu_like[0::2] = False
    x.masked_fill_(relu_like, 0)
    if N > 2:
        x[0] = 0
        x[1] = 255
    return x


def make_bits(cout, seed, kind):
    if kind == "fp32":
        return np.full(cout, 32, np.int32)
    if kind == "all2":
        return np.full(cout, 2, np.int32)
    return np.random.default_rng(seed).choice([2, 4, 6, 8], cout).astype(np.int32)


def sm_count():
    import slq_lib as L
    sms = ctypes.c_int32(0)
    L.check(L.lib().slq_device_info(ctypes.byref(sms), None, None))
    return sms.value


class Ref:
    """Exact accumulators of one ConvCase and the epilogue parameters of its launches.  The output scales are fitted
    to the data (~0.5 % of the outputs saturate), so the u8 / s8 ranges are really used."""

    def __init__(self, case, seed):
        self.case = case
        c = case
        self.relu = not c.w16  # the two-limb downsample convs produce signed tensors (s8; fp32 without ReLU)
        codes = torch.from_numpy(codes_ohwi(c.meta, c.cout, c.cin, c.k)).cuda()
        self.lo, self.hi, self.S = cr.conv_acc(c.xd, codes, c.stride, c.pad, bool(c.w16))
        rng = np.random.default_rng(seed)
        self.zf = np.array([m[2] for m in c.meta], np.float32)
        s = np.array([m[3] for m in c.meta], np.float32)
        self.wscale = (s * (0.5 + rng.random(c.cout))).astype(np.float32)
        self.bias = (rng.standard_normal(c.cout) * 0.2).astype(np.float32)
        s_in = np.float32(0.02)
        y = cr.epilogue(self.lo, self.S, self.zf, self.wscale, self.bias, s_in, "f32", hi=self.hi, relu=False)
        flat = y.view(-1)
        flat = flat[:: -(-flat.numel() // (1 << 23))]
        s_u8 = float(torch.quantile(flat[flat > 0], 0.995)) / 255.0
        s_s8 = float(torch.quantile(flat.abs().float(), 0.995)) / 127.0
        # act_scales: in, u8 out, s8 out, u8 residual, s8 residual
        self.scales = np.array([s_in, s_u8, s_s8, s_u8 * 0.25, s_u8 * 0.5], np.float32)
        g = torch.Generator("cuda").manual_seed(seed)
        self.res = torch.randint(0, 256, (c.M, c.cout), generator=g, device="cuda", dtype=torch.uint8)
        self.vec = [torch.from_numpy(v).cuda() for v in (self.wscale, self.zf, self.bias, self.scales)]

    # mode: "acc", "u8", "s8", "f32", with "+u8res" / "+s8res"
    def want(self, mode):
        out, _, res = mode.partition("+")
        res_kind = res[:2] if res else None
        o = {"u8": 1, "s8": 2}.get(out)
        r = {"u8": 3, "s8": 4}.get(res_kind)
        sc = self.scales
        return cr.epilogue(self.lo, self.S, self.zf, self.wscale, self.bias, sc[0], out,
                           s_out=sc[o] if o else None, hi=self.hi, res=self.res if res_kind else None,
                           s_res=sc[r] if r else None, res_signed=res_kind == "s8", relu=self.relu)

    def launch(self, mode, **kw):
        import slq_lib as L
        out, _, res = mode.partition("+")
        res_kind = res[:2] if res else None
        m = {"u8": L.OUT_U8, "s8": L.OUT_S8, "f32": L.OUT_F32}[out]
        ws, zf, b, sc = self.vec
        return self.case.launch_epi(m, ws, zf, b, sc, 0, {"u8": 1, "s8": 2}.get(out, 1),
                                    res=self.res if res_kind else None, res_id={"u8": 3, "s8": 4}.get(res_kind, -1),
                                    res_signed=1 if res_kind == "s8" else 0, relu=int(self.relu), **kw)


def first_diff(got, want):
    bad = (got.view(torch.int32) != want.view(torch.int32)) if got.dtype == torch.float32 else (got != want)
    n = int(bad.sum())
    idx = torch.nonzero(bad)[0].tolist() if n else None
    return "%d elements differ, first at (m, oc) = %s: got %s want %s" % (
        n, idx, got[tuple(idx)].item() if n else None, want[tuple(idx)].item() if n else None)


def assert_same(got, want, what):
    same = torch.equal(got.view(torch.int32), want.view(torch.int32)) if got.dtype == torch.float32 \
        else torch.equal(got, want)
    assert same, "%s: %s" % (what, first_diff(got, want))


def check_acc(ref, **kw):
    c = ref.case
    out, S = c.launch_acc(**kw)
    assert_same(S.view(-1, 1), ref.S.view(-1, 1), "window sums")
    assert_same(out[:, :c.cout], ref.lo, "accumulators")
    if c.w16:
        assert_same(out[:, c.cout:], ref.hi, "high-limb accumulators")


def check_out_rowsum(case, got):
    """Plane p of out_rowsum = the channel sum of n-tile p's output bytes (epilogue.cuh, EpiDev.out_rowsum)."""
    rs = case.out_rowsum
    P = rs.shape[0]
    want = got.view(case.M, P, case.cout // P).sum(-1, dtype=torch.int32).t()
    assert_same(rs, want, "out_rowsum (%d planes)" % P)


def check_mode(ref, mode, want, **kw):
    got = ref.launch(mode, **kw)
    assert_same(got, want, mode)
    out = mode.split("+")[0]
    if out in ("u8", "s8"):
        lo, hi = (0x80, 0x7F) if out == "s8" else (0, 255)
        assert bool((want == lo).any()) and bool((want == hi).any()), "%s: the range does not saturate" % mode
        assert int(torch.unique(want).numel()) > 200, "%s: too few distinct bytes" % mode
    if out == "u8":
        check_out_rowsum(ref.case, got)
    return got


# ---------------------------------------------------------------------------------------------------------------
# every shape at N = 256 in each of its engine modes
# ---------------------------------------------------------------------------------------------------------------
_PLAIN = ["u8", "f32"]
_EXPAND = ["u8+u8res", "u8+s8res", "f32+u8res", "f32+s8res"]
_BASIC = _PLAIN + _EXPAND
_R50_EXPAND = {(64, 256, 1, 1, 56), (128, 512, 1, 1, 28), (256, 1024, 1, 1, 14), (512, 2048, 1, 1, 7)}
# BasicBlock 3x3 stride-1 shapes are conv1 and conv2 (identity or downsample residual); the strided ones conv1 only
_R18_MODES = {s: (_BASIC if s[3] == 1 else _PLAIN) for s in R18_SHAPES}


def _shape_cases():
    cases = {}
    for s in R50_SHAPES:
        cases[s] = ("r50", list(_EXPAND if s in _R50_EXPAND else _PLAIN))
    for s in R18_SHAPES:
        if s in cases:
            tag, modes = cases[s]
            cases[s] = ("r50-r18", modes + [m for m in _R18_MODES[s] if m not in modes])
        else:
            cases[s] = ("r18", list(_R18_MODES[s]))
    out = [(tag, s, "mix", modes) for s, (tag, modes) in cases.items()]
    out.append(("r50", (64, 256, 1, 1, 56), "all2", list(_EXPAND)))
    out += [("ds", s, "fp32", ["s8", "f32"]) for s in DOWNSAMPLE_SHAPES]
    return out


SHAPE_CASES = _shape_cases()


def _case_id(c):
    tag, (cin, cout, k, s, h), bits, modes = c
    return "%s_c%d-%d_k%d_s%d_h%d_%s_%s" % (tag, cin, cout, k, s, h, bits, ",".join(["acc"] + modes))


@pytest.mark.parametrize("cfg", SHAPE_CASES, ids=_case_id)
def test_shape_modes_at_batch_256(cfg):
    import slq_lib as L
    tag, (cin, cout, k, stride, H), bits_kind, modes = cfg
    seed = cin * 7 + cout + k + stride + H
    x = make_x(N_PROD, H, cin, seed)
    case = ConvCase(N_PROD, H, cin, cout, k, stride, make_bits(cout, seed, bits_kind), seed=seed, x=x,
                    packed_b=bits_kind != "fp32")
    try:
        assert case.w16 == (1 if bits_kind == "fp32" else 0)
        ref = Ref(case, seed)
        check_acc(ref)
        lib = L.lib()
        for mode in modes:
            want = ref.want(mode)
            check_mode(ref, mode, want)
            if case.packed_gemm is not None:  # the same launch from the u8 GEMM-ready matrix
                L.check(lib.slq_conv_set_packed_weights(case.handle, None, None, None, None))
                check_mode(ref, mode, want)
                pg = case.packed_gemm
                L.check(lib.slq_conv_set_packed_weights(case.handle, pg.blob.data_ptr(), pg.tile_base.data_ptr(),
                                                        pg.seg_bytes.data_ptr(), pg.row_offsets.data_ptr()))
            del want
    finally:
        case.close()


# ---------------------------------------------------------------------------------------------------------------
# the rowsum contract of the 256-channel layers
# ---------------------------------------------------------------------------------------------------------------
def split_planes(rowsum, P, n_buf, stride, seed):
    """[n_buf, stride] int32 buffer whose first P planes split every pixel's sum at random cut points; the
    trailing planes and the stride padding hold a sentinel."""
    npix = rowsum.numel()
    buf = torch.full((n_buf, stride), 0x00ABCDEF, dtype=torch.int32, device="cuda")
    g = torch.Generator("cuda").manual_seed(seed)
    tot = rowsum.to(torch.int64)
    cuts = (torch.rand((P - 1, npix), generator=g, device="cuda", dtype=torch.float64) * (tot + 1).double()).floor()
    cuts = torch.sort(cuts.to(torch.int64), dim=0).values
    edges = torch.cat([torch.zeros((1, npix), dtype=torch.int64, device="cuda"), cuts, tot.view(1, -1)])
    buf[:P, :npix] = (edges[1:] - edges[:-1]).to(torch.int32)
    assert torch.equal(buf[:P, :npix].sum(0, dtype=torch.int32), rowsum)
    return buf


# the layers that run 256-channel tiles (Cout % 256 == 0, weights streamed) and the launches without residual
# gather S from the rowsum planes; the test asserts that through slq_conv_needs_rowsum
WIDE_SHAPES = [(256, 256, 3, 2, 28), (1024, 256, 1, 1, 14), (256, 256, 3, 1, 14), (1024, 512, 1, 1, 14),
               (512, 512, 3, 2, 14), (2048, 512, 1, 1, 7), (512, 512, 3, 1, 7), (128, 256, 3, 2, 28),
               (256, 512, 3, 2, 14),
               (1024, 2048, 1, 2, 14)]  # the stage-4 downsample with quantised rows: the strided 1x1 gather


@pytest.mark.parametrize("shape", WIDE_SHAPES, ids=lambda s: "c%d-%d_k%d_s%d_h%d" % s)
def test_wide_layer_rowsum_planes(shape):
    import slq_lib as L
    cin, cout, k, stride, H = shape
    seed = cin + cout * 3 + H
    x = make_x(N_PROD, H, cin, seed)
    case = ConvCase(N_PROD, H, cin, cout, k, stride, make_bits(cout, seed, "mix"), seed=seed, x=x)
    try:
        lib = L.lib()
        assert lib.slq_conv_needs_rowsum(case.handle, 0) == 1, "not a 256-channel layer"
        assert lib.slq_conv_rowsum_planes(case.handle, 0) == cout // 256
        ref = Ref(case, seed)
        npix = N_PROD * H * H
        n_buf = max(cin // 64, 1)  # what the engine allocates for a rowsum tensor
        stride_pl = npix + 1000  # larger than N*H*W
        u8_want = ref.want("u8")
        for P in sorted({1, cin // 128, cin // 64}):
            buf = split_planes(case.rowsum, P, n_buf, stride_pl, seed + P)
            check_acc(ref, in_rowsum=buf, in_planes=P)
            check_mode(ref, "u8", u8_want, in_rowsum=buf, in_planes=P)
            check_mode(ref, "f32", ref.want("f32"), in_rowsum=buf, in_planes=P)
        # sensitivity: one plane short gives a wrong S, and the comparison sees it
        P = cin // 64
        buf = split_planes(case.rowsum, P, n_buf, stride_pl, seed)
        _, S = case.launch_acc(in_rowsum=buf, in_planes=P - 1)
        assert not torch.equal(S, ref.S), "a missing rowsum plane went unnoticed (window sums)"
        got = ref.launch("u8", in_rowsum=buf, in_planes=P - 1)
        assert not torch.equal(got, u8_want), "a missing rowsum plane went unnoticed (u8 output)"
    finally:
        case.close()


# ---------------------------------------------------------------------------------------------------------------
# tile-walk edges
# ---------------------------------------------------------------------------------------------------------------
WALK_LAYERS = {  # name: (shape, launch mode, expected tiling)
    "resident64": ((64, 64, 3, 1, 56), "u8", "resident"),
    "resident128": ((128, 512, 1, 1, 28), "u8+u8res", "resident"),
    "streamed": ((128, 128, 3, 1, 28), "u8", "streamed"),
    "streamed_res": ((256, 256, 3, 1, 14), "u8+u8res", "streamed"),
    "wide3x3": ((256, 256, 3, 1, 14), "u8", "wide"),
    "wide1x1": ((2048, 512, 1, 1, 7), "u8", "wide"),
}


def launch_tiling(shape, kind):
    """(n_tiles, resident) of a launch: 64-channel tiles up to Cout = 64, 128-channel above, 256 when wide."""
    cin, cout, k, stride, H = shape
    if kind == "wide":
        return cout // 256, False
    return (cout + (127 if cout > 64 else 63)) // (128 if cout > 64 else 64), kind == "resident"


def walk(N, shape, kind, sms):
    """plan_grid + TileWalk: (m_tiles, grid, per-CTA tile counts)."""
    cin, cout, k, stride, H = shape
    Ho = (H + 2 * (k // 2) - k) // stride + 1
    M = N * Ho * Ho
    m_tiles = -(-M // 128)
    n_tiles, resident = launch_tiling(shape, kind)
    if resident:
        per_n = min(max(sms // n_tiles, 1), m_tiles)
        grid = per_n * n_tiles
        counts = [-(-(m_tiles - b // n_tiles) // per_n) for b in range(grid)]
    else:
        total = m_tiles * n_tiles
        grid = min(total, sms)
        counts = [-(-(total - b) // grid) for b in range(grid)]
    return M, m_tiles, grid, counts


EDGES = {  # predicate on (N, M, m_tiles, grid, per-CTA counts, n_tiles, SMs)
    "under": lambda N, M, mt, g, c, nt, sms: mt * nt < sms,
    "one_over": lambda N, M, mt, g, c, nt, sms: mt * nt > g,
    "cross3": lambda N, M, mt, g, c, nt, sms: set(c) == {3, 4},
    "cross6": lambda N, M, mt, g, c, nt, sms: set(c) == {6, 7},
    "ragged": lambda N, M, mt, g, c, nt, sms: N % 2 == 1 and M % 128 != 0 and max(c) >= 3,
}


def pick_n(shape, kind, edge, sms):
    """The N the edge is tested at: the largest N <= 2048 with fewer tiles than SMs for `under`; for `one_over` the
    N whose tiles exceed the grid by the least (one tile where m_tiles * n_tiles can be grid + 1); otherwise the
    smallest N with the property."""
    n_tiles, _ = launch_tiling(shape, kind)
    walks = {N: walk(N, shape, kind, sms) for N in range(1, 2049)}
    hits = [N for N, w in walks.items() if EDGES[edge](N, *w, n_tiles, sms)]
    assert hits, "no batch size reaches edge %s of %s" % (edge, shape)
    if edge == "one_over":
        return min(hits, key=lambda N: (walks[N][1] * n_tiles - walks[N][2], N))
    return hits[-1] if edge == "under" else hits[0]


def walk_table(sms=148):
    rows = []
    for name, (shape, mode, kind) in WALK_LAYERS.items():
        for edge in EDGES:
            N = pick_n(shape, kind, edge, sms)
            M, mt, g, c = walk(N, shape, kind, sms)
            rows.append((name, edge, N, mt, g, min(c), max(c), M % 128, mt * launch_tiling(shape, kind)[0] - g))
    return rows


@pytest.mark.parametrize("edge", list(EDGES))
@pytest.mark.parametrize("layer", list(WALK_LAYERS))
def test_tile_walk_edges(layer, edge):
    import slq_engine
    import slq_lib as L
    shape, mode, kind = WALK_LAYERS[layer]
    cin, cout, k, stride, H = shape
    N = pick_n(shape, kind, edge, sm_count())
    seed = 1000 + N + cin
    x = make_x(N, H, cin, seed)
    case = ConvCase(N, H, cin, cout, k, stride, make_bits(cout, seed, "mix"), seed=seed, x=x,
                    packed_b=kind == "resident")
    try:
        lib = L.lib()
        has_res = 1 if "res" in mode else 0
        bn_cols, n_tiles, _, _, resident = slq_engine.conv_tiling(case.desc)
        assert resident == (kind == "resident")
        assert lib.slq_conv_needs_rowsum(case.handle, has_res) == (kind == "wide")
        assert lib.slq_conv_rowsum_planes(case.handle, has_res) == launch_tiling(shape, kind)[0]
        if kind != "wide":
            assert n_tiles == launch_tiling(shape, kind)[0]
        if kind == "resident":
            assert case.packed_gemm is not None
        ref = Ref(case, seed)
        check_acc(ref)
        got = ref.launch(mode)
        assert_same(got, ref.want(mode), mode)
        check_out_rowsum(case, got)
    finally:
        case.close()


# ---------------------------------------------------------------------------------------------------------------
# one handle, several buffers: the output / residual maps are re-encoded when the pointers change
# ---------------------------------------------------------------------------------------------------------------
def test_handle_reuse_and_repeatability():
    cin, cout, k, stride, H = 128, 512, 1, 1, 28
    N = 64
    seed = 77
    case = ConvCase(N, H, cin, cout, k, stride, make_bits(cout, seed, "mix"), seed=seed, x=make_x(N, H, cin, seed))
    try:
        ref = Ref(case, seed)
        want_u8 = ref.want("u8+u8res")
        want_f32 = ref.want("f32+u8res")
        A = torch.full((case.M, cout), 11, dtype=torch.uint8, device="cuda")
        B = torch.full((case.M, cout), 13, dtype=torch.uint8, device="cuda")
        F32 = torch.full((case.M, cout), float("nan"), dtype=torch.float32, device="cuda")
        assert_same(ref.launch("u8+u8res", out=A), want_u8, "u8 into A")
        assert_same(ref.launch("u8+u8res", out=B), want_u8, "u8 into B")
        assert_same(ref.launch("f32+u8res", out=F32), want_f32, "f32")
        A.fill_(11)
        got = ref.launch("u8+u8res", out=A)
        assert_same(got, want_u8, "u8 into A again")
        rs1 = case.out_rowsum.clone()
        # a second residual buffer with the same bytes, then the first again
        res0 = ref.res
        ref.res = res0.clone()
        B.fill_(13)
        assert_same(ref.launch("u8+u8res", out=B), want_u8, "u8, second residual buffer")
        ref.res = res0
        # repeatability: the same launch twice, identical bytes and side tensor
        A.fill_(11)
        again = ref.launch("u8+u8res", out=A)
        assert torch.equal(again, want_u8) and torch.equal(case.out_rowsum, rs1)
    finally:
        case.close()
