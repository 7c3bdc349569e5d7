"""slq_engine.py -- host side of the B200 forward: turns a ResNet module tree (resnet.py) into a
static sequence of kernel launches over the C ABI (slq_lib) and runs it.

Data layout in HBM (DESIGN.md section 3):
  * activations: u8 NHWC per tensor, one static fp32 scale per tensor in ``act_scales`` (device
    array); a downsample branch that runs as its own launch (not post-ReLU) is s8 -- in the Bottleneck
    stages whose weights fit, it is fused into the block's conv3 launch and never exists in HBM;
  * weights: per conv a PackedLayer (bit/z/s32 per output channel + packed 2/4/8/16-bit codes) and
    the GEMM-ready u8 matrix the tcgen05 kernel streams with TMA;
  * everything is allocated once per (batch, H, W); a forward is launches only (CUDA-graph safe).

torch is plumbing here (allocation, streams); no torch op touches activations on the hot path.
"""
import ctypes
import os

import numpy as np
import torch

import slq_lib as L


def engine_batch(net, n):
    for (N, _h, _w, _d), _eng in getattr(net, "_slq_engines", {}).items():
        if N >= n:
            return N
    return n


def _align(v, a):
    return (v + a - 1) // a * a


class PackedLayer:
    """Packed store of one conv weight [Cout, K]: the mixed-precision model format (SURVEY N4).
    real weight of element e of channel oc = (code + z[oc]) * s[oc]."""

    def __init__(self, bits, z, s, offsets, blob, K):
        self.bits, self.z, self.s, self.offsets, self.blob, self.K = bits, z, s, offsets, blob, K

    @property
    def nbytes(self):
        return int(self.blob.numel())


def packed_offsets(bits_host, K):
    """Row start offsets (16-byte aligned) and blob size for rows with the given bit-widths."""
    lib = L.lib()
    sizes = np.array([_align(lib.slq_packed_row_bytes(K, int(b)), 16) for b in bits_host], np.int64)
    offs = np.zeros(len(sizes), np.int64)
    if len(sizes) > 1:
        offs[1:] = np.cumsum(sizes)[:-1]
    return offs, int(sizes.sum())


def classify_weights(weights, stream=None):
    """slq_classify_rows over a list of fp32 [Cout, K] device tensors, one host sync in total.
    Returns per tensor (bits_dev, z_dev, s_dev, bits_host, all_rows_exact)."""
    lib = L.lib()
    stream = L.current_stream() if stream is None else stream
    metas = []
    for w in weights:
        rows, K = w.shape[0], w[0].numel()
        meta = torch.empty((2, rows), dtype=torch.int32, device=w.device)  # bit | exact
        z = torch.empty(rows, dtype=torch.int32, device=w.device)
        s = torch.empty(rows, dtype=torch.float32, device=w.device)
        L.check(lib.slq_classify_rows(w.data_ptr(), rows, K, meta[0].data_ptr(), z.data_ptr(), s.data_ptr(),
                                      meta[1].data_ptr(), stream))
        metas.append((meta, z, s))
    all_meta = torch.cat([m[0] for m in metas], dim=1).cpu().numpy()  # the one sync
    out, pos = [], 0
    for (meta, z, s) in metas:
        n = meta.shape[1]
        out.append((meta[0], z, s, all_meta[0, pos:pos + n], bool(all_meta[1, pos:pos + n].all())))
        pos += n
    return out


class PackedGemm:
    """GEMM-ready weights of one conv in PACKED form (include/slq.h, slq_conv_set_packed_weights): what the
    tcgen05 kernel of a resident-weight layer fetches and unpacks in shared memory."""

    def __init__(self, blob, tile_base, seg_bytes, row_offsets):
        self.blob, self.tile_base, self.seg_bytes, self.row_offsets = blob, tile_base, seg_bytes, row_offsets
        self.used_bytes = 0

    @property
    def nbytes(self):
        return self.used_bytes


def conv_tiling(desc):
    lib = L.lib()
    v = [ctypes.c_int32(0) for _ in range(5)]
    L.check(lib.slq_conv_tiling(ctypes.byref(desc), *[ctypes.addressof(x) for x in v]))
    return tuple(int(x.value) for x in v)  # bn_cols, n_tiles, k_block, num_kb, resident


def alloc_packed_gemm(desc, device):
    """Persistent buffers for the packed operand of one layer (worst case: every row 8-bit), or None when the
    kernel does not keep this layer's weights resident.  Their ADDRESSES never change -- a re-pack rewrites the
    contents in place -- so conv handles and captured CUDA graphs stay valid."""
    bn_cols, n_tiles, k_block, num_kb, resident = conv_tiling(desc)
    if not resident:
        return None
    blob = torch.zeros(bn_cols * n_tiles * k_block * num_kb, dtype=torch.uint8, device=device)
    return PackedGemm(blob, torch.zeros(n_tiles, dtype=torch.int64, device=device),
                      torch.zeros(n_tiles, dtype=torch.int32, device=device),
                      torch.zeros((n_tiles, bn_cols + 1), dtype=torch.int16, device=device))


def build_packed_gemm(desc, packed, bits_host, device, stream=None, into=None):
    """Layout tables (numpy, from the per-channel bit-widths) + slq_build_packed_gemm_weights, written into the
    persistent buffers ``into`` (or fresh ones).  Returns None when the kernel does not keep this layer's weights
    resident (they are then streamed as u8 tiles) or the layer still has never-quantised rows."""
    lib = L.lib()
    bn_cols, n_tiles, k_block, num_kb, resident = conv_tiling(desc)
    if not resident or int(bits_host.max()) > 8:
        return None
    stream = L.current_stream() if stream is None else stream
    pg = into if into is not None else alloc_packed_gemm(desc, device)
    rows = bn_cols * n_tiles
    bits = np.full(rows, 4, np.int64)
    bits[:len(bits_host)] = bits_host
    seg = np.where(bits <= 4, k_block // 2, k_block).reshape(n_tiles, bn_cols)
    row_off = np.zeros((n_tiles, bn_cols + 1), np.int64)
    row_off[:, 1:] = np.cumsum(seg, axis=1)
    seg_bytes = row_off[:, -1].astype(np.int32)
    tile_base = np.zeros(n_tiles, np.int64)
    tile_base[1:] = np.cumsum(num_kb * seg_bytes.astype(np.int64))[:-1]
    pg.used_bytes = int(num_kb * seg_bytes.astype(np.int64).sum())
    assert row_off.max() < 65536 and pg.used_bytes <= pg.blob.numel()
    pg.tile_base.copy_(torch.from_numpy(tile_base), non_blocking=False)
    pg.seg_bytes.copy_(torch.from_numpy(seg_bytes), non_blocking=False)
    pg.row_offsets.copy_(torch.from_numpy(row_off.astype(np.uint16).view(np.int16)), non_blocking=False)
    L.check(lib.slq_build_packed_gemm_weights(ctypes.byref(desc), packed.blob.data_ptr(), packed.offsets.data_ptr(),
                                              packed.bits.data_ptr(), pg.tile_base.data_ptr(), pg.seg_bytes.data_ptr(),
                                              pg.row_offsets.data_ptr(), pg.blob.data_ptr(), stream))
    return pg


def encode_weight(w, bit, z, s, bits_host, stream=None):
    lib = L.lib()
    stream = L.current_stream() if stream is None else stream
    rows, K = w.shape[0], w[0].numel()
    offs, total = packed_offsets(bits_host, K)
    offsets = torch.from_numpy(offs).to(w.device)
    blob = torch.empty(max(total, 16), dtype=torch.uint8, device=w.device)
    L.check(lib.slq_encode_rows(w.data_ptr(), rows, K, bit.data_ptr(), z.data_ptr(), s.data_ptr(),
                                blob.data_ptr(), offsets.data_ptr(), stream))
    return PackedLayer(bit, z, s, offsets, blob, K)


class _ConvOp:
    pass


class _BlockTail:
    """conv3 + downsample conv of one Bottleneck (resnet.py:107-114) that can run as ONE launch
    (include/slq.h section 2b) while conv3 is quantised (<= 8-bit codes) and the downsample conv is not."""

    def __init__(self, dop, op3):
        self.dop, self.op3 = dop, op3
        self.handle, self.unsupported, self.fused, self.epi = None, False, False, {}


class Engine:
    def __init__(self, net, N, H, W, device, impl=L.IMPL_UMMA, a_mode=L.A_AUTO, stem="umma", packed_b=True,
                 fuse_tail=True):
        if device.type != "cuda":
            raise RuntimeError("slq Engine needs a CUDA device")
        self.lib = L.lib()
        self.net, self.N, self.H, self.W, self.device = net, N, H, W, device
        self.impl, self.a_mode = impl, a_mode
        self.packed_b = packed_b  # resident-weight layers fetch PACKED codes and unpack them in shared memory
        self.fuse_tail = fuse_tail  # conv3 + downsample conv of a stage's first block as one launch
        self.stem_kind = stem  # "umma": tcgen05 fp16 stem; "simt": exact-fp32 CUDA-core stem
        self.stem = None
        self.epoch = -1
        self.kernel_launches = 0
        self._graphs, self._seen = {}, set()  # CUDA graphs of the forward, one per input buffer (forward())
        self.use_graphs = os.environ.get("SLQ_NO_GRAPHS") is None
        with torch.cuda.device(device):
            self._plan()

    @classmethod
    def for_module(cls, net, x, **kw):
        """Engine for ANY module tree shaped like the reference's ResNet (resnet.py:121-202), e.g. the
        reference's own class patched per INTEGRATION.md B.2: cached on the module, layers whose
        tensors were written are re-packed on every call; calibrated on first use."""
        key = (tuple(x.shape), x.device.index)
        cached = getattr(net, "_slq_engine", None)
        if cached is None or cached[0] != key:
            eng = cls(net, x.shape[0], x.shape[2], x.shape[3], x.device, **kw)
            net._slq_engine = cached = (key, eng)
        eng = cached[1]
        eng.sync_weights()
        if not eng.calibrated:
            eng.calibrate(x)
        return eng

    # ------------------------------------------------------------------------------------------
    def _new_act(self, shape_nhwc, signed=False):
        """Reserves an activation tensor; the memory comes from ONE arena allocated when the plan is complete
        (_alloc_acts): 106 separate cudaMallocs cost 0.28 s per engine, a third of its set-up time."""
        self.act.append(None)
        self.act_shapes.append(tuple(int(v) for v in shape_nhwc))
        self.act_signed.append(signed)
        return len(self.act) - 1

    def _alloc_acts(self):
        sizes = [_align(int(np.prod(s)), 1024) for s in self.act_shapes]
        self.act_arena = torch.empty(max(sum(sizes), 1024), dtype=torch.uint8, device=self.device)
        off = 0
        for i, (s, n) in enumerate(zip(self.act_shapes, sizes)):
            self.act[i] = self.act_arena[off:off + int(np.prod(s))].view(s)
            off += n

    def _plan(self):
        net, N, dev = self.net, self.N, self.device
        if not net.conv1.weight.is_cuda:
            raise RuntimeError("model parameters must live on the CUDA device (call net.to(device))")
        Hc, Wc = (self.H + 6 - 7) // 2 + 1, (self.W + 6 - 7) // 2 + 1
        Hp, Wp = (Hc + 2 - 3) // 2 + 1, (Wc + 2 - 3) // 2 + 1
        self.act, self.act_shapes, self.act_signed, self.ops, self.tails, self.schedule = [], [], [], [], [], []
        self.stem_scratch = torch.empty(N * Hc * Wc * 64, dtype=torch.float32, device=dev)
        if self.stem_kind == "umma" and Wc > 128:
            self.stem_kind = "simt"  # one output row per 128-pixel tile: inputs wider than 256 px
        if self.stem_kind == "umma":
            nbytes = self.lib.slq_stem_workspace_bytes(N, self.H, self.W)
            self.stem_ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            h = ctypes.c_void_p()
            L.check(self.lib.slq_stem_create(N, self.H, self.W, self.stem_ws.data_ptr(), ctypes.byref(h)))
            self.stem = h
        x_id = self._new_act((N, Hp, Wp, 64))
        h, w = Hp, Wp
        max_out = N * Hp * Wp * 64
        for stage in (net.layer1, net.layer2, net.layer3, net.layer4):
            for blk in stage:
                convs = [c for c in ("conv1", "conv2", "conv3") if hasattr(blk, c)]
                res_id, res_signed = x_id, False
                cur, ch, cw = x_id, h, w
                pending = []
                for i, cname in enumerate(convs):
                    conv, bn = getattr(blk, cname), getattr(blk, "bn%d" % (i + 1))
                    op = self._make_op(conv, bn, cur, ch, cw, relu=True)
                    pending.append(op)
                    cur, ch, cw = op.out_id, op.Ho, op.Wo
                if blk.downsample is not None:
                    dop = self._make_op(blk.downsample[0], blk.downsample[1], x_id, h, w, relu=False, signed=True)
                    res_id, res_signed = dop.out_id, True
                    pending.insert(len(pending) - 1, dop)
                    if len(convs) == 3 and pending[-1].k == 1 and dop.k == 1:
                        self.tails.append(_BlockTail(dop, pending[-1]))
                last = pending[-1]
                last.res_id, last.res_signed = res_id, res_signed
                self.ops += pending
                x_id, h, w = last.out_id, last.Ho, last.Wo
        self._alloc_acts()
        for op in self.ops:
            max_out = max(max_out, op.M * op.Cout)
        self.final_id, self.final_hw, self.final_c = x_id, h * w, self.act[x_id].shape[3]
        # per-pixel channel sums ("rowsum") of the u8 activations that feed a layer running 256-channel tiles (the
        # K-heavy layers gather their window sums from it; everything else gets them from the tensor core): a stack
        # of planes per tensor, one per n-tile of the producing launch.  Allocated when a consumer first needs it.
        self.rowsum, self.rowsum_planes = {}, {}
        self.f32_scratch = torch.empty(max_out, dtype=torch.float32, device=dev)
        self.act_scales = torch.ones(len(self.act), dtype=torch.float32, device=dev)
        self.absmax_tmp = torch.zeros(1, dtype=torch.int32, device=dev)
        self.tail_ws = torch.empty(self.lib.slq_tail_workspace_bytes(N, self.final_c, net.fc.out_features) // 4,
                                   dtype=torch.float32, device=dev)
        self.logits = torch.empty((N, net.fc.out_features), dtype=torch.float32, device=dev)
        self.stem_w = torch.zeros_like(net.conv1.weight, dtype=torch.float32, device=dev)
        self.stem_a = torch.zeros(64, dtype=torch.float32, device=dev)
        self.stem_b = torch.zeros(64, dtype=torch.float32, device=dev)
        self.fc_w = torch.zeros_like(net.fc.weight, dtype=torch.float32, device=dev)
        self.fc_w_split = torch.zeros((2,) + tuple(net.fc.weight.shape), dtype=torch.float32, device=dev)  # {hi, lo} TF32 terms
        self.fc_b = torch.zeros_like(net.fc.bias, dtype=torch.float32, device=dev)
        self.ends_sig = None
        self.weights_version = 0   # bumped by every sync_weights() that changed something
        self.calibrated = False
        self.calib_hw = (self.H, self.W)
        self._graphs, self._seen = {}, set()

    def adopt_scales(self, other):
        """Takes over the activation scales of another engine of the same network (other batch size)."""
        self.act_scales.copy_(other.act_scales)
        self.calibrated = True

    def _make_op(self, conv, bn, in_id, h, w, relu, signed=False):
        op = _ConvOp()
        op.conv, op.bn, op.in_id, op.relu, op.signed = conv, bn, in_id, relu, signed
        op.Cin, op.Cout = conv.in_channels, conv.out_channels
        op.k, op.stride, op.pad = conv.kernel_size[0], conv.stride[0], conv.padding[0]
        op.H, op.W = h, w
        op.Ho = (h + 2 * op.pad - op.k) // op.stride + 1
        op.Wo = (w + 2 * op.pad - op.k) // op.stride + 1
        op.M = self.N * op.Ho * op.Wo
        op.out_id = self._new_act((self.N, op.Ho, op.Wo, op.Cout), signed)
        op.res_id, op.res_signed = -1, False
        op.handle, op.w16 = None, None
        op.variants = {}          # w16 -> (desc, GEMM-ready weight buffer, conv handle); created once, kept
        op.packed_gemm = None     # PackedGemm of the current weights (resident-weight layers)
        op.wsig = op.bsig = None  # what was packed last (see _sig)
        dev = self.device
        op.wscale = torch.zeros(op.Cout, dtype=torch.float32, device=dev)
        op.zf = torch.zeros(op.Cout, dtype=torch.float32, device=dev)
        op.bias = torch.zeros(op.Cout, dtype=torch.float32, device=dev)
        op.epi = {}
        return op

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _sig(*tensors):
        """What identifies the CONTENT of parameter tensors without reading them: storage pointer,
        autograd version counter (load_state_dict / any in-place op on the Parameter) and the write count
        the quantizer entry points keep per storage (resnet.note_weight_write: writes through ``.data``)."""
        import resnet
        return tuple((t.data_ptr(), t._version, resnet.weight_write_count(t)) for t in tensors)

    @staticmethod
    def _bn_tensors(bn):
        return (bn.weight, bn.bias, bn.running_mean, bn.running_var)

    def refresh_weights(self):
        """Re-derives every layer from the module tree's CURRENT fp32 parameters."""
        self.sync_weights(force=True)

    def sync_weights(self, force=False):
        """Brings the packed codes, GEMM-ready matrices and folded BN constants up to date with the module
        tree (content-derived, SURVEY.md H4 option b) -- only for the layers whose parameter tensors were
        written since they were packed last.  Device buffers keep their addresses (contents are updated in
        place), so conv handles, tensor maps and captured CUDA graphs stay valid; the activation scales are
        NOT touched (calibration is a separate, explicit step).  Returns the number of layers re-packed."""
        import resnet
        lib, dev = self.lib, self.device
        if self.epoch != resnet.WEIGHT_EPOCH[0]:
            force = True
            self.epoch = resnet.WEIGHT_EPOCH[0]
        todo, bn_todo = [], []
        for op in self.ops:
            wsig = self._sig(op.conv.weight)
            bsig = self._sig(*self._bn_tensors(op.bn))
            if force or wsig != op.wsig:
                todo.append((op, wsig, bsig))
            elif bsig != op.bsig:
                bn_todo.append((op, bsig))
        ends_sig = self._sig(self.net.conv1.weight, *self._bn_tensors(self.net.bn1), self.net.fc.weight, self.net.fc.bias)
        if not todo and not bn_todo and ends_sig == self.ends_sig and not force:
            return 0
        with torch.cuda.device(dev), torch.no_grad():
            stream = L.current_stream(dev)
            if todo:
                ws = [op.conv.weight.detach().to(torch.float32).reshape(op.Cout, -1).contiguous() for op, _, _ in todo]
                metas = classify_weights(ws, stream)
                for (op, wsig, bsig), w2d, (bit, z, s, bits_host, exact) in zip(todo, ws, metas):
                    op.packed = encode_weight(w2d, bit, z, s, bits_host, stream)
                    op.bits_host, op.packed_exact = bits_host, exact
                    w16 = 1 if int(bits_host.max()) > 8 else 0
                    var = op.variants.get(w16)
                    if var is None:  # first time this layer is seen in this mode: buffers + handle, kept for good
                        desc = L.ConvDesc(self.N, op.H, op.W, op.Cin, op.Cout, op.k, op.k, op.stride, op.pad,
                                          w16, self.impl, self.a_mode)
                        rows = lib.slq_gemm_weight_rows(ctypes.byref(desc))
                        wg = torch.empty((rows, op.k * op.k * op.Cin), dtype=torch.uint8, device=dev)
                        h = ctypes.c_void_p()
                        L.check(lib.slq_conv_create(ctypes.byref(desc), self.act[op.in_id].data_ptr(),
                                                    wg.data_ptr(), ctypes.byref(h)))
                        pgbuf = None
                        if w16 == 0 and self.packed_b and self.impl == L.IMPL_UMMA:
                            # resident-weight layers take their B operand PACKED (<= 4-bit rows two codes per byte),
                            # unpacked in shared memory; attached once, contents rewritten in place on every re-pack
                            pgbuf = alloc_packed_gemm(desc, dev)
                            if pgbuf is not None:
                                L.check(lib.slq_conv_set_packed_weights(h, pgbuf.blob.data_ptr(), pgbuf.tile_base.data_ptr(),
                                                                        pgbuf.seg_bytes.data_ptr(), pgbuf.row_offsets.data_ptr()))
                        var = op.variants[w16] = (desc, wg, h, pgbuf)
                    desc, wg, h, pgbuf = var
                    L.check(lib.slq_build_gemm_weights(ctypes.byref(desc), op.packed.blob.data_ptr(),
                                                       op.packed.offsets.data_ptr(), op.packed.bits.data_ptr(),
                                                       wg.data_ptr(), stream))
                    if pgbuf is not None:
                        build_packed_gemm(desc, op.packed, bits_host, dev, stream, into=pgbuf)
                    if op.w16 != w16:  # one-limb <-> two-limb: another kernel variant, graphs are stale
                        self._graphs, self._seen = {}, set()
                    op.packed_gemm = pgbuf
                    op.handle, op.w16, op.desc, op.wg = h, w16, desc, wg
                    op.s_dev, op.z_dev = s, z
                    self._fold_into(op)
                    op.wsig, op.bsig = wsig, bsig
            for op, bsig in bn_todo:
                self._fold_into(op)
                op.bsig = bsig
            if force or ends_sig != self.ends_sig:
                self.stem_w.copy_(self.net.conv1.weight.detach())
                if self.stem is not None:
                    L.check(lib.slq_stem_set_weights(self.stem, self.stem_w.data_ptr(), stream))
                a, b = self._fold_bn(self.net.bn1)
                self.stem_a.copy_(a)
                self.stem_b.copy_(b)
                self.fc_w.copy_(self.net.fc.weight.detach())
                L.check(lib.slq_tail_split_weights(self.fc_w.data_ptr(), self.fc_w.shape[0], self.fc_w.shape[1],
                                                   self.fc_w_split.data_ptr(), stream))
                self.fc_b.copy_(self.net.fc.bias.detach())
                self.ends_sig = ends_sig
        # the launch schedule: a block tail whose conv3 is quantised and whose downsample conv is not runs fused
        changed = False
        for bt in self.tails:
            want = self.fuse_tail and bt.op3.w16 == 0 and bt.dop.w16 == 1 and not bt.unsupported
            if want and bt.handle is None:
                dop, op3 = bt.dop, bt.op3
                desc = L.BlockTailDesc(self.N, dop.H, dop.W, dop.Cin, dop.stride, op3.Cin, op3.Cout, self.impl)
                h = ctypes.c_void_p()
                rc = lib.slq_blocktail_create(ctypes.byref(desc), self.act[op3.in_id].data_ptr(),
                                              self.act[dop.in_id].data_ptr(), op3.variants[0][1].data_ptr(),
                                              dop.variants[1][1].data_ptr(), ctypes.byref(h))
                if rc == L.SLQ_ERR_UNSUPPORTED:  # the two weight tiles do not fit one CTA: two launches
                    bt.unsupported, want = True, False
                else:
                    L.check(rc)
                    bt.handle = h
            if want != bt.fused:
                bt.fused, changed = want, True
        inside = {id(o): bt for bt in self.tails if bt.fused for o in (bt.dop, bt.op3)}
        self.schedule = []
        for op in self.ops:
            bt = inside.get(id(op))
            if bt is None:
                self.schedule.append(("conv", op))
            elif op is bt.op3:
                self.schedule.append(("tail", bt))
        # which activations need a rowsum side tensor (their consumer runs 256-channel tiles) and how many planes the
        # producer writes (n-tiles of the tiling its launch uses).  A layer that moved between the two-limb and the
        # one-limb mode changes both, and with them the epilogue descriptors of its neighbours.
        need = {op.in_id for kind, op in self.schedule if kind == "conv"
                and lib.slq_conv_needs_rowsum(op.handle, 1 if op.res_id >= 0 else 0)}
        planes = {0: 1}
        for kind, it in self.schedule:
            if kind == "tail":
                planes[it.op3.out_id] = max(int(lib.slq_blocktail_rowsum_planes(it.handle)), 1)
            elif not it.signed:
                planes[it.out_id] = max(int(lib.slq_conv_rowsum_planes(it.handle, 1 if it.res_id >= 0 else 0)), 1)
        changed = changed or set(self.rowsum) != need
        for i in need:
            if i not in self.rowsum:
                n_, h_, w_, c_ = self.act[i].shape
                self.rowsum[i] = torch.zeros((max(c_ // 64, 1), n_ * h_ * w_), dtype=torch.int32, device=dev)
            if self.rowsum_planes.get(i) != planes[i]:
                self.rowsum_planes[i], changed = planes[i], True
        for i in [i for i in self.rowsum if i not in need]:
            del self.rowsum[i]
            self.rowsum_planes.pop(i, None)
        if changed:
            for op in self.ops:
                op.epi = {}
            for bt in self.tails:
                bt.epi = {}
            self._graphs, self._seen = {}, set()
        self.weights_version += 1
        return len(todo)

    def _fold_into(self, op):
        """Per-channel epilogue constants of one layer, written IN PLACE (the epilogue descriptors and any
        captured graph hold these addresses)."""
        a, b = self._fold_bn(op.bn)
        op.wscale.copy_(op.s_dev * a)
        op.zf.copy_(op.z_dev.to(torch.float32))
        op.bias.copy_(b)

    @staticmethod
    def _fold_bn(bn):
        a = (bn.weight.detach() / torch.sqrt(bn.running_var.detach() + bn.eps)).to(torch.float32)
        b = (bn.bias.detach() - bn.running_mean.detach() * a).to(torch.float32)
        return a.contiguous(), b.contiguous()

    def _epilogue(self, op, mode, out_ptr, out_S=None):
        key = (mode, out_ptr)
        e = op.epi.get(key)
        if e is None:
            res = self.act[op.res_id].data_ptr() if op.res_id >= 0 else None
            rs_out = self.rowsum.get(op.out_id) if mode == L.OUT_U8 else None
            rs_in = self.rowsum.get(op.in_id)
            e = L.Epilogue(op.wscale.data_ptr(), op.zf.data_ptr(), op.bias.data_ptr(),
                           self.act_scales.data_ptr(), op.in_id, op.out_id, op.res_id, res,
                           1 if op.res_signed else 0, out_ptr, out_S, mode, 1 if op.relu else 0,
                           L.ptr(rs_in), L.ptr(rs_out), self.rowsum_planes.get(op.in_id, 0),
                           rs_in.shape[1] if rs_in is not None else 0)
            op.epi[key] = e
        return e

    def _tail_epilogue(self, bt, mode, out_ptr):
        key = (mode, out_ptr)
        e = bt.epi.get(key)
        if e is None:
            o3, od = bt.op3, bt.dop
            rs_out = self.rowsum.get(o3.out_id) if mode == L.OUT_U8 else None
            e = L.BlockTailEpilogue(o3.wscale.data_ptr(), o3.zf.data_ptr(), o3.bias.data_ptr(),
                                    od.wscale.data_ptr(), od.zf.data_ptr(), od.bias.data_ptr(),
                                    self.act_scales.data_ptr(), o3.in_id, od.in_id, o3.out_id, out_ptr, mode,
                                    L.ptr(rs_out))
            bt.epi[key] = e
        return e

    def launch_item(self, item, st, mode=None, out_ptr=None):
        """One entry of the launch schedule: ("conv", layer) or ("tail", fused block tail)."""
        kind, it = item
        if kind == "tail":
            mode = L.OUT_U8 if mode is None else mode
            out_ptr = self.act[it.op3.out_id].data_ptr() if out_ptr is None else out_ptr
            L.check(self.lib.slq_blocktail_launch(it.handle, ctypes.byref(self._tail_epilogue(it, mode, out_ptr)), st))
        else:
            mode = (L.OUT_S8 if it.signed else L.OUT_U8) if mode is None else mode
            out_ptr = self.act[it.out_id].data_ptr() if out_ptr is None else out_ptr
            L.check(self.lib.slq_conv_launch(it.handle, ctypes.byref(self._epilogue(it, mode, out_ptr)), st))

    def item_info(self, item):
        """Shape, arithmetic and algorithmic HBM bytes of one schedule entry (bench / tools)."""
        kind, it = item
        if kind == "tail":
            o3, od = it.op3, it.dop
            return dict(kind="tail", Cin=od.Cin, Cmid=o3.Cin, Cout=o3.Cout, k=1, stride=od.stride, H=od.H, M=o3.M,
                        w16=1, res=0, ops=2.0 * o3.M * o3.Cout * (o3.Cin + od.Cin),
                        bytes=self.act[o3.in_id].numel() + self.act[od.in_id].numel() + self.act[o3.out_id].numel()
                        + o3.wg.numel() + od.wg.numel())
        return dict(kind="conv", Cin=it.Cin, Cmid=0, Cout=it.Cout, k=it.k, stride=it.stride, H=it.H, M=it.M,
                    w16=it.w16, res=1 if it.res_id >= 0 else 0, ops=2.0 * it.M * it.Cout * it.k * it.k * it.Cin,
                    bytes=self.act[it.in_id].numel() + self.act[it.out_id].numel() + it.wg.numel()
                    + (self.act[it.res_id].numel() if it.res_id >= 0 else 0))

    # ------------------------------------------------------------------------------------------
    IN_KINDS = {torch.float32: L.IN_F32, torch.float16: L.IN_F16, torch.uint8: L.IN_U8}

    def _check_x(self, x):
        """The image batch as the loader hands it over: fp32 (the reference's format), fp16 (the same
        values rounded once; the stem rounds to fp16 anyway, so the logits are bit-identical) or raw u8
        pixels, normalised inside the stem with ``net.input_norm = (mean[3], std[3])`` exactly like
        torchvision's ToTensor + Normalize of reference imagenet.py:14-15."""
        if tuple(x.shape) != (self.N, 3, self.H, self.W) or x.dtype not in self.IN_KINDS or not x.is_cuda:
            raise ValueError("engine compiled for fp32 / fp16 / u8 CUDA input %s, got %s %s" %
                             ((self.N, 3, self.H, self.W), tuple(x.shape), x.dtype))
        kind = self.IN_KINDS[x.dtype]
        if kind != L.IN_F32 and self.stem is None:
            raise ValueError("fp16 / u8 inputs need the tensor-core stem (input width <= 256)")
        if kind == L.IN_U8:
            norm = getattr(self.net, "input_norm", None)
            if norm is None:
                raise ValueError("u8 input needs net.input_norm = (mean[3], std[3])")
            self.norm = (ctypes.c_float * 6)(*[float(v) for v in tuple(norm[0]) + tuple(norm[1])])
        self.in_kind = kind
        return x.contiguous()

    def calibrate(self, x, accumulate=False, headroom=1.0, images=None):
        """One pass with fp32 layer outputs: every activation tensor's static scale becomes
        absmax/255 (u8) or absmax/127 (s8) of this batch, times ``headroom``; with ``accumulate`` the
        larger of that and the scale it already has (running abs-max over several batches).  Each layer is
        then launched again in its quantised output mode, so the pass leaves exactly the bytes in HBM that
        forward(x) produces (and every later layer is calibrated on what it will really see).
        ``images``: only the first that many samples of x count (a padded short batch); None = all N."""
        lib = self.lib
        accumulate = accumulate and self.calibrated
        sc, tmp = self.act_scales.data_ptr(), self.absmax_tmp.data_ptr()
        old = self.act_scales.clone() if accumulate else None

        def observe(st, y, n, idx, qmax):
            L.check(lib.slq_absmax_scale(y, n, sc, idx, qmax, tmp, st))
            if headroom != 1.0:
                self.act_scales[idx:idx + 1].mul_(headroom)
            if old is not None:
                torch.maximum(self.act_scales[idx:idx + 1], old[idx:idx + 1], out=self.act_scales[idx:idx + 1])

        self._calib_walk(x, observe, images)
        self.calibrated = True

    def act_qmax(self):
        """Largest code of every activation tensor (device int32): 127 for s8 tensors, 255 for u8 ones."""
        return torch.tensor([127 if s else 255 for s in self.act_signed], dtype=torch.int32, device=self.device)

    def histogram(self, x, hist, rng, bins, images=None):
        """The calibration pass of ``calibrate`` with the scales in force left as they are: adds |y| of every
        layer output to its histogram (slq_act_histogram; hist [tensors, bins + 1] uint64, rng [tensors] fp32)."""
        lib = self.lib

        def observe(st, y, n, idx, qmax):
            L.check(lib.slq_act_histogram(y, n, rng.data_ptr(), idx, bins, hist.data_ptr(), st))

        self._calib_walk(x, observe, images)

    def hist_scales(self, hist, rng, bins, method, percentile=99.99, headroom=1.0):
        """Every activation scale from its histogram, in place (slq_hist_scales): captured graphs stay valid."""
        with torch.cuda.device(self.device):
            L.check(self.lib.slq_hist_scales(hist.data_ptr(), len(self.act), bins, rng.data_ptr(),
                                             self.act_qmax().data_ptr(), method, percentile, headroom,
                                             self.act_scales.data_ptr(), L.current_stream(self.device)))
        self.calibrated = True

    def _calib_walk(self, x, observe, images=None):
        """stem -> schedule: each layer once with fp32 output into f32_scratch, observe(stream, ptr, n, id, qmax)
        on it, then again in its quantised mode.  n covers the first ``images`` samples (NHWC: a prefix)."""
        lib = self.lib
        x = self._check_x(x)
        if any(op.handle is None for op in self.ops):
            raise RuntimeError("engine has no packed weights yet (call sync_weights())")
        images = self.N if images is None else images
        if not 0 < images <= self.N:
            raise ValueError("images=%d outside 1..%d" % (images, self.N))
        with torch.cuda.device(self.device), torch.no_grad():
            st = L.current_stream(self.device)
            f32 = self.f32_scratch.data_ptr()
            n0 = self.act[0].numel() // self.N * images
            self._stem(x.data_ptr(), f32, L.OUT_F32, st)
            observe(st, f32, n0, 0, 255)
            self._stem(x.data_ptr(), self.act[0].data_ptr(), L.OUT_U8, st)
            for item in self.schedule:
                op = item[1].op3 if item[0] == "tail" else item[1]   # the layer whose output tensor this writes
                if item[0] == "tail":
                    # the identity tensor does not exist on this path; its scale is still kept current for the day
                    # the block falls back to two launches (conv3 restored to fp32 weights)
                    dop = item[1].dop
                    self.launch_item(("conv", dop), st, L.OUT_F32, f32)
                    observe(st, f32, dop.M * dop.Cout // self.N * images, dop.out_id, 127)
                self.launch_item(item, st, L.OUT_F32, f32)
                observe(st, f32, op.M * op.Cout // self.N * images, op.out_id, 127 if op.signed else 255)
                self.launch_item(item, st)

    def forward(self, x):
        """Static-scale inference pass: stem -> conv launches -> tail.  Returns the engine's
        logits buffer [N, num_classes] (overwritten by the next call)."""
        if not self.calibrated:
            raise RuntimeError("engine is not calibrated (call calibrate(x) after refresh_weights())")
        x = self._check_x(x)
        # A forward is ~55 launches; replaying them as one CUDA graph saves ~0.3 ms of launch latency per
        # batch.  A graph bakes the input pointer in, so one is captured per input buffer the SECOND time
        # that buffer is seen (loaders and the caching allocator hand the same few buffers back), at most
        # four are kept, and all are dropped when weights or scales change.
        key = (x.data_ptr(), self.in_kind)
        g = self._graphs.get(key)
        if g is None and self.use_graphs:
            if key in self._seen:
                if len(self._graphs) >= 4:
                    self._graphs.pop(next(iter(self._graphs)))
                g = self._graphs[key] = self._capture(x)
            else:
                if len(self._seen) > 64:
                    self._seen.clear()
                self._seen.add(key)
        if g is not None:
            g.replay()
        else:
            self.launch_all(x.data_ptr(), L.current_stream(self.device))
        return self.logits

    def launch_all(self, x_ptr, st):
        lib = self.lib
        sc = self.act_scales.data_ptr()
        self._stem(x_ptr, self.act[0].data_ptr(), L.OUT_U8, st)
        for item in self.schedule:
            self.launch_item(item, st)
        L.check(lib.slq_tail_forward(self.act[self.final_id].data_ptr(), self.N, self.final_hw, self.final_c,
                                     sc, self.final_id, self.fc_w_split.data_ptr(), self.fc_b.data_ptr(),
                                     self.logits.shape[1], self.tail_ws.data_ptr(), self.logits.data_ptr(), st))
        self.kernel_launches = (1 if self.stem is not None else 2) + len(self.schedule) + 3

    def _stem(self, x_ptr, out_ptr, mode, st):
        lib, sc = self.lib, self.act_scales.data_ptr()
        if self.stem is not None:
            kind = getattr(self, "in_kind", L.IN_F32)
            norm = ctypes.cast(self.norm, ctypes.c_void_p) if kind == L.IN_U8 else None
            L.check(lib.slq_stem_launch_in(self.stem, x_ptr, kind, norm, self.stem_a.data_ptr(), self.stem_b.data_ptr(),
                                           sc, 0, out_ptr, mode, self.stem_scratch.data_ptr(),
                                           L.ptr(self.rowsum.get(0)), st))
        else:
            L.check(lib.slq_stem_forward(x_ptr, self.N, self.H, self.W, self.stem_w.data_ptr(),
                                         self.stem_a.data_ptr(), self.stem_b.data_ptr(), sc, 0,
                                         self.stem_scratch.data_ptr(), out_ptr, mode, L.ptr(self.rowsum.get(0)), st))

    # ------------------------------------------------------------------------------------------
    def capture_graph(self, x_static):
        """Captures one forward into a CUDA graph reading from x_static (fp32 / fp16 / u8 NCHW device buffer)."""
        x_static = self._check_x(x_static)
        self.graph, self.graph_x = self._capture(x_static), x_static
        return self.graph

    def _capture(self, x_static):
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream(self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            self.launch_all(x_static.data_ptr(), s.cuda_stream)  # warm-up outside capture
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
            self.launch_all(x_static.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        return g

    def weight_bytes(self):
        return sum(op.packed.nbytes for op in self.ops)

    def describe(self):
        rows = []
        for op in self.ops:
            bits, counts = np.unique(op.bits_host, return_counts=True)
            rows.append(dict(Cin=op.Cin, Cout=op.Cout, k=op.k, stride=op.stride, H=op.H, M=op.M, w16=op.w16,
                             bits={int(b): int(c) for b, c in zip(bits, counts)}))
        return rows

    def __del__(self):
        try:
            for op in getattr(self, "ops", []):
                for _desc, _wg, h, _pg in getattr(op, "variants", {}).values():
                    self.lib.slq_conv_destroy(h)
                op.variants, op.handle = {}, None
            for bt in getattr(self, "tails", []):
                if bt.handle is not None:
                    self.lib.slq_blocktail_destroy(bt.handle)
                    bt.handle = None
            if getattr(self, "stem", None) is not None:
                self.lib.slq_stem_destroy(self.stem)
                self.stem = None
        except Exception:
            pass
