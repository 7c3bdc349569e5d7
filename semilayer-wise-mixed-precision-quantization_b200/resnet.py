"""resnet.py -- drop-in mirror of the reference's ``resnet.py`` whose eval-mode CUDA forward runs on
the B200 engine (slq_engine.Engine: tcgen05 implicit-GEMM convs + fused epilogues) instead of
aten::convolution / native_batch_norm / relu_ / add_.

Boundary kept exactly (SURVEY.md 8b):
  * ``resnet18/34/50(pretrained=False, progress=True, **kwargs)``      reference resnet.py:235-265
  * module tree ``conv1, bn1, relu, maxpool, layer1..4[b].{conv1,bn1,conv2,bn2,conv3,bn3,relu,
    downsample}, avgpool, fc`` with torchvision-compatible ``state_dict`` keys   (resnet.py:121-202)
  * ``.weight`` of every conv is an fp32 Parameter ``[Cout,Cin,kh,kw]`` whose ``.data`` the mains
    re-assign after ``functions.channel_wise_quantizationperchan``       (resnet50_main.py:191)
  * ``net(x)``: fp32 NCHW in, fp32 logits out, same device               (resnet.py:204-223)
  * same construction + init order as the reference, so ``torch.manual_seed(s)`` followed by
    ``resnetXX(num_classes=1000)`` yields bit-identical parameters (tests/test_host_logic.py).

There is no eager-PyTorch or CPU fallback: a CPU tensor or training-mode call raises.
"""
import torch
import torch.nn as nn

try:
    from torch.hub import load_state_dict_from_url
except ImportError:  # pragma: no cover
    from torch.utils.model_zoo import load_url as load_state_dict_from_url

__all__ = ["ResNet", "resnet18", "resnet34", "resnet50"]

model_urls = {
    "resnet18": "https://download.pytorch.org/models/resnet18-5c106cde.pth",
    "resnet34": "https://download.pytorch.org/models/resnet34-333f7ec4.pth",
    "resnet50": "https://download.pytorch.org/models/resnet50-19c8e357.pth",
}

# ---- how the compiled engines learn that a weight tensor was written (SURVEY.md H4) ---------------------
# The mains mutate ``conv.weight.data`` in place through functions.channel_wise_quantizationperchan; a write
# through ``.data`` does not bump the Parameter's ``_version``.  Every quantizer entry point therefore notes
# the STORAGE it wrote (note_weight_write); an engine compares, per layer, (storage pointer, ``_version``,
# write count) with what it packed last and re-derives only the layers that differ.  ``load_state_dict``
# bumps ``_version`` and ``.to()`` / ``.data = ...`` change the pointer, so those are seen without a hook.
# WEIGHT_EPOCH is the conservative fallback for writers that cannot name a tensor (re-checks every layer).
WEIGHT_EPOCH = [0]
_WRITES = {}


def bump_weight_epoch():
    WEIGHT_EPOCH[0] += 1


def note_weight_write(tensor):
    key = tensor.untyped_storage().data_ptr()
    _WRITES[key] = _WRITES.get(key, 0) + 1


def weight_write_count(tensor):
    return _WRITES.get(tensor.untyped_storage().data_ptr(), 0)


def _conv(cin, cout, k, stride=1):
    return nn.Conv2d(cin, cout, kernel_size=k, stride=stride, padding=k // 2, bias=False)


class _Block(nn.Module):
    """One residual block.  ``kernels`` lists the conv kernel sizes of the main branch; the stride
    sits on the first 3x3 (ResNet v1.5 for Bottleneck, reference resnet.py:71-76)."""
    expansion = 1
    kernels = (3, 3)

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        widths = [planes] * (len(self.kernels) - 1) + [planes * self.expansion]
        cin = inplanes
        strided = False
        relu_registered = False
        for i, (k, cout) in enumerate(zip(self.kernels, widths), 1):
            s = 1
            if k == 3 and not strided:
                s, strided = stride, True
            setattr(self, "conv%d" % i, _conv(cin, cout, k, s))
            setattr(self, "bn%d" % i, nn.BatchNorm2d(cout))
            if self.expansion == 1 and not relu_registered:  # BasicBlock registers relu after bn1
                self.relu = nn.ReLU(inplace=True)
                relu_registered = True
            cin = cout
        if not relu_registered:
            self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):  # blocks only run inside ResNet.forward -> engine
        raise RuntimeError("residual blocks are executed by the B200 engine through ResNet.forward")


class BasicBlock(_Block):
    expansion = 1
    kernels = (3, 3)


class Bottleneck(_Block):
    expansion = 4
    kernels = (1, 3, 1)


class ResNet(nn.Module):
    # tests may install a checker (oracle) for CPU tensors; the product never sets this
    cpu_checker = None

    def __init__(self, block, layers, num_classes=1000):
        super().__init__()
        self.block_name = block.__name__
        self.arch = layers
        self.inplanes = 64
        self.conv1 = nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        self.relu = nn.ReLU(inplace=True)
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        for i, (planes, n) in enumerate(zip((64, 128, 256, 512), layers), 1):
            setattr(self, "layer%d" % i, self._make_layer(block, planes, n, stride=1 if i == 1 else 2))
        self.layers = [self.layer1, self.layer2, self.layer3, self.layer4]
        self.avgpool = nn.AdaptiveAvgPool2d((1, 1))
        self.fc = nn.Linear(512 * block.expansion, num_classes)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        self._slq_engines = {}
        self._slq_dirty = True

    def _make_layer(self, block, planes, blocks, stride):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = nn.Sequential(_conv(self.inplanes, planes * block.expansion, 1, stride),
                                       nn.BatchNorm2d(planes * block.expansion))
        seq = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * block.expansion
        seq += [block(self.inplanes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*seq)

    # ---- compiled-engine bookkeeping ---------------------------------------------------------
    def slq_invalidate(self):
        """Forces every layer to be re-packed on the next forward (for writers the engine cannot see,
        e.g. ``w.data.mul_(2)``: an in-place op through ``.data`` bumps no version counter)."""
        self._slq_dirty = True

    def _apply(self, fn, *a, **k):  # .to() / .cuda() / .float() ...
        before = (self.conv1.weight.data_ptr(), self.conv1.weight.dtype)
        out = super()._apply(fn, *a, **k)
        if (self.conv1.weight.data_ptr(), self.conv1.weight.dtype) != before:
            # storage moved or was converted: compiled pointers are stale.  A no-op ``net.to(device)``
            # (evaluate_acc_loss_softmax calls it before every evaluation, functions.py:97) keeps the
            # engine, its packed weights, its activation scales and its CUDA graphs.
            self._slq_engines = {}
            self._slq_dirty = True
        return out

    def __getstate__(self):  # copy.deepcopy / torch.save(net): engines own ctypes handles and GBs of HBM
        state = dict(self.__dict__)
        state["_slq_engines"] = {}
        state["_slq_dirty"] = True
        state.pop("_slq_donor", None)
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        self.__dict__.setdefault("_slq_engines", {})
        self._slq_dirty = True

    def slq_engine(self, x, **kw):
        """The compiled engine for inputs shaped like x (built on first use)."""
        import slq_engine
        key = (x.shape[0], x.shape[2], x.shape[3], x.device.index)
        eng = self._slq_engines.get(key)
        if eng is None:
            old = next(iter(self._slq_engines.values()), None)
            eng = slq_engine.Engine(self, x.shape[0], x.shape[2], x.shape[3], x.device, **kw)
            donor = getattr(self, "_slq_donor", None)
            if old is None and donor is not None:
                old = next((e for e in getattr(donor, "_slq_engines", {}).values()), None)
            if old is not None and old.calibrated and len(old.act) == len(eng.act) and old.calib_hw == (x.shape[2], x.shape[3]):
                eng.adopt_scales(old)  # same network, same image size (other batch size): ranges carry over
            self._slq_engines = {key: eng}  # one live shape at a time (activation buffers are large)
        return eng

    def slq_calibrated(self, hw=None):
        """True when a CUDA forward on images of size ``hw`` = (H, W) (None: of the size the net was calibrated at)
        runs under activation scales the net already holds (its engine's, or through slq_share_calibration its
        donor's); False when that forward calibrates them on its own batch (slq_engine() / forward())."""
        eng = next(iter(self._slq_engines.values()), None)
        donor = getattr(self, "_slq_donor", None)
        if eng is None and donor is not None:
            eng = next(iter(getattr(donor, "_slq_engines", {}).values()), None)
        return eng is not None and eng.calibrated and (hw is None or eng.calib_hw == tuple(hw))

    def slq_share_calibration(self, other):
        """Use ``other``'s activation scales (same architecture, same image size) instead of calibrating on
        the first batch: the un-quantised model and the candidates of a sweep must be compared under the SAME
        activation quantisation, or re-calibration noise lands on top of the effect being measured."""
        self._slq_donor = other

    CALIB_METHODS = ("absmax", "percentile", "mse", "entropy")
    CALIB_BINS = 2048

    def slq_calibrate(self, batches, headroom=1.0, method="absmax", percentile=99.99):
        """Explicit calibration of the static per-tensor activation scales (the reference never quantises
        activations, SURVEY.md F2, so this call has no counterpart there) over ``batches`` (a tensor, a list of
        tensors, or a loader of (x, y) pairs; CUDA or host), times ``headroom``:
          * ``"absmax"``      running abs-max over the batches (the default);
          * ``"percentile"``  the ``percentile``-th percentile of |y| over the batches, zeros included;
          * ``"mse"``         the clipping threshold with the least squared quantisation error of |y|;
          * ``"entropy"``     the clipping threshold whose quantised distribution of |y| has the least KL
                              divergence from the observed one (TensorRT's and pytorch-quantization's entropy
                              calibrator; zeros left out, candidates from bin 128 of 2048 up).
        The last three read a 2048-bin histogram of every layer output, whose range comes from an abs-max pass
        over the same batches: they iterate ``batches`` twice, so a one-shot iterator is refused.
        The scales then stay fixed -- through weight changes, state_dict reloads and later batches -- until
        the next slq_calibrate().  Without this call the first forward calibrates on its own batch."""
        import slq_lib as L
        if method not in self.CALIB_METHODS:
            raise ValueError("slq_calibrate: method %r is not one of %s" % (method, ", ".join(self.CALIB_METHODS)))
        if torch.is_tensor(batches):
            batches = [batches]
        # threshold rule of slq_hist_scales per histogram method; None: abs-max, no histogram
        rule = {"percentile": L.CALIB_PERCENTILE, "mse": L.CALIB_MSE, "entropy": L.CALIB_ENTROPY}.get(method)
        hist = rule is not None
        if hist and iter(batches) is batches:
            raise TypeError("slq_calibrate(method=%r) reads the batches twice: pass a list or a re-iterable "
                            "loader, not a one-shot iterator" % method)
        first, eng = True, None
        for eng, x, n in self._calib_batches(batches):
            # histogram methods: the abs-max pass only sets each tensor's range, over the images actually given
            eng.calibrate(x, accumulate=not first, headroom=1.0 if hist else headroom, images=n if hist else None)
            first = False
        if first:
            raise ValueError("slq_calibrate: no batches")
        if not hist:
            return
        bins = self.CALIB_BINS
        qmax = eng.act_qmax().to(torch.float32)
        rng = eng.act_scales * qmax
        counts = torch.zeros((len(eng.act), bins + 1), dtype=torch.int64, device=eng.device)
        for e, x, n in self._calib_batches(batches):
            if e is not eng:
                raise ValueError("slq_calibrate: the batches changed shape between the two passes")
            eng.histogram(x, counts, rng, bins, images=n)
        eng.hist_scales(counts, rng, bins, rule, percentile, headroom)

    def _calib_batches(self, batches):
        """(engine, batch on the device padded to the engine's batch size, images in it) per calibration batch."""
        import slq_engine
        dev = self.conv1.weight.device
        for item in batches:
            x = item[0] if isinstance(item, (tuple, list)) else item
            x = x.to(dev, non_blocking=True)
            n = x.shape[0]
            cap = slq_engine.engine_batch(self, n)
            if n < cap:
                xp = x.new_zeros((cap,) + tuple(x.shape[1:]))
                xp[:n] = x
                x = xp
            eng = self.slq_engine(x)
            eng.sync_weights(force=self._slq_dirty)
            self._slq_dirty = False
            yield eng, x, n

    def forward(self, x):
        if not x.is_cuda:
            if ResNet.cpu_checker is not None:
                return ResNet.cpu_checker(self, x)
            raise RuntimeError("this ResNet runs on the B200 engine: pass a CUDA tensor "
                               "(there is no CPU / eager fallback)")
        if self.training:
            raise RuntimeError("the B200 engine implements the eval-mode forward only; call net.eval()")
        import slq_engine
        n = x.shape[0]
        cap = slq_engine.engine_batch(self, n)
        if n < cap:  # short last batch of a loader: pad (static scales keep samples independent)
            xp = x.new_zeros((cap,) + tuple(x.shape[1:]))
            xp[:n] = x
        else:
            xp = x
        eng = self.slq_engine(xp)
        eng.sync_weights(force=self._slq_dirty)  # re-packs only the layers whose tensors were written
        self._slq_dirty = False
        if not eng.calibrated:
            eng.calibrate(xp)
        return eng.forward(xp)[:n].clone()


def _resnet(arch, block, layers, pretrained, progress, **kwargs):
    model = ResNet(block, layers, **kwargs)
    if pretrained:
        model.load_state_dict(load_state_dict_from_url(model_urls[arch], progress=progress), strict=False)
    return model


def resnet18(pretrained=False, progress=True, **kwargs):
    return _resnet("resnet18", BasicBlock, [2, 2, 2, 2], pretrained, progress, **kwargs)


def resnet34(pretrained=False, progress=True, **kwargs):
    return _resnet("resnet34", BasicBlock, [3, 4, 6, 3], pretrained, progress, **kwargs)


def resnet50(pretrained=False, progress=True, **kwargs):
    return _resnet("resnet50", Bottleneck, [3, 4, 6, 3], pretrained, progress, **kwargs)
