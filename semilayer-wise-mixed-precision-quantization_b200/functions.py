"""functions.py -- drop-in mirror of the reference's ``functions.py`` on top of the B200 path.

Same ten module-level entry points, same argument meaning, return values and error behaviour
(SURVEY.md 8b), so the unmodified ``resnet18/34/50_main.py`` run against this module:

  channel_wise_quantizationperchan / quantize_wgt   reference functions.py:9-43   -> slq_quantize_rows
  evaluate_loss / evaluate_acc_loss_softmax / KLdiv reference functions.py:45-149 (callers of net(x))
  make_divide_minusplusmodels                       reference functions.py:151-184
  make_semilayers_resnet18/34/50                    reference functions.py:186-588 (one shared body,
                                                    candidates sharded over torch.distributed ranks)
  make_quantizedlists                               reference functions.py:590-612

Extensions (not in the reference): ``quantize_rows`` (a whole semilayer / layer in one launch, returns the
packed codes), ``quantize_model`` (every layer of a model in one launch), ``make_semilayers`` (arch-generic
sweep, optional delta-loss metric), ``snapshot`` / ``restore`` (device-resident undo state instead of
torch.save / torch.load), ``save_packed`` / ``load_packed`` (packed model file) and
``make_deltaloss_table`` / ``write_deltaloss_csv`` (regenerates dataset/*_deltaloss.csv).
"""
import os

import numpy as np
import torch
import torch.nn

import imagenet
import resnet
import slq_lib as L

SENTINEL = [0, 0, 100, 0, 0, 0, 0, 0]


# ==============================================================================================
# quantizer
# ==============================================================================================
class PackedRows:
    """Result of quantize_rows: job j -> codes blob[offsets[j]:...], z[j], s32[j], status[j]."""

    def __init__(self, rows, bits, offsets, blob, z, s32, status, K):
        self.rows, self.bits, self.offsets, self.blob = rows, bits, offsets, blob
        self.z, self.s32, self.status, self.K = z, s32, status, K

    def codes(self, j):
        """Unpacked codes of job j as a uint8/int32 numpy array (host copy; for inspection/tests)."""
        bit = int(self.bits[j])
        nbytes = L.lib().slq_packed_row_bytes(self.K, bit)
        off = int(self.offsets[j])
        raw = self.blob[off:off + nbytes].cpu().numpy().astype(np.int64)
        if bit == 4:
            return np.stack([raw & 15, raw >> 4], 1).reshape(-1)[:self.K].astype(np.int32)
        if bit == 2:
            return np.stack([(raw >> (2 * i)) & 3 for i in range(4)], 1).reshape(-1)[:self.K].astype(np.int32)
        return raw[:self.K].astype(np.int32)


def packed_row_bytes(K, bits):
    """slq_packed_row_bytes (include/slq.h) for an array of bit-widths <= 8 at once -- a ctypes call per
    row would dominate a whole-model pass: 4-bit rows pack two codes per byte, 2-bit rows four, every other
    width one."""
    b64 = np.asarray(bits, dtype=np.int64)
    return np.where(b64 == 4, (K + 1) // 2, np.where(b64 == 2, (K + 3) // 4, K)).astype(np.int64)


def _div_mode_for(tensor, div_mode):
    if div_mode is not None:
        return div_mode
    forced = os.environ.get("SLQ_DIV_MODE")  # "true" | "recip": pin one flavour for a whole run (tests)
    if forced:
        return {"true": L.DIV_TRUE, "recip": L.DIV_RECIP}[forced]
    # what the reference's own ATen call does on that device (SURVEY.md F5)
    return L.DIV_RECIP if tensor.is_cuda else L.DIV_TRUE


def quantize_rows(tensor, rows, bits, write_back=True, want_codes=True, div_mode=None):
    """Quantises rows ``rows[j]`` of a contiguous fp32 weight tensor ``[Cout, ...]`` to ``bits[j]``
    bits in ONE kernel launch (reference: one quantize_wgt call = 7 launches + 2 syncs per row).
    In place when write_back (the contract of functions.py:22).  Raises ZeroDivisionError for a
    constant row like the reference (functions.py:40).  Returns PackedRows."""
    lib = L.lib()
    if tensor.dtype != torch.float32 or not tensor.is_contiguous():
        raise TypeError("quantize_rows needs a contiguous float32 tensor")
    n_rows = tensor.shape[0]
    K = tensor[0].numel()
    rows_h = np.ascontiguousarray(rows, dtype=np.int32).reshape(-1)
    bits_h = np.ascontiguousarray(bits, dtype=np.int32).reshape(-1)
    if rows_h.size != bits_h.size:
        raise ValueError("rows and bits must have the same length")
    if rows_h.size and (rows_h.min() < 0 or rows_h.max() >= n_rows):
        raise IndexError("row index out of range")
    if bits_h.size and (bits_h.min() < 1 or bits_h.max() > 8):
        raise ValueError("bit-width must be in 1..8")
    n_jobs = rows_h.size
    sizes = (packed_row_bytes(K, bits_h) + 15) // 16 * 16
    offs_h = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64) if n_jobs else np.zeros(0, np.int64)
    total = int(sizes.sum())
    dm = _div_mode_for(tensor, div_mode)
    if n_jobs == 0:
        e = torch.empty(0)
        return PackedRows(rows_h, bits_h, offs_h, e.to(torch.uint8), e.to(torch.int32), e, e.to(torch.int32), K)
    if tensor.is_cuda:
        dev = tensor.device
        with torch.cuda.device(dev):
            # job table in ONE host->device copy: offsets (int64) | rows | bits (int32)
            table = np.concatenate([offs_h.view(np.int32), rows_h, bits_h])
            table_d = torch.from_numpy(table).to(dev)
            offs_d = table_d[:2 * n_jobs].view(torch.int64)
            rows_d, bits_d = table_d[2 * n_jobs:3 * n_jobs], table_d[3 * n_jobs:]
            blob = torch.empty(max(total, 16), dtype=torch.uint8, device=dev) if want_codes else None
            z = torch.empty(n_jobs, dtype=torch.int32, device=dev)
            s32 = torch.empty(n_jobs, dtype=torch.float32, device=dev)
            status = torch.empty(n_jobs, dtype=torch.int32, device=dev)
            L.check(lib.slq_quantize_rows(tensor.data_ptr(), n_rows, K, rows_d.data_ptr(), bits_d.data_ptr(),
                                          n_jobs, dm, 1 if write_back else 0, L.ptr(blob), offs_d.data_ptr(),
                                          z.data_ptr(), s32.data_ptr(), status.data_ptr(), L.current_stream(dev)))
            st_h = status.cpu()  # the reference is synchronous too (.item())
    else:
        blob = torch.empty(max(total, 16), dtype=torch.uint8) if want_codes else None
        z = torch.empty(n_jobs, dtype=torch.int32)
        s32 = torch.empty(n_jobs, dtype=torch.float32)
        status = torch.zeros(n_jobs, dtype=torch.int32)
        rc = lib.slq_quantize_rows_host(tensor.data_ptr(), n_rows, K, rows_h.ctypes.data, bits_h.ctypes.data,
                                        n_jobs, dm, 1 if write_back else 0, L.ptr(blob), offs_h.ctypes.data,
                                        z.data_ptr(), s32.data_ptr(), status.data_ptr())
        if rc not in (L.SLQ_OK, L.SLQ_ERR_ZERO_RANGE):
            L.check(rc)
        st_h = status
    if write_back:
        resnet.note_weight_write(tensor)  # engines re-pack exactly this tensor's layer on their next forward
    if bool((st_h & L.ROW_ZERO_RANGE).any()):
        raise ZeroDivisionError("float division by zero")
    return PackedRows(rows_h, bits_h, offs_h, blob, z, s32, status, K)


def quantize_wgt(tensor, bit):
    """Per-tensor min/max affine fake-quantiser; returns a NEW tensor (reference functions.py:25-43)."""
    flat = tensor.detach().to(torch.float32).contiguous().reshape(1, -1).clone()
    quantize_rows(flat, [0], [bit], write_back=True, want_codes=False)
    return flat.reshape(tensor.shape)


def channel_wise_quantizationperchan(tensor, bit, i):
    """Overwrites output channel ``i`` of ``tensor`` with its ``bit``-bit fake-quantised value, in
    place, and returns the same tensor object (reference functions.py:9-23)."""
    if tensor.is_contiguous() and tensor.dtype == torch.float32:
        quantize_rows(tensor, [i], [bit], write_back=True, want_codes=False)
    else:
        tensor[i] = quantize_wgt(tensor[i], bit)
        resnet.note_weight_write(tensor)
    return tensor


class QuantPlan:
    """A whole bit assignment -- rows of SEVERAL weight tensors -- prepared as ONE multi-tensor job table on
    the device (slq_quantize_jobs).  ``run()`` is then a single kernel launch with no host work in front of it
    (the reference makes one quantize_wgt call, 7 launches and 2 syncs, per row: resnet50_main.py:189-197).

    ``items``: list of ``(tensor, rows, bits)`` with contiguous fp32 CUDA tensors ``[Cout, ...]`` on one
    device.  Arrays are in launch order (jobs sorted by row-length class); ``perm[j]`` is the position of
    launch-order job j in the caller's order (tensors in the order given, rows in the order given)."""

    def __init__(self, items, want_codes=True, div_mode=None):
        if not items:
            raise ValueError("QuantPlan: no tensors")
        dev = items[0][0].device
        rowp, Ks, bits_all, rows_all, item_of = [], [], [], [], []
        for i, (t, rows, bits) in enumerate(items):
            if t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda or t.device != dev:
                raise TypeError("QuantPlan needs contiguous float32 CUDA tensors on one device")
            K = t[0].numel()
            if K % 4 != 0 or K > 4608 or t.data_ptr() % 16 != 0:
                raise ValueError("QuantPlan: row length %d unsupported (use quantize_rows)" % K)
            r = np.ascontiguousarray(rows, dtype=np.int64).reshape(-1)
            b = np.ascontiguousarray(bits, dtype=np.int32).reshape(-1)
            if r.size != b.size:
                raise ValueError("rows and bits must have the same length")
            if r.size and (r.min() < 0 or r.max() >= t.shape[0]):
                raise IndexError("row index out of range")
            if b.size and (b.min() < 1 or b.max() > 8):
                raise ValueError("bit-width must be in 1..8")
            rowp.append(np.uint64(t.data_ptr()) + (r * (4 * K)).astype(np.uint64))
            Ks.append(np.full(r.size, K, np.int32))
            bits_all.append(b)
            rows_all.append(r)
            item_of.append(np.full(r.size, i, np.int32))
        rowp, Ks, bits_all = np.concatenate(rowp), np.concatenate(Ks), np.concatenate(bits_all)
        rows_all, item_of = np.concatenate(rows_all), np.concatenate(item_of)
        n = rowp.size
        if n == 0:
            raise ValueError("QuantPlan: no rows")
        cls = (Ks > 288).astype(np.int8) + (Ks > 1152).astype(np.int8)
        perm = np.argsort(cls, kind="stable")
        self.counts = [int(c) for c in np.bincount(cls, minlength=3)]
        sizes = (np.where(bits_all == 4, (Ks + 1) // 2, np.where(bits_all == 2, (Ks + 3) // 4, Ks)).astype(np.int64) + 15) // 16 * 16
        sizes_p = sizes[perm]
        offs = np.zeros(n, np.int64)
        offs[1:] = np.cumsum(sizes_p)[:-1]
        self.div_mode = _div_mode_for(items[0][0], div_mode)
        self.items, self.device, self.n = items, dev, n
        self.perm, self.item_of, self.rows, self.bits, self.K, self.offsets = \
            perm, item_of[perm], rows_all[perm], bits_all[perm], Ks[perm], offs
        with torch.cuda.device(dev):
            self.blob = torch.empty(max(int(sizes_p.sum()), 16), dtype=torch.uint8, device=dev) if want_codes else None
            jobs = np.empty(n, _QJOB)
            jobs["row"], jobs["K"], jobs["bit"] = rowp[perm], Ks[perm], bits_all[perm]
            jobs["codes"] = (np.uint64(self.blob.data_ptr()) + offs.astype(np.uint64)) if want_codes else 0
            self.jobs_d = torch.from_numpy(jobs.view(np.uint8).reshape(-1)).to(dev)  # the one host->device copy
            self.z = torch.empty(n, dtype=torch.int32, device=dev)
            self.s32 = torch.empty(n, dtype=torch.float32, device=dev)
            self.status = torch.empty(n, dtype=torch.int32, device=dev)

    @property
    def nbytes(self):
        return 0 if self.blob is None else int(self.blob.numel())

    def run(self, write_back=True):
        """ONE launch; nothing is synchronised."""
        with torch.cuda.device(self.device):
            L.check(L.lib().slq_quantize_jobs(self.jobs_d.data_ptr(), self.counts[0], self.counts[1], self.counts[2],
                                              self.div_mode, 1 if write_back else 0, self.z.data_ptr(),
                                              self.s32.data_ptr(), self.status.data_ptr(),
                                              L.current_stream(self.device)))
        if write_back:
            for t, _r, _b in self.items:
                resnet.note_weight_write(t)
        return self

    def check(self):
        """The one synchronisation: raises ZeroDivisionError like the reference (functions.py:40) if any
        row was constant."""
        st = self.status.cpu()
        if bool((st & L.ROW_ZERO_RANGE).any()):
            raise ZeroDivisionError("float division by zero")
        return st


PackedModel = QuantPlan  # what quantize_model returns: the plan, with its outputs filled in
_QJOB = np.dtype([("row", "<u8"), ("codes", "<u8"), ("K", "<i4"), ("bit", "<i4")])


def quantize_model(items, write_back=True, want_codes=True, div_mode=None, check=True):
    """Quantises rows of several weight tensors -- a whole model's bit assignment -- in ONE kernel launch:
    one host->device copy of the job table, one launch, and -- with ``check`` -- one synchronisation at the
    end.  Returns the QuantPlan (keep it and call ``run()`` again to re-quantise without any host work)."""
    plan = QuantPlan(items, want_codes=want_codes, div_mode=div_mode).run(write_back=write_back)
    if check:
        plan.check()
    return plan


# ==============================================================================================
# evaluation (callers of the forward)
# ==============================================================================================
def _fused_tail_ok(t):
    return torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.is_contiguous()


def _to_device(net, device):
    """``net.to(device)`` (reference functions.py:97), skipped when every parameter and buffer already lives there:
    the no-op walks ~6000 module / tensor objects (16 ms for ResNet-50) -- once per evaluation that was 1.6 s of a
    96-candidate sweep whose forward passes take 0.1 s."""
    dev = torch.device(device)
    if dev.type == "cuda" and dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    for t in net.parameters():
        if t.device != dev:
            return net.to(device)
    for t in net.buffers():
        if t.device != dev:
            return net.to(device)
    return net


_RESIDENT = {"key": None, "loader": None, "batches": None}


def _resident_batches(data_loader, device, rank=0, world=1):
    """An IN-MEMORY loader (a list / tuple of (x, y) host tensors, e.g. imagenet.synthetic_loader or a calibration
    set) is copied to the device once and the copies are reused by the following evaluations, as long as the
    loader object and its tensors are unchanged (pointer + version counter per tensor).  Every candidate of a
    sweep evaluates the same batches: the pageable 38.5 MB per 64 images were copied again for each of them.
    With ``world`` > 1 only the batches ``rank`` owns (batch i belongs to rank i % world) are returned, and only
    those are copied.  Streaming loaders (anything else) are passed through."""
    if not isinstance(data_loader, (list, tuple)):
        return data_loader
    mine = data_loader if world == 1 else data_loader[rank::world]
    dev = torch.device(device)
    if dev.type != "cuda" or os.environ.get("SLQ_NO_RESIDENT_LOADER"):
        return mine  # (a writer that goes through ``x.data`` bumps no version counter: set the variable then)
    try:
        sig = tuple((x.data_ptr(), x._version, tuple(x.shape), y.data_ptr(), y._version) for x, y in mine)
    except Exception:
        return mine
    if any(x.is_cuda for x, _y in mine):
        return mine
    key = (id(data_loader), str(dev), rank, world, sig)
    if _RESIDENT["key"] != key:
        _RESIDENT["batches"] = [(x.to(device), y.to(device)) for x, y in mine]
        _RESIDENT["key"], _RESIDENT["loader"] = key, data_loader  # the reference keeps id() from being recycled
    return _RESIDENT["batches"]


_RANK_LOADER = {"key": None, "loader": None, "batches": None}


def _subset_loader(data_loader, batch_ids):
    """A DataLoader over ``data_loader``'s dataset that yields exactly its batches ``batch_ids`` (the loader reads the
    dataset in order: batch i is the indices [i*B, (i+1)*B)), with the same collate function, workers and pinning."""
    from torch.utils.data import DataLoader
    B, N = data_loader.batch_size, len(data_loader.dataset)
    kw = dict(num_workers=data_loader.num_workers, collate_fn=data_loader.collate_fn,
              pin_memory=data_loader.pin_memory, worker_init_fn=data_loader.worker_init_fn,
              multiprocessing_context=data_loader.multiprocessing_context, timeout=data_loader.timeout)
    if data_loader.num_workers > 0:
        kw.update(prefetch_factor=data_loader.prefetch_factor, persistent_workers=data_loader.persistent_workers)
    return DataLoader(data_loader.dataset, batch_sampler=[list(range(i * B, min((i + 1) * B, N))) for i in batch_ids],
                      **kw)


def _rank_loader(data_loader, rank, world):
    """For a torch DataLoader that reads its dataset in order (a SequentialSampler, as ``shuffle=False`` makes): a
    DataLoader that yields only the batches of ``rank`` -- the same tensors the full loader yields for them, read and
    decoded by this rank's workers alone.  Cached per (loader, rank) like the resident batches.  None for any other
    loader."""
    from torch.utils.data import DataLoader, SequentialSampler
    if not (isinstance(data_loader, DataLoader) and isinstance(data_loader.sampler, SequentialSampler)
            and data_loader.sampler.data_source is data_loader.dataset and data_loader.batch_size is not None):
        return None
    key = (id(data_loader), rank, world, len(data_loader.dataset))
    if _RANK_LOADER["key"] != key:
        _RANK_LOADER["batches"] = _subset_loader(data_loader, range(rank, len(data_loader), world))
        _RANK_LOADER["key"], _RANK_LOADER["loader"] = key, data_loader
    return _RANK_LOADER["batches"]


def _rank_batches(data_loader, device, rank, world):
    """The batches ``rank`` of ``world`` evaluates, batch i belonging to rank i % world: -> (number of batches, or None
    when only a full pass tells; iterable of (i, (x, y)); first, a callable returning batch 0 when the iterable leaves
    it out, else None; batch 0's (H, W), or None when unknown without reading it).  Only a loader that is neither in
    memory nor a DataLoader reading its dataset in order is iterated in full; the caller skips other ranks' batches."""
    if world > 1 and isinstance(data_loader, (list, tuple)):
        n = len(data_loader)
        return n, zip(range(rank, n, world), _resident_batches(data_loader, device, rank, world)), \
            lambda: data_loader[0], tuple(data_loader[0][0].shape[2:]) if n else None
    sub = _rank_loader(data_loader, rank, world) if world > 1 else None
    if sub is not None:
        n = len(data_loader)
        return n, zip(range(rank, n, world), sub), lambda: next(iter(_subset_loader(data_loader, [0]))), None
    return None, enumerate(_resident_batches(data_loader, device)), None, None


def _calibrate_on_batch0(net, device, batch0, hw):
    """What a single process's first forward does to the activation scales: when the net holds none for batch 0's
    image size (``hw``; None: any size), calibrate them on batch 0."""
    if not net.slq_calibrated(hw):
        with torch.no_grad():
            net(batch0()[0].to(device))


def _all_gather(t, dist, world):
    """all_gather of one equally shaped tensor per rank -> the world tensors, in rank order: NCCL on the current CUDA
    device, any other backend through the host."""
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = t.to(dev)
    bufs = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(bufs, t)
    return bufs


_PROB_DTYPES = (torch.float32, torch.float64, torch.float16, torch.bfloat16)
_FUSED, _HOST = 1, 2  # which route a rank's batches took (bit mask, gathered with the records)


def _evaluate(net, device, data_loader, ref_outputs=None, want_probs=True, shard=True):
    """One pass over the loader: -> (acc, loss, [softmax per batch], KL(ref_outputs || outputs) or None).

    On CUDA the whole tail of every batch -- argmax, cross-entropy, softmax and, when ``ref_outputs`` (the
    stored softmax outputs of the un-quantised model) is given, the per-sample KL divergence -- is ONE fused
    kernel pass (slq_eval_tail) that writes the batch's record of four doubles on the device; the records are read
    back ONCE at the end and folded in batch order on the host, which adds the same values in the same order as one
    running accumulator would (the reference synchronises three times per evaluation, functions.py:129, and KLdiv
    loops over every sample in Python, functions.py:142-146).  CPU tensors take the stock-torch route, whose
    per-batch values are folded with the reference's fp32 adds.

    With ``shard`` and torch.distributed initialised with a world size above 1, the evaluation is data-parallel by
    batch: batch i is run (forward and tail) by rank i % world only, one all_gather exchanges the records and, when
    ``want_probs``, a second one the probabilities, and every rank returns what a single process returns, bit for
    bit.  Every rank must therefore make the same evaluations in the same order, as for make_semilayers."""
    _to_device(net, device)
    net.eval()
    dist, rank, world = _dist() if shard else (None, 0, 1)
    n, batches, first, hw0 = _rank_batches(data_loader, device, rank, world)
    try:
        slots = max(1, -(-len(data_loader) // world))
    except TypeError:
        slots = 64
    lib, dev_recs, host_recs, outputs = None, None, [], []
    criterion = torch.nn.CrossEntropyLoss()
    # An uncalibrated engine calibrates its activation scales on its first batch, which in one process is batch 0.
    # Every other rank, one that owns no batch too, runs batch 0 through the net first: then all ranks hold the same
    # scales, in this evaluation and in any unsharded one that follows (the sweep's candidates).
    calib0 = world > 1 and rank != 0 and torch.device(device).type == "cuda" and hasattr(net, "slq_calibrated")
    if calib0 and first is not None and n:
        _calibrate_on_batch0(net, device, first, hw0)
    n_seen = 0
    for bi, (x, y) in batches:
        n_seen = bi + 1
        if bi % world != rank:
            if bi == 0 and calib0:
                _calibrate_on_batch0(net, device, lambda: (x, y), tuple(x.shape[2:]))
            continue
        x, y = x.to(device), y.to(device)
        with torch.no_grad():
            out = net(x)
        ref = ref_outputs[bi] if ref_outputs is not None else None
        if _fused_tail_ok(out) and (ref is None or (_fused_tail_ok(ref) and ref.shape == out.shape)):
            k = len(outputs)
            if dev_recs is None or k == dev_recs.shape[0]:
                more = torch.zeros((slots, 4), dtype=torch.float64, device=out.device)
                dev_recs = more if dev_recs is None else torch.cat([dev_recs, more])
                lib = L.lib()
            B, C = out.shape
            y64 = y.to(torch.int64).contiguous()
            probs = torch.empty_like(out) if want_probs else None
            rows = torch.empty(3 * B, dtype=torch.float32, device=out.device)
            with torch.cuda.device(out.device):
                L.check(lib.slq_eval_tail(out.data_ptr(), y64.data_ptr(), B, C, L.ptr(probs), L.ptr(ref),
                                          rows.data_ptr(), dev_recs[k].data_ptr(), L.current_stream(out.device)))
        else:  # stock torch ops, the reference's per-batch values: (#correct, batch-mean CE, sum of KL, images)
            with torch.no_grad():
                probs = torch.softmax(out, dim=1)
                kl = (ref * (ref / probs).log()).sum(dim=1).sum() if ref is not None else out.new_zeros(())
                host_recs.append(torch.stack([(out.max(1)[1] == y).sum().double(), criterion(out, y).double(),
                                              kl.double(), out.new_tensor(float(y.numel()), dtype=torch.float64)]))
        outputs.append(probs)
    n = n_seen if n is None else n
    route = (_FUSED if dev_recs is not None else 0) | (_HOST if host_recs else 0)
    recs = dev_recs[:len(outputs)] if route == _FUSED else torch.stack(host_recs) if route == _HOST else None
    if world == 1:
        if recs is None or route == _FUSED | _HOST:
            _evaluation_error(route)
        a = recs.cpu().numpy()  # the one device->host read of the evaluation
    else:
        m = -(-n // world)  # batches per rank, the last ones padded
        C = outputs[0].shape[1] if outputs and want_probs else 0
        dtype = _PROB_DTYPES.index(outputs[0].dtype) if outputs and want_probs else 0
        send = torch.zeros((m + 1, 4), dtype=torch.float64, device=torch.device(device))
        if recs is not None:
            send[:len(outputs)] = recs.to(send.device)
        send[m] = torch.tensor([route, C, dtype, 0], dtype=torch.float64)
        gathered = torch.stack(_all_gather(send, dist, world)).cpu().numpy()  # the one device->host read
        route = int(np.bitwise_or.reduce(gathered[:, m, 0].astype(np.int64)))
        if route not in (_FUSED, _HOST):
            _evaluation_error(route)
        a = gathered[:, :m].transpose(1, 0, 2).reshape(-1, 4)[:n]  # row i = batch i (rank i % world, slot i // world)
        if want_probs:
            C, dtype = int(gathered[:, m, 1].max()), _PROB_DTYPES[int(gathered[:, m, 2].max())]
            sizes = a[:, 3].astype(np.int64)
            probs = torch.zeros((m, int(sizes.max()), C), dtype=dtype, device=torch.device(device))
            for k, p in enumerate(outputs):
                probs[k, :p.shape[0]] = p
            bufs = [b.to(probs.device) for b in _all_gather(probs, dist, world)]
            outputs = [bufs[i % world][i // world, :sizes[i]] for i in range(n)]
        else:
            outputs = [None] * n
    if route == _FUSED:
        s = [0.0, 0.0, 0.0, 0.0]  # the running accumulator of one process, fed the same records in the same order
        for rec in a.tolist():
            for j in range(4):
                s[j] += rec[j]
        acc = float(np.float32(s[0]) / np.float32(s[3]))
        loss = float(np.float32(s[1]) / np.float32(n))
        kl = float(np.float32(s[2] / s[3])) if ref_outputs is not None else None
        return acc, loss, outputs, kl
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)  # noqa: E731 -- the host records are fp32 values
    loss_sum, kl_sum = 0, None
    for rec in a.tolist():
        loss_sum = loss_sum + f32(rec[1])
        kl_sum = f32(rec[2]) if kl_sum is None else kl_sum + f32(rec[2])
    images = int(a[:, 3].sum())
    acc = f32(float(a[:, 0].sum())) / images  # an exact count, as the reference's sum of 0/1 floats
    kl = (kl_sum / images).item() if ref_outputs is not None else None
    return acc.item(), (loss_sum / n).item(), outputs, kl


def _evaluation_error(route):
    if route == _FUSED | _HOST:
        raise RuntimeError("evaluate: the loader mixed CUDA and host batches")
    raise RuntimeError("evaluate: the loader yielded no batches")


def evaluate_loss(net, device, data_loader):
    """Mean-of-batch-means cross-entropy (reference functions.py:45-82; unused by the mains).  Data-parallel over
    the ranks of a torch.distributed job like evaluate_acc_loss_softmax."""
    return _evaluate(net, device, data_loader, want_probs=False)[1]


def evaluate_acc_loss_softmax(net, device, data_loader):
    """-> (accuracy, mean-of-batch-means CE loss, [softmax per batch])  (reference functions.py:84-129).
    Under torch.distributed (world size > 1) each rank runs only the batches i with i % world == rank and every
    rank returns the full result, identical to a single process's; every rank must make the same calls."""
    acc, loss, outputs, _kl = _evaluate(net, device, data_loader)
    return acc, loss, outputs


def KLdiv(n_out, out):
    """Mean over samples of sum_c p*log(p/q), p = before, q = after (reference functions.py:131-149)."""
    if len(out) and all(_fused_tail_ok(p) and _fused_tail_ok(q) and p.shape == q.shape for p, q in zip(n_out, out)):
        lib = L.lib()
        dev = out[0].device
        accum = torch.zeros(4, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            for p, q in zip(n_out, out):
                B, C = q.shape
                rows = torch.empty(3 * B, dtype=torch.float32, device=dev)
                L.check(lib.slq_kl_rows(p.data_ptr(), q.data_ptr(), B, C, rows.data_ptr(), accum.data_ptr(),
                                        L.current_stream(dev)))
        a = accum.cpu().numpy()
        return float(np.float32(a[2] / a[3]))
    total, n = None, 0
    for p, q in zip(n_out, out):
        kl = (p * (p / q).log()).sum(dim=1)
        total = kl.sum() if total is None else total + kl.sum()
        n += kl.numel()
    return (total / n).item()


# ==============================================================================================
# semilayer bookkeeping
# ==============================================================================================
def make_divide_minusplusmodels(paramlists, dlists, index):
    """Splits channel rows into the 'minus' (deltaloss <= 0) and 'plus' semilayer lists; column 5
    becomes the per-layer sign flag 0,-1,-2,.. / 1,2,3,..  (reference functions.py:151-184)."""
    listminus, listplus = [], []
    mflag, pflag = 0, 1
    last = len(paramlists) - 1
    for i, p in enumerate(paramlists):
        if dlists[i][index] <= 0:
            listminus.append([p[0], p[1], p[2], p[3], p[4], mflag, p[6], p[7]])
        else:
            listplus.append([p[0], p[1], p[2], p[3], p[4], pflag, p[6], p[7]])
        if i == last:
            print('function debug:number of total channels=', len(listminus) + len(listplus),
                  'No.1:', len(listminus), 'No.2:', len(listplus))
            break
        if p[2] != paramlists[i + 1][2]:
            mflag -= 1
            pflag += 1
    return listminus, listplus


_CONVS_PER_BLOCK = {"resnet18": 2, "resnet34": 2, "resnet50": 3}


def _conv_of(arch, block, lnum):
    """Layer number -> conv module inside its block (functions.py:236-242 / :504-512)."""
    cpb = _CONVS_PER_BLOCK[arch]
    return getattr(block, "conv%d" % ((lnum - 1) % cpb + 1))


def _dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


def _semilayer_runs(listminus, listplus):
    """Candidates = runs of equal layer number inside each (sentinel-terminated) list."""
    semilayers = []
    for lst in (listminus, listplus):
        cur = []
        for i, row in enumerate(lst):
            if row[2] == 100:
                break
            cur.append(list(row[:8]))
            if row[2] != lst[i + 1][2]:
                semilayers.append(cur)
                cur = []
    return semilayers


def _gather_values(values, flags, dist, world):
    """ONE all_gather of [values | error flags]; entry i comes from its owner rank i % world."""
    bufs = _all_gather(torch.cat([values, flags]), dist, world)
    n = values.numel()
    for index in range(n):
        src = bufs[index % world].cpu()
        values[index] = src[index]
        flags[index] = src[n + index]
    # a rank may also have failed outside its own candidates (candidate 0 runs everywhere)
    for src in bufs:
        flags[:] = torch.maximum(flags, src.cpu()[n:])


def make_semilayers(arch, net, device, originaloutputs, listminus, listplus, metric=None, shard=True):
    """Sensitivity sweep (reference functions.py:186-588, three copies): one candidate per semilayer
    = quantise its channels on fresh pretrained weights, evaluate the whole loader, sensitivity =
    KL(before, after) / sum(numel * (32-bit)/32).

    Candidates are independent, so with torch.distributed initialised they are dealt round-robin
    to the ranks and the per-candidate values are exchanged with ONE all_gather (SURVEY.md 8e);
    every rank returns the full ``(semilayers, orders)``.

    "Fresh pretrained weights" (the reference builds a new ``resnetXX(pretrained='imagenet')`` per candidate,
    functions.py:258/393/528) is ONE work model per call here: the candidate's conv tensors are saved on the
    device, quantised in place, evaluated and restored, so a candidate costs its forward passes plus the
    re-packing of the one or two layers it touched; the work model shares the caller's activation scales.
    Candidate 0 runs on the CALLER's net object and mutates it (reference quirk Q3), on every rank.

    metric: 'kl' (reference) or 'dloss' (loss_candidate - loss_base; KL is NaN for random-init
    R34/R50, SURVEY.md Q10).  Default from $SLQ_SWEEP_METRIC, else 'kl'.
    A candidate that raises (e.g. ZeroDivisionError for a constant channel) does not strand the other ranks
    in the collective: the error is flagged, every rank reaches the all_gather, then every rank raises."""
    metric = metric or os.environ.get("SLQ_SWEEP_METRIC", "kl")
    dist, rank, world = _dist() if shard else (None, 0, 1)
    listminus.append(list(SENTINEL))  # the reference mutates the caller's lists the same way
    listplus.append(list(SENTINEL))
    semilayers = _semilayer_runs(listminus, listplus)
    factory = getattr(resnet, arch)
    # delta-loss needs the un-quantised loss from logits (the stored softmax underflows to exact zeros on
    # random-init R34/R50, which is what makes KL NaN there): one more evaluation of the caller's net,
    # before candidate 0 mutates it
    base = _evaluate(net, device, imagenet.val_loader, want_probs=False, shard=False)[1] if metric == "dloss" else None
    values = torch.zeros(len(semilayers), dtype=torch.float64)
    flags = torch.zeros(len(semilayers), dtype=torch.float64)
    work, first_error = None, None
    # When the caller's net IS the pretrained model (the mains' case: resnet50_main.py:41-46 builds it and passes it
    # in), "a fresh pretrained model" for candidates 1.. is the caller's net with candidate 0's layer put back: no
    # second model, no second engine (0.55 s of set-up per rank).  Candidate 0's quantised weights are re-applied at
    # the end, so the caller's net leaves exactly as the reference leaves it (quirk Q3).
    reuse_net = len(semilayers) > 1 and _is_pretrained(arch, net, device)
    cand0_quantised = []
    for index, rows in enumerate(semilayers):
        mine = (index % world) == rank
        if not mine and index != 0:
            continue
        saved = []
        try:
            if index == 0 or reuse_net:
                cand = net
            else:
                if work is None:
                    # built ON the device: the constructor's random init (overwritten by the pretrained state dict
                    # right away) costs 0.5-0.7 s on the host for ResNet-50 -- a third of an 8-GPU sweep
                    with torch.device(device if torch.device(device).type == "cuda" else "cpu"):
                        work = factory(num_classes=1000, pretrained='imagenet')
                    if hasattr(work, "slq_share_calibration"):
                        work.slq_share_calibration(net)
                    work.to(device)
                cand = work
            layers = [cand.layer1, cand.layer2, cand.layer3, cand.layer4]
            param = 0.0
            by_conv = {}
            for li, bi, lnum, cnum, w_bit, _flag, _sel, _gi in rows:
                conv = _conv_of(arch, layers[li][bi], lnum)
                by_conv.setdefault(id(conv), (conv, [], []))
                by_conv[id(conv)][1].append(cnum)
                by_conv[id(conv)][2].append(w_bit)
                param += conv.weight[cnum].data.numel() * ((32 - w_bit) / 32)
            for conv, chans, bits in by_conv.values():
                if cand is work or reuse_net:
                    saved.append((conv, conv.weight.data.clone()))
                # a semilayer's rows are distinct channels of one conv: one launch, same result as the
                # reference's per-channel loop
                conv.weight.data = _quantize_channels(conv.weight.data, chans, bits)
            if mine:
                want_kl = metric == "kl"
                _acc, loss, _after, kl = _evaluate(cand, device, imagenet.val_loader,
                                                   ref_outputs=originaloutputs if want_kl else None,
                                                   want_probs=False, shard=False)
                val = (loss - base) if metric == "dloss" else kl / param
                values[index] = val
                print(rows[0][4], 'bit', 'semilayer-No.', index, 'layernumber=', rows[0][2], 'channels=', len(rows),
                      'total KL divergence=' if metric == "kl" else 'delta loss=', val)
        except Exception as e:  # keep walking: the collective below must be reached by every rank
            flags[index] = 1.0
            first_error = first_error or e
        finally:
            if index == 0 and reuse_net:  # what candidate 0 left in the caller's net: re-applied after the sweep
                cand0_quantised = [(conv, conv.weight.data.clone()) for conv, _orig in saved]
            for conv, orig in saved:  # back to the pretrained weights for the next candidate
                conv.weight.data.copy_(orig)
                resnet.note_weight_write(conv.weight.data)
    for conv, q in cand0_quantised:
        conv.weight.data.copy_(q)
        resnet.note_weight_write(conv.weight.data)
    if world > 1:
        _gather_values(values, flags, dist, world)
    if bool(flags.any()):
        bad = [int(i) for i in flags.nonzero().flatten()]
        if first_error is not None:
            raise first_error
        raise RuntimeError("sensitivity sweep: candidates %s failed on another rank" % bad)
    orders = [[i, float(values[i])] for i in range(len(semilayers))]
    return semilayers, orders


def _is_pretrained(arch, net, device):
    """True iff every tensor of net's state dict equals the pretrained one the factories load
    (resnet.load_state_dict_from_url(resnet.model_urls[arch])), bit for bit, compared on the device."""
    try:
        sd = resnet.load_state_dict_from_url(resnet.model_urls[arch], progress=True)
        mine = net.state_dict()
        if set(sd.keys()) != set(mine.keys()):
            return False
        dev = torch.device(device)
        same = True
        for k, v in sd.items():
            m = mine[k]
            if m.device.type != dev.type or m.shape != v.shape or m.dtype != v.dtype:
                return False
            same = same and bool(torch.equal(m, v.to(m.device)))
            if not same:
                return False
        return True
    except Exception:
        return False


def _quantize_channels(weight, chans, bits):
    if weight.is_contiguous() and weight.dtype == torch.float32:
        quantize_rows(weight, chans, bits, write_back=True, want_codes=False)
        return weight
    for c, b in zip(chans, bits):
        weight = channel_wise_quantizationperchan(weight, b, c)
    return weight


def make_semilayers_resnet18(net, device, originaloutputs, listminus, listplus):
    return make_semilayers("resnet18", net, device, originaloutputs, listminus, listplus)


def make_semilayers_resnet34(net, device, originaloutputs, listminus, listplus):
    return make_semilayers("resnet34", net, device, originaloutputs, listminus, listplus)


def make_semilayers_resnet50(net, device, originaloutputs, listminus, listplus):
    return make_semilayers("resnet50", net, device, originaloutputs, listminus, listplus)


# ==============================================================================================
# accept / undo state and the packed model format (SURVEY.md 8f: N2, N4)
# ==============================================================================================
def snapshot(net):
    """Device-resident replacement of ``torch.save(net.state_dict(), pthname)`` (resnet50_main.py:212):
    quantised layers are kept as packed codes (slq_store.Snapshot), nothing touches the file system."""
    import slq_store
    return slq_store.snapshot(net)


def restore(net, snap):
    """Replacement of ``net.load_state_dict(torch.load(pthname))`` (resnet50_main.py:233-234)."""
    import slq_store
    return slq_store.restore(net, snap)


def save_packed(net, path):
    import slq_store
    return slq_store.save_packed(net, path)


def load_packed(path, net):
    import slq_store
    return slq_store.load_packed(path, net)


# ==============================================================================================
# delta-loss table generator (SURVEY.md 8f: N3)
# ==============================================================================================
_LAYER_DEPTHS = {"resnet18": [2, 2, 2, 2], "resnet34": [3, 4, 6, 3], "resnet50": [3, 4, 6, 3]}


def quantized_convs(arch, net):
    """[(layer number 1.., conv module)] in the order of the reference's tables (dataset/*_deltaloss.csv row 0;
    resnet50_main.py:81-136: block = (lnum-1)//convs_per_block in flattened stage order)."""
    cpb = _CONVS_PER_BLOCK[arch]
    blocks = [b for stage in (net.layer1, net.layer2, net.layer3, net.layer4) for b in stage]
    return [(i * cpb + j + 1, getattr(b, "conv%d" % (j + 1))) for i, b in enumerate(blocks) for j in range(cpb)]


def make_deltaloss_table(arch, net, device, data_loader, bits=(8, 6, 4), layers=None, channels=None, shard=True):
    """Regenerates the per-channel sensitivity table the reference ships as ``dataset/<arch>_deltaloss.csv``
    but cannot rebuild (its generator is the dead helper ``evaluate_loss``, functions.py:45-82):
    for every output channel c of every quantised conv layer and every bit-width b,
        deltaloss[b][c] = loss(net with ONLY channel c fake-quantised to b bits from fp32) - loss(net).
    One candidate = one row through the quantizer kernel + one pass over the loader; the row is restored
    from a device copy afterwards.  Candidates are dealt round-robin over the torch.distributed ranks and
    exchanged with ONE all_gather, like the semilayer sweep (22,656 x 3 candidates for ResNet-50).
    layers: iterable of layer numbers (default all); channels: callable(lnum, Cout) -> iterable of channel
    indices (default all).  Returns (lnums, cnums_1based, {bit: [deltaloss...]}) in table column order."""
    dist, rank, world = _dist() if shard else (None, 0, 1)
    net.to(device)
    net.eval()
    base = _evaluate(net, device, data_loader, want_probs=False, shard=False)[1]
    cols = []
    for lnum, conv in quantized_convs(arch, net):
        if layers is not None and lnum not in layers:
            continue
        chans = range(conv.out_channels) if channels is None else channels(lnum, conv.out_channels)
        cols += [(lnum, conv, int(c)) for c in chans]
    values = torch.zeros(len(cols) * len(bits), dtype=torch.float64)
    flags = torch.zeros_like(values)
    first_error = None
    for ci, (lnum, conv, c) in enumerate(cols):
        if ci % world != rank:
            continue
        w = conv.weight.data
        keep = w[c].clone()
        for bi, b in enumerate(bits):
            try:
                quantize_rows(w, [c], [b], write_back=True, want_codes=False)
                loss = _evaluate(net, device, data_loader, want_probs=False, shard=False)[1]
                values[ci * len(bits) + bi] = loss - base
            except Exception as e:
                flags[ci * len(bits) + bi] = 1.0
                first_error = first_error or e
            finally:
                w[c].copy_(keep)
                resnet.note_weight_write(w)
    if world > 1:
        _gather_values(values, flags, dist, world)
    if bool(flags.any()):
        if first_error is not None:
            raise first_error
        raise RuntimeError("delta-loss table: %d candidates failed on another rank" % int(flags.sum()))
    v = values.reshape(len(cols), len(bits)).numpy()
    return [c[0] for c in cols], [c[2] + 1 for c in cols], {int(b): v[:, i].tolist() for i, b in enumerate(bits)}


def write_deltaloss_csv(path, lnums, cnums, table, bits=(8, 6, 4)):
    """Writes the table in the reference's layout (resnet50_main.py:59-79 reads it back): UTF-8 with BOM,
    row 0 layer numbers, row 1 1-based channel numbers, then one row of delta-loss values per bit-width."""
    import csv
    with open(path, "w", encoding="utf-8-sig", newline="") as f:
        wr = csv.writer(f)
        wr.writerow(lnums)
        wr.writerow(cnums)
        for b in bits:
            wr.writerow([repr(float(x)) for x in table[int(b)]])


def make_quantizedlists(semilayers, orders):
    """Least-sensitive semilayer first: sorts ``orders`` in place by sensitivity and flattens the
    semilayers in that order, sentinel-terminated (reference functions.py:590-612)."""
    orders.sort(key=lambda o: o[1])
    flat = []
    for idx, _sens in orders:
        flat.extend(list(r[:8]) for r in semilayers[idx])
        print('debug layernum=', semilayers[idx][-1][2], 'number of channels=', len(semilayers[idx]))
    print('number of valuationfirsts list=', len(flat))
    flat.append(list(SENTINEL))
    return flat
