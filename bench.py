#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 hot path (BASELINE.json metric):
ResNet-50 semilayer-wise mixed 8/4-bit inference, batch 256 per GPU, synthetic 224x224 images,
random-init weights, policy-P0 bit assignment derived from the reference's delta-loss table.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own path on the host CPU cores
    python bench.py ... --dump-outputs DIR    # also writes the last timed step's logits to DIR/logits.npy

A "step" is one forward pass of one batch (256 images per GPU) through the whole hot path:
stem -> 52 quantised/fp32-weight convs on tcgen05 (fused dequant+BN+residual+ReLU epilogues)
-> avgpool+fc.  `value` has the inputs resident in HBM; `e2e` goes through the public call
`net(x)` with pinned-host inputs copied H2D and logits copied D2H inside the timed region.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "semilayer-wise-mixed-precision-quantization_b200")
sys.path.insert(0, PKG)
DUMP_LIMIT_BYTES = 64 << 20

METRIC = "ResNet-50 mixed 8/4-bit images/s"


def metric_name(arch):  # BASELINE.json's metric; the other architectures are parity / side configurations
    return METRIC.replace("ResNet-50", {"resnet18": "ResNet-18", "resnet34": "ResNet-34"}.get(arch, "ResNet-50"))
UNIT = "images/s"
GOP_PER_IMG = {"resnet50": 8.178, "resnet34": 7.328, "resnet18": 3.628}  # 2*MAC, convs + fc (SURVEY 8d)
ALGO_MB_PER_IMG = {"resnet50": 27.84, "resnet34": 9.17, "resnet18": 6.22}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, bf16=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """Timed region starts here: samples taken before this call (warm-up) are dropped, except
        the last one, so that even a region shorter than the sampling period has a reading."""
        self.rows = self.rows[-1:]

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _p0_rows(arch):
    import numpy as np
    return np.load(os.path.join(PKG, "data", "p0_bits.npz"))[arch]


def cpu_reference_forward(arch, batch, reps, threads=None):
    """The reference's path on the host cores: fp32 fake-quant forward of the same P0 model.

    kind "reference": the UNMODIFIED reference modules staged under oracle/_ref (oracle/make_ref.py: byte
    copies of /root/reference/{resnet,functions}.py) -- ``resnet.resnet50`` builds the model,
    ``functions.channel_wise_quantizationperchan`` applies the P0 bit assignment row by row and
    ``net(x)`` (resnet.py:204-223) is what is timed.  If oracle/_ref is not there, kind "port": the oracle's
    call-for-call restatement on stock torch ops.  Returns (times, threads, kind)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    if threads:
        torch.set_num_threads(threads)
    table = _p0_rows(arch)
    cpb = 3 if arch == "resnet50" else 2
    g = torch.Generator().manual_seed(1)
    x = torch.randn(batch, 3, 224, 224, generator=g)
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    kind = "reference" if os.path.isfile(os.path.join(ref_dir, "resnet.py")) else "port"
    if kind == "reference":
        import importlib
        import types
        saved = {k: sys.modules.pop(k, None) for k in ("functions", "resnet", "imagenet")}
        stub = types.ModuleType("imagenet")
        stub.val_loader, stub.train_loader = [], None
        sys.modules["imagenet"] = stub
        sys.path.insert(0, ref_dir)
        try:
            r_resnet = importlib.import_module("resnet")
            r_functions = importlib.import_module("functions")
            assert os.path.dirname(os.path.abspath(r_functions.__file__)) == ref_dir
            torch.manual_seed(0)
            net = getattr(r_resnet, arch)(num_classes=1000).eval()
            blocks = [b for s in (net.layer1, net.layer2, net.layer3, net.layer4) for b in s]
            for lnum, cn, bit in table:
                conv = getattr(blocks[(lnum - 1) // cpb], "conv%d" % ((lnum - 1) % cpb + 1))
                conv.weight.data = r_functions.channel_wise_quantizationperchan(conv.weight.data, int(bit), int(cn))
            fwd = lambda: net(x)
        finally:
            sys.path.remove(ref_dir)
            for k in ("functions", "resnet", "imagenet"):
                sys.modules.pop(k, None)
                if saved[k] is not None:
                    sys.modules[k] = saved[k]
    else:
        import slq_oracle as so
        import resnet
        torch.manual_seed(0)
        net = getattr(resnet, arch)(num_classes=1000).eval()
        blocks = [b for s in (net.layer1, net.layer2, net.layer3, net.layer4) for b in s]
        for lnum, cn, bit in table:  # oracle quantizer: the CPU restatement of functions.py:9-43
            conv = getattr(blocks[(lnum - 1) // cpb], "conv%d" % ((lnum - 1) % cpb + 1))
            so.channel_wise(conv.weight.data.reshape(conv.out_channels, -1).numpy(), int(bit), int(cn))
        fwd = lambda: so.torch_forward(net, x)
    with torch.no_grad():
        fwd()  # warm-up
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fwd()
            times.append(time.perf_counter() - t0)
    return times, torch.get_num_threads(), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = args.ref_batch
    # all the host threads this process may use: torchrun pins OMP_NUM_THREADS=1 per rank, and only rank 0
    # runs this arm, so take the cores of its affinity mask instead
    try:
        threads = len(os.sched_getaffinity(0))
    except AttributeError:
        threads = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = os.environ["MKL_NUM_THREADS"] = str(threads)  # before torch is imported
    times, threads, kind = cpu_reference_forward(args.arch, batch, args.steps + args.warmup, threads=threads)
    times = times[args.warmup:] if len(times) > args.warmup else times
    total = sum(times)
    val = batch * len(times) / total
    line = {
        "metric": metric_name(args.arch), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": "%s semilayer 8/4-bit (P0) inference, synthetic 224x224, random-init" % args.arch,
                   "sample": "batch %d per step on the host CPU" % batch, "batch_per_gpu": args.batch},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": "%d fp32 forwards of batch %d through %s (torch %s CPU)" %
                                   (len(times), batch, "the unmodified reference's resnet.ResNet.forward (oracle/_ref)"
                                    if kind == "reference" else "the oracle's restatement of it", __import__("torch").__version__)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def bind_to_gpu_numa_node(local):
    """Binds this process to the cores of the NUMA node its GPU hangs off BEFORE any pinned buffer is
    allocated (first touch then places the pages on that node), so that the host side of the per-step
    fp32 upload does not cross the inter-socket link.  Returns a short description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return {"numa_node": node, "bound": False, "why": "no NUMA affinity reported for the GPU"}
        cpulist = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        cpus = set()
        for part in cpulist.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = sorted(cpus & allowed)
        if not use:
            return {"numa_node": node, "bound": False, "why": "none of node %d's cores are in this process's affinity mask" % node}
        os.sched_setaffinity(0, use)
        nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
        return {"numa_node": node, "numa_nodes": nodes, "bound": True, "cores": len(use)}
    except Exception as e:  # sysfs layout differs / no permission: run unbound
        return {"bound": False, "why": "%s: %s" % (type(e).__name__, e)}


def dump_logits(out_dir, logits, rank, world):
    """Writes one rank's logits [batch, classes] as float32 .npy.  The files of all ranks together stay under
    DUMP_LIMIT_BYTES: past that, a fixed seeded sample of the rows (the same rows on every run) is written."""
    import numpy as np
    cap = max(1, DUMP_LIMIT_BYTES // world // (4 * logits.shape[1]))
    if logits.shape[0] > cap:
        logits = logits[np.sort(np.random.default_rng(0).choice(logits.shape[0], cap, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    name = "logits.npy" if world == 1 else "logits_rank%d.npy" % rank
    np.save(os.path.join(out_dir, name), np.ascontiguousarray(logits, dtype=np.float32))


def measure_i8_peak(lib, L, st, torch):
    """Dense kind::i8 tensor rate of THIS GPU (slq_probe_i8_peak: every SM streams M128 x N256 x K32 MMAs):
    burst = best of 5 launches of ~20 ms; sustained = one >= 2 s train of launches."""
    import ctypes
    ops = ctypes.c_int64(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 40000
    L.check(lib.slq_probe_i8_peak(4000, ctypes.byref(ops), st.cuda_stream))  # warm-up (smem opt-in, clocks)
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(5):
        e0.record(st)
        L.check(lib.slq_probe_i8_peak(iters, ctypes.byref(ops), st.cuda_stream))
        e1.record(st)
        torch.cuda.synchronize()
        best = max(best, ops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    n = max(1, int(2.2 / (ops.value / (best * 1e12))))
    e0.record(st)
    for _ in range(n):
        L.check(lib.slq_probe_i8_peak(iters, ctypes.byref(ops), st.cuda_stream))
    e1.record(st)
    torch.cuda.synchronize()
    secs = e0.elapsed_time(e1) * 1e-3
    return {"burst_tops": best, "sustained_tops": n * ops.value / secs / 1e12, "sustained_seconds": secs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arch", default="resnet50")
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--ref-batch", type=int, default=32, help="images per step of the CPU reference arm")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-agree", action="store_true", help="skip the fp32 agreement check (torch kernels)")
    ap.add_argument("--simt", action="store_true", help="run the dp4a checker kernels instead (debug)")
    ap.add_argument("--layers", default="", help="write the per-layer CUDA-event table to this file")
    ap.add_argument("--no-packed-b", action="store_true",
                    help="A/B: resident-weight layers take u8 weight tiles through TMA instead of packed codes unpacked in smem")
    ap.add_argument("--no-fuse-tail", action="store_true",
                    help="A/B: downsample conv and conv3 of a stage's first block as two launches (identity through HBM)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the logits of the last timed step to DIR/logits.npy (float32; "
                         "logits_rank<r>.npy per rank with several GPUs) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)  # before the first pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import slq_build
    slq_build.build()
    import functions
    import resnet
    import slq_engine
    import slq_lib as L

    # ---- model: seeded random init + P0 8/4-bit assignment through the product quantizer --------
    torch.manual_seed(0)
    net = getattr(resnet, args.arch)(num_classes=1000).to(dev).eval()
    table = np.load(os.path.join(PKG, "data", "p0_bits.npz"))[args.arch]
    cpb = 3 if args.arch == "resnet50" else 2
    blocks = [b for s in (net.layer1, net.layer2, net.layer3, net.layer4) for b in s]
    convs = dict(functions.quantized_convs(args.arch, net))
    items = [(convs[int(l)].weight.data, table[table[:, 0] == l][:, 1], table[table[:, 0] == l][:, 2])
             for l in np.unique(table[:, 0])]
    # ---- quantizer (HBM-bound): the whole P0 assignment of the model in ONE launch ----------------
    # Timed like a kernel in isolation: CUDA events around the launch, L2 flushed before every repetition
    # (the 83 MB of weights would otherwise sit in the 126 MB L2), median of 5.  Every repetition re-quantises
    # fp32 rows in place (the first from the random-init weights, the others from fake-quantised values:
    # the same reads, arithmetic and writes, SURVEY.md F6).
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    qe = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
    fresh = [t.clone() for t, _r, _b in items]
    functions.quantize_model([(torch.randn(8, 64, device=dev), [0, 1], [8, 4])])  # module load / first launch
    # allocator warm-up: the same call on copies of the weights, so that the timed call below does not pay the
    # cudaMallocs of its 15 MB code blob and job table (2.5 ms with a warm allocator, up to 18 ms cold)
    functions.quantize_model([(f.clone(), r, b) for (t, r, b), f in zip(items, fresh)], div_mode=L.DIV_TRUE)
    torch.cuda.synchronize()
    tq0 = time.perf_counter()
    pm = functions.quantize_model(items, div_mode=L.DIV_TRUE)  # wall clock incl. job table, H2D, status check
    quant_ms = 1e3 * (time.perf_counter() - tq0)
    packed_bytes = pm.nbytes
    keep_first = [t.clone() for t, _r, _b in items]  # the model the rest of the run uses: quantised ONCE from fp32
    q_times = []
    for a_, b_ in qe:
        for (t, _r, _b), f in zip(items, fresh):
            t.copy_(f)
        flush.zero_()
        a_.record(torch.cuda.current_stream(dev))
        pm.run()  # the prepared plan: ONE launch, no host work between the events
        b_.record(torch.cuda.current_stream(dev))
        torch.cuda.synchronize()
        q_times.append(a_.elapsed_time(b_))
    tq0 = time.perf_counter()
    pm.run().check()  # what a greedy step pays: the prepared plan again + the one status read-back, wall clock
    quant_replay_ms = 1e3 * (time.perf_counter() - tq0)
    for (t, _r, _b), f in zip(items, keep_first):
        t.copy_(f)
    del fresh, keep_first
    q_ms = statistics.median(q_times)
    n_w = sum(int(len(r)) * t[0].numel() for t, r, _b in items)
    q_bytes = 4 * n_w * 2 + packed_bytes + 12 * len(table)  # fp32 rows read + written back, codes, z/s32/status
    peaks0 = load_peaks()
    roofline_q = {"bound": "hbm", "achieved": q_bytes / (q_ms * 1e-3) / 1e9, "peak": peaks0["hbm"], "unit": "GB/s",
                  "frac": q_bytes / (q_ms * 1e-3) / 1e9 / peaks0["hbm"], "traffic": None,
                  "kernel": "quantize_jobs_kernel: all %d (row, bit) jobs of the %d quantised convs in one launch, "
                            "CUDA events on the launching stream, L2 flushed, median of 5" % (len(table), len(items)),
                  "algorithmic_bytes": q_bytes, "us": 1e3 * q_ms, "us_all": [1e3 * v for v in q_times],
                  "peak_source": "%s copy bandwidth (MEASURED_PEAKS.json)" % peaks0["src"]}

    B = args.batch
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    x = torch.randn(B, 3, 224, 224, generator=g, device=dev)
    x_host = x.cpu().pin_memory()
    impl = L.IMPL_SIMT if args.simt else L.IMPL_UMMA
    eng = net.slq_engine(x, impl=impl, packed_b=not args.no_packed_b, fuse_tail=not args.no_fuse_tail)
    eng.refresh_weights()
    eng.calibrate(x)
    eng.epoch = resnet.WEIGHT_EPOCH[0]
    net._slq_dirty = False
    logits = eng.forward(x).clone()
    torch.cuda.synchronize()

    # ---- accuracy side-channel: agreement with the fp32 torch restatement (not timed) -----------
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    agree = rel = None
    try:
        if args.no_agree:
            raise RuntimeError("skipped")
        import slq_oracle as so
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        nb = min(B, 64)
        ref = so.torch_forward(net, x[:nb])
        agree = float((ref.argmax(1) == logits[:nb].argmax(1)).float().mean())
        rel = float((ref - logits[:nb]).norm() / ref.norm())
    except Exception as e:  # the checker is optional here
        agree, rel = None, "unavailable: %s" % type(e).__name__

    use_graph = not args.no_graph
    if use_graph:
        try:
            eng.capture_graph(x)
        except Exception as e:
            print("graph capture failed (%s); timing direct launches" % e, file=sys.stderr)
            use_graph = False
    st = torch.cuda.current_stream(dev)

    def step():
        if use_graph:
            eng.graph.replay()
        else:
            eng.launch_all(x.data_ptr(), st.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for i in range(args.steps):
        if not use_graph and i == args.steps - 1:  # profiling hook: ncu --nvtx --nvtx-include "slq_step/"
            torch.cuda.nvtx.range_push("slq_step")
            step()
            torch.cuda.nvtx.range_pop()
        else:
            step()
    e1.record(st)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:  # before the e2e loops below overwrite the engine's logits buffer
        dump_logits(args.dump_outputs, eng.logits.cpu().numpy(), rank, world)
    ms = e0.elapsed_time(e1)
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    value = world * B * args.steps / (ms * 1e-3)

    # ---- e2e: the public call net(x) with host buffers: H2D + forward + D2H every step ---------
    # The loader-side pattern of the reference (functions.py:110-113: inputs.to(device); net(inputs))
    # with pinned memory and a copy stream: batch i+1 crosses PCIe while batch i computes; every
    # step's logits come back to the host (a blocking read), so nothing is deferred past the region.
    # as many steps as the headline loop (--steps); with only one or two, the figure is mostly the time to fill
    # the copy pipeline
    e2e_steps = args.steps
    copy_stream = torch.cuda.Stream(dev)
    NB = 3  # input buffers: the copy engine always has the next batch queued behind the one in flight
    dbuf = [torch.empty_like(x) for _ in range(NB)]
    landed = [torch.cuda.Event() for _ in range(NB)]
    out_pinned = torch.empty((B, net.fc.out_features), dtype=torch.float32).pin_memory()
    out_done = torch.cuda.Event()

    def e2e_loop(n, src=None, bufs=None):
        src = x_host if src is None else src
        bufs = dbuf if bufs is None else bufs

        def fetch(i):  # host -> device copy of step i's input on the copy stream
            with torch.cuda.stream(copy_stream):
                bufs[i % NB].copy_(src, non_blocking=True)
                landed[i % NB].record(copy_stream)

        fetch(0)
        if n > 1:
            fetch(1)
        out = None
        for i in range(n):
            st.wait_event(landed[i % NB])     # step i's input has landed
            if i + 2 < n:
                fetch(i + 2)                  # bufs[(i+2)%3] was last read by step i-1, which has finished
            logits_i = net(bufs[i % NB])      # forward (one CUDA graph replay)
            out_pinned.copy_(logits_i, non_blocking=True)  # D2H of the logits into pinned memory ...
            out_done.record(st)
            out_done.synchronize()            # ... and the host waits for exactly that event, every step
            out = out_pinned
        return out

    e2e_loop(2 * NB)  # every input buffer seen twice: its forward is a captured graph from here on
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(st)
    out_host = e2e_loop(e2e_steps)
    t1.record(st)
    barrier()
    e2e_ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_val = world * B * e2e_steps / (float(e2e_ms.item()) * 1e-3)

    # copy-only probe: the same pinned fp32 batch, the same copy stream, nothing else running on this rank --
    # what the host side of the upload can deliver per GPU when all ranks copy at once (max over ranks of
    # the time, like every multi-GPU number here)
    barrier()
    p0_, p1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(copy_stream):
        p0_.record(copy_stream)
        for i in range(8):
            dbuf[i % NB].copy_(x_host, non_blocking=True)
        p1_.record(copy_stream)
    barrier()
    h2d_ms = torch.tensor([p0_.elapsed_time(p1_)], device=dev)
    if world > 1:
        dist.all_reduce(h2d_ms, op=dist.ReduceOp.MAX)
    h2d_gbs = 8 * x_host.numel() * 4 / (float(h2d_ms.item()) * 1e-3) / 1e9

    # the same loop with the loader-side formats the stem also accepts (not the headline: the reference's
    # loader hands over fp32): the batch as fp16 (bit-identical logits) and as raw u8 pixels (normalised in
    # the stem kernel); same engine, same static scales
    import imagenet
    e2e_alt = {}
    net.input_norm = (imagenet.MEAN, imagenet.STD)
    for name, src in (("fp16", x_host.half().pin_memory()),
                      ("u8", torch.randint(0, 256, tuple(x.shape), dtype=torch.uint8).pin_memory())):
        bufs = [torch.empty(tuple(x.shape), dtype=src.dtype, device=dev) for _ in range(NB)]
        e2e_loop(2 * NB, src, bufs)
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(st)
        e2e_loop(e2e_steps, src, bufs)
        a1.record(st)
        barrier()
        tm = torch.tensor([a0.elapsed_time(a1)], device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e_alt[name] = {"value": world * B * e2e_steps / (float(tm.item()) * 1e-3), "unit": UNIT,
                         "h2d_bytes_per_step": int(src.numel() * src.element_size())}
        del bufs

    # ---- roofline of the dominant kernel (conv_umma_kernel), timed live per launch -------------
    peaks = load_peaks()
    conv_ms, conv_ops, conv_bytes = 0.0, 0.0, 0.0
    sched = list(eng.schedule)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in sched]
    torch.cuda.synchronize()
    for rep in range(3):
        for (a, b), item in zip(ev, sched):
            a.record(st)
            eng.launch_item(item, st.cuda_stream)
            b.record(st)
        torch.cuda.synchronize()
    per_layer = []
    for (a, b), item in zip(ev, sched):
        t = a.elapsed_time(b)
        info = eng.item_info(item)
        conv_ms += t
        conv_ops += info["ops"]
        conv_bytes += info["bytes"]
        per_layer.append((t, info))
    if args.layers and rank == 0:
        with open(args.layers, "w") as f:
            f.write("idx kind Cin Cmid Cout k s H M w16 res  us  TOPS  GB/s\n")
            for i, (t, d) in enumerate(per_layer):
                f.write("%2d %s %4d %4d %4d %d %d %3d %7d %d %d  %7.1f %7.1f %7.1f\n" % (
                    i, d["kind"], d["Cin"], d["Cmid"], d["Cout"], d["k"], d["stride"], d["H"], d["M"], d["w16"], d["res"],
                    1e3 * t, d["ops"] / (t * 1e-3) / 1e12, d["bytes"] / (t * 1e-3) / 1e9))
    achieved_tops = conv_ops / (conv_ms * 1e-3) / 1e12
    i8 = measure_i8_peak(eng.lib, L, st, torch)
    # the conv launches above are timed one by one, in isolation (a few ms in total): the BURST figure applies
    int8_peak = i8["burst_tops"]
    bf16_burst = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops") if peaks["src"] == "measured" else 1590.0
    # DRAM traffic of the same launches from the committed `ncu --set full` capture of one step
    traffic = None
    prof = os.path.join(ROOT, "profiles", "r2_ncu_full_step_summary.csv")
    if not os.path.exists(prof):
        prof = os.path.join(ROOT, "profiles", "r1_ncu_full_step_summary.csv")
    if args.arch == "resnet50" and B == 256 and os.path.exists(prof):
        import csv
        rows = [r for r in csv.DictReader(open(prof)) if "conv_umma" in r["kernel"] or "block_tail" in r["kernel"]]
        if len(rows) == len(sched):
            traffic = 1e6 * sum(float(r["dram_rd_MB"]) + float(r["dram_wr_MB"]) for r in rows) / len(rows)
    roofline = {"bound": "tensor", "achieved": achieved_tops, "peak": int8_peak, "unit": "TFLOP/s",
                "frac": achieved_tops / int8_peak, "traffic": traffic,
                "traffic_note": "mean DRAM bytes (read+write) per conv launch, %s; "
                                "algorithmic mean %.1f MB" % (os.path.relpath(prof, ROOT), conv_bytes / len(sched) / 1e6),
                "kernel": "conv_umma_kernel / block_tail_kernel: the %d conv launches of a step (%d of them fused block "
                          "tails = downsample conv + conv3), each timed with CUDA events on the launching stream; "
                          "achieved = sum(2*MAC) / sum(duration)" % (len(sched), sum(1 for k, _ in sched if k == "tail")),
                "peak_source": "measured i8: slq_probe_i8_peak on this GPU in this run, burst (best of 5 x ~20 ms); "
                               "sustained over %.1f s: %.0f TOPS" % (i8["sustained_seconds"], i8["sustained_tops"]),
                "peak_sustained": i8["sustained_tops"], "frac_vs_sustained_i8": achieved_tops / i8["sustained_tops"],
                "frac_vs_2x_bf16_burst": achieved_tops / (2.0 * bf16_burst),
                "whole_step_frac": (value / world) * GOP_PER_IMG[args.arch] * 1e9 / (i8["sustained_tops"] * 1e12),
                "whole_step_note": "whole step (stem + convs + tail, %.3f GOP/img) against the SUSTAINED measured i8 rate: "
                                   "the step is timed inside a long loop" % GOP_PER_IMG[args.arch],
                "hbm_achieved_gbs": conv_bytes / (conv_ms * 1e-3) / 1e9, "hbm_peak_gbs": peaks["hbm"],
                "hbm_frac": conv_bytes / (conv_ms * 1e-3) / 1e9 / peaks["hbm"],
                "conv_ms_per_step_serialised": conv_ms, "step_ms": ms / args.steps}

    line = {
        "metric": metric_name(args.arch), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "impl": "ours",
        "config": {"workload": "%s semilayer 8/4-bit (P0: %d of %d channels 4-bit) inference, batch %d per GPU, "
                               "synthetic 224x224, random-init" % (args.arch, int((table[:, 2] == 4).sum()), len(table), B),
                   "batch_per_gpu": B, "global_batch": B * world, "parallelism": "dp%d" % world,
                   "cuda_graph": use_graph, "kernels": "simt-checker" if args.simt else "tcgen05",
                   "weights": "resident-weight layers fetch PACKED codes (4-bit rows two per byte) and unpack them in shared "
                              "memory; K-heavy layers stream u8 tiles" if not args.no_packed_b else "u8 tiles everywhere (A/B)",
                   "l2": "per-step working set (u8 activations ~%.1f GB) >> 126 MB L2; no flush needed" %
                         (sum(a.numel() for a in eng.act) / 1e9),
                   "activation_quant": "static per-tensor u8 (calibrated on one batch)"},
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(x_host.numel() * 4),
                "d2h_bytes_per_step": int(out_host.numel() * 4), "steps": e2e_steps,
                "overlap": "pinned fp32 H2D two batches ahead on a copy stream; logits D2H into pinned memory, the host "
                           "waits on that copy's event every step",
                "efficiency_note": "e2e per GPU at N over e2e at N=1 is computed by the reader from the per-N lines",
                "h2d_probe_gbs_per_gpu": h2d_gbs,
                "h2d_needed_gbs_per_gpu_at_value": (value / world) * 3 * 224 * 224 * 4 / 1e9,
                "numa": numa},
        "e2e_other_input_formats": e2e_alt,
        "gpu_launches": int(eng.kernel_launches * args.steps),
        "roofline": roofline,
        "pct_int8_peak_whole_net": 100.0 * (value / world) * GOP_PER_IMG[args.arch] * 1e9 / (int8_peak * 1e12),
        "top1_agreement_vs_fp32": agree, "logits_rel_l2_vs_fp32": rel,
        "quantizer": {"ms_all_layers": quant_ms, "ms_all_layers_prepared_plan": quant_replay_ms,
                      "packed_bytes": packed_bytes, "launches": 1,
                      "note": "wall clock of functions.quantize_model for all %d rows (warm allocator): job table, one H2D, "
                              "ONE launch, one status read-back; prepared_plan = QuantPlan.run() + check() again" % len(table)},
        "roofline_quantizer": roofline_q,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            times, threads, kind = cpu_reference_forward(args.arch, 32, 12)
            v = 32 * len(times) / sum(times)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": kind,
                                    "sample": "%d fp32 forwards of batch 32 (%.1f s) on the host CPU after one warm-up, %s"
                                              % (len(times), sum(times), "unmodified reference modules from oracle/_ref"
                                                 if kind == "reference" else "oracle restatement on stock torch ops")}
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                    "sample": "failed: %s" % e}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
