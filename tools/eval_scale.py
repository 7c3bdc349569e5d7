"""tools/eval_scale.py -- wall time of ONE functions.evaluate_acc_loss_softmax over an ImageNet-val-sized loader on
ResNet-50, data-parallel over the ranks of a torchrun job (batch i on rank i % world).

    python tools/eval_scale.py --out profiles/eval_sharded_1gpu.json
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29513 \
        tools/eval_scale.py --out profiles/eval_sharded_Ngpu.json

Loader: a seeded synthetic torch DataLoader (``shuffle=False``, ``--workers`` worker processes, pinned memory) of
50,000 u8 224x224 images with ``net.input_norm`` set (normalisation runs in the stem kernel), batch 256: 196 batches,
the last one of 80 images.  Image i is image i % 1024 of a seeded pool and its label is seeded too, so the
"decode" is a copy out of the pool: this measures the evaluation and the loader machinery, not JPEG decoding.  The
same evaluation is also timed from an in-memory loader (a list of the same 196 batches, views of the pool), whose
batches the evaluation keeps resident on the device after the first call.

Time: host clock around a call that starts after a barrier and ends in a device synchronise, after one warm-up
evaluation of the same loader; the median over ``--reps`` calls, per rank, and the slowest rank's median.
Digest: sha256 over (acc, loss, every probability tensor), which must be the same at every world size and for both
loaders.  The card's name and power limit are read in the same run and written beside the numbers."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "semilayer-wise-mixed-precision-quantization_b200"))

N_IMAGES, BATCH, HW, POOL = 50000, 256, 224, 1024


class SyntheticVal(torch.utils.data.Dataset):
    def __init__(self, pool, labels):
        self.pool, self.labels = pool, labels

    def __len__(self):
        return len(self.labels)

    def __getitem__(self, i):
        return self.pool[i % POOL], self.labels[i]


def card():
    info = {"name": torch.cuda.get_device_name(torch.cuda.current_device())}
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                                     "-i", str(torch.cuda.current_device())], text=True).splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")]
    except (OSError, subprocess.CalledProcessError) as e:
        info["power_limit"] = "unknown (%s)" % e
    return info


def digest(acc, loss, probs):
    h = hashlib.sha256(np.array([acc, loss], np.float64).tobytes())
    for p in probs:
        h.update(p.cpu().numpy().tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workers", type=int, default=4, help="DataLoader worker processes per rank")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dev = torch.device("cuda", torch.cuda.current_device())
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import slq_build
    slq_build.build()
    import functions
    import imagenet
    import resnet

    g = torch.Generator().manual_seed(1)
    pool = torch.randint(0, 256, (POOL, 3, HW, HW), generator=g, dtype=torch.uint8)
    labels = torch.randint(0, 1000, (N_IMAGES,), generator=g)
    loader = torch.utils.data.DataLoader(SyntheticVal(pool, labels), batch_size=BATCH, shuffle=False,
                                         num_workers=args.workers, pin_memory=True)
    resident = [(pool[s % POOL:s % POOL + min(BATCH, N_IMAGES - s)], labels[s:s + BATCH])
                for s in range(0, N_IMAGES, BATCH)]
    assert len(loader) == len(resident) == 196
    torch.manual_seed(0)
    net = resnet.resnet50(num_classes=1000).to(dev)
    net.input_norm = (imagenet.MEAN, imagenet.STD)

    def timed(ld):
        out = functions.evaluate_acc_loss_softmax(net, dev, ld)  # warm-up (the first one also calibrates)
        times = []
        for _ in range(args.reps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = functions.evaluate_acc_loss_softmax(net, dev, ld)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        return out, times

    result = {"world": world, "card": card(), "images": N_IMAGES, "batch": BATCH, "batches": len(loader),
              "workers_per_rank": args.workers}
    for name, ld in (("dataloader", loader), ("resident", resident)):
        (acc, loss, probs), times = timed(ld)
        mine = {"median_s": statistics.median(times), "times_s": times, "sha256": digest(acc, loss, probs)}
        ranks = [mine]
        if world > 1:
            ranks = [None] * world
            dist.all_gather_object(ranks, mine)
        result[name] = {"median_s": max(r["median_s"] for r in ranks), "rank_median_s": [r["median_s"] for r in ranks],
                        "times_s_rank0": times, "sha256": mine["sha256"],
                        "ranks_agree": len({r["sha256"] for r in ranks}) == 1}
        result["acc"], result["loss"] = acc, loss
    result["same_result_both_loaders"] = result["dataloader"]["sha256"] == result["resident"]["sha256"]
    if rank == 0:
        line = json.dumps(result)
        print(line)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
