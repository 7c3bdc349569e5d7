"""Data-parallel evaluation on CPU: under torch.distributed (gloo, world sizes 2 and 3) every rank's
evaluate_acc_loss_softmax / evaluate_loss / KLdiv / fused-KL evaluation returns exactly what one process returns --
the same float bits, and probability tensors that are torch.equal -- over in-memory loaders of 1, 2, 5 and 7 batches
(some with a short last batch, some leaving ranks without a batch), a loader that is neither in memory nor a
DataLoader, and a DataLoader reading its dataset in order, of which each rank must read exactly its own batches.
The CUDA entry points are replaced by the oracle (tests/cpu_standins.py)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from helpers import ROOT

CASES = {"b1": (1, False), "b2": (2, True), "b5": (5, False), "b7": (7, True)}  # batches, short last batch
N_ITEMS, BATCH = 18, 4  # the DataLoader case: 5 batches, the last one of 2 images


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _Counting(torch.utils.data.Dataset):
    """Seeded (image, label) pairs that record every index read."""

    def __init__(self, n, seed):
        g = torch.Generator().manual_seed(seed)
        self.x = torch.randn(n, 3, 32, 32, generator=g)
        self.y = torch.randint(0, 1000, (n,), generator=g)
        self.calls = []

    def __len__(self):
        return len(self.x)

    def __getitem__(self, i):
        self.calls.append(int(i))
        return self.x[i], self.y[i]


class _Stream:
    """A loader that is neither a list nor a DataLoader: every rank iterates it in full."""

    def __init__(self, batches):
        self.batches = batches

    def __iter__(self):
        return iter(self.batches)


def _loader(n, short, seed):
    import imagenet
    batches = imagenet.synthetic_loader(n, BATCH, 32, seed=seed)
    if short:
        x, y = batches[-1]
        batches[-1] = (x[:3].clone(), y[:3].clone())
    return batches


def _worker(rank, world, port, out_dir):
    for p in ("semilayer-wise-mixed-precision-quantization_b200", "oracle", "tests"):
        sys.path.insert(0, os.path.join(ROOT, p))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    import cpu_standins
    import functions
    import resnet
    import slq_oracle as so
    torch.set_num_threads(2)
    functions.quantize_rows = cpu_standins.oracle_quantize_rows
    resnet.ResNet.cpu_checker = staticmethod(so.torch_forward)
    if world > 1:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    net = resnet.resnet18(num_classes=1000)
    res = {}
    for name, (n, short) in CASES.items():
        loader = _loader(n, short, seed=n)
        acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cpu", loader)
        shifted = [(x * 1.1, y) for x, y in loader]
        _, _, probs2 = functions.evaluate_acc_loss_softmax(net, "cpu", shifted)
        _, _, _, kl_fused = functions._evaluate(net, "cpu", shifted, ref_outputs=probs)
        res[name] = dict(acc=acc, loss=loss, probs=probs, kl=functions.KLdiv(probs, probs2), kl_fused=kl_fused,
                         eval_loss=functions.evaluate_loss(net, "cpu", loader))
    acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cpu", _Stream(_loader(5, True, seed=11)))
    res["stream"] = dict(acc=acc, loss=loss, probs=probs)
    ds = _Counting(N_ITEMS, seed=3)
    dl = torch.utils.data.DataLoader(ds, batch_size=BATCH, shuffle=False)
    acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cpu", dl)
    res["dataloader"] = dict(acc=acc, loss=loss, probs=probs, calls=list(ds.calls))
    ds.calls.clear()
    res["dataloader"]["eval_loss"] = functions.evaluate_loss(net, "cpu", dl)  # the cached rank loader, again
    res["dataloader"]["calls_again"] = list(ds.calls)
    dl2 = torch.utils.data.DataLoader(_Counting(N_ITEMS, seed=3), batch_size=BATCH, shuffle=False, num_workers=2)
    acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cpu", dl2)
    res["dataloader_workers"] = dict(acc=acc, loss=loss, probs=probs)
    torch.save(res, os.path.join(out_dir, "r%d_w%d.pt" % (rank, world)))
    if world > 1:
        dist.destroy_process_group()


def _bits(v):
    return None if v is None else int(np.float64(v).view(np.int64))


def _run(world, out_dir):
    mp.spawn(_worker, args=(world, _free_port(), str(out_dir)), nprocs=world, join=True)
    return [torch.load(out_dir / ("r%d_w%d.pt" % (r, world))) for r in range(world)]


@pytest.fixture(scope="module")
def single(tmp_path_factory):
    return _run(1, tmp_path_factory.mktemp("w1"))[0]


def _batch_indices(rank, world):
    n_batches = -(-N_ITEMS // BATCH)
    return [i for b in range(rank, n_batches, world) for i in range(b * BATCH, min((b + 1) * BATCH, N_ITEMS))]


def test_single_process_reads_every_batch_once(single):
    assert single["dataloader"]["calls"] == list(range(N_ITEMS))
    assert [len(p) for p in single["b7"]["probs"]] == [BATCH] * 6 + [3]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_evaluation_equals_single_process(world, single, tmp_path):
    for rank, got in enumerate(_run(world, tmp_path)):
        for case, want in single.items():
            have = got[case]
            for key in ("acc", "loss", "kl", "kl_fused", "eval_loss"):
                if key in want:
                    assert _bits(have[key]) == _bits(want[key]), (world, rank, case, key, have[key], want[key])
            assert len(have["probs"]) == len(want["probs"]), (world, rank, case)
            for p, q in zip(have["probs"], want["probs"]):
                assert p.dtype == q.dtype and torch.equal(p, q), (world, rank, case)
        # a DataLoader reading its dataset in order: this rank decoded exactly its own batches, every time
        assert got["dataloader"]["calls"] == _batch_indices(rank, world), (world, rank)
        assert got["dataloader"]["calls_again"] == _batch_indices(rank, world), (world, rank)
