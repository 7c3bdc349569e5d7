"""Data-parallel evaluation on the GPU: two processes on one device (gloo) give, on both ranks, exactly what one
process gives.

  * a fresh, UNCALIBRATED ResNet-18 and ResNet-50: its first forward calibrates the activation scales, which in one
    process happens on batch 0, so rank 1 (whose first batch is batch 1) must run batch 0 first.  Checked: the
    scales, (acc, loss, every softmax tensor), evaluate_loss and the fused KL, over in-memory loaders whose last batch
    is short (rank 1 owning a full batch, and rank 1 owning only the short one) and over a DataLoader;
  * the calls of resnet50_main.py, shortened (pretrained model, baseline evaluation, the sensitivity sweep over the
    first layers, then the greedy accept / undo loop with an evaluation and a KLdiv per semilayer): the same trace
    and the same final conv weights at world 2 as at world 1;
  * where the reference is staged (oracle/make_ref.py), the unmodified resnet50_main.py itself (oracle/run_main.py,
    the set-up of tests/test_reference_mains_gpu.py): the same output rows and final conv weights at world 2."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from helpers import ROOT

pytestmark = pytest.mark.gpu

HW = 64


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _loader(n, batch, last, seed):
    import imagenet
    batches = imagenet.synthetic_loader(n, batch, HW, seed=seed)
    x, y = batches[-1]
    batches[-1] = (x[:last].clone(), y[:last].clone())
    return batches


class _Images(torch.utils.data.Dataset):
    def __init__(self, n, seed):
        g = torch.Generator().manual_seed(seed)
        self.x = torch.randn(n, 3, HW, HW, generator=g)
        self.y = torch.randint(0, 1000, (n,), generator=g)

    def __len__(self):
        return len(self.x)

    def __getitem__(self, i):
        return self.x[i], self.y[i]


def _scales(net):
    return next(iter(net._slq_engines.values())).act_scales.cpu()


def _fresh_nets(functions, resnet):
    res = {}
    for arch in ("resnet18", "resnet50"):
        for case, (n, batch, last) in {"full": (3, 8, 5), "short": (2, 8, 3)}.items():
            loader = _loader(n, batch, last, seed=n)
            torch.manual_seed(0)
            net = getattr(resnet, arch)(num_classes=1000).cuda()  # uncalibrated: no engine yet
            acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cuda", loader)
            shifted = [(x * 1.05, y) for x, y in loader]
            _, _, _, kl = functions._evaluate(net, "cuda", shifted, ref_outputs=probs)
            res[arch, case] = dict(acc=acc, loss=loss, probs=[p.cpu() for p in probs], kl=kl, scales=_scales(net),
                                   eval_loss=functions.evaluate_loss(net, "cuda", loader))
        torch.manual_seed(0)
        net = getattr(resnet, arch)(num_classes=1000).cuda()
        dl = torch.utils.data.DataLoader(_Images(20, seed=5), batch_size=8, shuffle=False)
        acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cuda", dl)
        res[arch, "dataloader"] = dict(acc=acc, loss=loss, probs=[p.cpu() for p in probs], scales=_scales(net))
    return res


def _mini_main(functions, resnet, imagenet):
    """resnet50_main.py's calls on a seeded 'pretrained' ResNet-50, shortened to the first two layers' semilayers."""
    import run_main
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from sweep_run import rows_from_p0
    os.environ["SLQ_SWEEP_METRIC"] = "dloss"  # KL is NaN on a random-init ResNet-50 (softmax underflow)
    loader = _loader(3, 4, 3, seed=7)
    imagenet.val_loader = loader
    torch.manual_seed(0)
    sd = resnet.resnet50(num_classes=1000).state_dict()
    resnet.load_state_dict_from_url = lambda url, progress=True: {k: v.clone() for k, v in sd.items()}
    net = resnet.resnet50(pretrained="imagenet").cuda()
    preacc, preloss, orig = functions.evaluate_acc_loss_softmax(net, "cuda", loader)
    trace = [preacc, preloss]
    minus, plus = rows_from_p0("resnet50")
    minus, plus = [r for r in minus if r[2] <= 2], [r for r in plus if r[2] <= 2]
    semilayers, orders = functions.make_semilayers_resnet50(net, "cuda", orig, minus, plus)
    functions.make_quantizedlists(semilayers, orders)  # sorts orders in place
    trace += [v for _i, v in orders]
    layers = [net.layer1, net.layer2, net.layer3, net.layer4]
    for idx, _v in orders:
        saved = []
        for li, bi, lnum, cnum, w_bit, _f, _s, _g in semilayers[idx]:
            conv = functions._conv_of("resnet50", layers[li][bi], lnum)
            saved.append((conv, cnum, conv.weight.data[cnum].clone()))
            functions.channel_wise_quantizationperchan(conv.weight.data, w_bit - 2, cnum)
        acc, loss, probs = functions.evaluate_acc_loss_softmax(net, "cuda", loader)
        trace += [acc, loss, functions.KLdiv(orig, probs)]
        if acc < preacc or loss > preloss * 1.001:  # undo
            for conv, cnum, row in saved:
                conv.weight.data[cnum] = row
                resnet.note_weight_write(conv.weight.data)
    return dict(trace=trace, weights=run_main.conv_weights_sha256(net))


def _worker(rank, world, port, out_dir, what):
    for p in ("semilayer-wise-mixed-precision-quantization_b200", "oracle", "tests"):
        sys.path.insert(0, os.path.join(ROOT, p))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    torch.cuda.set_device(0)
    if world > 1:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    if what == "staged_main":
        import run_main
        res = run_main.run_main("resnet50", "b200", batches=3, batch=4, hw=64, loader_seed=1, model_seed=0)
        res = dict(rows=res["rows"], weights=res["weights_sha256"])
    else:
        import functions
        import imagenet
        import resnet
        res = _fresh_nets(functions, resnet) if what == "fresh" else _mini_main(functions, resnet, imagenet)
    torch.save(res, os.path.join(out_dir, "%s_r%d_w%d.pt" % (what, rank, world)))
    if world > 1:
        dist.destroy_process_group()


def _run(what, world, out_dir):
    mp.spawn(_worker, args=(world, _free_port(), str(out_dir), what), nprocs=world, join=True)
    return [torch.load(os.path.join(out_dir, "%s_r%d_w%d.pt" % (what, r, world))) for r in range(world)]


def _bits(v):
    return int(np.float64(v).view(np.int64))


def test_uncalibrated_nets_world2_equal_single_process(tmp_path):
    one = _run("fresh", 1, tmp_path)[0]
    for rank, got in enumerate(_run("fresh", 2, tmp_path)):
        for key, want in one.items():
            have = got[key]
            assert torch.equal(have["scales"], want["scales"]), (rank, key)
            for k in ("acc", "loss", "kl", "eval_loss"):
                if k in want:
                    assert _bits(have[k]) == _bits(want[k]), (rank, key, k, have[k], want[k])
            assert len(have["probs"]) == len(want["probs"])
            for p, q in zip(have["probs"], want["probs"]):
                assert torch.equal(p, q), (rank, key)


def test_resnet50_main_calls_world2_equal_single_process(tmp_path):
    one = _run("mini_main", 1, tmp_path)[0]
    assert len(one["trace"]) > 10
    for got in _run("mini_main", 2, tmp_path):
        assert [_bits(v) for v in got["trace"]] == [_bits(v) for v in one["trace"]]
        assert got["weights"] == one["weights"]


def test_unmodified_resnet50_main_world2_equals_single_process(tmp_path):
    import make_ref
    if not make_ref.staged():
        pytest.skip("the reference's resnet50_main.py is not staged under oracle/_ref")
    one = _run("staged_main", 1, tmp_path)[0]
    for got in _run("staged_main", 2, tmp_path):
        assert got["rows"] == one["rows"]
        assert got["weights"] == one["weights"]
