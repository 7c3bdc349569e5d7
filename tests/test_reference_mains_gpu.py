"""Integration test of the drop-in boundary (SURVEY.md section 4, last-but-one row; BASELINE north_star:
"the functions.py / resnet.py entry points and the *_main.py flow stay as they are"):

the reference's UNMODIFIED ``resnet50_main.py`` (staged byte for byte under oracle/_ref by oracle/make_ref.py)
is executed with this repo's ``functions`` / ``resnet`` / ``imagenet`` modules first on sys.path, on the GPU,
and what it writes to ``output/resnet50_output.csv`` is compared with the fixture
``tests/golden/main_resnet50.npz`` = the same script run against the reference's own modules on the CPU
(oracle/run_main.py, 2 batches of 4 synthetic 64x64 images, seeded random labels and weights).

With random labels the baseline accuracy is 0, so ``acc >= preacc`` (resnet50_main.py:209) accepts every
semilayer in every phase (SURVEY.md Appendix F): the run is the progressive 8 -> 6 -> 4 bit
re-quantisation of every channel.  What must then be IDENTICAL to the reference: the number of steps, the
bit / phase-flag / accuracy rows, the cumulative reduced-parameter total, per phase the multiset of
(layer number, channel count, parameter increment), and -- with the divide flavour pinned to the CPU one
(SURVEY.md F5) -- every final conv weight, bit for bit.  The ORDER of the semilayers inside a phase comes
from the KL/param ranking of the sweep, which this path perturbs by its u8 activation quantisation (the
reference never quantises activations, F2): it is reported (rank correlation), not asserted.

The driver script is the reference project's, not this repository's, so that test runs only where the
reference has been staged (oracle/make_ref.py).  The fixture alone pins the part of its outcome that needs no
driver: the package's evaluation on the fixture's seeded batches gives the accuracy row, so every semilayer is
accepted, every channel goes 8 -> 6 -> 4 bit, and the final weights are that progressive re-quantisation of the
seeded model through the package's drop-in quantizer."""
import os
from collections import Counter

import numpy as np
import pytest
import torch

from helpers import GOLD

pytestmark = pytest.mark.gpu


def _phases(rows):
    """-> {(bit, flag): sorted list of (layer number, channels, param increment)} from the 7 CSV rows."""
    params = [float(v) for v in rows[0]]
    out = {}
    for i in range(1, len(params)):
        key = (int(rows[3][i]), int(rows[4][i]))
        out.setdefault(key, []).append((int(rows[5][i]), int(rows[6][i]), params[i] - params[i - 1]))
    return {k: sorted(v) for k, v in out.items()}


def test_unmodified_resnet50_main_against_the_package(monkeypatch):
    import make_ref
    import run_main
    if not make_ref.staged():
        pytest.skip("the reference's resnet50_main.py is not staged under oracle/_ref")
    gold = np.load(os.path.join(GOLD, "main_resnet50.npz"))
    want = [r.split("\x1f") for r in gold["rows"]]
    b, n, hw, lseed, mseed = [int(v) for v in gold["config"]]
    monkeypatch.setenv("SLQ_DIV_MODE", "true")
    res = run_main.run_main("resnet50", "b200", batches=b, batch=n, hw=hw, loader_seed=lseed, model_seed=mseed)
    got = res["rows"]
    print("unmodified resnet50_main.py on the B200 path: %.1f s (reference on 6 CPU threads: %.1f s)" %
          (res["seconds"], float(gold["seconds"])))
    assert [len(r) for r in got] == [len(r) for r in want] == [280] * 7
    assert got[3] == want[3] and got[4] == want[4]          # bit-width and phase flag of every step
    assert [float(v) for v in got[1]] == [float(v) for v in want[1]]   # accuracy row (all 0.0)
    assert float(got[0][-1]) == float(want[0][-1]) == 18092032.0        # = 20,676,608 * 28 / 32
    assert _phases(got) == _phases(want)
    assert res["weights_sha256"] == str(gold["weights_sha256"])
    # order inside the 8-bit phase (sweep ranking): informative only
    g8 = [int(v) for v, bit in zip(got[5], got[3]) if bit == "8"]
    w8 = [int(v) for v, bit in zip(want[5], want[3]) if bit == "8"]
    same_pos = sum(1 for a, c in zip(g8, w8) if a == c)
    print("8-bit phase: %d of %d steps visit the same layer as the reference run" % (same_pos, len(w8)))
    kl = np.array([float(v) for v in got[2]])
    print("KL row, first steps: ours %s reference %s" % (kl[1:4], [float(v) for v in want[2][1:4]]))


def test_resnet50_main_fixture_weights_from_the_package_quantizer(monkeypatch):
    """The reference run of the fixture accepts every semilayer (the accuracy on its seeded batches never drops
    below the fp32 model's) and so visits every channel of the 48 quantised convs once per phase, at 8, then 6,
    then 4 bit.  On the package, the seeded model re-quantised that way with ``channel_wise_quantizationperchan``
    on the GPU must be evaluated (``evaluate_acc_loss_softmax``) to the fixture's accuracy row after every phase,
    and must end with the reference run's final conv weights bit for bit."""
    import functions
    import imagenet
    import resnet
    import run_main
    gold = np.load(os.path.join(GOLD, "main_resnet50.npz"))
    rows = [r.split("\x1f") for r in gold["rows"]]
    b, n, hw, lseed, mseed = [int(v) for v in gold["config"]]
    loader = imagenet.synthetic_loader(b, n, hw, seed=lseed)
    monkeypatch.setenv("SLQ_DIV_MODE", "true")
    torch.manual_seed(mseed)
    net = resnet.resnet50(num_classes=1000).cuda()
    convs = dict(functions.quantized_convs("resnet50", net))
    preacc = functions.evaluate_acc_loss_softmax(net, "cuda", loader)[0]
    params = [float(v) for v in rows[0]]
    bits = [int(v) for v in rows[3][1:]]
    assert len(params) == 280 and bits == sorted(bits, reverse=True) and sorted(set(bits)) == [4, 6, 8]
    previous = {8: 32, 6: 8, 4: 6}
    for bit in (8, 6, 4):
        visited, accs = Counter(), set()
        for i in range(1, len(params)):
            if int(rows[3][i]) != bit:
                continue
            lnum, channels = int(rows[5][i]), int(rows[6][i])
            K = convs[lnum].weight[0].numel()
            assert params[i] - params[i - 1] == channels * K * (previous[bit] - bit) / 32  # the reference's layer map
            visited[lnum] += channels
            accs.add(float(rows[1][i]))
        assert visited == {lnum: conv.out_channels for lnum, conv in convs.items()}
        for conv in convs.values():
            for c in range(conv.out_channels):
                functions.channel_wise_quantizationperchan(conv.weight.data, bit, c)
        acc = functions.evaluate_acc_loss_softmax(net, "cuda", loader)[0]
        assert acc >= preacc and accs == {acc}, (bit, preacc, acc, accs)
    assert params[-1] == 18092032.0
    assert run_main.conv_weights_sha256(net) == str(gold["weights_sha256"])


def test_reference_files_are_staged_unmodified():
    """oracle/_ref holds byte-for-byte copies (digest written by oracle/make_ref.py)."""
    import hashlib
    import make_ref
    if not make_ref.staged():
        pytest.skip("oracle/_ref not staged")
    digest = hashlib.sha256()
    for f in make_ref.FILES:
        digest.update(f.encode() + b"\0" + open(os.path.join(make_ref.DST, f), "rb").read())
    assert digest.hexdigest() == open(os.path.join(make_ref.DST, "SHA256")).read().strip()
