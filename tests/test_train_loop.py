"""`odevit_b200.train.train_classification_task` against the UNMODIFIED reference loop (train.py:18-110) on a CPU
stand-in model: same weights after an epoch with gradient accumulation, clipping, AdamW and a scheduler -- including
the reference's two quirks (JaSMin added twice; the clip only bites at the first optimizer step of a call because
`params` is a generator).  The live comparisons need the reference's sources (ref_import); the stored ones run
everywhere: tests/golden/train_loop_stub.npz (oracle/make_golden_train_loop.py) and tests/golden/experiment_vit_edo_keys.yaml."""
import copy
import importlib
import os
import sys

import numpy as np
import pytest
import torch
from torch import nn

import ref_import
from _util import GOLDEN_DIR

needs_reference = pytest.mark.skipif(not ref_import.reference_available(), reason="reference sources not present")


class Stub(nn.Module):
    """Returns what the train loop reads: logits, loss, jasmin_loss (a differentiable function of the weights)."""

    def __init__(self):
        super().__init__()
        self.fc = nn.Linear(12, 5)

    def forward(self, pixel_values, labels=None, **kw):
        logits = self.fc(pixel_values.flatten(1))
        return {"logits": logits, "loss": nn.functional.cross_entropy(logits, labels) * 3.0,
                "jasmin_loss": logits.square().mean()}


def _loader(n=7):
    from odevit_b200.data import PixelBatch
    g = torch.Generator().manual_seed(0)
    return [{"pixel_values": PixelBatch({"pixel_values": torch.randn(4, 3, 2, 2, generator=g) * 3}), "labels": torch.randint(0, 5, (4,), generator=g)}
            for _ in range(n)]


def _reference_train():
    ref_import.import_reference()
    shims = os.path.join(os.path.dirname(ref_import.__file__), "shims")
    if shims not in sys.path:
        sys.path.insert(0, shims)
    sys.modules.pop("train", None)
    return importlib.import_module("train")


def _run_ours(m, accum, loader, monkeypatch):
    from odevit_b200 import train as ours
    monkeypatch.setattr(ours, "device", "cpu")      # the stand-in model is a CPU module, also where a GPU is present
    opt = torch.optim.AdamW(m.parameters(), lr=1e-2, weight_decay=5e-2)
    sch = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=0.7)
    _, loss = ours.train_classification_task(loader, m, opt, None, sch, wandb_logger=None, epoch=1,
                                             num_accumulation_steps=accum, log_every=3)
    return loss, opt.param_groups[0]["lr"]


@pytest.mark.parametrize("accum", [1, 2, 3])
def test_train_loop_matches_stored_reference_run(accum, monkeypatch):
    """The same epoch against the stored run: initial weights, batches and results come from the file."""
    from odevit_b200.data import PixelBatch
    z = np.load(os.path.join(GOLDEN_DIR, "train_loop_stub.npz"))
    m = Stub()
    with torch.no_grad():
        m.fc.weight.copy_(torch.from_numpy(z["init/fc.weight"]))
        m.fc.bias.copy_(torch.from_numpy(z["init/fc.bias"]))
    loader = [{"pixel_values": PixelBatch({"pixel_values": torch.from_numpy(px)}), "labels": torch.from_numpy(lb)}
              for px, lb in zip(z["in/pixel_values"], z["in/labels"])]
    loss, lr = _run_ours(m, accum, loader, monkeypatch)
    assert loss == pytest.approx(float(z[f"a{accum}/loss"]), rel=1e-6)
    assert lr == pytest.approx(float(z[f"a{accum}/lr"]), rel=1e-12)
    for n, p in m.named_parameters():
        assert torch.allclose(p.detach(), torch.from_numpy(z[f"a{accum}/param/{n}"]), rtol=1e-6, atol=1e-7), n
        key = f"a{accum}/grad/{n}"
        assert (p.grad is None) == (key not in z.files), n          # the partial accumulation group left in .grad
        if p.grad is not None:
            assert torch.allclose(p.grad, torch.from_numpy(z[key]), rtol=1e-6, atol=1e-7), n


@needs_reference
@pytest.mark.parametrize("accum", [1, 2, 3])
def test_train_loop_matches_reference(accum):
    ref = _reference_train()
    from odevit_b200 import train as ours
    torch.manual_seed(0)
    base = Stub()
    results = []
    for fn in (ref.train_classification_task, ours.train_classification_task):
        m = copy.deepcopy(base)
        opt = torch.optim.AdamW(m.parameters(), lr=1e-2, weight_decay=5e-2)
        sch = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=0.7)
        _, loss = fn(_loader(), m, opt, None, sch, wandb_logger=None, epoch=1, num_accumulation_steps=accum, log_every=3)
        results.append((loss, [p.detach().clone() for p in m.parameters()], [None if p.grad is None else p.grad.clone() for p in m.parameters()],
                        opt.param_groups[0]["lr"]))
    (l0, p0, g0, lr0), (l1, p1, g1, lr1) = results
    assert l0 == pytest.approx(l1, rel=1e-6)
    assert lr0 == lr1
    for a, b in zip(p0, p1):
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-7)
    for a, b in zip(g0, g1):                     # the partial accumulation group left in .grad
        assert (a is None) == (b is None) and (a is None or torch.allclose(a, b, rtol=1e-6, atol=1e-7))


@needs_reference
def test_config_and_schedule_follow_the_shipped_yaml():
    _check_config_and_schedule(os.path.join(ref_import.REFERENCE_ROOT, "configs", "classification", "experiment_vit_edo.yaml"))


def test_config_and_schedule_follow_the_stored_yaml_keys():
    _check_config_and_schedule(os.path.join(GOLDEN_DIR, "experiment_vit_edo_keys.yaml"))


def _check_config_and_schedule(path):
    from odevit_b200 import train as ours
    cfg = ours.load_config(path, ["setup.dict.epochs=200", "modeling.inputs.solver=rk4"])
    assert cfg["modeling"]["inputs"]["embed_dim"] == 768 and cfg["modeling"]["inputs"]["solver"] == "rk4"
    assert cfg["setup"]["dict"]["epochs"] == 200 and cfg["data"]["collator"]["train"]["batch_size"] == 64
    opt = torch.optim.AdamW([nn.Parameter(torch.zeros(1))], lr=1e-4)
    sch = ours.restart_schedule(opt, 200, 10)
    lrs = []
    for _ in range(2000):
        opt.step()
        sch.step()
        lrs.append(opt.param_groups[0]["lr"])
    assert max(lrs) == pytest.approx(1e-4, rel=1e-3) and lrs[199] == pytest.approx(1e-4, rel=1e-2)   # 10 % warm-up
    assert lrs[1098] < 1e-6 and lrs[1100] > 9e-5                                                        # hard restart (2 cycles)
