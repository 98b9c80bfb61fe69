"""TEST INFRASTRUCTURE ONLY -- tests/golden/train_loop_stub.npz: one epoch of the classification train loop
(train.py:18-110) on the CPU stand-in model of tests/test_train_loop.py, for num_accumulation_steps 1, 2 and 3.

    python oracle/make_golden_train_loop.py

Stores the stand-in's initial weights, the seven batches, and per accumulation count the mean epoch loss, the weights
after the epoch, the partial gradient group left in .grad and the learning rate.  The loop that is recorded is the
reference's own `train.train_classification_task` when its sources are present (ref_import.reference_available()),
otherwise `odevit_b200.train.train_classification_task`; meta["source"] says which.  The stored file was recorded
from odevit_b200.train, unchanged since tests/test_train_loop.py matched it against the unmodified reference loop
(rtol 1e-6).
"""
import copy
import importlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, HERE, os.path.join(ROOT, "tests")]
OUT = os.path.join(ROOT, "tests", "golden", "train_loop_stub.npz")

import ref_import  # noqa: E402
from test_train_loop import Stub, _loader  # noqa: E402


def main():
    if ref_import.reference_available():
        ref_import.import_reference()
        sys.path.insert(0, os.path.join(HERE, "shims"))
        sys.modules.pop("train", None)
        fn, source = importlib.import_module("train").train_classification_task, "reference train.py"
    else:
        from odevit_b200 import train as ours
        fn, source = ours.train_classification_task, "odevit_b200.train"
    torch.manual_seed(0)
    base = Stub()
    loader = _loader()
    store = {"init/fc.weight": base.fc.weight.detach().numpy(), "init/fc.bias": base.fc.bias.detach().numpy(),
             "in/pixel_values": np.stack([b["pixel_values"]["pixel_values"].numpy() for b in loader]),
             "in/labels": np.stack([b["labels"].numpy() for b in loader])}
    for accum in (1, 2, 3):
        m = copy.deepcopy(base)
        opt = torch.optim.AdamW(m.parameters(), lr=1e-2, weight_decay=5e-2)
        sch = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=0.7)
        _, loss = fn(_loader(), m, opt, None, sch, wandb_logger=None, epoch=1, num_accumulation_steps=accum, log_every=3)
        store[f"a{accum}/loss"] = np.float64(loss)
        store[f"a{accum}/lr"] = np.float64(opt.param_groups[0]["lr"])
        for n, p in m.named_parameters():
            store[f"a{accum}/param/{n}"] = p.detach().numpy()
            if p.grad is not None:
                store[f"a{accum}/grad/{n}"] = p.grad.numpy()
    store["meta"] = json.dumps({"source": source, "torch": torch.__version__})
    np.savez_compressed(OUT, **store)
    print("wrote", OUT, "from", source)


if __name__ == "__main__":
    main()
