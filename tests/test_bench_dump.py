"""bench.py --dump-outputs: the last timed step's outputs as .npy files, within the size budget, comparable run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dir_bytes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_dump_fits_the_budget_with_the_same_sample_every_time(tmp_path):
    rng = np.random.default_rng(1)
    arrays = {"loss": np.float32(2.5), "small": rng.standard_normal(100),
              "big": rng.standard_normal((4000, 2500)), "bigger": rng.standard_normal(9_000_000)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
        assert _dir_bytes(tmp_path / d) <= bench.DUMP_BUDGET_BYTES
    a = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(a) == ["big.npy", "bigger.npy", "loss.npy", "small.npy"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert float(a["loss.npy"]) == 2.5 and np.array_equal(a["small.npy"], arrays["small"].astype(np.float32))
    assert a["big.npy"].size == a["bigger.npy"].size < 9_000_000           # both sampled to the same count
    assert np.isin(a["big.npy"], arrays["big"].astype(np.float32)).all()
    for f, v in a.items():
        assert np.array_equal(v, np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    import torch
    import odevit_b200 as ob
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c10b8", "--steps", "1", "--warmup", "1",
                            "--repeats", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           cwd=tmp_path, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 1 and line["value"] > 0
        assert _dir_bytes(out) <= bench.DUMP_BUDGET_BYTES
        d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
        assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in d.values())
        dumps.append(d)
    a, b = dumps
    assert {"loss", "logits", "param.head.weight", "grad.head.weight"} <= set(a) and set(a) == set(b)
    # the loss is the smoothed cross-entropy of the dumped logits: both come from the same step
    _, labels = bench.synthetic_batch(bench.C10, 8)
    ce = torch.nn.functional.cross_entropy(torch.from_numpy(a["logits"]).double(), labels, label_smoothing=0.05)
    assert float(a["loss"]) == pytest.approx(float(ce), rel=1e-4)
    # the weights are the seeded ones after exactly one AdamW step (lr 1e-4: every update is about lr)
    torch.manual_seed(0)
    init = dict(ob.ViTNeuralODE(**bench.C10).named_parameters())
    steps = {n: np.abs(a[f"param.{n}"] - p.detach().numpy()).max() for n, p in init.items() if f"param.{n}" in a}
    assert steps["head.weight"] > 1e-5 and max(steps.values()) < 3e-4, steps
    # two runs with the same arguments: the same inputs, so the same outputs up to the rounding of the gradient atomics
    for k in a:
        if not k.startswith("param."):
            assert np.abs(a[k] - b[k]).max() <= 1e-3 * np.abs(b[k]).max() + 1e-6, k
