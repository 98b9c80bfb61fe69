"""What torch.use_deterministic_algorithms(True) costs: ms per training step with the switch off and on, alternated
within one call, plus the per-launch device times of the weight-gradient GEMMs (G1, G2) at the bench shape.  One JSON
line per workload (card name and power limit read in the same call), also appended to --out.
    python tools/deterministic_cost.py [--rounds 3] [--steps 5] [--out profiles/deterministic_cost.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import odevit_b200 as ob  # noqa: E402
from odevit_b200 import _lib, ops  # noqa: E402
from odevit_b200.graphs import GraphedTrainStep  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C100 = dict(img_size=224, patch_size=16, num_classes=100, embed_dim=768, num_heads=12, mlp_ratio=1.0, emulate_depth=12,
            time_interval=1.0, num_eval_steps=24, solver="euler", register_tokens=10)
C10 = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
           time_interval=1.0, num_eval_steps=5, solver="rk4", register_tokens=4)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def switch(on):
    torch.use_deterministic_algorithms(on)
    ops._sync_deterministic()


def timed(fn, n):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def build(cfg, batch, graphed, adaptive=False):
    """A training step with the switch as it is now (a graph captures the kernels of the mode it was captured in)."""
    torch.manual_seed(0)
    m = ob.ViTNeuralODE(**cfg).cuda().train()
    m.precision = "bf16"
    if adaptive:
        m.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "differentiable": True}
    params = [p for p in m.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=5e-2, fused=True, capturable=graphed)
    S, C = cfg["img_size"], cfg["num_classes"]
    px = torch.randn(batch, 3, S, S, generator=torch.Generator().manual_seed(1234)).cuda()
    lb = torch.randint(0, C, (batch,), generator=torch.Generator().manual_seed(1235)).cuda()
    if graphed:
        stepper = GraphedTrainStep(m, opt, (px, lb), clip=1.0)
        return lambda: stepper(px, lb)

    def step():
        opt.zero_grad(set_to_none=True)
        m(px, labels=lb)["loss"].backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0, foreach=True)
        opt.step()
    return step


def in_process(name, cfg, batch, graphed, rounds, steps, adaptive=False):
    fns = {}
    for on in (False, True):
        switch(on)
        fns[on] = build(cfg, batch, graphed, adaptive)
        fns[on]()
    ms = {False: [], True: []}
    for _ in range(rounds):
        for on in (False, True):
            switch(on)
            ms[on].append(timed(fns[on], steps))
    switch(False)
    return {"workload": name, "ms_off": ms[False], "ms_on": ms[True],
            "ratio_median": sorted(ms[True])[rounds // 2] / sorted(ms[False])[rounds // 2]}


def distill(rounds, steps):
    # the distillation step of tools/distill_step.py (ViTTeacher, batch 64, eager), one process per run: alternated runs
    code = ("import sys, runpy, torch; torch.use_deterministic_algorithms(sys.argv.pop(1) == '1'); "
            "sys.argv[0] = 'tools/distill_step.py'; runpy.run_path('tools/distill_step.py', run_name='__main__')")
    ms = {False: [], True: []}
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    for _ in range(rounds):
        for on in (False, True):
            r = subprocess.run([sys.executable, "-c", code, "1" if on else "0", "--steps", str(steps)], cwd=ROOT, env=env,
                               capture_output=True, text=True)
            if r.returncode != 0:
                return {"workload": "distillation step", "error": r.stderr[-2000:]}
            ms[on].append(json.loads(r.stdout.strip().splitlines()[-1])["ms_per_step"])
    return {"workload": "distillation step (tools/distill_step.py, ViTTeacher, batch 64, eager)", "ms_off": ms[False],
            "ms_on": ms[True], "ratio_median": sorted(ms[True])[rounds // 2] / sorted(ms[False])[rounds // 2]}


def gemm_classes(iters):
    """Per-launch device time of the G1 / G2 classes (and the column-sum pieces) in one eager bench-shape step."""
    out = {}
    for on in (False, True):
        switch(on)
        step = build(C100, 64, graphed=False)
        step()
        torch.cuda.synchronize()
        _lib.profile_reserve(20000)
        _lib.profile_enable(True)
        for _ in range(iters):
            step()
        torch.cuda.synchronize()
        r = _lib.profile_read()
        _lib.profile_enable(False)
        out["on" if on else "off"] = {k: {"us_per_launch": 1e3 * ms / n, "launches_per_step": n / iters}
                                      for k, (ms, n) in r.items()
                                      if k in ("bwd_gemm_g1", "bwd_gemm_g2", "bwd_colsum", "det_sum", "weights", "bwd_gemm_doh")}
    switch(False)
    return {"workload": "bench-shape step kernel classes (C100, Euler T=24, batch 64, bf16, eager, profiled)", **out}


def default_differs():
    """Evidence, not a test: two identical eager bench-shape steps with the switch off -- do the weight gradients differ?"""
    switch(False)
    torch.manual_seed(0)
    m = ob.ViTNeuralODE(**C100).cuda().train()
    m.precision = "bf16"
    px = torch.randn(64, 3, 224, 224, generator=torch.Generator().manual_seed(1234)).cuda()
    lb = torch.randint(0, 100, (64,), generator=torch.Generator().manual_seed(1235)).cuda()
    grads = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        m(px, labels=lb)["loss"].backward()
        grads.append({n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None})
    differ = [n for n in grads[0] if not torch.equal(grads[0][n], grads[1][n])]
    return {"workload": "switch off: two identical bench-shape steps (C100, Euler T=24, batch 64, bf16)",
            "params_with_different_grads": len(differ), "of": len(grads[0]), "examples": differ[:6],
            "max_abs_diff": max((float((grads[0][n] - grads[1][n]).abs().max()) for n in differ), default=0.0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    gpu = card()
    jobs = [
        default_differs,
        lambda: in_process("bench training step: C100, Euler T=24, batch 64, bf16, graph-replayed", C100, 64, True, a.rounds,
                           a.steps),
        lambda: in_process("config 1: C10, RK4 T=5, batch 8, bf16, eager", C10, 8, False, a.rounds, a.steps),
        lambda: in_process("C10 training, RK4 T=5, batch 512, bf16, eager", C10, 512, False, a.rounds, a.steps),
        lambda: in_process("adaptive training step: C10, dopri5 rtol 1e-3, batch 64, bf16, eager", C10, 64, False, a.rounds,
                           a.steps, adaptive=True),
        lambda: distill(a.rounds, a.steps),
        lambda: gemm_classes(3),
    ]
    for job in jobs:
        ln = job()
        ln["gpu"] = gpu
        print(json.dumps(ln), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
            with open(a.out, "a") as f:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
