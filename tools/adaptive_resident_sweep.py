"""The capturable on-chip adaptive Dormand-Prince solve (odeint_adaptive(capturable=True), odevit_solve_adaptive_resident)
against the synchronising multi-kernel adaptive solve and the fixed-grid on-chip rk4, at the c10 shape of
tools/adaptive_sweep.py (32 px CIFAR-10, D 192, 3 heads, 69 tokens, batch 512, bf16, seeded reference_like_init weights
and images, t = [0, 1]).  One JSON line per rtol, atol = rtol / 100:
  ms per solve (host clock around `reps` solves that end synchronised, after a warm-up of every shape; the median and
  range over `trials` such windows) for the multi-kernel solve, the on-chip solve called eagerly, the on-chip solve
  replayed from a CUDA graph, and the on-chip rk4 with round(nfe_mean / 4) steps; field evaluations per second of the
  on-chip solve; NFE mean / min / max; launches per on-chip solve (odevit_launch_count); the max-relative difference of
  the final state against the multi-kernel solve; the card's name and power limit.

    python tools/adaptive_resident_sweep.py [--out profiles/adaptive_resident_sweep.jsonl] [--reps 10] [--trials 5]
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import odevit_b200 as ob  # noqa: E402
import odevit_oracle as orc  # noqa: E402
from adaptive_sweep import RTOLS, SHAPES, card  # noqa: E402


def timed(fn, reps, trials):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(trials):
        t0 = time.perf_counter()
        for _ in range(reps):
            out = fn()
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3 / reps)
    return ms, out


def summary(ms):
    return dict(median=round(statistics.median(ms), 3), min=round(min(ms), 3), max=round(max(ms), 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--trials", type=int, default=5)
    args = ap.parse_args()
    name, power = card()
    cfg, B = SHAPES["c10"]
    model = ob.ViTNeuralODE(**cfg)
    model.load_state_dict(orc.reference_like_init(cfg, cfg["num_classes"], seed=0), strict=True)
    model = model.cuda().eval()
    model.precision = "bf16"
    px = torch.randn(B, 3, cfg["img_size"], cfg["img_size"], generator=torch.Generator().manual_seed(1)).cuda()
    t = torch.tensor([0.0, 1.0])
    lines = []
    with torch.no_grad():
        x0 = model.patch_embed(px).contiguous()
        static_x = x0.clone()
        for rtol in RTOLS:
            atol = rtol / 100

            def multi():
                return ob.odeint_adaptive(model.odefunc, x0, t, rtol=rtol, atol=atol, return_stats=True)

            def onchip():
                return ob.odeint_adaptive(model.odefunc, static_x, t, rtol=rtol, atol=atol, return_stats=True,
                                          capturable=True)
            ms_multi, (s_multi, _) = timed(multi, args.reps, args.trials)
            ms_chip, (s_chip, st) = timed(onchip, args.reps, args.trials)
            torch.cuda.synchronize()
            ob.reset_launch_count()
            onchip()
            torch.cuda.synchronize()
            launches = ob.launch_count()
            g = torch.cuda.CUDAGraph()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                onchip()
            torch.cuda.current_stream().wait_stream(s)
            with torch.cuda.graph(g):
                s_graph, _ = onchip()
            ms_graph, _ = timed(g.replay, args.reps, args.trials)
            assert torch.equal(s_graph, s_chip)
            nfe = st["nfe"].double()
            steps = max(1, round(nfe.mean().item() / 4))
            grid = torch.linspace(0.0, 1.0, steps + 1)

            def fixed():
                return ob.odeint(model.odefunc, x0, grid, method="rk4", record_attention=False)
            ms_rk4, _ = timed(fixed, args.reps, args.trials)
            diff = ((s_chip[-1] - s_multi[-1]).abs().max() / s_multi[-1].abs().max()).item()
            evals = nfe.sum().item()
            line = dict(shape="c10", batch=B, tokens=x0.shape[1], dim=cfg["embed_dim"], precision="bf16", rtol=rtol,
                        atol=atol, nfe_mean=round(nfe.mean().item(), 2), nfe_min=int(nfe.min().item()),
                        nfe_max=int(nfe.max().item()), ms_multikernel=summary(ms_multi), ms_onchip=summary(ms_chip),
                        ms_onchip_graph=summary(ms_graph), rk4_steps=steps, ms_rk4_onchip=summary(ms_rk4),
                        onchip_field_evals_per_s=round(evals / statistics.median(ms_chip) * 1e3),
                        launches_per_onchip_solve=launches, final_maxrel_vs_multikernel=float(f"{diff:.3e}"),
                        reps=args.reps, trials=args.trials, gpu=name, power_limit=power)
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
