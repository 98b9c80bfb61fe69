"""Per-image adaptive Dormand-Prince solve (odevit_b200.odeint_adaptive) over tolerances, against the fixed-grid rk4
solve that spends the same number of field evaluations per image, at two model shapes in bf16:
  c10   32 px CIFAR-10 shape (D 192, 3 heads, 69 tokens), batch 512
  c100  224 px CIFAR-100 shape (D 768, 12 heads, 207 tokens), batch 64
with seeded random weights of the reference's init statistics (oracle.reference_like_init) and seeded random images,
integrated over the models' t = [0, 1].  One JSON line per (shape, rtol), atol = rtol / 100:
  rounds, nfe_mean / nfe_max per image, batch_efficiency = sum of attempted steps / (B * rounds),
  ms per solve and img/s (host clock around the call, which ends synchronised), the rk4 solve with
  round(nfe_mean / 4) steps timed the same way, the max-relative difference of the two final states,
  and the card's name and power limit.

    python tools/adaptive_sweep.py [--out profiles/adaptive_sweep.jsonl] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import odevit_b200 as ob  # noqa: E402
import odevit_oracle as orc  # noqa: E402

SHAPES = {
    "c10": (dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
                 time_interval=1.0, num_eval_steps=5, solver="rk4", register_tokens=4), 512),
    "c100": (dict(img_size=224, patch_size=16, num_classes=100, embed_dim=768, num_heads=12, mlp_ratio=1.0,
                  emulate_depth=12, time_interval=1.0, num_eval_steps=24, solver="euler", register_tokens=10), 64),
}
RTOLS = (1e-2, 1e-3, 1e-4)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shapes", default="c10,c100")
    args = ap.parse_args()
    name, power = card()
    lines = []
    for shape in args.shapes.split(","):
        cfg, B = SHAPES[shape]
        model = ob.ViTNeuralODE(**cfg)
        model.load_state_dict(orc.reference_like_init(cfg, cfg["num_classes"], seed=0), strict=True)
        model = model.cuda().eval()
        model.precision = "bf16"
        px = torch.randn(B, 3, cfg["img_size"], cfg["img_size"], generator=torch.Generator().manual_seed(1)).cuda()
        t = torch.tensor([0.0, 1.0])
        with torch.no_grad():
            x0 = model.patch_embed(px).contiguous()
            for rtol in RTOLS:
                atol = rtol / 100

                def adaptive():
                    return ob.odeint_adaptive(model.odefunc, x0, t, rtol=rtol, atol=atol, return_stats=True)
                ms, (states, st) = timed(adaptive, args.reps)
                nfe = st["nfe"].double()
                attempts = (st["accepted"] + st["rejected"]).sum().item()
                steps = max(1, round(nfe.mean().item() / 4))
                grid = torch.linspace(0.0, 1.0, steps + 1)

                def fixed():
                    return ob.odeint(model.odefunc, x0, grid, method="rk4", record_attention=False)
                ms_rk4, ref = timed(fixed, args.reps)
                diff = ((states[-1] - ref[-1]).abs().max() / ref[-1].abs().max()).item()
                line = dict(shape=shape, batch=B, tokens=x0.shape[1], dim=cfg["embed_dim"], precision="bf16",
                            rtol=rtol, atol=atol, rounds=st["rounds"], nfe_mean=round(nfe.mean().item(), 2),
                            nfe_max=int(nfe.max().item()), nfe_min=int(nfe.min().item()),
                            rejected_total=int(st["rejected"].sum().item()),
                            batch_efficiency=round(attempts / (B * st["rounds"]), 4),
                            ms_per_solve=round(ms, 3), img_per_s=round(B / ms * 1e3, 1),
                            rk4_steps=steps, rk4_nfe=4 * steps, rk4_ms_per_solve=round(ms_rk4, 3),
                            rk4_img_per_s=round(B / ms_rk4 * 1e3, 1), final_maxrel_vs_rk4=float(f"{diff:.3e}"),
                            reps=args.reps, gpu=name, power_limit=power)
                print(json.dumps(line), flush=True)
                lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
