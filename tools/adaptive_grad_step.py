"""Training through the per-image adaptive Dormand-Prince solve (model.adaptive_solve with "differentiable": True) at
two model shapes in bf16, with seeded random weights of the reference's init statistics and seeded random images:
  c10   32 px CIFAR-10 shape (D 192, 3 heads, 65 tokens), batch 512
  c100  224 px CIFAR-100 shape (D 768, 12 heads, 207 tokens), batch 64
integrated over t = [0, 0.5, 1].  One JSON line per shape:
  fwd_record_ms      the forward solve with its accepted-step record (ops.ode_solve_adaptive, differentiable)
  bwd_tape_ms / bwd_recompute_ms   its backward (odevit_solve_adaptive_bwd) with and without a tape
  replay_kernel_ms, reverse_kernel_ms, recompute_kernel_ms   kernel time of the backward by phase, from the library's
                     per-class event timing in separate profiled runs: forward-class kernels of the tape run (the
                     replay), backward-class kernels (the reverse sweep), and the forward-class kernels the recomputing
                     run adds
  nfe_fwd_mean, S, bwd_evals (6 S + 1 replay, + 6 S recomputed without a tape), bwd_vjps (6 S + 1)
  img_per_s of a full training step (model forward with loss, backward) against the fixed-grid rk4 step whose forward
  spends the same number of field evaluations (round(nfe_fwd_mean / 4) steps),
and the card's name and power limit.  Times are host clocks around work that ends synchronised.

    python tools/adaptive_grad_step.py [--out profiles/adaptive_grad_step.jsonl] [--reps 3]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import odevit_b200 as ob  # noqa: E402
import odevit_oracle as orc  # noqa: E402
from adaptive_sweep import card, timed  # noqa: E402
from odevit_b200 import _lib  # noqa: E402

SHAPES = {
    "c10": (dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
                 time_interval=1.0, num_eval_steps=5, solver="rk4", register_tokens=0), 512),
    "c100": (dict(img_size=224, patch_size=16, num_classes=100, embed_dim=768, num_heads=12, mlp_ratio=1.0,
                  emulate_depth=12, time_interval=1.0, num_eval_steps=24, solver="euler", register_tokens=10), 64),
}
FWD_CLASSES = ("center_rows", "gemm_in_qkv_fc1", "attn_qk", "softmax", "attn_pv", "gemm_out_rk", "fused_attn",
               "fused_attn_export")
RTOL, ATOL = 1e-3, 1e-5
T = torch.tensor([0.0, 0.5, 1.0])


def profiled(fn):
    """(forward-class ms, other-class ms) of the kernels `fn` launches."""
    torch.cuda.synchronize()
    _lib.profile_reserve(200000)
    _lib.profile_enable(True)
    fn()
    torch.cuda.synchronize()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    fwd = sum(ms for k, (ms, _) in prof.items() if k in FWD_CLASSES)
    return fwd, sum(ms for k, (ms, _) in prof.items() if k not in FWD_CLASSES)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="c10,c100")
    args = ap.parse_args()
    name, power = card()
    lines = []
    for shape in args.shapes.split(","):
        cfg, B = SHAPES[shape]
        model = ob.ViTNeuralODE(**cfg)
        model.load_state_dict(orc.reference_like_init(cfg, cfg["num_classes"], seed=0), strict=True)
        model = model.cuda().train()
        model.precision = "bf16"
        func = model.odefunc
        px = torch.randn(B, 3, cfg["img_size"], cfg["img_size"], generator=torch.Generator().manual_seed(1)).cuda()
        labels = torch.randint(0, cfg["num_classes"], (B,), generator=torch.Generator().manual_seed(2)).cuda()
        with torch.no_grad():
            x0 = model.patch_embed(px).contiguous()
        W = torch.randn((len(T),) + tuple(x0.shape), generator=torch.Generator().manual_seed(3)).cuda()

        def fwd():
            x = x0.clone().requires_grad_(True)
            return ob.odeint_adaptive(func, x, T, rtol=RTOL, atol=ATOL, differentiable=True, return_stats=True)

        def bwd(mode):
            func.block.backward_mode = mode
            states, _ = fwd()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            (states * W).sum().backward()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3

        fwd_ms, (states, st) = timed(fwd, args.reps)
        nfe = st["nfe"].double().mean().item()
        S = int(st["accepted"].max().item())
        bwd_ms = {}
        for mode in ("tape", "recompute"):
            bwd(mode)
            bwd_ms[mode] = sum(bwd(mode) for _ in range(args.reps)) / args.reps
        phases = {}
        for mode in ("tape", "recompute"):
            func.block.backward_mode = mode
            s_, _ = fwd()
            torch.cuda.synchronize()
            phases[mode] = profiled(lambda: (s_ * W).sum().backward())
        func.block.backward_mode = "auto"

        steps = max(1, round(nfe / 4))
        grid = torch.linspace(0.0, 1.0, steps + 1)

        def train_adaptive():
            model.zero_grad(set_to_none=True)
            model.adaptive_solve = {"rtol": RTOL, "atol": ATOL, "differentiable": True}
            out = model(px, labels=labels, t_grid=T)
            out["loss"].backward()
            model.adaptive_solve = None
            return out["loss"]

        def train_rk4():
            model.zero_grad(set_to_none=True)
            model.solver = "rk4"
            out = model(px, labels=labels, t_grid=grid)
            out["loss"].backward()
            return out["loss"]

        ms_ad, loss_ad = timed(train_adaptive, args.reps)
        ms_rk, loss_rk = timed(train_rk4, args.reps)
        line = dict(shape=shape, batch=B, tokens=x0.shape[1], dim=cfg["embed_dim"], precision="bf16", rtol=RTOL,
                    atol=ATOL, n_out=len(T), nfe_fwd_mean=round(nfe, 2), nfe_fwd_max=int(st["nfe"].max().item()), S=S,
                    accepted_mean=round(st["accepted"].double().mean().item(), 2),
                    rejected_total=int(st["rejected"].sum().item()), bwd_evals_tape=6 * S + 1,
                    bwd_evals_recompute=12 * S + 1, bwd_vjps=6 * S + 1,
                    fwd_record_ms=round(fwd_ms, 2), bwd_tape_ms=round(bwd_ms["tape"], 2),
                    bwd_recompute_ms=round(bwd_ms["recompute"], 2),
                    replay_kernel_ms=round(phases["tape"][0], 2), reverse_kernel_ms=round(phases["tape"][1], 2),
                    recompute_kernel_ms=round(phases["recompute"][0] - phases["tape"][0], 2),
                    train_step_ms=round(ms_ad, 2), train_img_per_s=round(B / ms_ad * 1e3, 1),
                    rk4_steps=steps, rk4_nfe_fwd=4 * steps, rk4_train_step_ms=round(ms_rk, 2),
                    rk4_train_img_per_s=round(B / ms_rk * 1e3, 1), loss=loss_ad.item(), rk4_loss=loss_rk.item(),
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
