"""What the attention outputs of the adaptive Dormand-Prince solve cost (ops.ode_solve_adaptive(want_p_last, jasmin),
odevit_solve_adaptive_attn / odevit_solve_adaptive_bwd_attn), bf16, seeded random weights of the reference's init
statistics and seeded random images, one JSON line each:
  solve     c10 shape (32 px, D 192, 3 heads, 65 tokens), batch 512, t = [0, 0.5, 1], rtol 1e-3 / atol 1e-5:
              fwd_ms            inference solve without attention outputs
              fwd_attn_ms       the same with p_last and the JaSMin window (W = 30, k = 2: statistic in the attention
                                kernel), one extra evaluation and one small kernel per evaluation expected
              fwd_record_ms / fwd_record_attn_ms   the differentiable forward (with the accepted-step record)
              bwd_ms / bwd_p_last_ms   its backward with a loss on the states, and on the states plus p_last
  distill   one ImageDistilTrainer-style step (student forward with control points, attentions and jasmin_loss, library
            ViT-B/16 teacher, the trajectory losses, backward, AdamW) on an adaptive student (differentiable, dropout 0) at
            the distillation shape (224 px, D 768, 12 heads, 207 tokens, 36 output times), batch 64
and the card's name and power limit.  Times are host clocks around work that ends synchronised.

    python tools/adaptive_attn_cost.py [--out profiles/adaptive_attn_cost.jsonl] [--reps 5]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import odevit_b200 as ob  # noqa: E402
from adaptive_sweep import card, timed  # noqa: E402
from distill_step import distillation_loss  # noqa: E402
from odevit_b200 import ops  # noqa: E402


def solve_line(reps):
    cfg = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
               time_interval=1.0, num_eval_steps=5, solver="rk4", register_tokens=0)
    torch.manual_seed(0)
    model = ob.ViTNeuralODE(**cfg).cuda()
    model.precision = "bf16"
    B = 512
    px = torch.randn(B, 3, 32, 32, generator=torch.Generator().manual_seed(1)).cuda()
    with torch.no_grad():
        x0 = model.patch_embed(px).contiguous()
    t = torch.tensor([0.0, 0.5, 1.0])
    blk = model.odefunc.block
    spec, w = blk.field_spec(model.odefunc.scaler), blk.field_weights()
    rtol, atol, W, k = 1e-3, 1e-5, 30, 2

    def fwd(attn):
        with torch.no_grad():
            return ops.ode_solve_adaptive(x0, t, spec, w, rtol, atol, want_p_last=attn, jasmin=(W, k) if attn else None)

    def rec(attn):
        x = x0.clone().requires_grad_(True)
        return x, ops.ode_solve_adaptive(x, t, spec, w, rtol, atol, differentiable=True, want_p_last=attn,
                                         jasmin=(W, k) if attn else None)

    g_s = torch.randn(len(t), *x0.shape, generator=torch.Generator().manual_seed(2)).cuda()
    g_p = torch.randn(B, 3, x0.shape[1], x0.shape[1], generator=torch.Generator().manual_seed(3)).cuda()

    def bwd(with_p):
        x, res = rec(with_p)
        torch.cuda.synchronize()
        loss = (res["states"] * g_s).sum() + ((res["p_last"] * g_p).sum() if with_p else 0.0)
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        loss.backward()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1)

    out = {"case": "solve", "batch": B, "tokens": x0.shape[1], "dim": 192, "precision": "bf16", "rtol": rtol,
           "atol": atol, "jas_window": W, "jas_k": k}
    base = fwd(False)
    out["nfe_mean"] = round(float(base["nfe"].float().mean()), 2)
    out["rounds"] = base["rounds"]
    for _ in range(2):   # alternate the two forms so drift hits both
        for name, fn in (("fwd_ms", lambda: fwd(False)), ("fwd_attn_ms", lambda: fwd(True)),
                         ("fwd_record_ms", lambda: rec(False)), ("fwd_record_attn_ms", lambda: rec(True))):
            ms, _ = timed(fn, reps)
            out[name] = min(out.get(name, 1e30), round(ms, 2))
        for name, flag in (("bwd_ms", False), ("bwd_p_last_ms", True)):
            bwd(flag)
            ms = min(bwd(flag) for _ in range(reps))
            out[name] = min(out.get(name, 1e30), round(ms, 2))
    return out


def distill_line(reps):
    from transformers import ViTConfig, ViTForImageClassification
    torch.manual_seed(1)
    hf = ViTForImageClassification(ViTConfig(num_labels=100, attn_implementation="eager")).cuda().eval()
    teacher = ob.ViTTeacher(hf, precision="bf16", attention_maps="last")
    cfg = dict(img_size=224, patch_size=16, num_classes=100, embed_dim=768, num_heads=12, mlp_ratio=4.0,
               emulate_depth=12, time_interval=1.0, num_eval_steps=36, solver="euler", register_tokens=10)
    torch.manual_seed(0)
    student = ob.ViTNeuralODE(**cfg).cuda().train()
    student.precision = "bf16"
    student.adaptive_solve = {"rtol": 1e-3, "atol": 1e-5, "differentiable": True, "attention_outputs": True}
    opt = torch.optim.AdamW(student.parameters(), lr=1e-4, weight_decay=5e-2)
    B = 64
    px = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(1234)).cuda()
    nfe = []

    def step():
        opt.zero_grad(set_to_none=True)
        s = student(px, output_hidden_states=True, output_control_points=True, output_attentions=True, jasmin_k=2)
        with torch.no_grad():
            t = teacher(pixel_values=px, output_hidden_states=True, output_attentions=True)
        loss = distillation_loss(s, t)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(student.parameters(), 1.0)
        opt.step()
        nfe.append(float(s["nfe"].float().mean()))
        return loss

    ms, loss = timed(step, reps)
    return {"case": "distill", "batch": B, "tokens": 207, "dim": 768, "precision": "bf16", "rtol": 1e-3, "atol": 1e-5,
            "n_out": 36, "nfe_mean": round(sum(nfe) / len(nfe), 2), "step_ms": round(ms, 1),
            "img_per_s": round(B * 1e3 / ms, 1), "loss": round(float(loss), 5)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, power = card()
    lines = [solve_line(a.reps), distill_line(max(2, a.reps // 2))]
    with open(a.out, "a") if a.out else open(os.devnull, "w") as f:
        for line in lines:
            line.update(gpu=name, power_limit=power, reps=a.reps)
            s = json.dumps(line)
            print(s)
            f.write(s + "\n")


if __name__ == "__main__":
    main()
