"""TEST INFRASTRUCTURE ONLY -- the attention outputs of the per-image dopri5 of oracle/adaptive_dp5.py (reused unchanged),
taken per image as odevit_solve_adaptive_attn defines them.

  dopri5_evaluations  dopri5 plus each image's evaluation sequence: the field is wrapped to log the state of every call
                      it receives, and dopri5's per-image `steps` say which rounds image b took part in (an image is
                      active from the first round until it finishes, so its attempts are rounds 0 .. len(steps[b]) - 1)
  jasmin_stat         the per-(image, head) JaSMin statistic of one map: ode_transformer_gpt.py:429-456 up to the
                      means (the row maximum of log(g_1 / (g_k + 1e-12) + 1e-12), or log(g_1 + 1e-12) for k = 0)
  window              image b's JaSMin window: the statistics of its last min(W, nfe_b) evaluations, in order

The reference's semantics, per image (torchdiffeq dopri5 on a batch of one): `block.attentions` is the map of the LAST
evaluation, k7 = f(y1) of the last accepted step; `attention_trajectory` lists every evaluation in order: f(x0), the
initial-step probe (when first_step is not given) and the 6 stages of every attempted step, rejected ones included.
"""
from typing import Callable, Optional

import torch

import adaptive_dp5 as dp
import odevit_oracle as orc


def dopri5_evaluations(f: Callable, y0: torch.Tensor, t, rtol: float, atol: float, first_step: Optional[float] = None,
                       max_num_steps: int = 2 ** 31 - 1):
    """dp.dopri5(..., record_steps=True) and, in "evaluations", per image b the list of its evaluations in order:
    dict(state = the field's input [N, D], step = index of the attempted step it belongs to (None for f(x0) and the
    probe), accepted = whether that step was accepted (None for f(x0) and the probe)).  Length 1 + probe + 6 attempts."""
    calls = []

    def logged(y):
        calls.append(y.detach().clone())
        return f(y)

    res = dp.dopri5(logged, y0, t, rtol, atol, first_step=first_step, max_num_steps=max_num_steps, record_steps=True)
    base = 1 if first_step is not None else 2
    assert len(calls) == base + 6 * res["rounds"]
    evals = []
    for b, steps in enumerate(res["steps"]):
        ev = [dict(state=calls[i][b], step=None, accepted=None) for i in range(base)]
        for r, (_t0, _h, ok, _ratio) in enumerate(steps):
            ev += [dict(state=calls[base + 6 * r + i][b], step=r, accepted=ok) for i in range(6)]
        evals.append(ev)
    res["evaluations"] = evals
    return res


def jasmin_stat(P: torch.Tensor, k: int) -> torch.Tensor:
    """[..., H, N, N] -> [..., H]"""
    P = torch.clamp(P, min=1e-12, max=1.0)
    P = P / (P.sum(dim=-1, keepdim=True) + 1e-12)
    g1 = orc.g_k(P, 1)
    v = torch.log(g1 + 1e-12) if k == 0 else torch.log(g1 / (orc.g_k(P, k) + 1e-12) + 1e-12)
    return v.max(dim=-1).values


def window(evals, W: int, field_map: Callable, k: int) -> torch.Tensor:
    """[min(W, len(evals)), H]: the statistic of each of the last min(W, nfe) evaluations of one image, in order.
    field_map(state [1, N, D]) -> its map [1, H, N, N]."""
    return torch.stack([jasmin_stat(field_map(e["state"][None]), k)[0] for e in evals[-W:]])
