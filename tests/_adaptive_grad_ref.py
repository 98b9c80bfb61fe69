"""TEST INFRASTRUCTURE ONLY -- the gradient odevit_solve_adaptive_bwd computes, restated on top of the per-image dopri5
of oracle/adaptive_dp5.py (which this module reuses unchanged: its tableau, interp_fit / interp_evaluate and the
`steps` list of dopri5(record_steps=True)).

  record_from_steps  dopri5's per-image `steps` -> the accepted steps in the layout of odevit_solve_adaptive_record
  replay             the forward with the accepted steps GIVEN: plain differentiable torch; its fp64 autograd is the
                     reference gradient (discretise-then-optimise, steps frozen)
  interp_vjp         the closed-form VJP of one step's dense output (what ad_interp_vjp_kernel computes)
"""
from typing import Callable

import torch

import adaptive_dp5 as dp


def _bcast(v: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """[B] -> [B, 1, ...] in like's dtype"""
    return v.to(like.dtype).reshape((-1,) + (1,) * (like.dim() - 1))


def record_from_steps(steps, t_out):
    """The accepted steps of dopri5's `steps` (per image: (t0, dt, accepted, ratio) of every attempt) as
    (step_t0, step_dt [S, B] float64, step_out [S, B] int64), S = max accepted, zero past an image's count.
    step_out is the first output index not yet written after the step: dopri5 writes output j from the accepted step
    that first has t_out[j] <= t0 + dt (the same fp64 sum)."""
    t = [float(v) for v in torch.as_tensor(t_out, dtype=torch.float64).flatten()]
    acc = [[(t0, h) for t0, h, ok, _ in s if ok] for s in steps]
    S, B = max(len(a) for a in acc), len(acc)
    step_t0 = torch.zeros(S, B, dtype=torch.float64)
    step_dt = torch.zeros(S, B, dtype=torch.float64)
    step_out = torch.zeros(S, B, dtype=torch.int64)
    for b, a in enumerate(acc):
        on = 1
        for s, (t0, h) in enumerate(a):
            t1 = t0 + h
            while on < len(t) and t[on] <= t1:
                on += 1
            step_t0[s, b], step_dt[s, b], step_out[s, b] = t0, h, on
    return step_t0, step_dt, step_out


def replay(f: Callable, y0: torch.Tensor, t_out, step_t0: torch.Tensor, step_dt: torch.Tensor,
           step_out: torch.Tensor) -> torch.Tensor:
    """The forward of dopri5 with the accepted steps given (layout of record_from_steps / odevit_solve_adaptive_record):
    round s runs step s of every image (dt = 0 past an image's count: an identity step) with dopri5's stage, FSAL and
    dense-output arithmetic, and writes the outputs step_out[s - 1] <= j < step_out[s] (from 1 for s = 0) from the
    step's quartic.  The steps, the outputs' positions x = (t_out[j] - t0) / dt and the rejected attempts are
    constants.  Returns states [len(t_out), B, ...]."""
    t = torch.as_tensor(t_out, dtype=torch.float64).flatten()
    S, B = step_dt.shape
    rows = [[None] * B for _ in range(t.numel())]
    rows[0] = list(y0.unbind(0))
    y = y0
    k1 = f(y)
    for s in range(S):
        h = step_dt[s].to(torch.float64)
        hb = _bcast(h, y)
        k = [k1]
        for i in range(5):
            yi = y + hb * sum(b * kk for b, kk in zip(dp.BETA[i], k) if b != 0)
            k.append(f(yi))
        y1 = y + hb * sum(c * kk for c, kk in zip(dp.BETA[5], k) if c != 0)
        k.append(f(y1))
        y_mid = y + hb * sum(c * kk for c, kk in zip(dp.DPS_C_MID, k) if c != 0)
        coeffs = dp.interp_fit(y, y1, y_mid, k[0], k[6], hb)
        for b in range(B):
            lo = int(step_out[s - 1, b]) if s else 1
            for j in range(lo, int(step_out[s, b])):
                x = ((t[j] - step_t0[s, b]) / h[b]).to(y.dtype)
                rows[j][b] = dp.interp_evaluate([c[b] for c in coeffs], x)
        y, k1 = y1, k[6]
    return torch.stack([torch.stack(r) for r in rows])


def interp_vjp(g_rows: torch.Tensor, xs: torch.Tensor, dt):
    """Closed-form VJP of the dense output of one step: g_rows [J, ...] are the cotangents of the outputs at positions
    xs [J] of a step of size dt.  The power sums S_p = sum_j x_j^p g_j are the cotangents of interp_fit's coefficients
    [e, d, c, b, a] = [S0, S1, S2, S3, S4]; interp_fit's linear map takes them to y0, y1, y_mid, f0 = k1 and f1 = k7, and
    y_mid = y0 + dt sum_l DPS_C_MID[l] k_l spreads its cotangent onto y0 and onto k_l with dt * DPS_C_MID[l].
    Returns dict(y0, y1, k = [cotangents of k1..k7])."""
    xs = xs.reshape((-1,) + (1,) * (g_rows.dim() - 1)).to(g_rows.dtype)
    S0, S1, S2, S3, S4 = [(xs ** p * g_rows).sum(0) for p in range(5)]
    g_mid = 16 * S2 - 32 * S3 + 16 * S4
    g_f0 = dt * (S1 - 4 * S2 + 5 * S3 - 2 * S4)
    g_f1 = dt * (S2 - 3 * S3 + 2 * S4)
    k = [dt * c * g_mid for c in dp.DPS_C_MID]
    k[0] = k[0] + g_f0
    k[6] = k[6] + g_f1
    return {"y0": S0 - 11 * S2 + 18 * S3 - 8 * S4 + g_mid, "y1": -5 * S2 + 14 * S3 - 8 * S4, "k": k}
