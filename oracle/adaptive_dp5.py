"""TEST INFRASTRUCTURE ONLY -- restatement of torchdiffeq's adaptive `dopri5` with the error norm taken PER IMAGE.

Published algorithm restated (torchdiffeq 0.2.x):
  * `_impl/dopri5.py`: the Dormand-Prince tableau with Shampine's embedded pair (`_DORMAND_PRINCE_SHAMPINE_TABLEAU`:
    alpha, beta, c_sol, c_error) and the dense-output midpoint weights `DPS_C_MID`;
  * `_impl/rk_common.py`: `_runge_kutta_step` (FSAL: k7 = f(y1) is the next step's k1; error = dt * sum c_error k;
    y_mid = y0 + dt * sum DPS_C_MID k), `RKAdaptiveStepsizeODESolver._adaptive_step` (accept iff ratio <= 1; the
    solver steps until t1 >= the output time and interpolates, it does not step to output times) and `_before_integrate`
    (first step from `_select_initial_step(order - 1 = 4)` unless `first_step` is given);
  * `_impl/interp.py`: `_interp_fit` (quartic through y0, y1, y_mid with slopes f0, f1) and `_interp_evaluate`;
  * `_impl/misc.py`: `_compute_error_ratio` (RMS of err / (atol + rtol max(|y0|, |y1|))), `_optimal_step_size`
    (safety 0.9, ifactor 10, dfactor 0.2, order 5; dfactor = 1 when ratio < 1) and `_select_initial_step` (Hairer's
    d0, d1, h0, d2, h1 rule with one probe evaluation at y0 + h0 f0).

Difference from torchdiffeq, on purpose (odevit_solve_adaptive does the same): the norm is taken over each image's
elements separately (dim 0 is the batch), so every image has its own t, dt, decisions and dense output, and an image's
result does not depend on the batch it sits in.  A batch of one is torchdiffeq's algorithm.  `max_num_steps` bounds the
attempted steps per image over the whole solve (torchdiffeq counts per output interval).  Only strictly increasing
output times.

The batch runs in ROUNDS, as on the GPU: one attempted step of every image per round, an image that has finished keeps
dt = 0 (its stage inputs equal y0; nothing of it changes).  Arithmetic in y0's dtype; time and dt in float64.
"""
from typing import Callable, Optional

import torch

ALPHA = [1 / 5, 3 / 10, 4 / 5, 8 / 9, 1.0, 1.0]
BETA = [
    [1 / 5],
    [3 / 40, 9 / 40],
    [44 / 45, -56 / 15, 32 / 9],
    [19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729],
    [9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656],
    [35 / 384, 0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84],
]
C_SOL = [35 / 384, 0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84, 0]
C_ERROR = [35 / 384 - 1951 / 21600, 0, 500 / 1113 - 22642 / 50085, 125 / 192 - 451 / 720,
           -2187 / 6784 + 12231 / 42400, 11 / 84 - 649 / 6300, -1 / 60]
DPS_C_MID = [6025192743 / 30085553152 / 2, 0, 51252292925 / 65400821598 / 2, -2691868925 / 45128329728 / 2,
             187940372067 / 1594534317056 / 2, -1776094331 / 19743644256 / 2, 11237099 / 235043384 / 2]
SAFETY, IFACTOR, DFACTOR, ORDER = 0.9, 10.0, 0.2, 5


class MaxStepsExceeded(RuntimeError):
    pass


def _bcast(v: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """[B] -> [B, 1, ...] in like's dtype"""
    return v.to(like.dtype).reshape((-1,) + (1,) * (like.dim() - 1))


def rms_per_image(x: torch.Tensor) -> torch.Tensor:
    """misc._rms_norm over each image's elements: [B, ...] -> [B] float64"""
    return x.double().pow(2).flatten(1).mean(1).sqrt()


def interp_fit(y0, y1, y_mid, f0, f1, dt):
    """interp._interp_fit: coefficients [e, d, c, b, a] of the quartic in x = (t - t0) / dt"""
    a = 2 * dt * (f1 - f0) - 8 * (y1 + y0) + 16 * y_mid
    b = dt * (5 * f0 - 3 * f1) + 18 * y0 + 14 * y1 - 32 * y_mid
    c = dt * (f1 - 4 * f0) - 11 * y0 - 5 * y1 + 16 * y_mid
    d = dt * f0
    e = y0
    return [e, d, c, b, a]


def interp_evaluate(coeffs, x):
    """interp._interp_evaluate at x (already (t - t0) / (t1 - t0))"""
    total = coeffs[0] + x * coeffs[1]
    xp = x
    for c in coeffs[2:]:
        xp = xp * x
        total = total + xp * c
    return total


def optimal_step_size(dt: torch.Tensor, ratio: torch.Tensor) -> torch.Tensor:
    """misc._optimal_step_size, elementwise over images (float64)"""
    dfactor = torch.where(ratio < 1, torch.ones_like(ratio), torch.full_like(ratio, DFACTOR))
    factor = torch.clamp(torch.maximum(SAFETY / ratio.clamp_min(1e-300) ** (1.0 / ORDER), dfactor), max=IFACTOR)
    return torch.where(ratio == 0, dt * IFACTOR, dt * factor)


def select_initial_step(f: Callable, y0, f0, rtol: float, atol: float):
    """misc._select_initial_step with order 4, per image: returns (dt0 [B] float64, the probe's evaluation count)"""
    scale = atol + y0.abs() * rtol
    d0 = rms_per_image(y0 / scale)
    d1 = rms_per_image(f0 / scale)
    h0 = torch.where((d0 < 1e-5) | (d1 < 1e-5), torch.full_like(d0, 1e-6), 0.01 * d0 / d1)
    y_probe = y0 + _bcast(h0, y0) * f0
    f1 = f(y_probe)
    d2 = rms_per_image((f1 - f0) / scale) / h0
    small = (d1 <= 1e-15) & (d2 <= 1e-15)
    h1 = torch.where(small, torch.maximum(torch.full_like(h0, 1e-6), h0 * 1e-3),
                     (0.01 / torch.maximum(d1, d2)) ** (1.0 / (4 + 1)))
    return torch.minimum(100 * h0, h1)


def dopri5(f: Callable, y0: torch.Tensor, t: torch.Tensor, rtol: float, atol: float,
           first_step: Optional[float] = None, max_num_steps: int = 2 ** 31 - 1, record_steps: bool = False):
    """Per-image adaptive Dormand-Prince 5(4) over the output times t (strictly increasing).

    f: [B, ...] -> [B, ...] (autonomous field, applied to the whole batch; it must treat images independently).
    Returns dict(states [len(t), B, ...], nfe, accepted, rejected ([B] int64), rounds, steps (per image: list of
    (t0, dt, accepted, error ratio) when record_steps))."""
    t = torch.as_tensor(t, dtype=torch.float64).flatten()
    if t.numel() < 2 or not bool((t[1:] > t[:-1]).all()):
        raise ValueError("t must hold >= 2 strictly increasing times")
    B = y0.shape[0]
    T = t.numel()
    states = torch.empty((T,) + tuple(y0.shape), dtype=y0.dtype)
    states[0] = y0
    y = y0.clone()
    k1 = f(y)
    nfe = torch.ones(B, dtype=torch.int64)
    if first_step is None:
        dt = select_initial_step(f, y, k1, rtol, atol)
        nfe += 1
    else:
        dt = torch.full((B,), float(first_step), dtype=torch.float64)
    t0 = torch.full((B,), float(t[0]), dtype=torch.float64)
    out_next = torch.ones(B, dtype=torch.int64)
    active = torch.ones(B, dtype=torch.bool)
    attempts = torch.zeros(B, dtype=torch.int64)
    accepted = torch.zeros(B, dtype=torch.int64)
    steps = [[] for _ in range(B)]
    rounds = 0
    while bool(active.any()):
        rounds += 1
        h = torch.where(active, dt, torch.zeros_like(dt))
        hb = _bcast(h, y)
        k = [k1]
        for i in range(5):
            yi = y + hb * sum(b * kk for b, kk in zip(BETA[i], k) if b != 0)
            k.append(f(yi))
        y1 = y + hb * sum(c * kk for c, kk in zip(BETA[5], k) if c != 0)
        k.append(f(y1))
        err = hb * sum(c * kk for c, kk in zip(C_ERROR, k) if c != 0)
        tol = atol + rtol * torch.maximum(y.abs(), y1.abs())
        ratio = rms_per_image(err / tol)
        attempts += active.long()
        if not bool(torch.isfinite(ratio[active]).all()):
            bad = [b for b in range(B) if active[b] and not torch.isfinite(ratio[b])]
            raise FloatingPointError(f"image {bad[0]}: non-finite error ratio")
        acc = active & (ratio <= 1)
        accepted += acc.long()
        y_mid = y + hb * sum(c * kk for c, kk in zip(DPS_C_MID, k) if c != 0)
        coeffs = interp_fit(y, y1, y_mid, k[0], k[6], hb)
        t1 = t0 + h
        for b in range(B):
            if record_steps and active[b]:
                steps[b].append((float(t0[b]), float(h[b]), bool(acc[b]), float(ratio[b])))
            if not acc[b]:
                continue
            while int(out_next[b]) < T and float(t[out_next[b]]) <= float(t1[b]):
                j = int(out_next[b])
                x = ((t[j] - t0[b]) / h[b]).to(y.dtype)
                states[j, b] = interp_evaluate([c[b] for c in coeffs], x)
                out_next[b] += 1
        dt_new = optimal_step_size(h, ratio)
        accb = _bcast(acc, y).bool()
        y = torch.where(accb, y1, y)
        k1 = torch.where(accb, k[6], k1)
        t0 = torch.where(acc, t1, t0)
        dt = torch.where(active, dt_new, dt)
        done = out_next >= T
        for b in range(B):
            if active[b] and not done[b]:
                if int(attempts[b]) >= max_num_steps:
                    raise MaxStepsExceeded(f"image {b}: max_num_steps ({max_num_steps}) exceeded")
                if float(t0[b] + dt[b]) == float(t0[b]):
                    raise FloatingPointError(f"image {b}: underflow in dt {float(dt[b])}")
        active = active & ~done
    nfe += 6 * attempts
    return {"states": states, "nfe": nfe, "accepted": accepted, "rejected": attempts - accepted, "rounds": rounds,
            "steps": steps}
