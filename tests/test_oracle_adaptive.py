"""Known-answer tests of the per-image adaptive Dormand-Prince restatement (oracle/adaptive_dp5.py), the reference
that tests/test_gpu_adaptive.py holds odevit_solve_adaptive to."""
import importlib.util
import os
from fractions import Fraction as Fr

import numpy as np
import pytest
import torch

import adaptive_dp5 as dp


# exact rationals of the tableau (dopri5.py writes them as fractions)
C_SOL_Q = [Fr(35, 384), Fr(0), Fr(500, 1113), Fr(125, 192), Fr(-2187, 6784), Fr(11, 84), Fr(0)]
C_HAT_Q = [Fr(1951, 21600), Fr(0), Fr(22642, 50085), Fr(451, 720), Fr(-12231, 42400), Fr(649, 6300), Fr(1, 60)]
BETA_Q = [[Fr(1, 5)], [Fr(3, 40), Fr(9, 40)], [Fr(44, 45), Fr(-56, 15), Fr(32, 9)],
          [Fr(19372, 6561), Fr(-25360, 2187), Fr(64448, 6561), Fr(-212, 729)],
          [Fr(9017, 3168), Fr(-355, 33), Fr(46732, 5247), Fr(49, 176), Fr(-5103, 18656)],
          [Fr(35, 384), Fr(0), Fr(500, 1113), Fr(125, 192), Fr(-2187, 6784), Fr(11, 84)]]
C_NODES = [Fr(0)] + [sum(r) for r in BETA_Q]


def _order_conditions(b, order):
    """Butcher order conditions up to `order` for weights b (7 stages, A = BETA_Q)."""
    A = [[Fr(0)] * 7 for _ in range(7)]
    for i, row in enumerate(BETA_Q):
        for j, v in enumerate(row):
            A[i + 1][j] = v
    c = C_NODES
    conds = [(sum(b), Fr(1))]
    if order >= 2:
        conds.append((sum(bi * ci for bi, ci in zip(b, c)), Fr(1, 2)))
    if order >= 3:
        conds.append((sum(bi * ci ** 2 for bi, ci in zip(b, c)), Fr(1, 3)))
        conds.append((sum(b[i] * A[i][j] * c[j] for i in range(7) for j in range(7)), Fr(1, 6)))
    if order >= 4:
        conds.append((sum(bi * ci ** 3 for bi, ci in zip(b, c)), Fr(1, 4)))
        conds.append((sum(b[i] * c[i] * A[i][j] * c[j] for i in range(7) for j in range(7)), Fr(1, 8)))
        conds.append((sum(b[i] * A[i][j] * c[j] ** 2 for i in range(7) for j in range(7)), Fr(1, 12)))
        conds.append((sum(b[i] * A[i][j] * A[j][k] * c[k] for i in range(7) for j in range(7) for k in range(7)),
                      Fr(1, 24)))
    if order >= 5:
        conds.append((sum(bi * ci ** 4 for bi, ci in zip(b, c)), Fr(1, 5)))
        conds.append((sum(b[i] * c[i] ** 2 * A[i][j] * c[j] for i in range(7) for j in range(7)), Fr(1, 10)))
        conds.append((sum(b[i] * c[i] * A[i][j] * c[j] ** 2 for i in range(7) for j in range(7)), Fr(1, 15)))
        conds.append((sum(b[i] * A[i][j] * c[j] ** 3 for i in range(7) for j in range(7)), Fr(1, 20)))
        Ac = [sum(A[i][j] * c[j] for j in range(7)) for i in range(7)]
        conds.append((sum(b[i] * Ac[i] ** 2 for i in range(7)), Fr(1, 20)))
        conds.append((sum(b[i] * c[i] * A[i][j] * A[j][k] * c[k] for i in range(7) for j in range(7)
                          for k in range(7)), Fr(1, 30)))
        conds.append((sum(b[i] * A[i][j] * c[j] * A[j][k] * c[k] for i in range(7) for j in range(7)
                          for k in range(7)), Fr(1, 40)))
        conds.append((sum(b[i] * A[i][j] * A[j][k] * c[k] ** 2 for i in range(7) for j in range(7)
                          for k in range(7)), Fr(1, 60)))
        conds.append((sum(b[i] * A[i][j] * A[j][k] * A[k][m] * c[m] for i in range(7) for j in range(7)
                          for k in range(7) for m in range(7)), Fr(1, 120)))
    return conds


def test_tableau_constants_match_the_rationals():
    assert dp.ALPHA == pytest.approx([float(x) for x in C_NODES[1:]], abs=1e-15)
    for row, rq in zip(dp.BETA, BETA_Q):
        assert row == pytest.approx([float(x) for x in rq], abs=1e-15)
    assert dp.C_SOL == pytest.approx([float(x) for x in C_SOL_Q], abs=1e-15)
    assert dp.C_ERROR == pytest.approx([float(s - h) for s, h in zip(C_SOL_Q, C_HAT_Q)], abs=1e-15)


def test_tableau_order_conditions():
    for got, want in _order_conditions(C_SOL_Q, 5):
        assert got == want                              # c_sol: order 5
    c_hat = [s - e for s, e in zip(C_SOL_Q, [s - h for s, h in zip(C_SOL_Q, C_HAT_Q)])]
    for got, want in _order_conditions(c_hat, 4):
        assert got == want                              # c_sol - c_error: order 4
    assert sum(dp.C_ERROR) == pytest.approx(0.0, abs=1e-16)
    assert sum(dp.DPS_C_MID) == pytest.approx(0.5, abs=1e-15)


def test_dense_output_endpoints_and_slope():
    g = torch.Generator().manual_seed(0)
    y0, y1, ym, f0, f1 = (torch.randn(5, dtype=torch.float64, generator=g) for _ in range(5))
    dt = 0.37
    c = dp.interp_fit(y0, y1, ym, f0, f1, dt)
    assert torch.allclose(dp.interp_evaluate(c, 0.0), y0, atol=1e-14)
    assert torch.allclose(dp.interp_evaluate(c, 1.0), y1, atol=1e-13)
    eps = 1e-7
    slope = (dp.interp_evaluate(c, eps) - dp.interp_evaluate(c, -eps)) / (2 * eps) / dt
    assert torch.allclose(slope, f0, atol=1e-6)
    slope1 = (dp.interp_evaluate(c, 1 + eps) - dp.interp_evaluate(c, 1 - eps)) / (2 * eps) / dt
    assert torch.allclose(slope1, f1, atol=1e-6)


def _linear_problem():
    g = torch.Generator().manual_seed(3)
    A = torch.randn(6, 6, dtype=torch.float64, generator=g) * 0.6
    y0 = torch.randn(3, 6, dtype=torch.float64, generator=g)
    return A, y0


def test_linear_system_against_expm_scales_with_rtol():
    from scipy.linalg import expm
    A, y0 = _linear_problem()
    t = torch.tensor([0.0, 0.3, 1.1, 2.0], dtype=torch.float64)
    exact = np.stack([y0.numpy() @ expm(A.numpy() * float(ti)).T for ti in t])
    errs = []
    for rtol in (1e-3, 1e-4, 1e-5, 1e-6, 1e-7, 1e-8):
        res = dp.dopri5(lambda y: y @ A.T, y0, t, rtol=rtol, atol=rtol * 1e-2)
        err = float(np.abs(res["states"].numpy() - exact).max() / np.abs(exact).max())
        errs.append(err)
        assert err < 200 * rtol, (rtol, err)
        assert int(res["nfe"].min()) >= 8
    assert errs[-1] < errs[0] * 1e-3   # the error follows the tolerance over five decades


def _nonlinear(y):
    # per-image coupled nonlinear system (elementwise, so batch size cannot change a single rounding)
    return torch.stack([y[:, 1], -y[:, 0] + 0.8 * (1 - y[:, 0] ** 2) * y[:, 1], torch.sin(y[:, 0]) - 0.3 * y[:, 2]], 1)


def test_nonlinear_against_dop853():
    from scipy.integrate import solve_ivp
    y0 = torch.tensor([[1.5, 0.0, 0.2], [0.3, -0.7, 1.0]], dtype=torch.float64)
    t = torch.linspace(0.0, 4.0, 9, dtype=torch.float64)
    res = dp.dopri5(_nonlinear, y0, t, rtol=1e-9, atol=1e-11)
    for b in range(2):
        ref = solve_ivp(lambda _t, y: _nonlinear(torch.from_numpy(y)[None])[0].numpy(), (0.0, 4.0), y0[b].numpy(),
                        method="DOP853", rtol=1e-13, atol=1e-15, t_eval=t.numpy())
        assert np.abs(res["states"][:, b].numpy() - ref.y.T).max() < 1e-7


def test_batched_equals_per_image_exactly():
    y0 = torch.tensor([[1.5, 0.0, 0.2], [0.3, -0.7, 1.0], [2.0, 0.5, -0.4]], dtype=torch.float64)
    y0[1] *= 1e-3    # very different step sequences within one batch
    t = torch.tensor([0.0, 0.5, 3.0], dtype=torch.float64)
    res = dp.dopri5(_nonlinear, y0, t, rtol=1e-6, atol=1e-9, record_steps=True)
    assert len({int(n) for n in res["nfe"]}) > 1
    for b in range(3):
        one = dp.dopri5(_nonlinear, y0[b:b + 1], t, rtol=1e-6, atol=1e-9, record_steps=True)
        assert torch.equal(one["states"][:, 0], res["states"][:, b])
        assert one["steps"][0] == res["steps"][b]
        assert int(one["nfe"][0]) == int(res["nfe"][b]) == 2 + 6 * len(one["steps"][0])
    assert res["rounds"] == max(len(s) for s in res["steps"])


def test_output_times_do_not_change_the_steps():
    y0 = torch.tensor([[1.5, 0.0, 0.2], [0.3, -0.7, 1.0]], dtype=torch.float64)
    coarse = dp.dopri5(_nonlinear, y0, torch.tensor([0.0, 3.0], dtype=torch.float64), 1e-5, 1e-8, record_steps=True)
    fine_t = torch.tensor([0.0, 0.1, 0.2, 1.0, 1.7, 2.9, 3.0], dtype=torch.float64)
    fine = dp.dopri5(_nonlinear, y0, fine_t, 1e-5, 1e-8, record_steps=True)
    assert coarse["steps"] == fine["steps"]
    assert torch.equal(coarse["states"][-1], fine["states"][-1])


def test_first_step_option_and_max_num_steps():
    y0 = torch.tensor([[1.5, 0.0, 0.2]], dtype=torch.float64)
    t = torch.tensor([0.0, 3.0], dtype=torch.float64)
    res = dp.dopri5(_nonlinear, y0, t, 1e-5, 1e-8, first_step=0.01, record_steps=True)
    assert res["steps"][0][0][1] == 0.01   # (t0, dt, accepted, ratio) of the first attempt
    assert int(res["nfe"][0]) == 1 + 6 * len(res["steps"][0])
    with pytest.raises(dp.MaxStepsExceeded, match="image 0"):
        dp.dopri5(_nonlinear, y0, t, 1e-8, 1e-10, max_num_steps=5)
    with pytest.raises(ValueError):
        dp.dopri5(_nonlinear, y0, torch.tensor([1.0, 0.0], dtype=torch.float64), 1e-5, 1e-8)


def _real_torchdiffeq():
    spec = importlib.util.find_spec("torchdiffeq")
    if spec is None or spec.origin is None:
        return None
    if os.sep + "shims" + os.sep in spec.origin:   # the fixed-grid stand-in under oracle/shims
        return None
    import torchdiffeq
    return torchdiffeq if hasattr(torchdiffeq, "odeint") else None


@pytest.mark.skipif(_real_torchdiffeq() is None, reason="torchdiffeq is not installed")
def test_batch_of_one_matches_torchdiffeq_dopri5():
    tde = _real_torchdiffeq()
    y0 = torch.tensor([[1.5, 0.0, 0.2]], dtype=torch.float64)
    t = torch.tensor([0.0, 0.4, 1.3, 3.0], dtype=torch.float64)
    want = tde.odeint(lambda _t, y: _nonlinear(y), y0, t, method="dopri5", rtol=1e-6, atol=1e-9)
    got = dp.dopri5(_nonlinear, y0, t, 1e-6, 1e-9)["states"]
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-13)
