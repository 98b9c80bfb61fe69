"""CPU tests of the gradient of the adaptive Dormand-Prince solve as tests/_adaptive_grad_ref.py states it on top of
oracle/adaptive_dp5.py: `replay` (the forward with the accepted steps given) and `interp_vjp` (the closed-form VJP of
the dense output), the reference that tests/test_gpu_adaptive_grad.py holds odevit_solve_adaptive_bwd to; and the new
C-ABI symbols."""
import ctypes

import torch

import _adaptive_grad_ref as ref
import adaptive_dp5 as dp
from odevit_b200 import _lib

T_OUT = torch.tensor([0.0, 0.3, 0.35, 1.0, 1.5], dtype=torch.float64)


def _field(seed=0, n=6):
    """A small nonlinear autonomous field acting on each image separately: [B, 2, n] -> [B, 2, n]."""
    g = torch.Generator().manual_seed(seed)
    W = (torch.randn(n, n, generator=g, dtype=torch.float64) / n ** 0.5).requires_grad_(True)
    c = (0.3 * torch.randn(n, generator=g, dtype=torch.float64)).requires_grad_(True)
    return (lambda y: torch.tanh(y @ W + c) * y.roll(1, -1) - 0.5 * y), (W, c)


def _x0(B=3, n=6, seed=1):
    x = torch.randn(B, 2, n, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    x[1] *= 3.0   # a stiffer image: more steps than its batch-mates
    return x


def _solve(f, x0, rtol=1e-4, atol=1e-6):
    with torch.no_grad():
        r = dp.dopri5(f, x0, T_OUT, rtol, atol, record_steps=True)
    r["step_t0"], r["step_dt"], r["step_out"] = ref.record_from_steps(r["steps"], T_OUT)
    return r


def test_record_layout():
    f, _ = _field()
    r = _solve(f, _x0())
    acc = r["accepted"].tolist()
    S, B = r["step_dt"].shape
    assert S == max(acc) and B == 3
    for b in range(B):
        steps = [s for s in r["steps"][b] if s[2]]
        assert len(steps) == acc[b]
        assert r["step_t0"][:acc[b], b].tolist() == [s[0] for s in steps]
        assert r["step_dt"][:acc[b], b].tolist() == [s[1] for s in steps]
        assert (r["step_dt"][acc[b]:, b] == 0).all() and (r["step_out"][acc[b]:, b] == 0).all()
        assert int(r["step_out"][acc[b] - 1, b]) == len(T_OUT)
        assert (r["step_out"][1:acc[b], b] >= r["step_out"][:acc[b] - 1, b]).all()


def test_replay_reproduces_dopri5_bitwise():
    f, _ = _field()
    x0 = _x0()
    r = _solve(f, x0)
    assert len(set(r["accepted"].tolist())) > 1   # the images take different numbers of steps
    assert r["rejected"].sum() > 0                # and some attempts were rejected
    with torch.no_grad():
        states = ref.replay(f, x0, T_OUT, r["step_t0"], r["step_dt"], r["step_out"])
    assert torch.equal(states, r["states"])


def test_replay_gradcheck():
    f, (W, c) = _field(n=3)
    x0 = _x0(n=3)
    r = _solve(f, x0, rtol=1e-3, atol=1e-5)
    assert len(set(r["accepted"].tolist())) > 1
    rec = (r["step_t0"], r["step_dt"], r["step_out"])

    def fn(x, W_, c_):
        g = lambda y: torch.tanh(y @ W_ + c_) * y.roll(1, -1) - 0.5 * y   # noqa: E731
        return ref.replay(g, x, T_OUT, *rec)

    assert torch.autograd.gradcheck(fn, (x0.clone().requires_grad_(True), W.detach().clone().requires_grad_(True),
                                         c.detach().clone().requires_grad_(True)))


def test_interp_vjp_closed_form():
    g = torch.Generator().manual_seed(3)
    shape = (2, 5)
    y0, y1, k1, k3, k4, k5, k6, k7 = [torch.randn(shape, generator=g, dtype=torch.float64).requires_grad_(True)
                                      for _ in range(8)]
    k2 = torch.randn(shape, generator=g, dtype=torch.float64).requires_grad_(True)
    ks = [k1, k2, k3, k4, k5, k6, k7]
    dt = 0.37
    xs = torch.tensor([0.1, 0.55, 1.0], dtype=torch.float64)
    y_mid = y0 + dt * sum(c * k for c, k in zip(dp.DPS_C_MID, ks) if c != 0)
    coeffs = dp.interp_fit(y0, y1, y_mid, k1, k7, dt)
    out = torch.stack([dp.interp_evaluate(coeffs, x) for x in xs])
    g_rows = torch.randn(out.shape, generator=g, dtype=torch.float64)
    want = torch.autograd.grad(out, [y0, y1] + ks, g_rows, allow_unused=True)
    got = ref.interp_vjp(g_rows, xs, dt)
    torch.testing.assert_close(got["y0"], want[0], rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(got["y1"], want[1], rtol=1e-12, atol=1e-12)
    for i in range(7):
        w = want[2 + i] if want[2 + i] is not None else torch.zeros(shape, dtype=torch.float64)
        torch.testing.assert_close(got["k"][i], w, rtol=1e-12, atol=1e-12)


def test_replay_gradient_is_batch_independent():
    f, (W, c) = _field()
    x0 = _x0()
    r = _solve(f, x0)
    G = torch.randn(r["states"].shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    x = x0.clone().requires_grad_(True)
    (ref.replay(f, x, T_OUT, r["step_t0"], r["step_dt"], r["step_out"]) * G).sum().backward()
    for b in range(3):
        rb = _solve(f, x0[b:b + 1])
        xb = x0[b:b + 1].clone().requires_grad_(True)
        (ref.replay(f, xb, T_OUT, rb["step_t0"], rb["step_dt"], rb["step_out"]) * G[:, b:b + 1]).sum().backward()
        torch.testing.assert_close(xb.grad[0], x.grad[b], rtol=1e-12, atol=1e-12)


def test_new_symbols_and_workspace_kind():
    L = _lib.lib()
    for name in ("odevit_solve_adaptive_record", "odevit_solve_adaptive_bwd", "odevit_adaptive_tape_bytes"):
        assert hasattr(L, name) and name in _lib.DECLARED_SYMBOLS
    d = _lib.Desc()
    d.abi_version = _lib.ABI_VERSION
    d.batch, d.tokens, d.dim, d.heads, d.hidden = 2, 19, 64, 2, 128
    d.variant, d.precision, d.scaler = _lib.FIELD_PARALLEL, _lib.FP32, 12.0
    assert _lib.WS_SOLVE_ADAPTIVE_BWD == 5
    assert L.odevit_workspace_bytes(ctypes.byref(d), _lib.WS_SOLVE_ADAPTIVE_BWD, 0) > 0
    assert L.odevit_adaptive_tape_bytes(ctypes.byref(d), 3) > L.odevit_adaptive_tape_bytes(ctypes.byref(d), 1) > 0
    assert L.odevit_adaptive_tape_bytes(ctypes.byref(d), 0) == 0
    assert L.odevit_abi_version() == 8
