"""GPU tests of the fixed-grid reverse sweep (odevit_solve_bwd through ops.ode_solve) with cotangents injected at the
trajectory rows: on `states`, on `final`, on `rows` with repeated indices, and on `p_last`, against fp64 autograd through
orc.odeint_fixed.  The row indices send more terms to the last row than the one-pass seed takes, and more terms to an
interior row than fit the epilogue of its stage-0 VJP, so the sweep's fallback passes run; the same objective with the
cotangents summed to one term per row takes the fused paths."""
import dataclasses
import functools

import pytest
import torch

import odevit_oracle as orc
from _util import Golden, cosine, max_rel
from test_gpu_adaptive import _model, _tokens

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-3, "bf16": 3e-2}   # the bars of the fixed-grid reverse sweep
T = torch.tensor([0.0, 0.25, 0.5, 1.0])
# row 3 (the last): g_states, g_final and three rows -> five terms, more than the one-pass seed's four;
# row 1: g_states and six rows -> seven terms, more than the stage-0 epilogue holds next to any method's stage mus
ROWS = (3, 1, 1, 3, 1, 2, 1, 1, 3, 1, 0)
# the fallback launches the overflowing rows add: at the last row an axpy per term and the seed combine in place of
# the one-pass seed (5 + 1 - 1), at row 1 an axpy per term and the seed combine of step 0 (7 + 1)
FALLBACK_LAUNCHES = 13


def _cotangents(x0, heads, with_p, seed=5):
    g = torch.Generator().manual_seed(seed)
    B, N, D = x0.shape
    Ws = torch.randn((len(T), B, N, D), generator=g, dtype=torch.float64)
    Wf = torch.randn((B, N, D), generator=g, dtype=torch.float64)
    Wr = torch.randn((len(ROWS), B, N, D), generator=g, dtype=torch.float64)
    Wp = torch.randn((B, heads, N, N), generator=g, dtype=torch.float64) if with_p else None
    return Ws, Wf, Wr, Wp


def _objective(states, final, rows, p_last, W, summed):
    Ws, Wf, Wr, Wp = (w.to(states.device, states.dtype) if w is not None else None for w in W)
    if summed:   # the same objective, one cotangent term per row
        Ws = Ws.clone()
        Ws[-1] += Wf
        for i, r in enumerate(ROWS):
            Ws[r] += Wr[i]
        L = (states * Ws).sum()
    else:
        L = (states * Ws).sum() + (final * Wf).sum() + (rows * Wr).sum()
    return L if Wp is None else L + (p_last * Wp).sum()


def _gpu(func, x0, method, mode, W, summed):
    """(g_x0, {parameter name: grad}, odevit launches of the backward)"""
    import odevit_b200 as ob
    from odevit_b200 import ops
    spec = dataclasses.replace(func.block.field_spec(func.scaler), backward=mode)
    func.zero_grad(set_to_none=True)
    x = x0.detach().clone().requires_grad_(True)
    out = ops.ode_solve(x, T, spec, method, func.block.field_weights(), row_index=ROWS, want_p_last=W[3] is not None)
    L = _objective(out["states"], out["final"], out["rows"], out["p_last"], W, summed)
    torch.cuda.synchronize()
    ob.reset_launch_count()
    L.backward()
    torch.cuda.synchronize()
    n = ob.launch_count()
    return x.grad, {k: p.grad.clone() for k, p in func.named_parameters() if p.grad is not None}, n


def _oracle(sd, field, x0, method, W):
    """fp64 autograd: (g_x0, {state-dict key: grad})"""
    sd64 = {k: v.detach().double().requires_grad_(True) for k, v in sd.items()}
    xo = x0.detach().cpu().double().requires_grad_(True)
    last_p = []

    def f(y):
        dy, p = field(y, sd64)
        last_p[:] = [p]
        return dy
    states = orc.odeint_fixed(f, xo, T.double(), method)
    rows = states.index_select(0, torch.tensor(ROWS))
    _objective(states, states[-1], rows, last_p[0], W, False).backward()
    return xo.grad, {k: v.grad for k, v in sd64.items() if v.grad is not None}


def _check(got, want, key_prefix, precision):
    g_x0, grads = got[0], got[1]
    pairs = [("x0", g_x0, want[0])] + [(n, grads[n], want[1][key_prefix + n]) for n in grads]
    assert len(pairs) >= 9
    for n, a, b in pairs:
        assert torch.isfinite(a).all(), n
        if precision == "fp32":
            assert max_rel(a, b) <= TOL["fp32"], n
        else:
            assert max_rel(a, b) <= TOL["bf16"] and cosine(a, b) >= 0.999, n


@functools.lru_cache(maxsize=None)
def _parallel_case(method):
    model, sd = _model("fp32")
    x0 = _tokens(model, 2)
    W = _cotangents(x0, 3, True)
    field = lambda y, s: orc.field_parallel(y, s, 3, 12.0)   # noqa: E731
    return x0, W, _oracle(sd, field, x0, method, W)


@pytest.mark.parametrize("mode", ["tape", "recompute"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("method", ["euler", "midpoint", "rk4"])
def test_injected_cotangents_match_oracle(method, precision, mode):
    x0, W, want = _parallel_case(method)
    model, _ = _model(precision)
    func = model.odefunc
    split = _gpu(func, x0, method, mode, W, summed=False)
    summed = _gpu(func, x0, method, mode, W, summed=True)
    _check(split, want, "odefunc.", precision)
    _check(summed, want, "odefunc.", precision)
    assert split[2] - summed[2] == FALLBACK_LAUNCHES


def _d64_case(kind, method, with_p, field):
    import odevit_b200 as ob
    g = Golden("fields_d64")
    if kind == "l2":
        f = ob.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=1.0, l2_attention=True)
    else:
        f = ob.macaron.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=3.0)
    sd = g.group(kind + "/sd")
    f.load_state_dict(sd, strict=True)
    f = f.cuda()
    f.block.precision = "fp32"
    x0 = g.get(kind + "/x").cuda()
    W = _cotangents(x0, 2, with_p)
    want = _oracle(sd, field, x0, method, W)
    for summed in (False, True):
        _check(_gpu(f, x0, method, "tape", W, summed), want, "", "fp32")


def test_l2_injected_cotangents_match_oracle():
    _d64_case("l2", "midpoint", True, lambda y, s: orc.field_parallel(y, s, 2, 12.0, prefix="block.", l2=True))


def test_macaron_injected_cotangents_match_oracle():
    _d64_case("macaron", "rk4", False, lambda y, s: (orc.field_macaron(y, s, 2, 1.0, prefix="block."), None))
