"""GPU tests of the reverse sweep through the adaptive Dormand-Prince solve (odevit_solve_adaptive_record,
odevit_solve_adaptive_bwd, ops.ode_solve_adaptive(differentiable=True), the models' adaptive_solve["differentiable"])
against fp64 autograd through `replay` (tests/_adaptive_grad_ref.py), driven by the steps the GPU recorded."""
import ctypes

import pytest
import torch

import _adaptive_grad_ref as ref
import odevit_oracle as orc
from _util import Golden, cosine, max_rel
from test_gpu_adaptive import T_OUT, _model, _tokens

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-3, "bf16": 3e-2}   # the bars of the fixed-grid reverse sweep


def _weights(func):
    w = func.block.field_weights()
    names = tuple(k for k, v in w.items() if v is not None)
    return func.block.field_spec(func.scaler), names, [w[k].detach() for k in names]


def _record(func, x0, t, rtol, atol, cap=256):
    """The record entry point directly: (status, states, counts [3,B], (step_t0, step_dt, step_out) [S,B] on the CPU)."""
    from odevit_b200 import ops
    spec, names, ws = _weights(func)
    B = x0.shape[0]
    rec = (cap, torch.empty(cap, B, dtype=torch.float64, device="cuda"),
           torch.empty(cap, B, dtype=torch.float64, device="cuda"), torch.empty(cap, B, dtype=torch.int32, device="cuda"))
    t_c = (ctypes.c_float * len(t))(*t.tolist())
    with torch.no_grad():
        st, states, counts = ops._adaptive_call(x0.detach(), t_c, len(t), spec, names, ws, rtol, atol, 0.0,
                                                ops.DOPRI5_MAX_NUM_STEPS, rec)
    S = int(counts[1].max()) if st == 0 else 0
    return st, states, counts, (rec[1][:S].cpu(), rec[2][:S].cpu(), rec[3][:S].cpu().long())


def _functional(shape, seed=9):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def _gpu_grads(func, x0, t, rtol, atol, W):
    """L = sum_j <W_j, states[j]> through odeint_adaptive(differentiable=True): (g_x0, {param name: grad}, states)."""
    import odevit_b200 as ob
    func.zero_grad(set_to_none=True)
    x = x0.detach().clone().requires_grad_(True)
    states = ob.odeint_adaptive(func, x, t, rtol=rtol, atol=atol, differentiable=True)
    (states * W.cuda()).sum().backward()
    return x.grad, {n: p.grad.clone() for n, p in func.named_parameters() if p.grad is not None}, states.detach()


def _check_against_oracle(func, sd, key_prefix, field, x0, t, rtol, atol, precision):
    st, _, counts, rec = _record(func, x0, t, rtol, atol)
    assert st == 0
    W = _functional((len(t),) + tuple(x0.shape))
    g_x0, grads, _ = _gpu_grads(func, x0, t, rtol, atol, W)
    sd64 = {k: v.detach().double().requires_grad_(True) for k, v in sd.items()}
    xo = x0.detach().cpu().double().requires_grad_(True)
    (ref.replay(lambda y: field(y, sd64), xo, t.double(), *rec) * W.double()).sum().backward()
    pairs = [("x0", g_x0, xo.grad)]
    for n in grads:
        want = sd64[key_prefix + n].grad
        assert want is not None, n
        pairs.append((n, grads[n], want))
    assert len(pairs) >= 9
    for n, got, want in pairs:
        assert torch.isfinite(got).all(), n
        if precision == "fp32":
            assert max_rel(got, want) <= TOL["fp32"], n
        else:
            assert max_rel(got, want) <= TOL["bf16"] and cosine(got, want) >= 0.999, n


def test_record_matches_plain_solve():
    import odevit_b200 as ob
    model, _ = _model("fp32")
    x0 = _tokens(model, 4)
    st, states, counts, rec = _record(model.odefunc, x0, T_OUT, 1e-3, 1e-4)
    assert st == 0
    with torch.no_grad():
        plain, stats = ob.odeint_adaptive(model.odefunc, x0, T_OUT, rtol=1e-3, atol=1e-4, return_stats=True)
    assert torch.equal(states, plain)
    assert torch.equal(counts[0], stats["nfe"]) and torch.equal(counts[1], stats["accepted"])
    assert torch.equal(counts[2], stats["rejected"])
    t0, dtr, out = rec
    for b, n in enumerate(stats["accepted"].tolist()):
        assert int((dtr[:, b] > 0).sum()) == n and (dtr[n:, b] == 0).all()
        assert int(out[n - 1, b]) == len(T_OUT) and (out[n:, b] == 0).all()
        assert (t0[1:n, b] == t0[:n - 1, b] + dtr[:n - 1, b]).all()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_parallel_grads_match_oracle(precision):
    model, sd = _model(precision)
    x0 = _tokens(model, 2)
    field = lambda y, s: orc.field_parallel(y, s, 3, 12.0)[0]   # noqa: E731
    _check_against_oracle(model.odefunc, sd, "odefunc.", field, x0, T_OUT, 1e-3, 1e-4, precision)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_l2_grads_match_oracle(precision):
    import odevit_b200 as ob
    g = Golden("fields_d64")
    f = ob.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=1.0, l2_attention=True)
    f.load_state_dict(g.group("l2/sd"), strict=True)
    f = f.cuda()
    f.block.precision = precision
    field = lambda y, s: orc.field_parallel(y, s, 2, 12.0, prefix="block.", l2=True)[0]   # noqa: E731
    _check_against_oracle(f, g.group("l2/sd"), "", field, g.get("l2/x").cuda(), torch.tensor([0.0, 0.05, 0.1]), 1e-4,
                          1e-6, precision)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_macaron_grads_match_oracle(precision):
    import odevit_b200 as ob
    g = Golden("fields_d64")
    f = ob.macaron.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=3.0)
    f.load_state_dict(g.group("macaron/sd"), strict=True)
    f = f.cuda()
    f.block.precision = precision
    field = lambda y, s: orc.field_macaron(y, s, 2, 1.0, prefix="block.")   # noqa: E731
    _check_against_oracle(f, g.group("macaron/sd"), "", field, g.get("macaron/x").cuda(),
                          torch.tensor([0.0, 0.1, 0.3]), 1e-3, 1e-5, precision)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batch_independence(precision):
    model, _ = _model(precision)
    base = _tokens(model, 5, seed=2)
    for scale in (0.25, 4.0, 0.05, 16.0):   # image 3 scaled until its step count differs from its batch-mates'
        x0 = base.clone()
        x0[3] *= scale
        _, _, counts, _ = _record(model.odefunc, x0, T_OUT, 1e-3, 1e-4)
        acc = counts[1].tolist()
        if len(set(acc)) > 1:
            break
    assert len(set(acc)) > 1, acc
    W = _functional((len(T_OUT),) + tuple(x0.shape))
    g_x0, grads, _ = _gpu_grads(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W)
    summed = {}
    for b in range(5):
        g1, gr1, _ = _gpu_grads(model.odefunc, x0[b:b + 1].contiguous(), T_OUT, 1e-3, 1e-4, W[:, b:b + 1].contiguous())
        assert max_rel(g1[0], g_x0[b]) < 1e-6, b
        for n, v in gr1.items():
            summed[n] = summed.get(n, 0) + v
    assert summed.keys() == grads.keys()
    for n in grads:
        assert max_rel(grads[n], summed[n]) < 1e-4, n


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_tape_equals_recompute_and_is_deterministic(precision):
    """g_x0 has no atomics on its path: bitwise.  The weight gradients are summed by split-K atomics (as in the
    fixed-grid reverse sweep): equal up to the order of those sums."""
    model, _ = _model(precision)
    x0 = _tokens(model, 3)
    W = _functional((len(T_OUT),) + tuple(x0.shape))
    runs = {}
    for mode in ("tape", "recompute", "tape2"):
        model.odefunc.block.backward_mode = mode.rstrip("2")
        runs[mode] = _gpu_grads(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W)
    model.odefunc.block.backward_mode = "auto"
    for other in ("recompute", "tape2"):
        assert torch.equal(runs["tape"][0], runs[other][0]), other
        for n in runs["tape"][1]:
            assert max_rel(runs["tape"][1][n], runs[other][1][n]) < 1e-5, (other, n)


def test_record_retry_path(monkeypatch):
    from odevit_b200 import ops
    model, _ = _model("fp32")
    x0 = _tokens(model, 3)
    W = _functional((len(T_OUT),) + tuple(x0.shape))
    model.odefunc.block.backward_mode = "recompute"
    base = _gpu_grads(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W)
    monkeypatch.setattr(ops, "ADAPTIVE_STEP_CAP", 1)
    got = _gpu_grads(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W)
    model.odefunc.block.backward_mode = "auto"
    assert torch.equal(got[2], base[2])
    assert torch.equal(got[0], base[0])
    for n in base[1]:
        assert max_rel(got[1][n], base[1][n]) < 1e-5, n
    st, _, _, _ = _record(model.odefunc, x0, T_OUT, 1e-3, 1e-4, cap=1)
    assert st == -2   # ODEVIT_ERR_WORKSPACE: the record is full
    from odevit_b200 import _lib
    assert b"image" in _lib.lib().odevit_last_error_string() and b"step_cap" in _lib.lib().odevit_last_error_string()


def _check_model_training(model, px, labels, compose):
    model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "differentiable": True}
    model.zero_grad(set_to_none=True)
    out = model(px, labels=labels)
    out["loss"].backward()
    field = {n: p for n, p in model.odefunc.named_parameters()}
    for n, p in model.named_parameters():
        if p.grad is not None:
            assert torch.isfinite(p.grad).all(), n
    for n, p in field.items():
        assert p.grad is not None, n
    got = {n: p.grad.clone() for n, p in field.items()}
    model.zero_grad(set_to_none=True)
    compose().backward()
    for n, p in field.items():
        assert max_rel(got[n], p.grad) < 1e-5, n
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4)
    before = [p.detach().clone() for p in model.parameters()]
    opt.step()
    assert any(not torch.equal(b, p) for b, p in zip(before, model.parameters()))
    model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4}
    with pytest.raises(RuntimeError, match="inference-only"):
        model(px)
    model.adaptive_solve = None


def test_model_training_vit_neural_ode():
    import torch.nn.functional as F

    import odevit_b200 as ob
    model, _ = _model("fp32")
    model.train()
    px = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(7)).cuda()
    labels = torch.tensor([1, 4, 7], device="cuda")

    def compose():
        tokens = model.patch_embed(px)
        states = ob.odeint_adaptive(model.odefunc, tokens, model.t_grid, rtol=1e-3, atol=1e-4, differentiable=True)
        return F.cross_entropy(model.head(states[-1][:, 0]), labels, label_smoothing=0.05)

    _check_model_training(model, px, labels, compose)
    with pytest.raises(ValueError, match="output_attentions"):
        model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "differentiable": True}
        model(px, output_attentions=True)
    model.adaptive_solve = None


def test_model_training_macaron():
    import torch.nn.functional as F

    import odevit_b200 as ob
    cfg = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0,
               emulate_depth=1, time_interval=2.0, num_eval_steps=3, solver="rk4")
    torch.manual_seed(11)
    model = ob.ViTMacaron(**cfg).cuda().train()
    model.precision = "bf16"
    px = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(3)).cuda()
    labels = torch.tensor([2, 5], device="cuda")

    def compose():
        tokens = model.embed(px)
        states = ob.odeint_adaptive(model.odefunc, tokens, model.t_grid, rtol=1e-3, atol=1e-4, differentiable=True)
        return F.cross_entropy(model.head(model.norm_head(states[-1][:, 0])), labels)

    _check_model_training(model, px, labels, compose)


# ---- error paths ------------------------------------------------------------------------------------------------------
def _raw_bwd(func, x0, t, rec, n_steps, g_states, g_x0, ckpt, spec=None, ws_bytes=None):
    from odevit_b200 import _lib, ops
    spec0, names, ws = _weights(func)
    spec = spec or spec0
    B, N, D = x0.shape
    desc = spec.desc(B, N)
    w, keep = ops._pack_weights(names, ws)
    gw, gts = ops._alloc_grads(names, ws, [True] * len(ws))
    t_c = (ctypes.c_float * len(t))(*t.tolist())
    n_c = (ctypes.c_int32 * B)(*n_steps)
    cap, t0, dtr, out = rec
    buf, wsp, wsn = ops._workspace(desc, _lib.WS_SOLVE_ADAPTIVE_BWD, 0, torch.device("cuda", torch.cuda.current_device()))
    p = lambda z: ctypes.c_void_p(z.data_ptr())   # noqa: E731
    return _lib.lib().odevit_solve_adaptive_bwd(ctypes.byref(desc), ctypes.byref(w), p(x0), t_c, len(t), p(t0), p(dtr),
                                                p(out), cap, n_c, p(g_states), p(g_x0), ctypes.byref(gw), p(ckpt), None,
                                                0, wsp, wsn if ws_bytes is None else ws_bytes, ops._stream())


def test_bwd_error_paths():
    import dataclasses

    from odevit_b200 import _lib
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    func = model.odefunc
    cap = 64
    B = 2
    rec = (cap, torch.empty(cap, B, dtype=torch.float64, device="cuda"),
           torch.empty(cap, B, dtype=torch.float64, device="cuda"), torch.empty(cap, B, dtype=torch.int32, device="cuda"))
    from odevit_b200 import ops
    spec, names, ws = _weights(func)
    t_c = (ctypes.c_float * len(T_OUT))(*T_OUT.tolist())
    st, states, counts = ops._adaptive_call(x0, t_c, len(T_OUT), spec, names, ws, 1e-3, 1e-4, 0.0, 1000, rec)
    assert st == 0
    n = counts[1].tolist()
    S = max(n)
    g_states = torch.randn_like(states)
    g_x0 = torch.empty_like(x0)
    ckpt = torch.empty(S + 1, *x0.shape, device="cuda")
    assert _raw_bwd(func, x0, T_OUT, rec, n, g_states, g_x0, ckpt) == 0
    drop = dataclasses.replace(spec, attn_drop=0.1)
    assert _raw_bwd(func, x0, T_OUT, rec, n, g_states, g_x0, ckpt, spec=drop) == -1
    assert b"dropout" in _lib.lib().odevit_last_error_string()
    assert _raw_bwd(func, x0, T_OUT, rec, n, g_states.cpu(), g_x0, ckpt) == -5
    assert _raw_bwd(func, x0, T_OUT, rec, n, g_states, g_x0, ckpt.cpu()) == -5
    assert _raw_bwd(func, x0, T_OUT, rec, [n[0], cap + 1], g_states, g_x0, ckpt) == -1
    assert b"step_cap" in _lib.lib().odevit_last_error_string()
    assert _raw_bwd(func, x0, T_OUT, rec, n, g_states, g_x0, ckpt, ws_bytes=4096) == -2
    assert _raw_bwd(func, x0, T_OUT, rec, n, g_states, g_x0, ckpt) == 0   # usable afterwards
    with pytest.raises(Exception, match="dropout"):
        ops.ode_solve_adaptive(x0.requires_grad_(True), T_OUT, drop, func.block.field_weights(), 1e-3, 1e-4,
                               differentiable=True)
