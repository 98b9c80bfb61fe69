"""GPU tests of the per-image adaptive Dormand-Prince solve (odevit_solve_adaptive, ops.ode_solve_adaptive,
odevit_b200.odeint_adaptive, the models' `adaptive_solve`) against the restatement in oracle/adaptive_dp5.py."""
import ctypes

import pytest
import torch

import adaptive_dp5 as dp
import odevit_oracle as orc
from _util import Golden, max_rel

pytestmark = pytest.mark.gpu

CFG = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
           time_interval=1.0, num_eval_steps=5, solver="rk4", register_tokens=4)
T_OUT = torch.tensor([0.0, 0.25, 0.5, 1.0])


def _model(precision, seed=0):
    import odevit_b200 as ob
    sd = orc.reference_like_init(CFG, 10, seed=seed)
    model = ob.ViTNeuralODE(**CFG)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    model.precision = precision
    return model, sd


def _tokens(model, B, seed=1):
    px = torch.randn(B, 3, 32, 32, generator=torch.Generator().manual_seed(seed))
    with torch.no_grad():
        return model.patch_embed(px.cuda()).detach().contiguous()


def _solve(model, x0, t=T_OUT, rtol=1e-3, atol=1e-4, **kw):
    import odevit_b200 as ob
    with torch.no_grad():
        states, stats = ob.odeint_adaptive(model.odefunc, x0, t, rtol=rtol, atol=atol, options=kw or None,
                                           return_stats=True)
    return states, stats


def _oracle(sd, x0, t=T_OUT, rtol=1e-3, atol=1e-4, prefix="odefunc.block.", l2=False, macaron=False, heads=3,
            scaler=12.0):
    # the fp32 field of the restatement; stage combines, norms and time in fp64
    def f(y):
        if macaron:
            return orc.field_macaron(y.float(), sd, heads, scaler, prefix=prefix).double()
        return orc.field_parallel(y.float(), sd, heads, scaler, prefix=prefix, l2=l2)[0].double()
    with torch.no_grad():
        return dp.dopri5(f, x0.detach().cpu().double(), t.double(), rtol, atol)


def _counts(stats):
    return stats["accepted"].cpu().tolist(), stats["rejected"].cpu().tolist()


# seed 0 of reference_like_init: no image's error ratio lies within 1e-4 of 1 at rtol 1e-3 (checked against the oracle
# when the test was written; the counts would otherwise depend on rounding, not on the algorithm)
def test_fp32_matches_oracle_counts_and_states():
    model, sd = _model("fp32")
    x0 = _tokens(model, 4)
    states, stats = _solve(model, x0)
    want = _oracle(sd, x0)
    assert _counts(stats) == (want["accepted"].tolist(), want["rejected"].tolist())
    assert stats["nfe"].cpu().tolist() == want["nfe"].tolist()
    assert stats["rounds"] == int((want["accepted"] + want["rejected"]).max())
    assert max_rel(states, want["states"]) < 1e-4


def test_bf16_matches_oracle():
    model, sd = _model("bf16")
    x0 = _tokens(model, 4)
    states, stats = _solve(model, x0)
    want = _oracle(sd, x0)
    assert max_rel(states, want["states"]) < 2e-2
    assert states.shape == (len(T_OUT), 4, x0.shape[1], 192)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batch_independence(precision):
    model, _ = _model(precision)
    x0 = _tokens(model, 5, seed=2)
    x0[3] *= 0.25    # an image with a different step sequence in the same batch
    states, stats = _solve(model, x0)
    acc, rej = _counts(stats)
    for b in range(5):
        s1, st1 = _solve(model, x0[b:b + 1].contiguous())
        assert _counts(st1) == ([acc[b]], [rej[b]]), b
        assert max_rel(s1[:, 0], states[:, b]) < 1e-6, b


def test_tight_tolerance_agrees_with_fine_fixed_grid():
    import odevit_b200 as ob
    model, _ = _model("fp32")
    x0 = _tokens(model, 2)
    states, _ = _solve(model, x0, t=torch.tensor([0.0, 1.0]), rtol=1e-7, atol=1e-9)
    with torch.no_grad():
        ref = ob.odeint(model.odefunc, x0, torch.linspace(0.0, 1.0, 513), method="rk4", record_attention=False)
    assert max_rel(states[-1], ref[-1]) < 1e-4


def test_more_output_times_keep_the_counts():
    model, _ = _model("fp32")
    x0 = _tokens(model, 3)
    _, st_a = _solve(model, x0, t=torch.tensor([0.0, 1.0]))
    s_b, st_b = _solve(model, x0, t=torch.linspace(0.0, 1.0, 17))
    assert _counts(st_a) == _counts(st_b)
    assert st_a["nfe"].cpu().tolist() == st_b["nfe"].cpu().tolist()


def test_first_step_option_and_nfe():
    model, sd = _model("fp32")
    x0 = _tokens(model, 2)
    states, stats = _solve(model, x0, first_step=0.05)
    want = dp.dopri5(lambda y: orc.field_parallel(y.float(), sd, 3, 12.0)[0].double(), x0.cpu().double(),
                     T_OUT.double(), 1e-3, 1e-4, first_step=0.05)
    acc, rej = _counts(stats)
    assert acc == want["accepted"].tolist() and rej == want["rejected"].tolist()
    assert stats["nfe"].cpu().tolist() == [1 + 6 * (a + r) for a, r in zip(acc, rej)]
    assert max_rel(states, want["states"]) < 1e-4


def test_counts_are_deterministic():
    model, _ = _model("bf16")
    x0 = _tokens(model, 8)
    runs = [_solve(model, x0) for _ in range(3)]
    for s, st in runs[1:]:
        assert _counts(st) == _counts(runs[0][1])
        assert torch.equal(s, runs[0][0])


def test_l2_field_matches_oracle():
    import odevit_b200 as ob
    g = Golden("fields_d64")
    f = ob.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=1.0, l2_attention=True)
    f.load_state_dict(g.group("l2/sd"), strict=True)
    f = f.cuda()
    f.block.precision = "fp32"
    x0 = g.get("l2/x").cuda()
    t = torch.tensor([0.0, 0.05, 0.1])
    with torch.no_grad():
        states, stats = ob.odeint_adaptive(f, x0, t, rtol=1e-4, atol=1e-6, return_stats=True)
    want = _oracle(g.group("l2/sd"), x0, t=t, rtol=1e-4, atol=1e-6, prefix="block.", l2=True, heads=2, scaler=12.0)
    assert _counts(stats) == (want["accepted"].tolist(), want["rejected"].tolist())
    assert max_rel(states, want["states"]) < 1e-4


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 2e-2)])
def test_macaron_field_matches_oracle(precision, tol):
    import odevit_b200 as ob
    g = Golden("fields_d64")
    f = ob.macaron.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=3.0)
    assert f.scaler == 1.0
    f.load_state_dict(g.group("macaron/sd"), strict=True)
    f = f.cuda()
    f.block.precision = precision
    x0 = g.get("macaron/x").cuda()
    t = torch.tensor([0.0, 0.1, 0.3])
    with torch.no_grad():
        states, stats = ob.odeint_adaptive(f, x0, t, rtol=1e-3, atol=1e-5, return_stats=True)
    want = _oracle(g.group("macaron/sd"), x0, t=t, rtol=1e-3, atol=1e-5, prefix="block.", macaron=True, heads=2,
                   scaler=1.0)
    if precision == "fp32":
        assert _counts(stats) == (want["accepted"].tolist(), want["rejected"].tolist())
    assert int((stats["accepted"] + stats["rejected"]).max()) <= 10
    assert max_rel(states, want["states"]) < tol


def test_model_adaptive_solve_logits_are_head_of_final_state():
    import odevit_b200 as ob
    model, _ = _model("fp32")
    px = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(7)).cuda()
    with torch.no_grad():
        plain = model(px)
        model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4}
        out = model(px, output_hidden_states=True)
        tokens = model.patch_embed(px)
        states, stats = ob.odeint_adaptive(model.odefunc, tokens, model.t_grid, rtol=1e-3, atol=1e-4,
                                           return_stats=True)
    assert max_rel(out["states"], states) < 1e-6
    assert torch.equal(out["nfe"], stats["nfe"])
    with torch.no_grad():
        assert torch.equal(out["logits"], model.head(out["states"][-1][:, 0]))
        assert max_rel(out["logits"], model.head(states[-1][:, 0])) < 1e-6
    assert out["finite_difference_upper_bound"]["batched_upper_bound"].shape == (3,)
    with pytest.raises(ValueError, match="output_attentions"):
        with torch.no_grad():
            model(px, output_attentions=True)
    with pytest.raises(RuntimeError, match="inference-only"):
        model(px)   # gradients enabled and the parameters require them
    model.adaptive_solve = None
    with torch.no_grad():
        assert torch.equal(model(px)["logits"], plain["logits"])


def test_macaron_model_adaptive_solve():
    import odevit_b200 as ob
    cfg = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0,
               emulate_depth=1, time_interval=2.0, num_eval_steps=3, solver="rk4")
    torch.manual_seed(11)
    model = ob.ViTMacaron(**cfg).cuda().eval()
    model.precision = "bf16"
    model.adaptive_solve = {"rtol": 1e-2, "atol": 1e-3, "max_num_steps": 50}
    px = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(3)).cuda()
    with torch.no_grad():
        out = model(px, output_hidden_states=True)
    assert out["states"].shape[0] == 3 and out["nfe"].shape == (2,)
    assert torch.allclose(out["logits"], model.head(model.norm_head(out["states"][-1][:, 0])))


# ---- error paths ------------------------------------------------------------------------------------------------------
def test_max_num_steps_raises():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    with pytest.raises(ob.NotConvergedError, match="image .*max_num_steps"):
        _solve(model, x0, rtol=1e-8, atol=1e-10, max_num_steps=3)
    _solve(model, x0)   # the library is usable afterwards


def test_bad_times_raise():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    for t in (torch.tensor([0.0, 0.5, 0.4]), torch.tensor([1.0, 0.0]), torch.tensor([0.0, 0.0, 1.0]),
              torch.tensor([0.0])):
        with pytest.raises(ob.OdevitError, match="t_out"):
            _solve(model, x0, t=t)


def test_gradient_request_raises():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    with pytest.raises(ob.OdevitError, match="inference-only"):
        ob.odeint_adaptive(model.odefunc, x0.requires_grad_(True), T_OUT)
    with pytest.raises(ob.OdevitError, match="inference-only"):
        ob.odeint_adaptive(model.odefunc, x0.detach(), T_OUT)   # the weights require grad


def test_capture_is_refused():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    _solve(model, x0)   # workspace allocated outside the capture
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), pytest.raises(ob.OdevitError, match="captured"):
        with torch.cuda.graph(g, stream=s):
            ob.odeint_adaptive(model.odefunc, x0, T_OUT)


def _raw_call(spec, x0, states, t, counts=None):
    """The C ABI directly (what ops.ode_solve_adaptive checks before it gets there is bypassed)."""
    from odevit_b200 import _lib, ops
    B, N, D = x0.shape
    desc = spec.desc(B, N)
    model_w = _RAW_W
    w, keep = ops._pack_weights(tuple(model_w), [model_w[k] for k in model_w])
    t_c = (ctypes.c_float * len(t))(*t)
    buf, ws, ws_bytes = ops._workspace(desc, _lib.WS_SOLVE_ADAPTIVE, 0, torch.device("cuda", torch.cuda.current_device()))
    return _lib.lib().odevit_solve_adaptive(ctypes.byref(desc), ctypes.byref(w), ctypes.c_void_p(x0.data_ptr()), t_c,
                                            len(t), 1e-3, 1e-4, 0.0, 100, ctypes.c_void_p(states.data_ptr()),
                                            ctypes.c_void_p(counts.data_ptr()) if counts is not None else None,
                                            None, None, ws, ws_bytes, ops._stream())


_RAW_W = {}


def test_c_abi_rejects_dropout_and_host_pointers():
    import dataclasses
    from odevit_b200 import _lib
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    _RAW_W.clear()
    _RAW_W.update({k: v.detach() for k, v in model.odefunc.block.field_weights().items() if v is not None})
    spec = model.odefunc.block.field_spec(model.odefunc.scaler)
    states = torch.empty(3, *x0.shape, device="cuda")
    assert _raw_call(spec, x0, states, [0.0, 0.5, 1.0]) == 0
    drop = dataclasses.replace(spec, attn_drop=0.1)
    assert _raw_call(drop, x0, states, [0.0, 0.5, 1.0]) == -1
    assert b"dropout" in _lib.lib().odevit_last_error_string()
    host_states = torch.empty(3, *x0.shape)
    assert _raw_call(spec, x0, host_states, [0.0, 0.5, 1.0]) == -5
    host_counts = torch.zeros(2, dtype=torch.int32)
    assert _raw_call(spec, x0, states, [0.0, 0.5, 1.0], counts=host_counts) == -5
    assert _raw_call(spec, x0.cpu(), states, [0.0, 0.5, 1.0]) == -5
