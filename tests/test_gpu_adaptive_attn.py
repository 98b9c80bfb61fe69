"""GPU tests of the attention outputs of the adaptive Dormand-Prince solve (odevit_solve_adaptive_attn,
odevit_solve_adaptive_bwd_attn, ops.ode_solve_adaptive(want_p_last, jasmin), the models' output_attentions with
`adaptive_solve = {..., "attention_outputs": True}`) against the per-image evaluation sequence of the oracle
(tests/_adaptive_attn_ref.py) and fp64 autograd through `replay` plus the map (tests/_adaptive_grad_ref.py) on the steps
the GPU recorded."""
import ctypes

import pytest
import torch

import _adaptive_attn_ref as aref
import _adaptive_grad_ref as gref
import odevit_oracle as orc
from _util import Golden, cosine, max_rel
from test_gpu_adaptive import T_OUT, _model, _tokens
from test_gpu_adaptive_grad import _functional, _weights

pytestmark = pytest.mark.gpu

TOL_P = {"fp32": 1e-4, "bf16": 5e-2}   # bf16: the bar of the exported map in tests/test_distill_trainer.py
TOL_S = {"fp32": 1e-4, "bf16": 2e-2}   # the end state against the oracle's: the bars of tests/test_gpu_adaptive.py
# the bars of the adaptive reverse sweep without a map cotangent; in bf16 the map's cotangent enters through the bf16
# attention VJP on top.  A loss on p_last alone is checked in fp32 only: in bf16 its gradients are the attention VJP's
# rounding throughout (measured 9.6e-2 on norm_attn.bias, cosine 0.9975), so bf16 is checked, as the fixed grid's
# reverse sweep is (tests/test_gpu_solve_bwd.py), with the map cotangent added to a loss on the states
TOL_G = {"fp32": 2e-3, "bf16": 5e-2}


def _l2_field():
    import odevit_b200 as ob
    g = Golden("fields_d64")
    f = ob.ViT_ODEFunc(dim=64, num_heads=2, mlp_ratio=2.0, emulate_depth=12, time_interval=1.0, l2_attention=True)
    f.load_state_dict(g.group("l2/sd"), strict=True)
    return f.cuda(), g.group("l2/sd"), g.get("l2/x").cuda()


def _cases(precision):
    """(func, state dict, key prefix, oracle field (y, sd) -> (dx, P), x0, t, rtol, atol) of the PARALLEL and L2 fields"""
    model, sd = _model(precision)
    model.odefunc.block.precision = precision
    par = (model.odefunc, sd, "odefunc.", lambda y, s: orc.field_parallel(y, s, 3, 12.0), _tokens(model, 3), T_OUT)
    f, sd2, x2 = _l2_field()
    f.block.precision = precision
    l2 = (f, sd2, "", lambda y, s: orc.field_parallel(y, s, 2, 12.0, prefix="block.", l2=True), x2,
          torch.tensor([0.0, 0.05, 0.1]))
    return {"parallel": par, "l2": l2}


def _solve(func, x0, t, rtol, atol, W=None, k=0, cap=256, first_step=None):
    """odevit_solve_adaptive_attn with a record, p_last and (W given) the window"""
    from odevit_b200 import _lib, ops
    spec, names, ws = _weights(func)
    B = x0.shape[0]
    rec = (cap, torch.empty(cap, B, dtype=torch.float64, device="cuda"),
           torch.empty(cap, B, dtype=torch.float64, device="cuda"), torch.empty(cap, B, dtype=torch.int32, device="cuda"))
    attn = ops._adaptive_attn_outputs(x0, spec, True, (W, k) if W else None)
    t_c = (ctypes.c_float * len(t))(*t.tolist())
    with torch.no_grad():
        st, states, counts = ops._adaptive_call(x0.detach(), t_c, len(t), spec, names, ws, rtol, atol,
                                                first_step or 0.0, ops.DOPRI5_MAX_NUM_STEPS, rec, attn)
    assert st == 0, _lib.lib().odevit_last_error_string()
    S = int(counts[1].max())
    out = {"states": states, "counts": counts, "p_last": attn[0],
           "rec": (rec[1][:S].cpu(), rec[2][:S].cpu(), rec[3][:S].cpu().long())}
    if W:
        out["ring"], out["count"] = attn[1][0], attn[1][1]
    return out


def _window(ring, count, b):
    """image b's window from the ring, in evaluation order: [min(W, n_b), H]"""
    W, n = ring.shape[0], int(count[b])
    return torch.stack([ring[e % W, b] for e in range(max(0, n - W), n)])


def _map64(field, sd):
    sd64 = {k: v.double() for k, v in sd.items()}
    return lambda y: field(y.double(), sd64)[1]


def _oracle(field, sd, x0, t, rtol, atol, first_step=None):
    # the fp32 field of the restatement, stage combines, norms and time in fp64 (as tests/test_gpu_adaptive.py)
    with torch.no_grad():
        return aref.dopri5_evaluations(lambda y: field(y.float(), sd)[0].double(), x0.detach().cpu().double(), t.double(),
                                       rtol, atol, first_step=first_step)


def _replay(field, sd, x0, t, rec):
    """the fp64 replay of the GPU's recorded steps: (states, each image's y1 of its last accepted step)"""
    calls, n = [], (rec[1] > 0).sum(0).tolist()
    sd64 = {k: v.double() for k, v in sd.items()}

    def logged(y):
        calls.append(y)
        return field(y, sd64)[0]

    with torch.no_grad():
        states = gref.replay(logged, x0.detach().cpu().double(), t.double(), *rec)
    return states, torch.stack([calls[1 + 6 * (n[b] - 1) + 5][b] for b in range(len(n))])


def _end_states(func, x0, t, got):
    """every image's y1 on the GPU: ckpt[S] of odevit_solve_adaptive_bwd's replay of the recorded steps"""
    from odevit_b200 import _lib, ops
    spec, names, ws = _weights(func)
    B, N, D = x0.shape
    n = got["counts"][1].cpu().tolist()
    S = max(n)
    rec = [r.cuda().contiguous() for r in got["rec"]]
    rec[2] = rec[2].int()
    ck = torch.empty(S + 1, B, N, D, device="cuda")
    w, keep = ops._pack_weights(names, ws)
    gw, gts = ops._alloc_grads(names, ws, [True] * len(ws))
    buf, wsp, wsn = ops._workspace(spec.desc(B, N), _lib.WS_SOLVE_ADAPTIVE_BWD, 0, x0.device)
    t_c = (ctypes.c_float * len(t))(*t.tolist())
    p = lambda z: ctypes.c_void_p(z.data_ptr())   # noqa: E731
    st = _lib.lib().odevit_solve_adaptive_bwd(ctypes.byref(spec.desc(B, N)), ctypes.byref(w), p(x0), t_c, len(t),
                                              p(rec[0]), p(rec[1]), p(rec[2]), S, (ctypes.c_int32 * B)(*n),
                                              p(torch.zeros_like(got["states"])), p(torch.empty_like(x0)),
                                              ctypes.byref(gw), p(ck), None, 0, wsp, wsn, ops._stream())
    assert st == 0
    return ck[S].contiguous()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", ["parallel", "l2"])
def test_p_last_matches_oracle_last_evaluation(precision, case):
    """p_last is the map of the last evaluation, k7 = f(y1) of the last accepted step: the GPU's end state against the
    fp64 replay of the steps it took, within the solve's bars, and p_last against the oracle field's map of that state.
    The oracle's own last state is not the reference: where the steps agree in number, the sizes still differ by the
    rounding of the fp32 error estimate (a cancelling sum), so its y1 sits at another t1 (measured 3e-3 away on the PARALLEL
    field, 1e-1 on L2); the dense outputs at t_out agree within 1e-4 (tests/test_gpu_adaptive.py)."""
    func, sd, _, field, x0, t = _cases(precision)[case]
    tols = [(1e-3, 1e-4), (1e-5, 1e-7)] if case == "parallel" else [(1e-4, 1e-6), (1e-6, 1e-8)]
    for rtol, atol in tols:
        got = _solve(func, x0, t, rtol, atol)
        if precision == "fp32" and rtol >= 1e-4:   # the evaluation count is the oracle's
            want = _oracle(field, sd, x0, t, rtol, atol)
            assert got["counts"][0].cpu().tolist() == want["nfe"].tolist()
        _, y1 = _replay(field, sd, x0, t, got["rec"])
        mine = _end_states(func, x0, t, got)
        assert max_rel(mine, y1) <= TOL_S[precision], (rtol, max_rel(mine, y1))
        ref = _map64(field, sd)(mine.cpu())
        assert max_rel(got["p_last"], ref) <= TOL_P[precision], (rtol, max_rel(got["p_last"], ref))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_p_last_is_the_in_solve_map_bitwise(precision):
    """The extra evaluation at the end state repeats the solve's last k7 = f(y1): the same map as exporting it from that
    evaluation (the replay writes y1 bitwise as the forward did: ckpt[S])."""
    import odevit_b200 as ob
    from odevit_b200 import ops
    model, _ = _model(precision)
    x0 = _tokens(model, 4)
    x0[2] *= 0.25
    got = _solve(model.odefunc, x0, T_OUT, 1e-3, 1e-4)
    func = model.odefunc
    with torch.no_grad():
        plain = ob.odeint_adaptive(func, x0, T_OUT, rtol=1e-3, atol=1e-4)
    assert torch.equal(plain, got["states"])
    spec = func.block.field_spec(func.scaler)
    with torch.no_grad():
        _, p_ref = ops.field_eval(_end_states(func, x0, T_OUT, got), spec, func.block.field_weights())
    assert torch.equal(got["p_last"], p_ref)


@pytest.mark.parametrize("k", [0, 2, 10])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_jasmin_window_matches_oracle_per_image(precision, k):
    """Images with different nfe, one with nfe < W; k <= 3 in bf16 forms the statistic inside the fused attention
    kernel, k = 10 and fp32 from the exported map (jasmin_rowmax)."""
    model, sd = _model(precision)
    field = lambda y, s: orc.field_parallel(y, s, 3, 12.0)   # noqa: E731
    x0 = _tokens(model, 3, seed=2)
    x0[1] *= 0.05
    # (bf16 with k > 3 exports every map: the export kernel rounds O differently, so the steps may differ from k <= 3's)
    got = _solve(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W=1, k=k)
    nfe = got["counts"][0].cpu().tolist()
    assert len(set(nfe)) > 1, nfe
    W = (min(nfe) + max(nfe)) // 2
    assert min(nfe) < W < max(nfe)
    got = _solve(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W=W, k=k)
    assert got["count"].cpu().tolist() == nfe
    # the statistic is the log of a near-cancelling g_1 (see test_distill_trainer) of maps whose logits amplify the
    # state's rounding (test_p_last_matches_oracle_last_evaluation): measured up to 2.2e-3 at the window's end
    tol = 5e-3
    for b in range(3):
        alone = _solve(model.odefunc, x0[b:b + 1].contiguous(), T_OUT, 1e-3, 1e-4, W=W, k=k)
        assert torch.equal(_window(alone["ring"], alone["count"], 0), _window(got["ring"], got["count"], b))
        if precision == "fp32":
            want = _oracle(field, sd, x0[b:b + 1], T_OUT, 1e-3, 1e-4)
            ev = want["evaluations"][0]
            assert len(ev) == nfe[b]
        else:
            ev = None
        if ev is not None:
            ref = aref.window(ev, W, _map64(field, sd), k)
            win = _window(got["ring"], got["count"], b)
            assert win.shape == ref.shape == (min(W, nfe[b]), 3)
            assert max_rel(win, ref) <= tol, (b, max_rel(win, ref))


def test_jasmin_window_bf16_against_fp32_map():
    """bf16 steps are not the oracle's: the window's last entry, formed inside the fused attention kernel (k <= 3) or from
    the exported map (k = 10), against odevit_jasmin_rowmax of the same evaluation's map, p_last.  The k <= 3 solve
    does not export its maps, so its states are those of the plain solve."""
    import odevit_b200 as ob
    from odevit_b200 import ops
    model, _ = _model("bf16")
    x0 = _tokens(model, 2)
    with torch.no_grad():
        plain = ob.odeint_adaptive(model.odefunc, x0, T_OUT, rtol=1e-3, atol=1e-4)
    for k in (2, 10):
        a = _solve(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W=40, k=k)
        if k == 2:
            assert torch.equal(a["states"], plain)
        assert torch.equal(a["count"], a["counts"][0])
        with torch.no_grad():
            last = ops.jasmin_rowmax(a["p_last"][None], k)[0]
        for i in range(2):
            assert max_rel(_window(a["ring"], a["count"], i)[-1], last[i]) < 2e-2, (k, i)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batch_of_300_is_each_image_alone(precision):
    model, _ = _model(precision)
    x0 = _tokens(model, 300, seed=5)
    x0[::7] *= 0.1
    W = 30
    got = _solve(model.odefunc, x0, T_OUT, 1e-3, 1e-4, W=W, k=2)
    nfe = got["counts"][0].cpu()
    assert len(set(nfe.tolist())) > 1
    picks = sorted(set([int(nfe.argmin()), int(nfe.argmax())] + list(range(0, 300, 13))))
    for b in picks:
        alone = _solve(model.odefunc, x0[b:b + 1].contiguous(), T_OUT, 1e-3, 1e-4, W=W, k=2)
        assert torch.equal(alone["states"][:, 0], got["states"][:, b]), b
        assert torch.equal(alone["p_last"][0], got["p_last"][b]), b
        assert torch.equal(_window(alone["ring"], alone["count"], 0), _window(got["ring"], got["count"], b)), b


def _gpu_grads(func, x0, t, rtol, atol, Ws, Wp):
    """L = <Ws, states> + <Wp, p_last> through ops.ode_solve_adaptive(differentiable=True, want_p_last=True)"""
    from odevit_b200 import ops
    func.zero_grad(set_to_none=True)
    x = x0.detach().clone().requires_grad_(True)
    res = ops.ode_solve_adaptive(x, t, func.block.field_spec(func.scaler), func.block.field_weights(), rtol, atol,
                                 differentiable=True, want_p_last=True)
    loss = (res["p_last"] * Wp.cuda()).sum()
    if Ws is not None:
        loss = loss + (res["states"] * Ws.cuda()).sum()
    loss.backward()
    return x.grad, {n: p.grad.clone() for n, p in func.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("mode", ["tape", "recompute"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", ["parallel", "l2"])
def test_grads_with_a_p_last_loss_match_fp64_autograd(case, precision, mode):
    func, sd, prefix, field, x0, t = _cases(precision)[case]
    rtol, atol = (1e-3, 1e-4) if case == "parallel" else (1e-4, 1e-6)
    got = _solve(func, x0, t, rtol, atol)
    rec = got["rec"]
    Ws = _functional((len(t),) + tuple(x0.shape))
    Wp = _functional(tuple(got["p_last"].shape), seed=4)
    func.block.backward_mode = mode
    try:
        for with_states in ((False, True) if precision == "fp32" else (True,)):
            g_x0, grads = _gpu_grads(func, x0, t, rtol, atol, Ws if with_states else None, Wp)
            sd64 = {k: v.detach().double().requires_grad_(True) for k, v in sd.items()}
            xo = x0.detach().cpu().double().requires_grad_(True)
            calls = []

            def logged(y):
                dx, P = field(y, sd64)
                calls.append(P)
                return dx

            states = gref.replay(logged, xo, t.double(), *rec)
            n = (rec[1] > 0).sum(0).tolist()
            p_last = torch.stack([calls[1 + 6 * (n[b] - 1) + 5][b] for b in range(len(n))])
            loss = (p_last * Wp.double()).sum()
            if with_states:
                loss = loss + (states * Ws.double()).sum()
            loss.backward()
            pairs = [("x0", g_x0, xo.grad)] + [(nm, grads[nm], sd64[prefix + nm].grad) for nm in grads]
            assert len(pairs) >= 9
            for nm, a, b in pairs:
                assert b is not None, nm
                assert torch.isfinite(a).all(), nm
                assert max_rel(a, b) <= TOL_G[precision], (with_states, nm, max_rel(a, b))
                if precision == "bf16":
                    assert cosine(a.flatten().double().cpu(), b.flatten()) >= 0.995, nm
    finally:
        func.block.backward_mode = "auto"


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_deterministic_mode_is_bitwise(precision):
    model, _ = _model(precision)
    x0 = _tokens(model, 3)
    Ws = _functional((len(T_OUT),) + tuple(x0.shape))
    Wp = _functional((3, 3, x0.shape[1], x0.shape[1]), seed=4)
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        runs = [_gpu_grads(model.odefunc, x0, T_OUT, 1e-3, 1e-4, Ws, Wp) for _ in range(2)]
    finally:
        torch.use_deterministic_algorithms(was)
    assert torch.equal(runs[0][0], runs[1][0])
    for n in runs[0][1]:
        assert torch.equal(runs[0][1][n], runs[1][1][n]), n


def test_odeint_adaptive_record_attention():
    import odevit_b200 as ob
    model, _ = _model("fp32")
    x0 = _tokens(model, 2)
    got = _solve(model.odefunc, x0, T_OUT, 1e-3, 1e-4)
    model.odefunc.block.attentions = None
    with torch.no_grad():
        states = ob.odeint_adaptive(model.odefunc, x0, T_OUT, rtol=1e-3, atol=1e-4, record_attention=True)
    assert torch.equal(states, got["states"]) and torch.equal(model.odefunc.block.attentions, got["p_last"])


def test_model_output_attentions():
    """attentions / attentions_register_tokens slice the last-evaluation map as the fixed grid does; jasmin_loss is the
    mean over images of each image's own window mean"""
    model, _ = _model("fp32")
    R = model.patch_embed.num_register_tokens
    px = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(7)).cuda()
    model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "attention_outputs": True}
    try:
        with torch.no_grad():
            out = model(px, output_attentions=True, jasmin_k=2)
            tokens = model.patch_embed(px)
    finally:
        model.adaptive_solve = None
    W = int(model.num_eval_steps * 0.85)
    got = _solve(model.odefunc, tokens, model.t_grid, 1e-3, 1e-4, W=W, k=2)
    assert torch.equal(out["attentions"], got["p_last"][:, :, :-R, :-R])
    assert torch.equal(out["attentions_register_tokens"], got["p_last"][:, :, -R:, :])
    per_image = torch.stack([_window(got["ring"], got["count"], b).double().mean() for b in range(3)])
    assert float(out["jasmin_loss"]) == pytest.approx(float(per_image.mean()), rel=1e-6)


def test_model_attention_outputs_are_opt_in():
    """Without "attention_outputs": True a request keeps refusing output_attentions (and adds no evaluation); with it
    the outputs come, and the trajectory list still raises."""
    model, _ = _model("fp32")
    px = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(7)).cuda()
    try:
        model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4}
        with torch.no_grad():
            plain = model(px)
            with pytest.raises(ValueError, match="attention_outputs"):
                model(px, output_attentions=True)
        model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "attention_outputs": True}
        with torch.no_grad():
            out = model(px, output_attentions=True, jasmin_k=2)
            assert torch.equal(out["logits"], plain["logits"]) and torch.equal(out["nfe"], plain["nfe"])
            assert torch.equal(model(px)["logits"], plain["logits"])
            with pytest.raises(ValueError, match="output_attention_trajectory"):
                model(px, output_attentions=True, output_attention_trajectory=True)
        model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "attention_output": True}
        with pytest.raises(ValueError, match="attention_outputs"):
            with torch.no_grad():
                model(px)
    finally:
        model.adaptive_solve = None


def test_model_training_through_attentions():
    """A differentiable request with attention outputs: the model's gradients are those of the same loss composed from
    ops.ode_solve_adaptive(differentiable=True, want_p_last=True)."""
    import torch.nn.functional as F

    from odevit_b200 import ops
    model, _ = _model("fp32")
    model.train()
    R = model.patch_embed.num_register_tokens
    px = torch.randn(3, 3, 32, 32, generator=torch.Generator().manual_seed(7)).cuda()
    labels = torch.tensor([1, 4, 7], device="cuda")
    model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "differentiable": True, "attention_outputs": True}
    try:
        model.zero_grad(set_to_none=True)
        out = model(px, labels=labels, output_attentions=True)
        (out["loss"] + out["attentions"].square().sum()).backward()
    finally:
        model.adaptive_solve = None
    field = dict(model.odefunc.named_parameters())
    got = {n: p.grad.clone() for n, p in field.items()}
    for n, g in got.items():
        assert torch.isfinite(g).all() and g.abs().max() > 0, n
    model.zero_grad(set_to_none=True)
    blk = model.odefunc.block
    res = ops.ode_solve_adaptive(model.patch_embed(px), model.t_grid, blk.field_spec(model.odefunc.scaler),
                                 blk.field_weights(), 1e-3, 1e-4, differentiable=True, want_p_last=True)
    loss = F.cross_entropy(model.head(res["final"][:, 0]), labels, label_smoothing=0.05)
    (loss + res["p_last"][:, :, :-R, :-R].square().sum()).backward()
    for n, p in field.items():
        assert max_rel(got[n], p.grad) < 1e-5, n


def test_distill_trainer_step_on_an_adaptive_student():
    """One ImageDistilTrainer step, unchanged, on a student with a differentiable adaptive_solve that asks for attention
    outputs, and the library teacher:
    every loss term against the same terms composed from the oracle's outputs (its dense output at the control points,
    each image's last-evaluation map and JaSMin window)."""
    import odevit_b200 as ob
    from odevit_b200.loss_trainer import ImageDistilTrainer
    from test_distill_trainer import _teacher
    g = Golden("distill_trainer_tiny")
    cfg = g.meta["student"]
    student = ob.ViTNeuralODE(**cfg)
    sd = g.group("sd")
    student.load_state_dict(sd, strict=True)
    student = student.cuda()
    student.precision = "fp32"
    student.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "differentiable": True, "attention_outputs": True}
    teacher = ob.ViTTeacher(_teacher(g).cuda(), precision="fp32", attention_maps="last")
    opt = torch.optim.SGD(student.parameters(), lr=0.0)
    tr = ImageDistilTrainer(teacher_model=teacher, student_model=student, optimizer=opt, **g.meta["trainer"])
    px, lb = g.get("in/pixel_values").cuda(), g.get("in/labels").cuda()
    out = tr({"pixel_values": px}, lb, epoch=0)
    assert torch.isfinite(out["loss"])
    for n, p in student.odefunc.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n
    s_out = out["student_output"]

    # the oracle's student outputs over the same tokens
    R = student.patch_embed.num_register_tokens
    heads, k = cfg["num_heads"], g.meta["trainer"]["jasmin_k"]
    field = lambda y, s: orc.field_parallel(y, s, heads, student.odefunc.scaler)   # noqa: E731
    m32 = lambda y: field(y.float(), sd)[1]   # noqa: E731  (the reference's fp32 maps: JaSMin of near-one-hot rows)
    with torch.no_grad():
        tokens = student.patch_embed(px)
    # the trajectory and the last map from the fp64 replay of the steps the step's solve took (the solve is
    # deterministic: a second one records them), the window from the oracle's own evaluations
    got = _solve(student.odefunc, tokens, student.t_grid, 1e-3, 1e-4)
    assert torch.equal(got["counts"][0], s_out["nfe"])
    states, y1 = _replay(field, sd, tokens, student.t_grid, got["rec"])
    want = _oracle(field, sd, tokens, student.t_grid, 1e-3, 1e-4)
    assert s_out["nfe"].cpu().tolist() == want["nfe"].tolist()
    m64 = _map64(field, sd)
    W = int(student.num_eval_steps * 0.85)
    p_last = m64(y1)
    jas = torch.stack([aref.window(ev, W, m32, k).double().mean() for ev in want["evaluations"]]).mean()
    idx = student.get_proportional_control_points_with_temperature(temperature=30, num_eval_steps=student.num_eval_steps)
    ref_out = {"control_points": states[idx][:, :, :-R].float().cuda(),
               "attentions": p_last[:, :, :-R, :-R].float().cuda()}
    with torch.no_grad():
        t_out = teacher(pixel_values=px, output_hidden_states=True, output_attentions=True)
        rep = tr.train_batch_representation(ref_out, t_out)
    # this fixture's maps are near one-hot (see tests/test_distill_trainer.py): the fp32 solve's 1e-4 state rounding
    # moves them by up to 1.8e-3 (measured), and the L1 term sits behind a slope-40 sigmoid of their cumulative mass
    assert max_rel(s_out["attentions"], ref_out["attentions"]) <= 5e-3
    assert max_rel(s_out["control_points"], ref_out["control_points"]) <= 1e-4
    assert float(out["mse_loss"]) == pytest.approx(float(rep["mse_loss"]), rel=1e-3)
    assert float(out["kl_loss"]) == pytest.approx(float(rep["kl_loss"]), rel=2e-2)
    assert float(out["jasmin_loss"]) == pytest.approx(float(jas), rel=5e-3)
    total = float(rep["loss"]) + float(jas)
    assert float(out["loss"]) == pytest.approx(total, rel=2e-2)


def test_error_paths():
    import dataclasses

    import odevit_b200 as ob
    from odevit_b200 import _lib, ops
    model, _ = _model("bf16")
    func = model.odefunc
    x0 = _tokens(model, 2)
    spec, names, ws = _weights(func)
    w = func.block.field_weights()
    with pytest.raises(ob.OdevitError, match="capturable"):
        with torch.no_grad():
            ops.ode_solve_adaptive(x0, T_OUT, spec, w, 1e-3, 1e-4, capturable=True, want_p_last=True)
    with pytest.raises(ob.OdevitError, match="capturable"):
        with torch.no_grad():
            ops.ode_solve_adaptive(x0, T_OUT, spec, w, 1e-3, 1e-4, capturable=True, jasmin=(4, 2))
    drop = dataclasses.replace(spec, attn_drop=0.1)
    with pytest.raises(ob.OdevitError, match="dropout"):
        ops.ode_solve_adaptive(x0.clone().requires_grad_(True), T_OUT, drop, w, 1e-3, 1e-4, differentiable=True,
                               want_p_last=True)
    with pytest.raises(ValueError, match="jasmin window"):
        with torch.no_grad():
            ops.ode_solve_adaptive(x0, T_OUT, spec, w, 1e-3, 1e-4, jasmin=(0, 2))
    model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4}
    px = torch.randn(2, 3, 32, 32, generator=torch.Generator().manual_seed(7)).cuda()
    try:
        with pytest.raises(ValueError, match="output_attention_trajectory is not built"):
            with torch.no_grad():
                model(px, output_attention_trajectory=True)
        model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "capturable": True, "attention_outputs": True}
        with pytest.raises(ValueError, match="capturable"):
            with torch.no_grad():
                model(px, output_attentions=True)
    finally:
        model.adaptive_solve = None
    # the C ABI: jas_k / jas_window out of range, MACARON, a partial record, a NULL g_p_last
    B, N, D = x0.shape
    t_c = (ctypes.c_float * len(T_OUT))(*T_OUT.tolist())
    states = torch.empty(len(T_OUT), B, N, D, device="cuda")
    ring = torch.empty(4, B, 3, device="cuda")
    cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    p = lambda z: ctypes.c_void_p(z.data_ptr()) if z is not None else None   # noqa: E731
    wts, keep = ops._pack_weights(names, ws)
    buf, wsp, wsn = ops._workspace(spec.desc(B, N), _lib.WS_SOLVE_ADAPTIVE, 0, x0.device)

    def call(desc, k=2, window=4, t0=None):
        return _lib.lib().odevit_solve_adaptive_attn(ctypes.byref(desc), ctypes.byref(wts), p(x0), t_c, len(T_OUT),
                                                     1e-3, 1e-4, 0.0, 1000, p(states), None, None, None, 4, p(t0), None,
                                                     None, None, k, window, p(ring), p(cnt), wsp, wsn, ops._stream())
    desc = spec.desc(B, N)
    assert call(desc, k=N + 1) == -1 and b"jas_k" in _lib.lib().odevit_last_error_string()
    assert call(desc, window=0) == -1 and b"jas_window" in _lib.lib().odevit_last_error_string()
    assert call(desc, t0=torch.empty(4, B, dtype=torch.float64, device="cuda")) == -1
    assert b"all three or none" in _lib.lib().odevit_last_error_string()
    assert call(desc) == 0   # usable afterwards
    assert _lib.lib().odevit_solve_adaptive_bwd_attn(ctypes.byref(desc), ctypes.byref(wts), p(x0), t_c, len(T_OUT), None,
                                                     None, None, 1, (ctypes.c_int32 * B)(1, 1), None, None, None, None,
                                                     None, None, 0, wsp, wsn, ops._stream()) == -1
    assert b"g_p_last" in _lib.lib().odevit_last_error_string()
    mac = dataclasses.replace(spec, variant=_lib.FIELD_MACARON)
    with pytest.raises(ob.OdevitError, match="MACARON"):
        with torch.no_grad():
            ops.ode_solve_adaptive(x0, T_OUT, mac, w, 1e-3, 1e-4, want_p_last=True)
