"""torch.use_deterministic_algorithms(True): the library's backward kernels sum every floating-point reduction in a fixed
order (split-K partial slabs, column-sum partials, the unfold and res_scale partials, extract_mass's blur transpose as a
gather), so the same seeded training step gives bitwise-identical losses and gradients run after run.

The switch is process-wide: the fixture turns it on and always restores what was there before."""
import pytest
import torch

from _util import cosine, max_rel

pytestmark = pytest.mark.gpu

C10 = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
           time_interval=1.0)
C100 = dict(img_size=224, patch_size=16, num_classes=100, embed_dim=768, num_heads=12, mlp_ratio=1.0, emulate_depth=12,
            time_interval=1.0)


@pytest.fixture(autouse=True)
def deterministic_switch(monkeypatch):
    # (PyTorch refuses cuBLAS under the switch without this; the library's own kernels do not need it)
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    before, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(before, warn_only=warn)
        _sync()


def _sync():
    from odevit_b200 import ops
    ops._sync_deterministic()


def _lib():
    from odevit_b200 import _lib
    return _lib


def _inputs(cfg, batch, seed=1234):
    S, C = cfg["img_size"], cfg["num_classes"]
    px = torch.randn(batch, 3, S, S, generator=torch.Generator().manual_seed(seed)).cuda()
    lb = torch.randint(0, C, (batch,), generator=torch.Generator().manual_seed(seed + 1)).cuda()
    return px, lb


def _model(cfg, precision="bf16", macaron=False, **kw):
    import odevit_b200 as ob
    torch.manual_seed(0)
    m = (ob.ViTMacaron if macaron else ob.ViTNeuralODE)(**cfg, **kw).cuda().train()
    m.precision = precision
    return m


def _step(model, px, lb, seed=5):
    """One seeded training step: (loss, {name: grad}) plus the library launches it took and the profiled scopes."""
    L = _lib()
    torch.manual_seed(seed)
    model.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    L.lib().odevit_reset_launch_count()
    L.profile_enable(True)
    loss = model(px, labels=lb)["loss"]
    loss.backward()
    torch.cuda.synchronize()
    scopes = sum(n for _, n in L.profile_read().values())
    L.profile_enable(False)
    launches = int(L.lib().odevit_launch_count())
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return loss.detach().clone(), grads, launches - scopes


def _assert_equal_runs(runs):
    (l0, g0, _), rest = runs[0], runs[1:]
    for l1, g1, _ in rest:
        assert torch.equal(l0, l1)
        assert g0.keys() == g1.keys()
        for n in g0:
            assert torch.equal(g0[n], g1[n]), n


def _check(model, px, lb, n_runs=2, tol=2e-2, cos_min=0.9999):
    base = _step(model, px, lb)                      # the default (atomic) kernels
    with _on():
        runs = [_step(model, px, lb) for _ in range(n_runs)]
    _assert_equal_runs(runs)
    # the forward has no order-dependent reduction: its loss is the same bits with the switch on and off
    assert torch.equal(runs[0][0], base[0])
    for n, g in base[1].items():
        got = runs[0][1][n]
        if g.abs().max() == 0:
            continue
        assert max_rel(got, g) < tol, (n, max_rel(got, g))
        if g.numel() > 1:
            assert cosine(got, g) > cos_min, (n, cosine(got, g))
    return base, runs


class _on:
    """The switch on for a block (the fixture restores what was there before the test)."""

    def __enter__(self):
        torch.use_deterministic_algorithms(True)

    def __exit__(self, *a):
        torch.use_deterministic_algorithms(False)
        _sync()


def _split_k_gemms(base, det):
    """Split-K GEMMs that went through partial slabs: in the deterministic mode each adds one det_sum launch inside the
    GEMM's own profiled scope (launches beyond scopes), nothing else does."""
    return det[2] - base[2]


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_c10_rk4(precision):
    m = _model(dict(C10, num_eval_steps=5, solver="rk4"), precision)
    px, lb = _inputs(C10, 16)     # K = 16 x 65 tokens: the weight-gradient GEMMs split K
    base, runs = _check(m, px, lb, n_runs=3, tol=2e-2 if precision == "bf16" else 1e-3)
    assert _split_k_gemms(base, runs[0]) > 0
    # back to the default kernels
    assert _lib().lib().odevit_deterministic() == 0
    again = _step(m, px, lb)
    assert again[2] == base[2]
    assert torch.equal(again[0], base[0])


@pytest.mark.parametrize("mode", ["tape", "recompute"])
def test_bench_shape(mode):
    m = _model(dict(C100, num_eval_steps=24, solver="euler"))
    m.odefunc.block.backward_mode = mode
    px, lb = _inputs(C100, 64)
    base, runs = _check(m, px, lb)
    assert _split_k_gemms(base, runs[0]) > 0


def test_dropout():
    m = _model(dict(C10, num_eval_steps=5, solver="rk4"), attn_drop=0.3, proj_drop=0.3, mlp_drop=0.3)
    px, lb = _inputs(C10, 16)
    with _on():
        runs = [_step(m, px, lb, seed=7) for _ in range(3)]
    _assert_equal_runs(runs)


def test_macaron_field():
    cfg = dict(C10, num_eval_steps=4, solver="rk4")
    m = _model(cfg, macaron=True)
    px, lb = _inputs(C10, 16)
    _check(m, px, lb)


def test_adaptive_solve():
    m = _model(dict(C10, num_eval_steps=5, solver="rk4"))
    m.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "differentiable": True}
    px, lb = _inputs(C10, 16)
    _check(m, px, lb)


@pytest.mark.parametrize("l2", [False, True], ids=["softmax", "l2"])
def test_initial_state_gradient(l2):
    """g_x0 and the field's gradients of a bare solve (odeint) under the switch, C10 shape, batch 16, RK4; the L2 field
    here (the model's forward computes a bound the L2 attention does not define)."""
    import odevit_b200 as ob
    m = _model(dict(C10, num_eval_steps=5, solver="rk4"), l2_attention=l2)
    x0 = torch.randn(16, 65, 192, generator=torch.Generator().manual_seed(3)).cuda()
    t = torch.linspace(0, 1, 6)

    def run():
        x = x0.clone().requires_grad_(True)
        m.zero_grad(set_to_none=True)
        ys = ob.odeint(m.odefunc, x, t, method="rk4")
        (ys[-1] * ys[-1]).sum().backward()
        return x.grad.clone(), {n: p.grad.clone() for n, p in m.odefunc.named_parameters() if p.grad is not None}
    with _on():
        a, b = run(), run()
    assert torch.equal(a[0], b[0])
    for n in a[1]:
        assert torch.equal(a[1][n], b[1][n]), n


def test_distillation_step():
    import odevit_b200 as ob
    from _util import Golden
    from odevit_b200.loss_trainer import ImageDistilTrainer
    from test_distill_trainer import _teacher
    g = Golden("distill_trainer_tiny")
    student = ob.ViTNeuralODE(**g.meta["student"])
    student.load_state_dict(g.group("sd"), strict=True)
    student = student.cuda()
    student.precision = "bf16"
    teacher = _teacher(g).cuda()
    opt = torch.optim.SGD(student.parameters(), lr=0.0)
    tr = ImageDistilTrainer(teacher_model=teacher, student_model=student, optimizer=opt, **g.meta["trainer"])
    px, lb = g.get("in/pixel_values").cuda(), g.get("in/labels").cuda()

    def run():
        torch.manual_seed(3)
        student.zero_grad(set_to_none=True)
        out = tr({"pixel_values": px}, lb, epoch=201)
        return out["loss"].detach().clone(), {n: p.grad.clone() for n, p in student.named_parameters() if p.grad is not None}
    with _on():
        a, b = run(), run()
    assert torch.equal(a[0], b[0])
    for n in a[1]:
        assert torch.equal(a[1][n], b[1][n]), n


def test_extract_mass_backward():
    from odevit_b200 import ops
    rows = torch.rand(8, 3, 196, generator=torch.Generator().manual_seed(2)).cuda()
    gm = torch.randn(8, 196, generator=torch.Generator().manual_seed(4)).cuda()

    def run():
        x = rows.clone().requires_grad_(True)
        (ops.extract_mass(x, smooth=True)[0].reshape(8, 196) * gm).sum().backward()
        return x.grad.clone()
    base = run()
    with _on():
        a, b = run(), run()
    assert torch.equal(a, b)
    assert max_rel(a, base) < 1e-5


def test_graphed_train_step():
    from odevit_b200.graphs import GraphedTrainStep
    cfg = dict(C10, num_eval_steps=5, solver="rk4")
    px, lb = _inputs(C10, 16)

    def run():
        m = _model(cfg)
        params = [p for p in m.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-3, fused=True, capturable=True)
        torch.manual_seed(9)
        stepper = GraphedTrainStep(m, opt, (px, lb), clip=1.0)
        stepper(px, lb)
        stepper(px, lb)
        torch.cuda.synchronize()
        return [p.detach().clone() for p in params]
    with _on():
        a, b = run(), run()
    for x, y in zip(a, b):
        assert torch.equal(x, y)
