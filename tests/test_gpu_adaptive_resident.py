"""GPU tests of the capturable adaptive Dormand-Prince solve inside the on-chip-state kernel
(odevit_solve_adaptive_resident, ops.ode_solve_adaptive(capturable=True), odeint_adaptive(capturable=True), the models'
adaptive_solve with "capturable") against oracle/adaptive_dp5.py and the multi-kernel adaptive solve."""
import pytest
import torch

import adaptive_dp5 as dp
import odevit_oracle as orc
from _util import max_rel
from test_gpu_adaptive import CFG, T_OUT, _model, _oracle, _tokens

pytestmark = pytest.mark.gpu


def _solve(model, x0, t=T_OUT, rtol=1e-3, atol=1e-4, capturable=True, **kw):
    import odevit_b200 as ob
    with torch.no_grad():
        return ob.odeint_adaptive(model.odefunc, x0, t, rtol=rtol, atol=atol, options=kw or None, return_stats=True,
                                  capturable=capturable)


def _counts(stats):
    return stats["accepted"].cpu().tolist(), stats["rejected"].cpu().tolist()


def test_forced_schedule_pins_stages_and_dense_output():
    # atol 1e9 accepts every attempt and each step is 10x the last: [0, 0.0125], then [0.0125, 0.1375].  t = 0.01 lies
    # inside the first step, t = 0.0125 at its end, 0.05 and 0.1 inside the second (FSAL k1 = k7 of the first).  (With
    # t up to 1 the second step would be 1.25 long: there the bf16 field alone puts both bf16 solves ~3e-2 from the
    # fp32 oracle, and 3e-2 from each other.)
    model, sd = _model("bf16")
    x0 = _tokens(model, 4)
    t = torch.tensor([0.0, 0.01, 0.0125, 0.05, 0.1])
    states, stats = _solve(model, x0, t=t, rtol=1e-3, atol=1e9, first_step=0.0125)
    assert _counts(stats) == ([2] * 4, [0] * 4)
    assert stats["status"].cpu().tolist() == [0] * 4
    want = dp.dopri5(lambda y: orc.field_parallel(y.float(), sd, 3, 12.0)[0].double(), x0.cpu().double(), t.double(),
                     1e-3, 1e9, first_step=0.0125)
    assert want["accepted"].tolist() == [2] * 4
    assert max_rel(states, want["states"]) < 2e-2
    ref, _ = _solve(model, x0, t=t, rtol=1e-3, atol=1e9, first_step=0.0125, capturable=False)
    assert max_rel(states, ref) < 1e-2


def test_real_tolerance_matches_oracle():
    # The counts are not compared with the fp32 oracle's: on this fixture (seed 0, tokens seed 1, B 4) the bf16 field
    # moves accept / reject decisions, for the multi-kernel bf16 solve as for this one (accepted [5, 6, 6, 6] and
    # [5, 6, 5, 6] against the oracle's [5, 5, 5, 5] when the test was written).  The test_gpu_adaptive.py fp32 tests pin
    # the controller's arithmetic; here the counts must agree with the NFE formula and the states with the oracle.
    model, sd = _model("bf16")
    x0 = _tokens(model, 4)
    states, stats = _solve(model, x0)
    want = _oracle(sd, x0)
    assert max_rel(states, want["states"]) < 2e-2
    acc, rej = _counts(stats)
    assert stats["nfe"].cpu().tolist() == [2 + 6 * (a + r) for a, r in zip(acc, rej)]
    assert stats["status"].cpu().tolist() == [0] * 4


def test_batch_independence_and_dealing_bitwise():
    model, _ = _model("bf16")
    x0 = _tokens(model, 300, seed=2)
    x0[::7] *= 0.25     # images that finish early: the CTAs that drew them take more images
    states, stats = _solve(model, x0)
    again, _ = _solve(model, x0)
    assert torch.equal(states, again)
    acc, rej = _counts(stats)
    assert len(set(zip(acc, rej))) > 1
    for b in (0, 1, 7, 150, 299):
        s1, st1 = _solve(model, x0[b:b + 1].contiguous())
        assert _counts(st1) == ([acc[b]], [rej[b]]), b
        assert torch.equal(s1[:, 0], states[:, b]), b


def test_graph_capture_replays_on_device_decisions():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x_a = _tokens(model, 6, seed=3)
    x_b = _tokens(model, 6, seed=4) * 0.25     # fewer steps than x_a
    static_x = x_a.clone()
    eager_a, st_a = _solve(model, x_a)
    eager_b, st_b = _solve(model, x_b)
    assert _counts(st_a) != _counts(st_b)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _solve(model, static_x)                # warm-up (workspace, kernel attributes)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g):
        out, stats = ob.odeint_adaptive(model.odefunc, static_x, T_OUT, rtol=1e-3, atol=1e-4, return_stats=True,
                                        capturable=True)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager_a)
    assert _counts(stats) == _counts(st_a)
    static_x.copy_(x_b)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager_b)
    assert _counts(stats) == _counts(st_b)
    assert int(stats["rounds"]) == max(a + r for a, r in zip(*_counts(st_b)))


def test_graph_capture_of_a_whole_model():
    model, _ = _model("bf16")
    model.adaptive_solve = {"rtol": 1e-3, "atol": 1e-4, "capturable": True}
    px = torch.randn(4, 3, 32, 32, generator=torch.Generator().manual_seed(5)).cuda()
    with torch.no_grad():
        eager = model(px)["logits"]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            model(px)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = model(px)
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out["logits"], eager)


def test_one_launch_per_solve():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x0 = _tokens(model, 8)
    launches, nfe = [], []
    for rtol in (1e-2, 1e-4):
        _solve(model, x0, rtol=rtol, atol=rtol / 100)   # warm-up
        torch.cuda.synchronize()
        ob.reset_launch_count()
        _, stats = _solve(model, x0, rtol=rtol, atol=rtol / 100)
        torch.cuda.synchronize()
        launches.append(ob.launch_count())
        nfe.append(float(stats["nfe"].float().mean()))
    assert nfe[0] < nfe[1]
    # the weight conversion of the call and the one solve kernel, whatever the number of steps
    assert launches[0] == launches[1] <= 8


def test_per_image_failure():
    import odevit_b200 as ob
    model, _ = _model("bf16")
    x0 = _tokens(model, 6, seed=6)
    x0[::2] *= 0.05     # these meet the tolerance in fewer steps than the others
    _, free = _solve(model, x0, rtol=1e-2, atol=1e-3)
    attempts = [a + r for a, r in zip(*_counts(free))]
    limit = min(attempts)   # the images that need more attempts fail
    assert max(attempts) > limit
    kw = dict(rtol=1e-2, atol=1e-3, max_num_steps=limit)
    with pytest.raises(ob.NotConvergedError, match=r"image .*max_num_steps"):
        _solve(model, x0, **kw)
    static_x = x0.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g):
        out, stats = ob.odeint_adaptive(model.odefunc, static_x, T_OUT, rtol=kw["rtol"], atol=kw["atol"],
                                        options={"max_num_steps": limit}, return_stats=True, capturable=True)
    g.replay()
    torch.cuda.synchronize()
    status = stats["status"].cpu().tolist()
    assert status == [1 if n > limit else 0 for n in attempts]
    for b in range(6):
        if status[b]:
            assert torch.isnan(out[-1, b]).all(), b
            assert not torch.isnan(out[0, b]).any(), b
        else:
            s1, st1 = _solve(model, x0[b:b + 1].contiguous(), **kw)
            assert torch.equal(s1[:, 0], out[:, b]), b
    # the library works afterwards
    s_ok, st_ok = _solve(model, x0[1:2].contiguous() * 0.05, rtol=1e-2, atol=1e-3)
    assert st_ok["status"].cpu().tolist() == [0] and torch.isfinite(s_ok).all()


def _field(cls=None, dim=192, heads=3, **kw):
    import odevit_b200 as ob
    cls = cls or ob.ViT_ODEFunc
    f = cls(dim=dim, num_heads=heads, mlp_ratio=4.0, emulate_depth=12, time_interval=1.0, **kw).cuda().eval()
    f.block.precision = "bf16"
    return f


def test_envelope_and_argument_errors():
    import odevit_b200 as ob
    x0 = torch.randn(2, 69, 192, generator=torch.Generator().manual_seed(0)).cuda()

    def solve(f, x=x0, t=T_OUT, **kw):
        with torch.no_grad():
            return ob.odeint_adaptive(f, x, t, rtol=1e-3, atol=1e-4, capturable=True, **kw)

    base = _field(l2_attention=False)
    solve(base)   # inside the envelope
    fp32 = _field(l2_attention=False)
    fp32.block.precision = "fp32"
    with pytest.raises(ob.OdevitError, match="bf16"):
        solve(fp32)
    with pytest.raises(ob.OdevitError, match="PARALLEL"):
        solve(_field(l2_attention=True))
    with pytest.raises(ob.OdevitError, match="PARALLEL"):
        solve(_field(ob.macaron.ViT_ODEFunc))
    with pytest.raises(ob.OdevitError, match="dim"):
        solve(_field(dim=256, heads=4, l2_attention=False), x=torch.randn(2, 69, 256).cuda())
    drop = _field(l2_attention=False, mlp_drop=0.1).train()
    with pytest.raises(ob.OdevitError, match="dropout"):
        solve(drop)
    with pytest.raises(ob.OdevitError, match="differentiable"):
        ob.odeint_adaptive(base, x0.clone().requires_grad_(True), T_OUT, rtol=1e-3, atol=1e-4, differentiable=True,
                           capturable=True)
    with pytest.raises(ob.OdevitError, match="t_out"):
        solve(base, t=torch.linspace(0.0, 1.0, 130))
    with pytest.raises(ob.OdevitError, match="t_out"):
        solve(base, t=torch.tensor([0.0, 0.5, 0.25]))


def test_more_than_96_tokens():
    import odevit_b200 as ob
    cfg = dict(CFG, embed_dim=64, num_heads=1, mlp_ratio=2.0, img_size=40, patch_size=4, register_tokens=11)
    sd = orc.reference_like_init(cfg, 10, seed=0)
    model = ob.ViTNeuralODE(**cfg)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    model.precision = "bf16"
    px = torch.randn(3, 3, 40, 40, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        x0 = model.patch_embed(px.cuda()).contiguous()
    assert x0.shape[1] > 96
    states, stats = _solve(model, x0)
    want = _oracle(sd, x0, heads=1)
    assert max_rel(states, want["states"]) < 2e-2
