"""CPU tests of the per-image evaluation sequence of the adaptive dopri5 restatement (tests/_adaptive_attn_ref.py), the
reference that tests/test_gpu_adaptive_attn.py holds the adaptive solve's p_last and JaSMin window to."""
import pytest
import torch

import _adaptive_attn_ref as aref
import _adaptive_grad_ref as gref
import adaptive_dp5 as dp

T_OUT = torch.tensor([0.0, 0.3, 1.0], dtype=torch.float64)


def _field():
    # images of different stiffness: different step counts per image
    rate = torch.tensor([0.5, 4.0, 20.0], dtype=torch.float64).reshape(3, 1, 1)
    return lambda y: -rate * y + 0.3 * torch.sin(y.flip(-1))


def _y0():
    return torch.randn(3, 4, 5, generator=torch.Generator().manual_seed(3), dtype=torch.float64)


@pytest.mark.parametrize("first_step", [None, 0.05])
def test_evaluation_count_and_order(first_step):
    res = aref.dopri5_evaluations(_field(), _y0(), T_OUT, 1e-6, 1e-8, first_step=first_step)
    want = dp.dopri5(_field(), _y0(), T_OUT, 1e-6, 1e-8, first_step=first_step, record_steps=True)
    assert torch.equal(res["states"], want["states"]) and res["steps"] == want["steps"]   # outputs unchanged
    probe = 1 if first_step is None else 0
    assert len(set(res["nfe"].tolist())) > 1 and int(res["rejected"].sum()) > 0
    for b, ev in enumerate(res["evaluations"]):
        acc, rej = int(res["accepted"][b]), int(res["rejected"][b])
        assert len(ev) == 1 + probe + 6 * (acc + rej) == int(res["nfe"][b])
        assert torch.equal(ev[0]["state"], _y0()[b])
        assert all(e["step"] is None for e in ev[:1 + probe])
        steps = [e["step"] for e in ev[1 + probe:]]
        assert steps == [r for r in range(acc + rej) for _ in range(6)]
        assert [e["accepted"] for e in ev[1 + probe::6]] == [s[2] for s in res["steps"][b]]
        assert ev[-1]["accepted"] is True


def test_last_evaluation_is_f_of_y1_of_the_last_accepted_step():
    """Replaying the accepted steps (no rejections, no probe) and logging its calls: the k7 = f(y1) of each image's last
    accepted step is the oracle's last evaluation of that image."""
    f = _field()
    res = aref.dopri5_evaluations(f, _y0(), T_OUT, 1e-6, 1e-8)
    rec = gref.record_from_steps(res["steps"], T_OUT)
    calls = []

    def logged(y):
        calls.append(y.clone())
        return f(y)

    gref.replay(logged, _y0(), T_OUT, *rec)
    for b, ev in enumerate(res["evaluations"]):
        n = int(res["accepted"][b])
        y1 = calls[1 + 6 * (n - 1) + 5][b]
        assert torch.allclose(ev[-1]["state"], y1, rtol=0, atol=1e-13)


def test_window_takes_the_last_evaluations():
    torch.manual_seed(0)
    H, N = 2, 4
    M = torch.randn(H, N, 5, dtype=torch.float64)

    def field_map(y):   # any per-image map [1, H, N, N] of the state
        s = torch.einsum("bnd,hmd->bhnm", y, M)
        return torch.softmax(s, dim=-1)

    res = aref.dopri5_evaluations(_field(), _y0(), T_OUT, 1e-6, 1e-8)
    ev = res["evaluations"][0]
    for W in (3, len(ev), len(ev) + 5):
        for k in (0, 2):
            got = aref.window(ev, W, field_map, k)
            assert got.shape == (min(W, len(ev)), H)
            want = aref.jasmin_stat(field_map(ev[-1]["state"][None]), k)[0]
            assert torch.equal(got[-1], want)
