"""CPU checks of tests/engine_state_ref.py: the float64 clip + Adam step the GPU engine-state tests hold every optimiser step
against is torch's clip_grad_norm_ + Adam, and its tolerance separates fp32 rounding from a stale operand."""
import pytest
import torch

import engine_state_ref as ES
from oracle import restate as R


@pytest.mark.parametrize("nseg", [1, 2])
def test_clip_adam_step_equals_torch_adam(nseg):
    """Three steps (the second below the clip norm, so coef = 1) over one or two LR segments, against torch.optim.Adam per
    segment after one clip_grad_norm_ over all of them -- the optimisers of nn/ppo.py:40-42,110-129 -- in float64, with the
    betas rounded to fp32 as the engine holds them."""
    g = torch.Generator().manual_seed(7)
    n, cut = 1000, 337
    segs = [0, n] if nseg == 1 else [0, cut, n]
    lrs = [2e-4] if nseg == 1 else [5e-5, 1e-3]
    p0 = torch.randn(n, generator=g, dtype=torch.float64)
    ref = [p0[segs[i]:segs[i + 1]].clone().requires_grad_(True) for i in range(nseg)]
    opts = [torch.optim.Adam([ref[i]], lrs[i], betas=(ES.fp32(0.9), ES.fp32(0.999))) for i in range(nseg)]
    lr = torch.cat([torch.full((segs[i + 1] - segs[i],), lrs[i], dtype=torch.float64) for i in range(nseg)])
    p, m, v = p0.clone(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    for step in range(1, 4):
        grad = torch.randn(n, generator=g, dtype=torch.float64) * (0.005 if step == 2 else 1.0)
        for i in range(nseg):
            ref[i].grad = grad[segs[i]:segs[i + 1]].clone()
        total = float(torch.nn.utils.clip_grad_norm_(ref, 0.5))
        for o in opts:
            o.step()
        p, m, v, norm = ES.clip_adam_step(p, grad, m, v, step, lr)
        assert abs(norm - total) <= 1e-12 * total
        assert torch.allclose(p, torch.cat([r.detach() for r in ref]), rtol=0, atol=1e-13)
        m_ref = torch.cat([opts[i].state[ref[i]]["exp_avg"] for i in range(nseg)])
        v_ref = torch.cat([opts[i].state[ref[i]]["exp_avg_sq"] for i in range(nseg)])
        assert torch.allclose(m, m_ref, rtol=1e-12, atol=0) and torch.allclose(v, v_ref, rtol=1e-12, atol=0)


def test_adam_tolerance_takes_fp32_rounding_and_rejects_a_stale_gradient():
    """The engine steps in fp32: the reference rounded to fp32 must pass.  A step taken with the gradient of a parameter one
    Adam step old is off by ~1e-3 of the gradient: it must not."""
    g = torch.Generator().manual_seed(3)
    n = 4096
    p = torch.randn(n, generator=g) * 0.05
    m = torch.randn(n, generator=g) * 1e-3
    v = torch.rand(n, generator=g) * 1e-6
    grad = torch.randn(n, generator=g) * 1e-2
    ref = ES.clip_adam_step(p, grad, m, v, 7, 1e-3)
    assert not ES.adam_mismatch(p, [t.float() for t in ref[:3]], ref[:3])
    stale = ES.clip_adam_step(p, grad * (1 + 1e-3 * torch.randn(n, generator=g)), m, v, 7, 1e-3)
    bad = ES.adam_mismatch(p, [t.float() for t in stale[:3]], ref[:3])
    assert "m" in bad and "v" in bad, bad
    wrong_step = ES.clip_adam_step(p, grad, m, v, 6, 1e-3)            # the step scalars of another step
    assert "p" in ES.adam_mismatch(p, [t.float() for t in wrong_step[:3]], ref[:3])


@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_element_lrs_follow_the_optimisers_of_the_reference(kind):
    spec = R.SPECS[kind]
    table = R.param_table(spec)
    names, sizes = [n for n, _ in table], [int(torch.Size(s).numel()) for _, s in table]
    lr = ES.element_lrs(spec, names, sizes)
    assert lr.numel() == sum(sizes)
    if spec.shared:
        assert bool((lr == 2e-4).all())
    else:
        cut = sum(sizes[:names.index("critic.critic_linear.weight")])
        assert bool((lr[:cut] == 5e-5).all()) and bool((lr[cut:] == 1e-3).all())
