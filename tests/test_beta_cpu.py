"""Beta actor without a GPU: the float64 restatement (tests/beta_ref.py) itself, BetaActor's parameter table and bound
validation, the create_net / make_net mapping, and that a Beta net on the CPU fails loudly like every other net."""
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.special as sp
import scipy.stats as st
import torch

import beta_ref as BR
from oracle import restate as R


# ---------------------------------------------------------------------------------------------------------- the restatement
def test_inverse_is_the_inverse_of_the_incomplete_beta():
    a = np.array([1.0, 1.001, 2.0, 10.0, 100.0, 1e3, 1e4])
    u = np.array([1e-7, 1e-3, 0.1, 0.5, 0.9, 0.999, 1 - 6e-8])
    A, Bt, U = np.meshgrid(a, a, u, indexing="ij")
    x = sp.betaincinv(A, Bt, U)
    assert np.all((x >= 0) & (x <= 1))
    assert np.allclose(sp.betainc(A, Bt, x), U, rtol=1e-9, atol=1e-12)


def test_sample_stays_inside_the_bounds_and_play_mode_is_the_mean():
    g = torch.Generator().manual_seed(0)
    head = 40 * torch.randn(500, 6, generator=g)        # concentrations from 1 to ~120, softplus' identity branch included
    low, high = torch.tensor([-1.0, 0.0, -0.5]), torch.tensor([1.0, 3.0, -0.25])
    u = torch.rand(500, 3, generator=g)
    a = BR.sample(head, low, high, u)
    assert bool(((a >= low) & (a <= high)).all())
    al, be = BR.concentrations(head)
    m = BR.mean_action(head, low, high)
    assert torch.allclose(m.double(), (low + (high - low) * al / (al + be)).double(), rtol=1e-6)


def test_log_prob_and_entropy_match_the_closed_forms():
    g = torch.Generator().manual_seed(1)
    head = 2 * torch.randn(64, 4, generator=g)
    low, high = torch.tensor([-1.0, 2.0]), torch.tensor([1.0, 5.0])
    a = BR.sample(head, low, high, torch.rand(64, 2, generator=g))
    al, be = (t.double().numpy() for t in BR.concentrations(head.double()))
    w = (high - low).double().numpy()
    x = np.clip((a.double().numpy() - low.double().numpy()) / w, 1e-6, 1 - 1e-6)
    lp = ((al - 1) * np.log(x) + (be - 1) * np.log1p(-x) - sp.betaln(al, be) - np.log(w)).sum(-1)
    assert np.allclose(BR.log_prob(head, low, high, a).numpy(), lp, rtol=1e-12, atol=1e-12)
    ent = st.beta(al, be).entropy() + np.log(w)
    assert np.allclose(BR.entropy(head, low, high).numpy(), ent, rtol=1e-10, atol=1e-12)


def test_loss_reduces_to_plain_ppo_and_the_ratio_is_one_on_policy():
    g = torch.Generator().manual_seed(2)
    head = torch.randn(32, 4, generator=g)
    low, high = torch.full((2,), -1.0), torch.full((2,), 1.0)
    a = BR.sample(head, low, high, torch.rand(32, 2, generator=g))
    lp = BR.log_prob(head, low, high, a)
    adv, ret, v = (torch.randn(32, generator=g) for _ in range(3))
    out, dh, _ = BR.loss_and_grads(head, low, high, a, lp, adv, ret, v, R.PPOHyper(), shared=False)
    assert out["ApproxKL"] == 0.0 and out["ClipFrac"] == 0.0
    assert out["actor"] == pytest.approx(-float(adv.double().mean()), rel=1e-12)
    out2, dh2, _ = BR.loss_and_grads(head, low, high, a, lp, adv, ret, v, R.PPOHyper(), shared=False, prox=lp)
    assert out2["actor"] == out["actor"] and torch.equal(dh, dh2) and out2["BehaviourKL"] == 0.0


# ---------------------------------------------------------------------------------------------------------- BetaActor
def test_parameter_table_is_the_oracles_with_a_2A_head():
    from ddrl4nav_b200.runner import make_net
    for kind, spec in BR.SPECS.items():
        net = make_net(kind, device=None)
        assert [(n, tuple(p.shape)) for n, p in net.named_parameters()] == R.param_table(spec), kind
        assert dict(net.named_parameters())["actor.actor_linear.weight"].shape == (4, 512)
        assert not any("log_std" in n or "low" in n or "high" in n for n in net.state_dict())
        net.load_state_dict(R.init_params(spec, seed=3))


def test_bounds_are_configuration_broadcast_and_validated():
    from ddrl4nav_b200._lib import DDRLError
    from ddrl4nav_b200.nn import BetaActor
    act = BetaActor(3, last_input_dim=8, low=-2, high=[1, 2, 3.5])
    assert act.action_low == (-2.0, -2.0, -2.0) and act.action_high == (1.0, 2.0, 3.5)
    assert list(act.state_dict()) == ["actor_linear.weight", "actor_linear.bias"]
    assert BetaActor(2, last_input_dim=8).action_low == (-1.0, -1.0)
    bad = [dict(low=1.0, high=1.0), dict(low=[0.0, 2.0], high=[1.0, 1.0]), dict(low=float("nan")), dict(high=float("inf")),
           dict(low=[0.0, 0.0, 0.0]), dict(low="a"), dict(low=True), dict(high=1e39)]
    for kw in bad:
        with pytest.raises(DDRLError):
            BetaActor(2, last_input_dim=8, **kw)
    with pytest.raises(DDRLError):
        BetaActor(0, last_input_dim=8)


# ---------------------------------------------------------------------------------------------------------- factories
def _configs(actor_cls, share, **nn_extra):
    config = SimpleNamespace(TASK_TYPE="robot_nav", TASK_NAME="t", MODULE_KEY="MODEL")
    config_nn = SimpleNamespace(DEVICE="cpu", AC_INPUT_DIM=512, ACTOR_CLASS=actor_cls, ACTION_OUTPUT_DIM=2, SOFT_MAX_GRID=True,
                                MODULE_TENSOR_DTYPE=torch.float32, SHARE_CNN_NET=share, NETWORK_TYPE="ppo", **nn_extra)
    config_env = {"image_batch": 1, "ped_sim": {"total": 0}}
    return {"config": config, "config_nn": config_nn, "config_env": config_env}


def test_create_net_takes_the_beta_actor_and_its_bounds():
    from ddrl4nav_b200._lib import DDRLError
    from ddrl4nav_b200.nn import BetaActor
    from ddrl4nav_b200.runner import create_net
    net = create_net(_configs(BetaActor, False, ACTION_LOW=[0.0, -0.8], ACTION_HIGH=[0.6, 0.8]))
    assert type(net.actor) is BetaActor and net._spec()["act_dim"] == 2 and net._spec()["dist"] == "beta"
    assert net.actor.action_low == (0.0, np.float32(-0.8)) and net.actor.action_high == (np.float32(0.6), np.float32(0.8))
    assert [(n, tuple(p.shape)) for n, p in net.named_parameters()] == R.param_table(BR.SPECS["navlaser_beta"])
    shared = create_net(_configs(BetaActor, True))
    assert shared.actor.action_low == (-1.0, -1.0) and shared._spec()["shared"]
    for bad in (dict(ACTION_LOW=1.0, ACTION_HIGH=0.0), dict(ACTION_LOW=[0.0]), dict(ACTION_HIGH=float("nan"))):
        with pytest.raises(DDRLError):
            create_net(_configs(BetaActor, False, **bad))


def test_make_net_beta_kinds():
    from ddrl4nav_b200.nn import BetaActor, NavPreNet, NavPreNet1D
    from ddrl4nav_b200.runner import make_net
    a = make_net("navlaser_beta", device=None, ACTION_LOW=[0.0, -1.0], ACTION_HIGH=[0.5, 1.0])
    assert type(a.actor) is BetaActor and a.prenet is None and type(a.actor.pre) is NavPreNet1D
    assert a.actor.action_low == (0.0, -1.0) and a.actor.action_high == (0.5, 1.0)
    b = make_net("navimg_beta", device=None)
    assert type(b.actor) is BetaActor and type(b.prenet) is NavPreNet and b._spec()["act_dim"] == 2


def test_cpu_beta_net_fails_loudly():
    from ddrl4nav_b200._lib import DDRLError
    from ddrl4nav_b200.runner import make_net
    net = make_net("navlaser_beta", device=None)
    states = R.synth_states("navlaser", 2)
    with pytest.raises(DDRLError):
        net.act(states)
    with pytest.raises(DDRLError):
        net.actor(torch.zeros(2, 512))
