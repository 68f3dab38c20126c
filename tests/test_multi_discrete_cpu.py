"""MultiDiscrete actor without a GPU: the float64 restatement (tests/multi_discrete_ref.py) against an explicit product of torch
Categoricals, masks included; the MultiCategorical distribution object; nvec validation through the actor, create_net and
make_net; and the parameter tables of the navimg_md and navlaser_md kinds."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from torch.distributions.categorical import Categorical

import action_mask_ref as M
import multi_discrete_ref as MD
from oracle import restate as R

NVECS = [(6,), (4, 7), (5, 9), (2, 3, 1, 8), (1, 1), (8,) * 8]


def _product(logits, mask, nvec):
    """torch's own product of Categoricals: one Categorical(logits.masked_fill(~m, -inf)) per branch."""
    out = []
    for lo, hi in MD.slices(nvec):
        x = logits[:, lo:hi]
        if mask is not None:
            x = x.masked_fill(~M.effective_mask(mask[:, lo:hi]), float("-inf"))
        out.append(Categorical(logits=x))
    return out


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("nvec", NVECS)
def test_restatement_is_a_product_of_categoricals(nvec, masked):
    B = 300
    g = torch.Generator().manual_seed(sum(nvec) + len(nvec))
    logits = (2 * torch.randn(B, sum(nvec), generator=g)).double()
    mask = MD.random_mask(B, nvec, seed=3) if masked else None
    a = MD.sample(logits, mask, nvec, g)
    dists = _product(logits, mask, nvec)
    lp = sum(d.log_prob(a[:, i].long()) for i, d in enumerate(dists))
    ent = sum(d.entropy() for d in dists)
    # the restatement keeps torch's Categorical(probs) chain, clamp(q, eps, 1 - eps) with the fp32 eps: ~1e-7 per branch
    assert torch.allclose(MD.log_prob(logits, mask, a, nvec), lp, rtol=0, atol=2e-7 * len(nvec))
    assert torch.allclose(MD.entropy(logits, mask, nvec), ent, rtol=0, atol=2e-6 * len(nvec))
    if masked:
        eff = MD.effective_mask(mask, nvec)
        assert all(bool(eff[torch.arange(B), lo + a[:, i].long()].all()) for i, (lo, hi) in enumerate(MD.slices(nvec)))
        assert (MD.branch_probs(logits, mask, nvec)[~eff] == 0).all()


def test_one_branch_is_the_categorical_restatement():
    g = torch.Generator().manual_seed(5)
    logits = torch.randn(200, 28, generator=g).double()
    mask = M.random_mask(200, 28, seed=6)
    a = torch.randint(0, 28, (200,), generator=g).float()
    assert torch.equal(MD.log_prob(logits, mask, a[:, None], (28,)), M.log_prob(logits, mask, a))
    assert torch.equal(MD.entropy(logits, mask, (28,)), M.entropy(logits, mask))


def test_empty_branch_rule_is_per_branch():
    mask = torch.ones(3, 11, dtype=torch.uint8)
    mask[0, :4] = 0                          # branch 0 allows nothing: all-ones there, branch 1 untouched
    mask[1, 4:6] = 0
    eff = MD.effective_mask(mask, (4, 7))
    assert eff[0].all() and not eff[1, 4:6].any() and eff[1, :4].all() and eff[1, 6:].all()


def test_multicategorical_object():
    from ddrl4nav_b200.nn import MultiCategorical
    nvec = (3, 5)
    g = torch.Generator().manual_seed(1)
    p = MD.branch_probs(torch.randn(50, 8, generator=g).double(), None, nvec).float()
    d = MultiCategorical(p, nvec)
    torch.manual_seed(0)
    a = d.sample()
    assert a.shape == (50, 2) and (a[:, 0] < 3).all() and (a[:, 1] < 5).all()
    assert d.sample((4,)).shape == (4, 50, 2)
    want = Categorical(p[:, :3]).log_prob(a[:, 0]) + Categorical(p[:, 3:]).log_prob(a[:, 1])
    assert torch.equal(d.log_prob(a.float()), want)
    assert torch.equal(d.entropy(), Categorical(p[:, :3]).entropy() + Categorical(p[:, 3:]).entropy())


# ------------------------------------------------------------------------------------------------------------ validation
@pytest.mark.parametrize("nvec", [(), [0], (3, -1), (2.0, 3), (True, 2), "ab", 5, None, (1,) * 9, (40, 25), [64, 1]])
def test_actor_rejects_bad_nvec(nvec):
    from ddrl4nav_b200 import DDRLError
    from ddrl4nav_b200.nn import MultiCategoricalActor
    with pytest.raises(DDRLError):
        MultiCategoricalActor(nvec)


@pytest.mark.parametrize("nvec", [(1,), (64,), [4, 7], (8,) * 8, np.array([5, 9]), torch.tensor([2, 2, 2])])
def test_actor_accepts_good_nvec(nvec):
    from ddrl4nav_b200.nn import MultiCategoricalActor
    a = MultiCategoricalActor(nvec, last_input_dim=16)
    assert a.nvec == tuple(int(n) for n in nvec) and a.actor_linear.out_features == sum(a.nvec)
    assert [n for n, _ in a.named_parameters()] == ["actor_linear.weight", "actor_linear.bias"]


def test_actor_checks_action_output_dim():
    from ddrl4nav_b200 import DDRLError
    from ddrl4nav_b200.nn import MultiCategoricalActor
    assert MultiCategoricalActor((4, 7), action_output_dim=11).action_output_dim == 11
    with pytest.raises(DDRLError):
        MultiCategoricalActor((4, 7), action_output_dim=28)


def _configs(**nn_kw):
    from ddrl4nav_b200.nn import MultiCategoricalActor
    config = SimpleNamespace(TASK_TYPE="robot_nav", DEVICE=None, TASK_NAME="t-127.0.0.1", MODULE_KEY="MODEL")
    cfg = dict(DEVICE=None, AC_INPUT_DIM=512, ACTOR_CLASS=MultiCategoricalActor, ACTION_OUTPUT_DIM=11, SOFT_MAX_GRID=True,
               MODULE_TENSOR_DTYPE=torch.float32, SHARE_CNN_NET=True, NETWORK_TYPE="ppo")
    cfg.update(nn_kw)
    env = {"image_batch": 1, "ped_sim": {"total": 0}}
    return {"config": config, "config_nn": SimpleNamespace(**cfg), "config_env": env}


def test_create_net_reads_action_nvec():
    from ddrl4nav_b200 import DDRLError
    from ddrl4nav_b200.runner import create_net
    cfgs = _configs(ACTION_NVEC=(4, 7))
    cfgs["config"].DEVICE = "cpu"
    cfgs["config_nn"].DEVICE = "cpu"
    net = create_net(cfgs)
    assert net.actor.nvec == (4, 7) and net.actor.DIST == "multi_categorical"
    for bad in (dict(), dict(ACTION_NVEC=(4, 8)), dict(ACTION_NVEC=(0, 11))):
        cfgs = _configs(**bad)
        cfgs["config"].DEVICE = cfgs["config_nn"].DEVICE = "cpu"
        with pytest.raises(DDRLError):
            create_net(cfgs)


def test_make_net_kinds_and_override():
    from ddrl4nav_b200 import DDRLError
    from ddrl4nav_b200.runner import make_net
    assert make_net("navimg_md", device=None).actor.nvec == (4, 7)
    assert make_net("navlaser_md", device=None).actor.nvec == (5, 9)
    net = make_net("navlaser_md", device=None, ACTION_NVEC=(3, 3, 2))
    assert net.actor.nvec == (3, 3, 2) and net.actor.actor_linear.out_features == 8
    assert make_net("navimg_md", device=None, ACTION_NVEC=[28]).actor.nvec == (28,)
    assert make_net("navimg_md", device=None, ACTION_MASK=True).action_mask
    for bad in ((), (65,), (1,) * 9):
        with pytest.raises(DDRLError):
            make_net("navimg_md", device=None, ACTION_NVEC=bad)


@pytest.mark.parametrize("kind,spec", [("navimg_md", R.NetSpec("nav", 1, 11, "categorical", True)),
                                       ("navlaser_md", R.NetSpec("nav1d", 3, 14, "categorical", False))])
def test_parameter_tables(kind, spec):
    """A MultiDiscrete kind has the parameter table of a categorical net of head width sum n: nvec adds no parameter and no
    state_dict key."""
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None)
    assert [(n, tuple(p.shape)) for n, p in net.named_parameters()] == [(n, tuple(s)) for n, s in R.param_table(spec)]
    assert list(net.state_dict()) == [n for n, _ in R.param_table(spec)]


def test_action_mask_is_refused_for_continuous_actors_only():
    from ddrl4nav_b200 import DDRLError
    from ddrl4nav_b200.runner import make_net
    make_net("navlaser_md", device=None, ACTION_MASK=True)
    with pytest.raises(DDRLError):
        make_net("navlaser_beta", device=None, ACTION_MASK=True)
