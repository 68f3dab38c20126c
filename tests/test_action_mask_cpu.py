"""Invalid-action masking (ACTION_MASK) without a GPU: self-checks of the float64 restatement the GPU tests compare against
(tests/action_mask_ref.py), option validation, NORM_OBS's treatment of the mask slot, the factories, Experience.batch_data and the
C ABI (the new symbols, and the engine's slot table, which needs no device)."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import action_mask_ref as M
from oracle import restate as R


def _net(kind="navimg", **hyper):
    from ddrl4nav_b200.runner import make_net
    return make_net(kind, device=None, **hyper)


def _batch(B, A, seed):
    g = torch.Generator().manual_seed(seed)
    logits = 2 * torch.randn(B, A, generator=g, dtype=torch.float64)
    v, ret, adv = (torch.randn(B, generator=g, dtype=torch.float64) for _ in range(3))
    return logits, v, ret, adv, g


# ---------------------------------------------------------------------------------------------------------- restatement
@pytest.mark.parametrize("shared", [True, False])
def test_all_ones_mask_is_the_unmasked_chain(shared):
    B, A = 64, 6
    logits, v, ret, adv, g = _batch(B, A, 0)
    a = torch.randint(0, A, (B,), generator=g)
    old = M.log_prob(logits, None, a).detach() + 0.2 * torch.randn(B, generator=g, dtype=torch.float64)
    ones = torch.ones(B, A, dtype=torch.uint8)
    assert torch.equal(M.masked_probs(logits, ones), M.masked_probs(logits, None))
    r1, g1, v1 = M.loss_and_grads(logits, ones, a, old, adv, ret, v, R.PPOHyper(), shared)
    r0, g0, v0 = M.loss_and_grads(logits, None, a, old, adv, ret, v, R.PPOHyper(), shared)
    assert r1 == r0 and torch.equal(g1, g0) and torch.equal(v1, v0)
    # ... and the unmasked chain is the oracle's
    want = R.categorical_log_prob(torch.softmax(logits, -1), a)
    assert torch.equal(M.log_prob(logits, None, a), want)


def test_a_row_that_allows_nothing_is_an_all_ones_row():
    B, A = 8, 5
    logits, v, ret, adv, g = _batch(B, A, 1)
    a = torch.randint(0, A, (B,), generator=g)
    zero, ones = torch.zeros(B, A), torch.ones(B, A)
    assert torch.equal(M.masked_probs(logits, zero), M.masked_probs(logits, ones))
    rz, gz, _ = M.loss_and_grads(logits, zero, a, a.double() * 0 - 1.5, adv, ret, v, R.PPOHyper(), True)
    ro, go, _ = M.loss_and_grads(logits, ones, a, a.double() * 0 - 1.5, adv, ret, v, R.PPOHyper(), True)
    assert rz == ro and torch.equal(gz, go) and all(np.isfinite(list(rz.values())))


@pytest.mark.parametrize("shared", [True, False])
def test_masked_logits_get_zero_gradient_and_add_nothing_to_the_entropy(shared):
    B, A = 200, 28
    logits, v, ret, adv, g = _batch(B, A, 2)
    mask = M.random_mask(B, A, seed=3)
    eff = M.effective_mask(mask)
    q = M.masked_probs(logits, mask)
    assert (q[~eff] == 0).all() and torch.allclose(q.sum(-1), torch.ones(B, dtype=torch.float64))
    # taken actions: allowed ones, except a few rows that hold a masked action (corrupt data: log(eps), zero gradient)
    a = torch.multinomial(q, 1, generator=g).squeeze(-1)
    bad = [r for r in range(B) if not eff[r].all()][:3]
    for r in bad:
        a[r] = int(torch.nonzero(~eff[r])[0])
    lp = M.log_prob(logits, mask, a)
    assert torch.allclose(lp[bad], torch.full((len(bad),), np.log(np.float32(np.finfo(np.float32).eps)), dtype=torch.float64))
    old = lp.detach() + 0.3 * torch.randn(B, generator=g, dtype=torch.float64)
    _, glog, _ = M.loss_and_grads(logits, mask, a, old, adv, ret, v, R.PPOHyper(), shared,
                                  old_values=v + 0.1, value_clip=0.2, prox=old - 0.1, is_clip=1.5)
    assert torch.isfinite(glog).all() and (glog[~eff] == 0).all()
    ent_masked = M.entropy(logits, mask)
    ent_sub = torch.stack([R.categorical_entropy(torch.softmax(logits[r][eff[r]], -1)) for r in range(B)])
    assert torch.allclose(ent_masked, ent_sub, rtol=1e-12, atol=1e-12)


def test_inverse_cdf_falls_back_to_the_first_allowed_action():
    q = np.array([[0.0, 0.25, 0.5], [0.25, 0.25, 0.5], [0.0, 0.0, 0.5]], np.float32)     # rows 0 and 2 sum to less than u
    mask = torch.tensor([[0, 1, 1], [1, 1, 1], [0, 0, 1]])
    u = np.array([0.99999994, 0.3, 0.9], np.float32)
    assert M.sample_on_q(q, u, mask).tolist() == [1, 1, 2]
    assert M.sample_on_q(q, np.array([0.1, 0.1, 0.1], np.float32), mask).tolist() == [1, 0, 2]


# ---------------------------------------------------------------------------------------------------------- the option
@pytest.mark.parametrize("bad", [1, 0, "yes", None, 1.0, [True]])
def test_action_mask_must_be_a_bool(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="ACTION_MASK"):
        _net(ACTION_MASK=bad)


@pytest.mark.parametrize("kind", ["navlaser", "navlaser_beta", "navimg_beta"])
def test_action_mask_needs_a_categorical_actor(kind):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="ACTION_MASK needs a CategoricalActor"):
        _net(kind, ACTION_MASK=True)
    assert _net(kind, ACTION_MASK=False).action_mask is False


@pytest.mark.parametrize("kind", ["pong", "navimg", "navped", "mlp"])
def test_make_net_takes_the_option_and_adds_no_state(kind):
    on, off = _net(kind, ACTION_MASK=True), _net(kind)
    assert on.action_mask is True and off.action_mask is False and np.bool_(True) == _net(kind, ACTION_MASK=np.bool_(True)).action_mask
    assert list(on.state_dict()) == list(off.state_dict())
    on.load_state_dict(off.state_dict(), strict=True)
    assert on.model_bytes() == off.model_bytes()


def test_create_net_takes_the_option():
    from ddrl4nav_b200.nn import CategoricalActor
    from ddrl4nav_b200.runner import create_net
    config = SimpleNamespace(DEVICE="cpu", TASK_TYPE="robot_nav", TASK_NAME="t-127.0.0.1", MODULE_KEY="MODEL")
    config_nn = SimpleNamespace(DEVICE="cpu", AC_INPUT_DIM=512, ACTOR_CLASS=CategoricalActor, ACTION_OUTPUT_DIM=28,
                                SOFT_MAX_GRID=True, MODULE_TENSOR_DTYPE=torch.float32, SHARE_CNN_NET=True, NETWORK_TYPE="ppo",
                                ACTION_MASK=True)
    net = create_net({"config": config, "config_nn": config_nn, "config_env": {"image_batch": 1, "ped_sim": {"total": 0}}})
    assert net.action_mask is True


def test_norm_obs_leaves_the_mask_slot_out():
    from ddrl4nav_b200._lib import DDRLError
    from ddrl4nav_b200.nn.obs_rms import ObsRMS
    elems = {0: 2304, 1: 9, 2: 6912, 3: 28}.__getitem__           # navped: three encoder slots, the mask in slot 3
    every = ObsRMS(None, 10.0)
    every.bind(4, elems, "cpu", mask_slot=3)
    assert every.slots == (0, 1, 2) and "mean_3" not in dict(every.named_buffers())
    listed = ObsRMS((0, 2), 10.0)
    listed.bind(4, elems, "cpu", mask_slot=3)
    assert listed.slots == (0, 2)
    with pytest.raises(DDRLError, match="ACTION_MASK slot"):
        ObsRMS((1, 3), 10.0).bind(4, elems, "cpu", mask_slot=3)
    plain = ObsRMS(None, 10.0)
    plain.bind(4, elems, "cpu")                                   # without a mask every slot is normalised, as before
    assert plain.slots == (0, 1, 2, 3)


def test_experience_batch_data_carries_the_mask_slot():
    from ddrl4nav_b200.data import Experience
    states = [s.numpy() for s in R.synth_states("navimg", 6, seed=1)]
    masks = M.random_mask(6, 28, seed=2).numpy()
    exps = [Experience(states=[s[i:i + 3] for s in states] + [masks[i:i + 3]], advs=np.zeros(3, np.float32),
                       actions=np.zeros(3, np.float32), old_logps=np.zeros(3, np.float32), values=np.zeros((1, 3), np.float32))
            for i in (0, 3)]
    b = Experience.batch_data(exps)
    assert len(b.states) == 3 and b.states[2].dtype == np.uint8 and np.array_equal(b.states[2], masks)
    b.to_tensor(device="cpu")
    assert b.states[2].dtype == torch.float32 and torch.equal(b.states[2], torch.from_numpy(masks).float())


# ---------------------------------------------------------------------------------------------------------- C ABI
def _lib():
    import os
    from ddrl4nav_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    return L


def test_new_symbols_are_exported_and_bound():
    L = _lib()
    raw = C.CDLL(L.LIB_PATH)
    for name in ("ddrl_categorical_head_m", "ddrl_ppo_loss_categorical_m", "ddrl_logp_actions_categorical_m",
                 "ddrl_net_set_action_mask"):
        assert hasattr(raw, name) and name in L.SIGNATURES
    lib = L.load()
    # argument checks run before any device work
    assert lib.ddrl_categorical_head_m(None, 65, None, 1, 65, None, None, None, None, None) == -1       # A > 64
    assert lib.ddrl_logp_actions_categorical_m(None, 6, None, 0, 6, None, None, None) == 0             # B = 0: nothing to do


@pytest.mark.parametrize("kind,enc_slots", [("pong", 1), ("navimg", 2), ("navped", 3)])
def test_engine_adds_the_mask_slot(kind, enc_slots):
    L = _lib()
    lib = L.load()
    spec = R.SPECS[kind]
    desc = L.NetDesc(L.ARCH[spec.arch], spec.in_ch, spec.act_dim, L.DIST[spec.dist], int(spec.shared), spec.feat, 0, 0)
    h = C.c_void_p()
    assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) == 0
    try:
        assert lib.ddrl_net_num_obs(h) == enc_slots
        elems = [lib.ddrl_net_obs_elems(h, i) for i in range(enc_slots)]
        assert lib.ddrl_net_set_action_mask(h, 1) == 0
        assert lib.ddrl_net_num_obs(h) == enc_slots + 1
        assert [lib.ddrl_net_obs_elems(h, i) for i in range(enc_slots)] == elems
        assert lib.ddrl_net_obs_elems(h, enc_slots) == spec.act_dim
        assert lib.ddrl_net_set_action_mask(h, 0) == 0 and lib.ddrl_net_num_obs(h) == enc_slots
    finally:
        lib.ddrl_net_destroy(h)


def test_engine_rejects_the_mask_on_a_continuous_net():
    L = _lib()
    lib = L.load()
    for dist in ("gaussian", "beta"):
        desc = L.NetDesc(L.ARCH["nav1d"], 3, 2, L.DIST[dist], 0, 512, 0, 0)
        h = C.c_void_p()
        assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) == 0
        try:
            assert lib.ddrl_net_set_action_mask(h, 1) == -1
            assert lib.ddrl_net_num_obs(h) == 3
        finally:
            lib.ddrl_net_destroy(h)
    assert lib.ddrl_net_set_action_mask(None, 1) == -1
