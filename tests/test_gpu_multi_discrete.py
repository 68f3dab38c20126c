"""MultiDiscrete actor (MultiCategoricalActor) on the GPU: K = 1 against the categorical actor bit for bit (head kernel and whole
learner), per-branch inverse-CDF sampling and play mode with masks, log-prob bit equality of the head, pre-pass and loss kernels,
the fused loss against the float64 restatement (tests/multi_discrete_ref.py) with every option, whole-net gradients against the
oracle encoders, learn() with graphs and determinism, the engine's branch-table checks, the Forward module and ForwardThread, and
two-GPU parity."""
import ctypes as C
import socket
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import action_mask_ref as M
import multi_discrete_ref as MD
from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")
U_TOP = 1.0 - 2.0 ** -24                     # the largest fp32 below 1
NVECS = [(4, 7), (5, 9), (2, 3, 1, 8), (8,) * 8, (1, 6)]
# the oracle parameter tables of the MultiDiscrete kinds (a categorical head of width sum n) and their observations
SPECS = {"navimg_md": R.NetSpec("nav", 1, 11, "categorical", True), "navlaser_md": R.NetSpec("nav1d", 3, 14, "categorical", False)}
STATES_OF = {"navimg_md": "navimg", "navlaser_md": "navlaser"}
NVEC_OF = {"navimg_md": (4, 7), "navlaser_md": (5, 9)}


@pytest.fixture
def deterministic():
    from ddrl4nav_b200 import kernels
    was = kernels.set_deterministic(True)
    yield
    kernels.set_deterministic(was)


def _logits(B, A, seed):
    g = torch.Generator().manual_seed(seed)
    logits = 3 * torch.randn(B, A, generator=g)
    logits[:8] = torch.round(logits[:8])     # ties
    return logits, g


def _draw(B, K, g):
    u = torch.rand(B, K, generator=g)
    u[:4] = torch.tensor([0.0, U_TOP, 0.5, 1e-7])[:, None]
    return u


# ---------------------------------------------------------------------------------------------------------- 1. head kernel
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("A", [2, 6, 28, 64])
def test_one_branch_head_is_the_categorical_head(A, masked):
    from ddrl4nav_b200 import kernels
    B = 3000
    logits, g = _logits(B, A, A)
    u = _draw(B, 1, g)
    mask = M.random_mask(B, A, seed=A).to(DEV) if masked else None
    for draw in (u.to(DEV), None):
        want = kernels.categorical_head_m(logits.to(DEV), None if draw is None else draw[:, 0], mask)
        got = kernels.multi_categorical_head(logits.to(DEV), (A,), draw, mask)
        assert got[0].shape == (B, 1) and torch.equal(got[0][:, 0], want[0])
        assert torch.equal(got[1], want[1]) and torch.equal(got[2], want[2])


@pytest.mark.parametrize("nvec", NVECS)
def test_head_samples_each_branch_on_its_own_q(nvec):
    from ddrl4nav_b200 import kernels
    B, K, A = 3000, len(nvec), sum(nvec)
    logits, g = _logits(B, A, 100 + A)
    u = _draw(B, K, g)
    mask = MD.random_mask(B, nvec, seed=A, empty_rows=3)
    a, lp, q = kernels.multi_categorical_head(logits.to(DEV), nvec, u.to(DEV), mask.to(DEV))
    a, lp, q = a.cpu(), lp.cpu(), q.cpu()
    eff = MD.effective_mask(mask, nvec)
    assert (q[~eff] == 0).all()
    assert np.array_equal(a.numpy().astype(np.int64), MD.sample_on_q(q.numpy(), u.numpy(), mask, nvec))
    for i, (lo, hi) in enumerate(MD.slices(nvec)):
        assert bool(eff[torch.arange(B), lo + a[:, i].long()].all())                  # never a masked action
    ref = MD.branch_probs(logits.double(), mask, nvec)
    for lo, hi in MD.slices(nvec):
        assert torch.allclose(q[:, lo:hi].double(), ref[:, lo:hi] / ref[:, lo:hi].sum(-1, keepdim=True), rtol=1e-5, atol=1e-7)
    assert torch.allclose(lp.double(), MD.log_prob(logits, mask, a, nvec), rtol=1e-5, atol=1e-6 * K)


@pytest.mark.parametrize("nvec", [(4, 7), (2, 3, 1, 8)])
def test_head_falls_back_to_each_branch_first_allowed_action(nvec):
    """u[:, i] set to the fp32 sum of branch i's own q: no prefix sum exceeds it, so every branch takes its first allowed action."""
    from ddrl4nav_b200 import kernels
    B, K, A = 512, len(nvec), sum(nvec)
    logits, _ = _logits(B, A, 7)
    mask = MD.random_mask(B, nvec, seed=8, p_allowed=0.5, empty_rows=0)
    for lo, hi in MD.slices(nvec):
        mask[:, lo] = 0
        mask[:, hi - 1] = 1
    _, _, q = kernels.multi_categorical_head(logits.to(DEV), nvec, torch.zeros(B, K, device=DEV), mask.to(DEV))
    q = q.cpu().numpy()
    top = np.stack([np.cumsum(q[:, lo:hi], axis=1, dtype=np.float32)[:, -1] for lo, hi in MD.slices(nvec)], 1)
    a, lp, _ = kernels.multi_categorical_head(logits.to(DEV), nvec, torch.from_numpy(top).to(DEV), mask.to(DEV))
    first = np.stack([M.first_allowed(mask[:, lo:hi]) for lo, hi in MD.slices(nvec)], 1)
    assert np.array_equal(a.cpu().numpy().astype(np.int64), first)
    assert all((first[:, i] > 0).all() for i, (lo, hi) in enumerate(MD.slices(nvec)) if hi - lo > 1)
    assert torch.equal(lp, kernels.logp_actions_multi_categorical(logits.to(DEV), nvec, a, mask.to(DEV)))


@pytest.mark.parametrize("nvec", [(4, 7), (5, 9)])
def test_head_play_mode_is_the_per_branch_first_max(nvec):
    from ddrl4nav_b200 import kernels
    B, A = 1000, sum(nvec)
    logits, _ = _logits(B, A, 9)
    mask = MD.random_mask(B, nvec, seed=10, empty_rows=50)
    a, lp, p = kernels.multi_categorical_head(logits.to(DEV), nvec, None, mask.to(DEV))
    assert (lp == 0).all()
    assert np.array_equal(a.cpu().numpy().astype(np.int64), MD.first_max(p.cpu().numpy(), mask, nvec))
    ref = MD.branch_probs(logits.double(), mask, nvec)
    assert torch.allclose(p.cpu().double(), ref, rtol=1e-5, atol=1e-7)


def test_head_entry_validates_the_branch_table():
    from ddrl4nav_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(4, 64, device=DEV)
    out = torch.empty(4, 8, device=DEV)
    lp = torch.empty(4, device=DEV)
    call = lambda K, nv: lib.ddrl_multi_categorical_head(_lib.ptr(x), 64, None, 4, K, (C.c_int32 * max(len(nv), 1))(*nv),
                                                         _lib.ptr(out), _lib.ptr(lp), None, None, None)
    assert call(2, [32, 32]) == 0 and call(8, [8] * 8) == 0
    assert call(0, []) == -1 and call(9, [1] * 9) == -1 and call(2, [0, 4]) == -1
    assert call(2, [40, 25]) == -4                                                    # DDRL_E_UNSUPPORTED: sum > 64
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------- 2. log-prob bits
@pytest.mark.parametrize("nvec", NVECS + [(28,)])
def test_act_prepass_and_loss_log_probs_are_equal_bits(nvec):
    """The head kernel's log-prob of the actions it emitted, the pre-pass's and the loss kernel's (ppo_clip 0 with old = prox =
    that log-prob counts any r != 1 in ClipFrac) are the same bits."""
    from ddrl4nav_b200 import kernels
    B, K, A = 2000, len(nvec), sum(nvec)
    logits, g = _logits(B, A, 20 + A)
    u = _draw(B, K, g).to(DEV)
    mask = MD.random_mask(B, nvec, seed=A + 1).to(DEV)
    x = logits.to(DEV)
    a, lp_act, _ = kernels.multi_categorical_head(x, nvec, u, mask)
    assert torch.equal(lp_act, kernels.logp_actions_multi_categorical(x, nvec, a, mask))
    v, ret, adv = (torch.randn(B, generator=g).to(DEV) for _ in range(3))
    hp = kernels.make_hparams(ppo_clip=0.0, ppo_stats=True)
    _, _, sums = kernels.ppo_loss_multi_categorical(x, nvec, a, lp_act, adv, ret, v, hp, True, mask=mask)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0
    _, _, sums = kernels.ppo_loss_multi_categorical(x, nvec, a, lp_act - 0.3, adv, ret, v, hp, True, mask=mask, prox_logp=lp_act)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0


# ---------------------------------------------------------------------------------------------------------- 3. loss kernel
OPTIONS = ["none", "dual_clip", "VALUE_CLIP", "value_norm", "prox", "prox_is_clip", "mask", "all"]


@pytest.mark.parametrize("opt", OPTIONS)
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("nvec", [(4, 7), (2, 3, 1, 8)])
def test_loss_kernel_matches_the_restatement(nvec, shared, opt):
    from ddrl4nav_b200 import kernels
    B, A = 777, sum(nvec)
    logits, g = _logits(B, A, A + 10 * shared + 100 * OPTIONS.index(opt))
    logits = logits.double() / 2
    mask = MD.random_mask(B, nvec, seed=A + 3) if opt in ("mask", "all") else None
    a = MD.sample(logits, mask, nvec, g)
    if mask is not None:
        eff = MD.effective_mask(mask, nvec)
        for r in [r for r in range(B) if not eff[r, :nvec[0]].all()][:4]:          # corrupt rows: a masked taken action
            a[r, 0] = float(torch.nonzero(~eff[r, :nvec[0]])[0])
    lp = MD.log_prob(logits, mask, a, nvec)
    old = (lp + 0.3 * torch.randn(B, generator=g, dtype=torch.float64)).float()
    v, ret = torch.randn(B, generator=g), torch.randn(B, generator=g)
    adv = torch.randn(B, generator=g) * (3.0 if opt == "dual_clip" else 1.0)
    kw, ref_kw = {}, {}
    hp_kw = dict(ppo_stats=True)
    if opt in ("VALUE_CLIP", "all"):
        ov = v + 0.5 * torch.randn(B, generator=g)
        hp_kw["value_clip"] = 0.2
        kw["old_values"], ref_kw["old_values"], ref_kw["value_clip"] = ov.to(DEV), ov, 0.2
    if opt in ("value_norm", "all"):
        vn = torch.tensor([0.3, 1.7, 1 / 1.7], dtype=torch.float32)
        kw["value_norm"], ref_kw["value_norm"] = vn.to(DEV), (0.3, 1.7)
    if opt in ("prox", "prox_is_clip", "all"):
        prox = (lp + 0.2 * torch.randn(B, generator=g, dtype=torch.float64)).float()
        kw["prox_logp"], ref_kw["prox"] = prox.to(DEV), prox
        if opt != "prox":
            kw["is_clip"] = ref_kw["is_clip"] = 1.3
    if opt == "dual_clip":
        hp_kw["dual_clip"] = 1.5
    hp = kernels.make_hparams(**hp_kw)
    hyper = R.PPOHyper()
    if opt == "dual_clip":
        hyper.dual_clip = 1.5
    d = lambda t: None if t is None else t.to(DEV)
    dl, dv, sums = kernels.ppo_loss_multi_categorical(d(logits.float()), nvec, d(a), d(old), d(adv), d(ret), d(v), hp, shared,
                                                      mask=d(mask), **kw)
    ref, rdl, rdv = MD.loss_and_grads(logits.float(), mask, a, nvec, old, adv, ret, v, hyper, shared, **ref_kw)
    s = sums.cpu().double().tolist()
    for i, k in enumerate(("actor", "v", "entropy", "ApproxKL")):
        assert s[i] == pytest.approx(ref[k], rel=1e-5, abs=1e-7), k
    assert s[4] == pytest.approx(ref["ClipFrac"], abs=2.0 / B)
    if "prox" in ref_kw:
        assert s[5] == pytest.approx(ref["BehaviourKL"], rel=2e-5)
    for got, want in ((dl, rdl), (dv, rdv)):
        got = got.cpu().double()
        assert torch.allclose(got, want, rtol=0, atol=1e-5 * float(want.abs().max())), float((got - want).abs().max())
    if mask is not None:
        assert (dl.cpu()[~MD.effective_mask(mask, nvec)] == 0).all()


def test_one_branch_loss_is_the_categorical_loss(deterministic):
    from ddrl4nav_b200 import kernels
    B, A = 1500, 28
    logits, g = _logits(B, A, 3)
    mask = M.random_mask(B, A, seed=4).to(DEV)
    a, lp, _ = kernels.categorical_head_m(logits.to(DEV), torch.rand(B, generator=g).to(DEV), mask)
    old, adv, ret, v = lp + 0.2, *(torch.randn(B, generator=g).to(DEV) for _ in range(3))
    hp = kernels.make_hparams(ppo_stats=True, value_clip=0.2)
    for shared in (True, False):
        kw = dict(mask=mask, old_values=v + 0.1, prox_logp=lp - 0.1, is_clip=1.5)
        want = kernels.ppo_loss_categorical_m(logits.to(DEV), a, old, adv, ret, v, hp, shared, **kw)
        got = kernels.ppo_loss_multi_categorical(logits.to(DEV), (A,), a[:, None], old, adv, ret, v, hp, shared, **kw)
        for w, x in zip(want, got):
            assert torch.equal(w, x)


# ---------------------------------------------------------------------------------------------------------- 4. whole net
def make(kind, seed=11, **hyper):
    from ddrl4nav_b200.runner import make_net
    spec = SPECS[kind] if kind in SPECS else R.SPECS[kind]
    if "ACTION_NVEC" in hyper:
        spec = R.NetSpec(spec.arch, spec.in_ch, sum(hyper["ACTION_NVEC"]), "categorical", spec.shared)
    net = make_net(kind, device=None, **hyper)
    net.load_state_dict(R.init_params(spec, seed=seed), strict=False)
    return net.to(DEV)


def batch(kind, B, net, seed=9, mask=None):
    """(states [+ mask], actions [B, K], old log-probs, advantages, values [1, B]) on the device; actions sampled by `net`, old
    log-probs its log-probs plus N(0, 0.15) noise."""
    g = torch.Generator().manual_seed(seed)
    nvec = net.actor.nvec
    states = [s.to(DEV) for s in R.synth_states(STATES_OF.get(kind, kind), B, seed=seed)]
    if net.action_mask:
        states.append((MD.random_mask(B, nvec, seed=seed + 1) if mask is None else mask).to(DEV).float())
    u = torch.rand(B, len(nvec), generator=g).to(DEV)
    a, lp, _ = net.act(states, draw=u)
    old = lp + 0.15 * torch.randn(B, generator=g).to(DEV)
    adv, ret = torch.randn(B, generator=g).to(DEV), torch.randn(B, generator=g).to(DEV)
    return states, a, old, adv, ret[None]


def experience(states, a, old, adv, values):
    from ddrl4nav_b200.data import Experience
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values)


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("kind,B", [("navimg_md", 6), ("navlaser_md", 5), ("navimg_md", 33)])
def test_net_gradients_match_the_oracle(kind, B, masked):
    net = make(kind, ACTION_MASK=masked)
    nvec = NVEC_OF[kind]
    states, a, old, adv, values = batch(kind, B, net)
    mask = states[-1].cpu() if masked else None
    net.backward_only(states, adv, a, old, values)
    grads = {n: g.detach().cpu().double() for n, g in net.named_grads().items()}
    enc_states = [s.cpu() for s in (states[:-1] if masked else states)]
    losses, raw = MD.net_grads(SPECS[kind], R.init_params(SPECS[kind], seed=11), enc_states, mask, a.cpu(), nvec, old.cpu(),
                               adv.cpu(), values[0].cpu())
    for n in raw:
        err = float((grads[n] - raw[n]).abs().max())
        assert err <= 2e-5 * float(raw[n].abs().max()), (n, err)
    sums = net._grads[net._P:net._P + 3].cpu().numpy()
    assert np.allclose(sums, [losses["ActorLoss"], losses["VLoss"], losses["EntLoss"]], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------- 5. learn()
@pytest.fixture
def pong_md(monkeypatch):
    """A `pong_md` kind: Pong's encoder with a MultiDiscrete actor."""
    from ddrl4nav_b200 import runner
    from ddrl4nav_b200.nn import AtariPreNet
    monkeypatch.setitem(runner._KINDS, "pong_md", (lambda: AtariPreNet(4, 512), "multi_categorical", (6,), False))
    monkeypatch.setitem(SPECS, "pong_md", R.SPECS["pong"])
    monkeypatch.setitem(STATES_OF, "pong_md", "pong")


@pytest.mark.parametrize("opts", [dict(), dict(MINI_BATCH_NUM=4, MINI_BATCH_SEED=3),
                                  dict(DECOUPLED_PPO=True, PPO_STATS=True, ACTION_MASK=True)])
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_one_branch_learns_the_categorical_bits(deterministic, pong_md, kind, opts):
    """nvec = (A,): the same actions, log-probs, probabilities, losses and parameters as the CategoricalActor."""
    B = 48
    A = R.SPECS[kind].act_dim
    cat = make(kind, TRAINING_ITER_TIME=3, **opts)
    md = make(kind + "_md", TRAINING_ITER_TIME=3, ACTION_NVEC=(A,), **opts)
    states = [s.to(DEV) for s in R.synth_states(kind, B, seed=5)]
    if opts.get("ACTION_MASK"):
        states.append(M.random_mask(B, A, seed=6).to(DEV).float())
    g = torch.Generator().manual_seed(7)
    u = torch.rand(B, generator=g).to(DEV)
    a, lp, v, pi = cat.act(states, draw=u, want_pi=True)
    a2, lp2, v2, pi2 = md.act(states, draw=u[:, None], want_pi=True)
    assert torch.equal(a, a2[:, 0]) and torch.equal(lp, lp2) and torch.equal(v, v2) and torch.equal(pi, pi2)
    old = lp + 0.15 * torch.randn(B, generator=g).to(DEV)
    adv, ret = torch.randn(B, generator=g).to(DEV), torch.randn(B, generator=g).to(DEV)
    keys = KEYS + (("ApproxKL", "ClipFrac", "BehaviourKL") if opts.get("PPO_STATS") else ())
    lc = [[l[k] for k in keys] for l, _, _ in cat.learn(experience(states, a, old, adv, ret[None]))]
    lm = [[l[k] for k in keys] for l, _, _ in md.learn(experience(states, a[:, None], old, adv, ret[None]))]
    assert lc == lm and torch.equal(cat._flat, md._flat)


@pytest.mark.parametrize("M_", [1, 4])
@pytest.mark.parametrize("kind", ["navimg_md", "navlaser_md"])
def test_learn_with_every_option(kind, M_):
    net = make(kind, ACTION_MASK=True, MINI_BATCH_NUM=M_, MINI_BATCH_SEED=1, NORM_ADV=True, VALUE_CLIP=0.2, PPO_STATS=True,
               TARGET_KL=10.0, NORM_OBS=True, NORM_VALUE=True, DECOUPLED_PPO=True, DECOUPLED_IS_CLIP=2.0, DUEL_PPO_CLIP=2.0)
    states, a, old, adv, values = batch(kind, 96, net)
    before = net._flat.clone()
    logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, values))]
    assert len(logs) == 10 * M_ and logs[0]["ApproxKL"] == 0.0                        # a fresh decoupled batch starts at r == 1
    assert all(np.isfinite([l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")]).all() for l in logs)
    assert not torch.equal(before, net._flat) and torch.isfinite(net._flat).all()
    a2, lp2, _ = net.act(states, draw=torch.rand(96, len(net.actor.nvec), device=DEV))
    eff = MD.effective_mask(states[-1].cpu(), net.actor.nvec)
    for i, (lo, hi) in enumerate(MD.slices(net.actor.nvec)):
        assert bool(eff[torch.arange(96), lo + a2[:, i].cpu().long()].all())
    assert torch.isfinite(lp2).all()


def test_extra_critics():
    from ddrl4nav_b200.nn import Critic
    net = make("navimg_md", TRAINING_ITER_TIME=2, VALUE_CLIP=0.2, DECOUPLED_PPO=True, MINI_BATCH_NUM=2)
    for _ in range(2):
        net.add_critic(Critic(device=DEV, last_input_dim=512).to(DEV))
    net.gail_critic = True
    states, a, old, adv, values = batch("navimg_md", 64, net)
    v3 = torch.cat([values, values * 0.5, values * 2], 0)
    logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, v3))]
    assert len(logs) == 4 and all(np.isfinite([l[k] for k in KEYS]).all() for l in logs)


def test_deterministic_mode_is_bit_reproducible(deterministic):
    def run():
        net = make("navlaser_md", TRAINING_ITER_TIME=3, PPO_STATS=True)
        states, a, old, adv, values = batch("navlaser_md", 70, net)
        logs = [[l[k] for k in KEYS] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        return logs, net._flat.clone()

    (l1, f1), (l2, f2) = run(), run()
    assert l1 == l2 and torch.equal(f1, f2)


@pytest.mark.parametrize("M_", [1, 4])
def test_graph_replay_equals_stream_launches(deterministic, monkeypatch, M_):
    """Two learn calls on the same tensors, the actions and the mask rewritten in place (same addresses) between them: the graphs
    read the new contents when they replay."""
    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make("navimg_md", ACTION_MASK=True, TRAINING_ITER_TIME=3, MINI_BATCH_NUM=M_, MINI_BATCH_SEED=2, PPO_STATS=True,
                   DECOUPLED_PPO=True)
        states, a, old, adv, values = batch("navimg_md", 40, net)
        keys = KEYS + ("ApproxKL", "ClipFrac")
        logs = [[l[k] for k in keys] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        states[-1].copy_(MD.random_mask(40, (4, 7), seed=77).to(DEV))
        g = torch.Generator().manual_seed(78)
        a.copy_(torch.stack([torch.randint(0, 4, (40,), generator=g), torch.randint(0, 7, (40,), generator=g)], 1).float().to(DEV))
        logs += [[l[k] for k in keys] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        return logs, net._flat.clone()

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])


# ---------------------------------------------------------------------------------------------------------- 6. engine checks
def test_engine_checks_the_branch_table():
    from ddrl4nav_b200 import _lib
    lib = _lib.load()
    arr = lambda v: (C.c_int32 * len(v))(*v)
    desc = _lib.NetDesc(_lib.ARCH["mlp"], 4, 11, _lib.DIST["multi_categorical"], 1, 16, _lib.GEMM_MODE["tc3"], 0)
    h = C.c_void_p()
    assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) == 0
    try:
        params = torch.zeros(lib.ddrl_net_num_params(h), device=DEV)
        assert lib.ddrl_net_bind(h, _lib.ptr(params), None, None, None) == 0
        assert lib.ddrl_net_forward(h, None, 1, 1, None, None, None, None, None, None) == -3     # branches not set: E_STATE
        assert lib.ddrl_net_set_action_branches(h, 2, arr([4, 8])) == -1                        # sum != act_dim
        assert lib.ddrl_net_set_action_branches(h, 2, arr([0, 11])) == -1
        assert lib.ddrl_net_set_action_branches(h, 9, arr([1] * 9)) == -1
        assert lib.ddrl_net_set_action_branches(h, 2, arr([4, 7])) == 0
        assert lib.ddrl_net_set_action_mask(h, 1) == 0
        assert lib.ddrl_net_forward(h, None, 1, 1, None, None, None, None, None, None) == -1     # now it checks the observations
    finally:
        lib.ddrl_net_destroy(h)
    desc.dist = _lib.DIST["categorical"]
    assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) == 0
    assert lib.ddrl_net_set_action_branches(h, 2, arr([4, 7])) == -1                            # not a MultiDiscrete net
    lib.ddrl_net_destroy(h)
    desc.dist, desc.act_dim = _lib.DIST["multi_categorical"], 65
    assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) == -4
    net = make("navimg_md")
    batch("navimg_md", 4, net)
    assert lib.ddrl_net_set_action_branches(net._h, 2, arr([4, 7])) == -3                       # after a pass: E_STATE


# ---------------------------------------------------------------------------------------------------------- 7. Forward module
def test_forward_module_replies_and_weight_blob():
    from oracle.ref_shim import _FakeRedis
    from ddrl4nav_b200.runner import make_net
    from ddrl4nav_b200.server import ForwardModule, encode_forward_replies
    net = make("navlaser_md")
    B_env, n_env = 5, 7
    B = B_env * n_env
    states = [s.numpy() for s in R.synth_states("navlaser", B, seed=4)]
    payload = b"".join(R.easybytes_encode_forward_states("10.1.2.3", 100 + j, [s[j * B_env:(j + 1) * B_env] for s in states])
                       for j in range(n_env))
    draw = torch.rand(B, 2, generator=torch.Generator().manual_seed(6)).to(DEV)
    a, lp, v = net.act([torch.from_numpy(s).to(DEV) for s in states], draw=draw)
    assert a.shape == (B, 2)
    want = [a.cpu().numpy(), lp.cpu().numpy(), v.cpu().numpy()]
    fm = ForwardModule(net, device=DEV)
    got = fm.step(states, draw=draw)
    assert all(np.array_equal(x, y.reshape(x.shape)) for x, y in zip(got, want))
    _, replies = fm.step_bytes_replies(payload, B_env, draw=draw)
    assert replies == encode_forward_replies(want, [B_env] * n_env)
    assert R.easybytes_decode_data(replies[0])[0].shape == (B_env, 2)                           # act_cols = K
    # a predictor built with the same nvec gets the same bits from the weight blob
    mid = _FakeRedis()
    net.nn2redis(mid.pipeline(), "upd")
    pred = make_net("navlaser_md", device=DEV)
    pred.updatenn_by_redis(mid, net.model_key)
    for x, y in zip(net.act([torch.from_numpy(s).to(DEV) for s in states], draw=draw),
                    pred.act([torch.from_numpy(s).to(DEV) for s in states], draw=draw)):
        assert torch.equal(x, y)
    # forward(): a MultiCategorical, and the per-branch softmax in play mode
    (pi, log_p), _ = net.forward([torch.from_numpy(s).to(DEV) for s in states], act=a)
    assert torch.allclose(log_p, lp, rtol=1e-4, atol=1e-4) and pi.sample().shape == (B, 2)
    (p, _), _ = net.forward([torch.from_numpy(s).to(DEV) for s in states], play_mode=True)
    assert p.shape == (B, 14) and torch.allclose(p[:, :5].sum(-1), torch.ones(B, device=DEV), atol=1e-5)


def test_forward_thread_one_tick():
    from oracle.ref_shim import _FakeRedis
    from ddrl4nav_b200.server import ForwardThread
    from test_threads import _configs, _Logger
    B_env, n_env = 3, 2
    net = make("navimg_md")
    cfgs = _configs("navimg", B_env, "fwd-md")
    mid = _FakeRedis("fwd-md", 2)
    net.conn, net.model_key = mid, "tMODEL"
    net.nn2redis(mid.pipeline(), "tupd")
    th = ForwardThread(net, 0, _Logger(), None, types.SimpleNamespace(value=b"0"), cfgs)
    states = [s.numpy() for s in R.synth_states("navimg", B_env * n_env, seed=3)]
    payload = b"".join(R.easybytes_encode_forward_states("10.0.0.7", pid, [s[j * B_env:(j + 1) * B_env] for s in states])
                       for j, pid in enumerate((4, 9)))
    draw = torch.rand(B_env * n_env, 2, generator=torch.Generator().manual_seed(5)).to(DEV)
    assert th.tick(payload, draw=draw) == n_env
    wa, wlp, wv = net.act([torch.from_numpy(s).to(DEV) for s in states], draw=draw)
    pre = _FakeRedis("fwd-md", 1)
    for j, pid in enumerate((4, 9)):
        item = pre.blpop("tact10.0.0.7_%d" % pid)
        assert item is not None
        a, lp, v = R.easybytes_decode_data(item[1])
        sl = slice(j * B_env, (j + 1) * B_env)
        assert a.shape == (B_env, 2) and np.array_equal(a, wa.cpu().numpy()[sl]) and np.array_equal(lp, wlp.cpu().numpy()[sl])
        assert np.array_equal(v.reshape(-1), wv.cpu().numpy().reshape(-1)[sl])


# ---------------------------------------------------------------------------------------------------------- 8. two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, q):
    import torch.distributed as tdist
    from ddrl4nav_b200 import kernels
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    kernels.set_deterministic(True)
    tdist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world, device_id=dev)
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net
    kind, B = "navimg_md", 81
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, PPO_STATS=True, DECOUPLED_PPO=True, ACTION_MASK=True)
    net.load_state_dict(R.init_params(SPECS[kind], seed=11))
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    states, a, old, adv, values = batch(kind, B, net)
    lo, hi = (0, 41) if rank == 0 else (41, 81)
    exp = Experience(states=[s[lo:hi].to(dev) for s in states], advs=adv[lo:hi].to(dev), actions=a[lo:hi].to(dev),
                     old_logps=old[lo:hi].to(dev), values=values[:, lo:hi].to(dev))
    logs = [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")] for l, _, _ in net.learn(exp)]
    q.put((rank, logs, net._flat.cpu().numpy()))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_replicas_are_identical():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, logs, flat = q.get(timeout=600)
        res[r] = (logs, flat)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (l0, f0), (l1, f1) = res[0], res[1]
    assert l0 == l1 and np.array_equal(f0, f1)
    assert all(np.isfinite(l).all() for l in l0)
