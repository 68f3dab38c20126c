"""Beta actor on the GPU: the inverse-CDF sampler against scipy, log-prob bit equality of the head, pre-pass and loss kernels,
the fused loss against the float64 restatement (tests/beta_ref.py) with every PPO option, whole-net gradients against the
oracle, learn() with the options, the Forward module and the weight blob, and two-GPU parity."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import beta_ref as BR
from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")


@pytest.fixture
def deterministic():
    from ddrl4nav_b200 import kernels
    was = kernels.set_deterministic(True)
    yield
    kernels.set_deterministic(was)


def z_of(conc):
    """Head value whose 1 + softplus is `conc` (1 -> -100: softplus underflows to 0)."""
    c = torch.as_tensor(conc, dtype=torch.float64)
    return torch.where(c <= 1, torch.full_like(c, -100.0), torch.where(c - 1 > 20, c - 1, torch.log(torch.expm1(c - 1)))).float()


def bounds(A, lo=-2.0, hi=3.0):
    return torch.full((A,), lo), torch.full((A,), hi)


# ---------------------------------------------------------------------------------------------------------- 1. sampler
def test_sampler_matches_scipy_on_the_grid():
    from ddrl4nav_b200 import kernels
    grid = [1.0, 1.001, 2.0, 10.0, 100.0, 1e3, 1e4]
    us = [1e-7, 1e-4, 0.01, 0.3, 0.5, 0.7, 0.99, 1 - 1e-4, 1 - 6e-8]
    al, be, u = (torch.tensor(t).reshape(-1, 1) for t in np.meshgrid(grid, grid, us, indexing="ij"))
    head = torch.cat([z_of(al), z_of(be)], 1)
    low, high = bounds(1)
    a, lp, conc = kernels.beta_head(head.to(DEV), low.to(DEV), high.to(DEV), u.float().to(DEV))
    ref = BR.sample(head, low, high, u.float())
    err = (a.cpu().double() - ref.double()).abs()
    assert float(err.max()) <= 1e-6 * 5.0, (float(err.max()), int(err.argmax()))
    al32, be32 = BR.concentrations(head)
    assert torch.allclose(conc.cpu(), torch.cat([al32, be32], 1), rtol=2e-7, atol=0)
    assert torch.allclose(lp.cpu().double(), BR.log_prob(head, low, high, a.cpu()), rtol=1e-5, atol=1e-4)


def test_sampler_terminates_on_huge_and_non_finite_concentrations():
    """Concentrations of 1e6 give an action inside the bounds; a NaN or +inf head value gives a NaN action and log-prob (the
    documented result), and a NaN draw does too."""
    from ddrl4nav_b200 import kernels
    low, high = bounds(1)
    z = torch.tensor([[1e6, 1e6], [1e6, -100.0], [-100.0, 1e6], [float("nan"), 0.0], [float("inf"), 0.0], [0.0, 0.0]])
    u = torch.tensor([[0.5], [1e-7], [1 - 6e-8], [0.5], [0.5], [float("nan")]])
    a, lp, _ = kernels.beta_head(z.to(DEV), low.to(DEV), high.to(DEV), u.to(DEV))
    torch.cuda.synchronize()
    a, lp = a.cpu(), lp.cpu()
    assert bool(((a[:3] >= low) & (a[:3] <= high)).all())
    assert abs(float(a[0]) - 0.5) < 1e-2                      # Beta(1e6, 1e6) sits at the centre of [-2, 3]
    assert torch.isnan(a[3:]).all() and torch.isnan(lp[3:]).all()


def test_play_mode_returns_the_mean():
    from ddrl4nav_b200 import kernels
    g = torch.Generator().manual_seed(0)
    head = 3 * torch.randn(300, 6, generator=g)
    low, high = torch.tensor([-1.0, 0.0, 0.5]), torch.tensor([1.0, 2.0, 0.75])
    a, lp, conc = kernels.beta_head(head.to(DEV), low.to(DEV), high.to(DEV), None)
    assert torch.allclose(a.cpu(), BR.mean_action(head, low, high), rtol=1e-6, atol=1e-7)
    assert (lp == 0).all()


# ---------------------------------------------------------------------------------------------------------- 2. log-prob bits
def _head_batch(B, A, seed):
    g = torch.Generator().manual_seed(seed)
    head = 1.5 * torch.randn(B, 2 * A, generator=g)
    low = -1.0 - torch.rand(A, generator=g)
    high = 0.5 + 2 * torch.rand(A, generator=g)
    u = torch.rand(B, A, generator=g)
    a = BR.sample(head, low, high, u)
    v, ret, adv = (torch.randn(B, generator=g) for _ in range(3))
    return head, low, high, u, a, v, ret, adv, g


@pytest.mark.parametrize("A", [1, 2, 8])
def test_act_prepass_and_loss_log_probs_are_equal_bits(A):
    """The head kernel's log-prob of the action it emitted, ddrl_logp_actions_beta's, and the loss kernel's (ppo_clip 0 with
    old = prox = that log-prob counts any r != 1 in ClipFrac) are the same bits."""
    from ddrl4nav_b200 import kernels
    head, low, high, u, _, v, ret, adv, _ = _head_batch(1000, A, seed=A)
    d = lambda t: t.to(DEV)
    a, lp_act, _ = kernels.beta_head(d(head), d(low), d(high), d(u))
    lp_pre = kernels.logp_actions_beta(d(head), d(low), d(high), a)
    assert torch.equal(lp_act, lp_pre)
    hp = kernels.make_hparams(ppo_clip=0.0, ppo_stats=True)
    _, _, sums = kernels.ppo_loss_beta(d(head), d(low), d(high), a, lp_act, d(adv), d(ret), d(v), hp, True)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0
    _, _, sums = kernels.ppo_loss_beta(d(head), d(low), d(high), a, lp_act - 0.3, d(adv), d(ret), d(v), hp, True, prox_logp=lp_act)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0
    assert torch.allclose(lp_act.cpu().double(), BR.log_prob(head, low, high, a.cpu()), rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------- 3. loss kernel
OPTIONS = ["none", "VALUE_CLIP", "value_norm", "prox", "prox_is_clip", "all"]


@pytest.mark.parametrize("opt", OPTIONS)
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("A", [2, 5])
def test_loss_kernel_matches_the_restatement(A, shared, opt):
    from ddrl4nav_b200 import kernels
    B = 777
    head, low, high, _, a, v, ret, adv, g = _head_batch(B, A, seed=A + 10 * shared + 100 * OPTIONS.index(opt))
    lp = BR.log_prob(head, low, high, a)
    old = (lp + 0.3 * torch.randn(B, generator=g, dtype=torch.float64)).float()
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
    hp = kernels.make_hparams(**hp_kw)
    d = lambda t: t.to(DEV)
    dh, dv, sums = kernels.ppo_loss_beta(d(head), d(low), d(high), d(a), d(old), d(adv), d(ret), d(v), hp, shared, **kw)
    ref, rdh, rdv = BR.loss_and_grads(head, low, high, a, old, adv, ret, v, R.PPOHyper(), shared, **ref_kw)
    s = sums.cpu().double().tolist()
    for i, k in enumerate(("actor", "v", "entropy", "ApproxKL")):
        assert s[i] == pytest.approx(ref[k], rel=1e-5, abs=1e-7), k
    assert s[4] == pytest.approx(ref["ClipFrac"], abs=2.0 / B)
    if "prox" in ref_kw:
        assert s[5] == pytest.approx(ref["BehaviourKL"], rel=2e-5)
    for got, want in ((dh, rdh), (dv, rdv)):
        got = got.cpu().double()
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-5 * float(want.abs().max())), float((got - want).abs().max())


# ---------------------------------------------------------------------------------------------------------- 4. whole net
def make(kind, seed=11, **hyper):
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None, **hyper)
    net.load_state_dict(R.init_params(BR.SPECS[kind], seed=seed), strict=False)     # option buffers keep their initial values
    return net.to(DEV)


def batch(kind, B, seed=9, net=None):
    """(states, actions, old log-probs, advantages, values [1, B]) on the device; actions sampled by `net` (or the seed-11
    net), old log-probs are its log-probs plus N(0, 0.15) noise."""
    g = torch.Generator().manual_seed(seed)
    states = [s.to(DEV) for s in R.synth_states(BR.STATES_OF[kind], B, seed=seed)]
    net = net or make(kind)
    u = torch.rand(B, 2, generator=g).to(DEV)
    a, lp, _ = net.act(states, draw=u)
    old = lp + 0.15 * torch.randn(B, generator=g).to(DEV)
    adv, ret = torch.randn(B, generator=g).to(DEV), torch.randn(B, generator=g).to(DEV)
    return states, a, old, adv, ret[None]


def experience(states, a, old, adv, values):
    from ddrl4nav_b200.data import Experience
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values)


@pytest.mark.parametrize("kind,B", [("navlaser_beta", 4), ("navimg_beta", 6), ("navlaser_beta", 33)])
def test_net_gradients_match_the_oracle(kind, B):
    net = make(kind, ACTION_LOW=[-0.5, 0.0], ACTION_HIGH=[1.0, 2.0])
    states, a, old, adv, values = batch(kind, B, net=net)
    net.backward_only(states, adv, a, old, values)
    grads = {n: g.detach().cpu().double() for n, g in net.named_grads().items()}
    low, high = torch.tensor([-0.5, 0.0]), torch.tensor([1.0, 2.0])
    losses, raw = BR.net_grads(kind, R.init_params(BR.SPECS[kind], seed=11), [s.cpu() for s in states], a.cpu(), old.cpu(),
                               adv.cpu(), values[0].cpu(), low, high)
    worst = max(float((grads[n] - raw[n]).abs().max()) / max(float(raw[n].abs().max()), 1e-30) for n in raw)
    assert worst < 2e-5, worst
    sums = net._grads[net._P:net._P + 3].cpu().numpy()
    assert np.allclose(sums, [losses["ActorLoss"], losses["VLoss"], losses["EntLoss"]], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------- 5. learn()
@pytest.mark.parametrize("M", [1, 4])
@pytest.mark.parametrize("kind", ["navlaser_beta", "navimg_beta"])
def test_learn_with_the_ppo_options(kind, M):
    net = make(kind, MINI_BATCH_NUM=M, MINI_BATCH_SEED=1, NORM_ADV=True, VALUE_CLIP=0.2, PPO_STATS=True)
    data = batch(kind, 96)
    net._ensure_engine()
    before = net._flat.clone()
    logs = [l for l, _, _ in net.learn(experience(*data))]
    assert len(logs) == 10 * M
    assert all(np.isfinite([l[k] for k in KEYS + ("ApproxKL", "ClipFrac")]).all() for l in logs)
    assert not torch.equal(before, net._flat) and torch.isfinite(net._flat).all()


@pytest.mark.parametrize("kind", ["navlaser_beta", "navimg_beta"])
def test_decoupled_ppo(deterministic, kind):
    """A fresh batch starts at r == 1 exactly; on on-policy data the decoupled learner is the option-off learner bit for bit."""
    states, a, old, adv, values = batch(kind, 40)
    net = make(kind, DECOUPLED_PPO=True, PPO_STATS=True, TRAINING_ITER_TIME=3)
    logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, values))]
    assert logs[0]["ApproxKL"] == 0.0 and logs[0]["ClipFrac"] == 0.0 and logs[1]["ApproxKL"] > 0.0
    from ddrl4nav_b200 import kernels
    A = make(kind, DECOUPLED_PPO=True, TRAINING_ITER_TIME=2)
    B = make(kind, TRAINING_ITER_TIME=2)
    on_policy = kernels.net_log_prob(B, states, a).clone()
    for (la, _, _), (lb, _, _) in zip(A.learn(experience(states, a, on_policy, adv, values)),
                                      B.learn(experience(states, a, on_policy, adv, values))):
        assert [la[k] for k in KEYS] == [lb[k] for k in KEYS]
        assert torch.equal(A._flat, B._flat)


@pytest.mark.parametrize("opt", ["NORM_OBS", "NORM_VALUE"])
def test_norm_obs_and_norm_value_run(opt):
    net = make("navlaser_beta", TRAINING_ITER_TIME=3, **{opt: True})
    data = batch("navlaser_beta", 64)
    logs = [l for l, _, _ in net.learn(experience(*data))]
    assert all(np.isfinite([l[k] for k in KEYS]).all() for l in logs)
    a, lp, v = net.act(data[0])
    assert torch.isfinite(a).all() and torch.isfinite(lp).all() and torch.isfinite(v).all()


def test_deterministic_mode_is_bit_reproducible(deterministic):
    data = batch("navimg_beta", 200)
    runs = []
    for _ in range(2):
        net = make("navimg_beta", TRAINING_ITER_TIME=3, PPO_STATS=True)
        logs = [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac")] for l, _, _ in net.learn(experience(*data))]
        runs.append((logs, net._flat.clone()))
    assert runs[0][0] == runs[1][0] and torch.equal(runs[0][1], runs[1][1])


@pytest.mark.parametrize("M", [1, 4])
def test_graph_replay_equals_stream_launches(deterministic, monkeypatch, M):
    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make("navlaser_beta", TRAINING_ITER_TIME=3, MINI_BATCH_NUM=M, MINI_BATCH_SEED=2, PPO_STATS=True, DECOUPLED_PPO=True)
        logs = []
        for call in range(2):
            logs += [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")]
                     for l, _, _ in net.learn(experience(*batch("navlaser_beta", 40, seed=call)))]
        return logs, net._flat.clone()

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])


def test_bounds_are_required_and_validated_by_the_engine():
    import ctypes as C
    from ddrl4nav_b200 import _lib
    net = make("navlaser_beta")
    net._ensure_engine()
    lib = _lib.load()
    f2 = lambda *v: (C.c_float * 2)(*v)
    assert lib.ddrl_net_set_action_bounds(net._h, f2(0.0, 0.0), f2(1.0, 0.0)) != 0                  # low == high
    assert lib.ddrl_net_set_action_bounds(net._h, f2(0.0, float("nan")), f2(1.0, 1.0)) != 0
    assert lib.ddrl_net_set_action_bounds(net._h, f2(-1.0, -1.0), f2(1.0, 1.0)) == 0
    from ddrl4nav_b200._lib import NetDesc
    desc = NetDesc(_lib.ARCH["nav1d"], 3, 2, _lib.DIST["beta"], 0, 512, _lib.GEMM_MODE["tc3"], 0)
    h = C.c_void_p()
    assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) == 0
    try:
        flat = torch.zeros(lib.ddrl_net_num_params(h), device=DEV)
        assert lib.ddrl_net_bind(h, _lib.ptr(flat), None, None, None) == 0
        states = [s.to(DEV) for s in R.synth_states("navlaser", 2)]
        arr = (C.c_void_p * 3)(*[s.data_ptr() for s in states])
        out = torch.empty(8, device=DEV)
        rc = lib.ddrl_net_forward(h, arr, 3, 2, None, _lib.ptr(out), _lib.ptr(out[4:]), _lib.ptr(out[6:]), None, None)
        assert rc == -3                                             # DDRL_E_STATE: no bounds yet
    finally:
        lib.ddrl_net_destroy(h)
    desc.act_dim = 9
    assert lib.ddrl_net_create(C.byref(desc), C.byref(h)) != 0      # A <= 8


# ---------------------------------------------------------------------------------------------------------- 6. Forward module
def test_forward_module_replies_and_weight_blob():
    from oracle.ref_shim import _FakeRedis
    from ddrl4nav_b200.server import ForwardModule, encode_forward_replies
    lo, hi = [0.0, -0.6], [0.8, 0.6]
    net = make("navlaser_beta", ACTION_LOW=lo, ACTION_HIGH=hi)
    B_env, n_env = 5, 7
    states = [s.numpy() for s in R.synth_states("navlaser", B_env * n_env, seed=4)]
    payload = b"".join(R.easybytes_encode_forward_states("10.1.2.3", 100 + j, [s[j * B_env:(j + 1) * B_env] for s in states])
                       for j in range(n_env))
    draw = torch.rand(B_env * n_env, 2, generator=torch.Generator().manual_seed(6)).to(DEV)
    fm = ForwardModule(net, device=DEV)
    _, got = fm.step_bytes_replies(payload, B_env, draw=draw)
    a, lp, v = net.act([torch.from_numpy(s).to(DEV) for s in states], draw=draw)
    assert bool(((a >= torch.tensor(lo, device=DEV)) & (a <= torch.tensor(hi, device=DEV))).all())
    want = encode_forward_replies([a.cpu().numpy(), lp.cpu().numpy(), v.cpu().numpy()], [B_env] * n_env)
    assert got == want
    # nn2redis -> updatenn_by_redis into a predictor built with the same bounds: the same bits
    mid = _FakeRedis()
    net.nn2redis(mid.pipeline(), "upd")
    from ddrl4nav_b200.runner import make_net
    pred = make_net("navlaser_beta", device=DEV, ACTION_LOW=lo, ACTION_HIGH=hi)
    pred.updatenn_by_redis(mid, net.model_key)
    a2, lp2, v2 = pred.act([torch.from_numpy(s).to(DEV) for s in states], draw=draw)
    assert torch.equal(a, a2) and torch.equal(lp, lp2) and torch.equal(v, v2)
    # forward(): the Beta mapped onto the bounds, and the mean in play mode
    (pi, log_p), _ = net.forward([torch.from_numpy(s).to(DEV) for s in states], act=a)
    assert torch.allclose(log_p.double(), lp.double(), rtol=1e-4, atol=1e-4)
    (mean, _), _ = net.forward([torch.from_numpy(s).to(DEV) for s in states], play_mode=True)
    low, high = torch.tensor(lo, device=DEV), torch.tensor(hi, device=DEV)
    assert torch.allclose(mean, low + (high - low) * pi.base_dist.mean, rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------- 7. two ranks
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
    kind, B = "navlaser_beta", 81
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, PPO_STATS=True, DECOUPLED_PPO=True)
    net.load_state_dict(R.init_params(BR.SPECS[kind], seed=11))
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    states, a, old, adv, values = batch(kind, B)
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
