"""Decoupled PPO (DECOUPLED_PPO, DECOUPLED_IS_CLIP) on the GPU: with the option off the learner is the default path, launch for
launch and bit for bit; the _dc loss kernels against the float64 restatement (tests/decoupled_ref.py) and the pre-pass
log-probs against the loss kernels' own; r == 1 at the first step of a call; bit-identical equivalence with an option-off
learner on on-policy data and fp32-close equivalence on a stale batch with the weight moved into the advantages; graph
replay; the TARGET_KL stop; micro-batched rows; a full-size Pong run; and two-GPU parity."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import decoupled_ref as D
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


def make(kind, seed=11, **hyper):
    """A net of `kind` with fixed initial weights (the same for every hyper-parameter set)."""
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None, **hyper)
    if kind in R.SPECS:
        net.load_state_dict(R.init_params(R.SPECS[kind], seed=seed), strict=False)
    else:
        torch.manual_seed(seed)
        net.load_state_dict(make_net(kind, device=None).state_dict(), strict=False)
    return net.to(DEV)


def batch(kind, B, seed=9):
    """(states, actions, old log-probs, advantages, values [1, B]) on the device; old log-probs are the initial net's plus
    N(0, 0.15) noise: a stale behaviour policy."""
    g = torch.Generator().manual_seed(seed)
    if kind == "mlp":
        states = [torch.randn(B, 4, generator=g)]
        a = torch.randint(0, 2, (B,), generator=g).float()
        old = -0.69 + 0.15 * torch.randn(B, generator=g)
        adv = torch.randn(B, generator=g)
    else:
        spec = R.SPECS[kind]
        states = R.synth_states(kind, B, seed=seed)
        a, old, adv, _ = R.synth_learn_batch(spec, R.init_params(spec, seed=11), states, seed=seed)
    ret = torch.randn(B, generator=g)
    return [s.to(DEV) for s in states], a.to(DEV), old.to(DEV), adv.to(DEV), ret.to(DEV)[None]


def experience(states, a, old, adv, values):
    from ddrl4nav_b200.data import Experience
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values)


def prox_of(net, states, a):
    from ddrl4nav_b200 import kernels
    return kernels.net_log_prob(net, states, a).clone()


# ---------------------------------------------------------------------------------------------------------- 1. off = default
@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("kind", ["pong", "mlp"])
def test_option_off_is_the_default_path(deterministic, kind, M):
    from ddrl4nav_b200 import kernels
    data = batch(kind, 40)
    out = []
    for hyper in ({}, dict(DECOUPLED_PPO=False)):
        net = make(kind, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=3, PPO_STATS=True, **hyper)
        kernels.launch_count_reset()
        logs = [l for l, _, _ in net.learn(experience(*data))]
        n = kernels.launch_count()
        out.append(([[l[k] for k in KEYS + ("ApproxKL", "ClipFrac")] for l in logs], net._flat.clone(), n, net.model_bytes(),
                    sorted(logs[0])))
    assert out[0][0] == out[1][0] and torch.equal(out[0][1], out[1][1])
    assert out[0][2] == out[1][2] and out[0][3] == out[1][3]
    assert out[0][4] == out[1][4] and "BehaviourKL" not in out[1][4]


# ---------------------------------------------------------------------------------------------------------- 2. kernels
def _head_batch(dist, B, A, seed):
    g = torch.Generator().manual_seed(seed)
    head = 1.5 * torch.randn(B, A, generator=g)
    if dist == "categorical":
        a = torch.randint(0, A, (B,), generator=g).float()
    else:
        a = head + torch.randn(B, A, generator=g)
    log_std = -0.5 + 0.3 * torch.randn(A, generator=g)
    v = torch.randn(B, generator=g)
    ret = torch.randn(B, generator=g)
    adv = torch.randn(B, generator=g)
    return head, a, log_std, v, ret, adv, g


@pytest.mark.parametrize("is_clip", [None, 1.3])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("dist,A", [("categorical", 2), ("categorical", 7), ("categorical", 64), ("gaussian", 1),
                                    ("gaussian", 3), ("gaussian", 8)])
def test_dc_loss_kernels_match_the_restatement(dist, A, shared, is_clip):
    from ddrl4nav_b200 import kernels
    B = 777
    head, a, log_std, v, ret, adv, g = _head_batch(dist, B, A, seed=A + 10 * shared)
    hp = kernels.make_hparams(ppo_stats=True)
    if dist == "categorical":
        lp = R.categorical_log_prob(torch.softmax(head.double(), -1), a)
    else:
        lp = R.gaussian_log_prob(head.double(), log_std.double(), a.double())
    prox = (lp + 0.2 * torch.randn(B, generator=g, dtype=torch.float64)).float()
    old = (prox.double() + 0.5 * torch.randn(B, generator=g, dtype=torch.float64)).float()
    d = lambda t: t.to(DEV)
    if dist == "categorical":
        dh, dv, sums = kernels.ppo_loss_categorical_dc(d(head), d(a), d(old), d(adv), d(ret), d(v), hp, shared, d(prox), is_clip)
        dls = None
    else:
        dh, dv, dls, sums = kernels.ppo_loss_gaussian_dc(d(head), d(log_std), d(a), d(old), d(adv), d(ret), d(v), hp, shared,
                                                         d(prox), is_clip)
    ref, rdh, rdv, rdls = D.loss_and_grads(dist, head, a, old, prox, adv, ret, v, R.PPOHyper(), shared, is_clip,
                                           log_std if dist == "gaussian" else None)
    s = sums.cpu().double().tolist()
    for i, k in enumerate(("actor", "v", "entropy", "ApproxKL")):
        assert s[i] == pytest.approx(ref[k], rel=2e-5, abs=1e-6), k
    assert s[4] == pytest.approx(ref["ClipFrac"], abs=2.0 / B)
    assert s[5] == pytest.approx(ref["BehaviourKL"], rel=2e-5)
    for got, want in ((dh, rdh), (dv, rdv)) + (((dls, rdls),) if dls is not None else ()):
        got = got.cpu().double()
        assert torch.allclose(got, want, rtol=0, atol=2e-5 * float(want.abs().max())), float((got - want).abs().max())


@pytest.mark.parametrize("dist,A", [("categorical", 2), ("categorical", 64), ("gaussian", 1), ("gaussian", 8)])
def test_prepass_log_probs_are_the_loss_kernels_own(dist, A):
    """prox = logp_actions(head): the loss kernel then sees r == 1 on every row, exactly (ppo_clip 0 counts any r != 1)."""
    from ddrl4nav_b200 import kernels
    B = 1000
    head, a, log_std, v, ret, adv, _ = _head_batch(dist, B, A, seed=3)
    d = lambda t: t.to(DEV)
    hp = kernels.make_hparams(ppo_clip=0.0, ppo_stats=True)
    if dist == "categorical":
        lp = kernels.logp_actions_categorical(d(head), d(a))
        want = R.categorical_log_prob(torch.softmax(head.double(), -1), a)
        _, _, sums = kernels.ppo_loss_categorical_dc(d(head), d(a), lp - 0.3, d(adv), d(ret), d(v), hp, True, lp)
    else:
        lp = kernels.logp_actions_gaussian(d(head), d(log_std), d(a))
        want = R.gaussian_log_prob(head.double(), log_std.double(), a.double())
        _, _, _, sums = kernels.ppo_loss_gaussian_dc(d(head), d(log_std), d(a), lp - 0.3, d(adv), d(ret), d(v), hp, True, lp)
    assert torch.allclose(lp.cpu().double(), want, rtol=1e-5, atol=1e-5)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0


# ---------------------------------------------------------------------------------------------------------- 3. step 1
def test_first_step_has_unit_ratio_exactly_within_one_micro_batch():
    states, a, old, adv, values = batch("pong", 40)
    net = make("pong", DECOUPLED_PPO=True, PPO_STATS=True, TRAINING_ITER_TIME=3)
    for call in range(2):
        logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        assert logs[0]["ApproxKL"] == 0.0 and logs[0]["ClipFrac"] == 0.0, call
        assert logs[1]["ApproxKL"] > 0.0
        assert logs[0]["BehaviourKL"] == pytest.approx(D.behaviour_kl(net.last_prox_logps.cpu(), old.cpu()), rel=1e-4, abs=1e-7)
        assert all(l["BehaviourKL"] == logs[0]["BehaviourKL"] for l in logs)     # the proximal policy holds for the call


@pytest.mark.parametrize("M,micro", [(1, "16"), (4, None)])
def test_first_step_ratio_with_micro_batches_or_minibatches(monkeypatch, M, micro):
    if micro:
        monkeypatch.setenv("DDRL_MICRO_BATCH", micro)
    states, a, old, adv, values = batch("navimg", 40)
    net = make("navimg", DECOUPLED_PPO=True, PPO_STATS=True, TRAINING_ITER_TIME=1, MINI_BATCH_NUM=M, MINI_BATCH_SEED=1)
    logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, values))]
    assert abs(logs[0]["ApproxKL"]) <= 1e-6 and logs[0]["ClipFrac"] == 0.0
    assert logs[0]["BehaviourKL"] > 1e-3


# ---------------------------------------------------------------------------------------------------------- 4. on-policy
@pytest.mark.parametrize("opt", ["VALUE_CLIP", "NORM_ADV", "NORM_VALUE"])
@pytest.mark.parametrize("M", [1, 4])
@pytest.mark.parametrize("kind", ["pong", "navlaser", "navimg", "mlp"])
def test_on_policy_batch_equals_the_option_off_learner(deterministic, kind, M, opt):
    """old_logps := the proximal log-probs: w == 1 and r is the plain ratio, so losses, gradients and parameters are the
    option-off learner's, bit for bit.  (Both nets run the pre-pass once per call, so their workspaces match.)"""
    hyper = dict(TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=4, **{opt: 0.5 if opt == "VALUE_CLIP" else True})
    A = make(kind, DECOUPLED_PPO=True, DECOUPLED_IS_CLIP=2.0, **hyper)
    B = make(kind, **hyper)
    for call in range(2):
        states, a, _, adv, values = batch(kind, 40, seed=20 + call)
        on_policy = prox_of(B, states, a)
        n = 0
        for (la, _, _), (lb, _, _) in zip(A.learn(experience(states, a, on_policy, adv, values)),
                                          B.learn(experience(states, a, on_policy, adv, values))):
            n += 1
            assert [la[k] for k in KEYS] == [lb[k] for k in KEYS], (call, n)
            assert torch.equal(A.flat_grads(), B.flat_grads()), (call, n)
            assert torch.equal(A._flat, B._flat), (call, n)
        assert n == 2 * M
        assert torch.equal(A.last_prox_logps, on_policy)


# ---------------------------------------------------------------------------------------------------------- 5. stale batch
@pytest.mark.parametrize("kind", ["pong", "navlaser", "mlp"])
def test_stale_batch_equals_weighted_advantages(kind):
    """A batch sampled at theta_0, a learner at theta_1: the decoupled learner on (old_logps, advs) is an option-off learner on
    (prox_logps, w * advs) up to fp32 rounding of w * term against term(w * A)."""
    states, a, _, adv, values = batch(kind, 64)
    src = make(kind, TRAINING_ITER_TIME=4)
    old = prox_of(src, states, a)                          # behaviour policy theta_0
    list(src.learn(experience(states, a, old - 0.1, adv, values)))      # theta_0 -> theta_1
    A = make(kind, DECOUPLED_PPO=True, PPO_STATS=True, TRAINING_ITER_TIME=1)
    B = make(kind, PPO_STATS=True, TRAINING_ITER_TIME=1)
    for net in (A, B):
        net.load_state_dict(src.state_dict())
    prox = prox_of(B, states, a)
    w = torch.exp(prox - old)
    (la, _, _), = A.learn(experience(states, a, old, adv, values))
    (lb, _, _), = B.learn(experience(states, a, prox, w * adv, values))
    for k in KEYS + ("ApproxKL", "ClipFrac"):
        assert la[k] == pytest.approx(lb[k], rel=1e-5, abs=1e-7), k
    # fp32 (rho - 1) - log rho cancels near rho = 1: about 1e-8 absolute per row
    assert la["BehaviourKL"] == pytest.approx(D.behaviour_kl(prox.cpu(), old.cpu()), rel=1e-4, abs=1e-7)
    assert la["BehaviourKL"] > 1e-6
    # gradients of the one step: one more backward of each learner on its batch at theta_1
    for net in (A, B):
        net.load_state_dict(src.state_dict())
    A.backward_only(states, adv, a, old, values, prox_logps=prox)
    B.backward_only(states, w * adv, a, prox, values)
    ga, gb = A.flat_grads().double(), B.flat_grads().double()
    assert float((ga - gb).abs().max()) <= 2e-5 * float(gb.abs().max())


# ---------------------------------------------------------------------------------------------------------- 6. graphs
@pytest.mark.parametrize("M", [1, 4])
def test_graph_replay_equals_stream_launches_and_keeps_the_workspace(deterministic, monkeypatch, M):
    from ddrl4nav_b200 import _lib, kernels

    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make("pong", DECOUPLED_PPO=True, PPO_STATS=True, TRAINING_ITER_TIME=3, MINI_BATCH_NUM=M, MINI_BATCH_SEED=2)
        logs, launches, ws = [], [], []
        for call in range(3):
            kernels.launch_count_reset()
            logs += [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")]
                     for l, _, _ in net.learn(experience(*batch("pong", 40, seed=call)))]
            launches.append(kernels.launch_count())
            ws.append(_lib.load().ddrl_net_workspace_bytes(net._h))
        return logs, net._flat.clone(), launches, ws

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])
    # the pre-pass sizes the backward's workspace: calls 2 and 3 replay the graphs captured before, with the same launches
    assert g[2][1] == g[2][2] and g[3][0] == g[3][1] == g[3][2]


# ---------------------------------------------------------------------------------------------------------- 7. TARGET_KL
def test_target_kl_is_measured_against_the_proximal_policy(deterministic):
    """The stale batch puts the plain learner's first-step KL above a tiny target, so it stops at step 1; the decoupled
    learner's first-step KL is exactly 0 (the call has not moved the policy yet), so it stops at step 2."""
    states, a, old, adv, values = batch("navimg", 40)
    plain = [l for l, _, _ in make("navimg", TARGET_KL=1e-9, TRAINING_ITER_TIME=5).learn(experience(states, a, old, adv, values))]
    dc = [l for l, _, _ in make("navimg", TARGET_KL=1e-9, TRAINING_ITER_TIME=5, DECOUPLED_PPO=True).learn(
        experience(states, a, old, adv, values))]
    assert len(plain) == 1 and plain[0]["ApproxKL"] > 1e-9
    assert len(dc) == 2 and dc[0]["ApproxKL"] == 0.0 and dc[1]["ApproxKL"] > 1e-9


# ---------------------------------------------------------------------------------------------------------- 8. micro-batches
def test_micro_batched_rows_equal_the_option_off_learner_on_policy(deterministic, monkeypatch):
    monkeypatch.setenv("DDRL_MICRO_BATCH", "16")
    hyper = dict(TRAINING_ITER_TIME=2, PPO_STATS=True)
    A = make("navlaser", DECOUPLED_PPO=True, **hyper)
    B = make("navlaser", **hyper)
    states, a, _, adv, values = batch("navlaser", 40)
    on_policy = prox_of(B, states, a)
    for (la, _, _), (lb, _, _) in zip(A.learn(experience(states, a, on_policy, adv, values)),
                                      B.learn(experience(states, a, on_policy, adv, values))):
        assert [la[k] for k in KEYS] == [lb[k] for k in KEYS]
        assert torch.equal(A._flat, B._flat)
        assert la["BehaviourKL"] == 0.0


# ---------------------------------------------------------------------------------------------------------- 9. full size
def test_full_size_pong():
    B = 8192
    states, a, old, adv, values = batch("pong", B)
    net = make("pong", DECOUPLED_PPO=True, DECOUPLED_IS_CLIP=2.0, PPO_STATS=True)
    for call in range(2):
        out = [l for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        assert len(out) == 10
        assert all(np.isfinite([l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")]).all() for l in out)
        assert out[0]["ApproxKL"] == 0.0 and out[0]["ClipFrac"] == 0.0
        assert out[0]["BehaviourKL"] == pytest.approx(D.behaviour_kl(net.last_prox_logps.cpu(), old.cpu()), rel=1e-4, abs=1e-7)
    assert torch.isfinite(net._flat).all()


# ---------------------------------------------------------------------------------------------------------- 10. two ranks
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
    kind, B = "navlaser", 81
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, DECOUPLED_PPO=True, PPO_STATS=True)
    net.load_state_dict(R.init_params(R.SPECS[kind], seed=11), strict=False)
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    states, a, old, adv, values = batch(kind, B)
    lo, hi = (0, 41) if rank == 0 else (41, 81)
    exp = Experience(states=[s[lo:hi].to(dev) for s in states], advs=adv[lo:hi].to(dev), actions=a[lo:hi].to(dev),
                     old_logps=old[lo:hi].to(dev), values=values[:, lo:hi].to(dev))
    logs = [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")] for l, _, _ in net.learn(exp)]
    q.put((rank, logs, net._flat.cpu().numpy(), net.last_prox_logps.cpu().numpy()))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_replicas_are_identical_and_the_behaviour_kl_is_global():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, logs, flat, prox = q.get(timeout=600)
        res[r] = (logs, flat, prox)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (l0, f0, p0), (l1, f1, p1) = res[0], res[1]
    assert l0 == l1 and np.array_equal(f0, f1)
    states, a, old, adv, values = batch("navlaser", 81)
    prox = torch.from_numpy(np.concatenate([p0, p1]))
    assert l0[0][6] == pytest.approx(D.behaviour_kl(prox, old.cpu()), rel=1e-4, abs=1e-7)
    one = make("navlaser", TRAINING_ITER_TIME=2, DECOUPLED_PPO=True, PPO_STATS=True)
    ref = [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")]
           for l, _, _ in one.learn(experience(states, a, old, adv, values))]
    assert np.allclose(np.array(l0), np.array(ref), rtol=1e-4, atol=1e-6)
    assert np.allclose(f0, one._flat.cpu().numpy(), rtol=0, atol=1e-4)
