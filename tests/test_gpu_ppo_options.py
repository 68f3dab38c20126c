"""PPO training options of the learner on the GPU (NORM_ADV, VALUE_CLIP, PPO_STATS, TARGET_KL): with every option off the learner
is the default path, launch for launch and bit for bit; the one-block advantage normaliser against torch; the clipped value loss
and the statistics of the fused loss kernel against the CPU restatement (tests/ppo_options_ref.py); a minibatch step against a
full-batch step on its rows with every option on; graph replay; the KL early stop; a full-size run; and two-GPU parity."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import ppo_options_ref as O
from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")
STATS = ("ApproxKL", "ClipFrac")
ALL_ON = dict(NORM_ADV=True, VALUE_CLIP=1.0, PPO_STATS=True)
ALL_OFF = dict(NORM_ADV=False, VALUE_CLIP=None, PPO_STATS=False, TARGET_KL=None)


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


@pytest.fixture
def deterministic():
    from ddrl4nav_b200 import kernels
    was = kernels.set_deterministic(True)
    yield
    kernels.set_deterministic(was)


def make(kind, seed=11, **hyper):
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None, **hyper)
    net.load_state_dict(R.init_params(R.SPECS[kind], seed=seed), strict=True)
    return net.to(DEV)


def batch(kind, B, seed=9):
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=11)
    states = R.synth_states(kind, B, seed=5)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=seed)
    return [s.to(DEV) for s in states], a.to(DEV), old.to(DEV), adv.to(DEV), ret.to(DEV)[None]


def experience(states, a, old, adv, values, rows=None, old_values=None):
    from ddrl4nav_b200.data import Experience
    if rows is not None:
        r = rows.long()
        states = [s.index_select(0, r) for s in states]
        a, old, adv, values = a.index_select(0, r), old.index_select(0, r), adv.index_select(0, r), values.index_select(1, r)
        old_values = None if old_values is None else old_values.index_select(0, r)
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values, old_values=old_values)


def run_logs(net, exp, keys=KEYS + STATS):
    """[(losses, params after the step)] of every step of one learn call"""
    return [([l[x] for x in keys], net._flat.clone()) for l, _, _ in net.learn(exp)]


# ---------------------------------------------------------------------------------------------------------- 1. off = default
@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_options_off_is_the_default_path(deterministic, kind, M):
    from ddrl4nav_b200 import kernels
    states, a, old, adv, values = batch(kind, 40)
    out = []
    for hyper in ({}, ALL_OFF):
        net = make(kind, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=3, **hyper)
        kernels.launch_count_reset()
        logs = list(net.learn(experience(states, a, old, adv, values)))
        out.append(([[l[x] for x in KEYS] for l, _, _ in logs], net._flat.clone(), kernels.launch_count(),
                    [set(l) for l, _, _ in logs]))
    assert out[0][0] == out[1][0]
    assert torch.equal(out[0][1], out[1][1])
    assert out[0][2] == out[1][2]
    assert all(k == set(KEYS) | {"PpoBackUpTime"} for k in out[1][3])
    assert len(out[1][3]) == 2 * M


# ---------------------------------------------------------------------------------------------------------- 2. normaliser
@pytest.mark.parametrize("n", [2, 13, 8192, 65536])
def test_normaliser_matches_torch(n):
    from ddrl4nav_b200 import kernels
    g = torch.Generator(device=DEV).manual_seed(n)
    a = torch.randn(n, generator=g, device=DEV) * 2.5 + 0.7
    ref = (a - a.mean()) / (a.std() + 1e-8)
    out = kernels.adv_normalize(a)
    assert rel_err(out, ref) < 1e-6, rel_err(out, ref)
    assert torch.equal(kernels.adv_normalize(a), out)                     # two runs: the same bits
    b = a.clone()
    assert kernels.adv_normalize(b, out=b) is b and torch.equal(b, out)   # in place = out of place
    m3 = kernels.adv_moments(a)
    want = torch.tensor([n, float(a.double().sum()), float((a.double() ** 2).sum())], dtype=torch.float64)
    assert torch.allclose(m3.cpu(), want, rtol=1e-12)
    assert rel_err(kernels.adv_normalize(a, m3), out) < 1e-7               # given moments = the one-launch path


def test_normaliser_passes_one_row_through():
    from ddrl4nav_b200 import kernels
    a = torch.tensor([3.5], device=DEV)
    assert torch.equal(kernels.adv_normalize(a), a)
    assert torch.equal(kernels.adv_normalize(a, kernels.adv_moments(a)), a)
    e = torch.empty(0, device=DEV)
    assert kernels.adv_normalize(e).numel() == 0 and kernels.adv_moments(e).tolist() == [0.0, 0.0, 0.0]


# ---------------------------------------------------------------------------------------------------------- 3. vs the restatement
@pytest.mark.parametrize("smooth_l1", [False, True])
@pytest.mark.parametrize("given", [True, False])
@pytest.mark.parametrize("kind", ["pong", "navimg", "navlaser"])
def test_value_clip_and_stats_match_the_restatement(kind, given, smooth_l1):
    B, c = 48, 1.0
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=11)
    states, a, old, adv, values = batch(kind, B)
    adv0 = adv.clone()
    cpu = lambda t: t.detach().cpu()
    ret = cpu(values[0])
    with torch.no_grad():
        v_now = R.ppo_forward(spec, params, [cpu(s) for s in states])["values"].squeeze()
    if given:
        ov = v_now + 1.2 * torch.randn(B, generator=torch.Generator().manual_seed(17))
    else:
        ov = ret - cpu(adv)                                       # the learner's fallback: values[0] - advs
    frac = float(((v_now - ov).abs() > c).float().mean())
    assert 0.2 <= frac <= 0.8, frac                               # both branches of the clip run
    norm = given                                                  # normalisation on in half of the cases
    net = make(kind, TRAINING_ITER_TIME=1, VALUE_CLIP=c, PPO_STATS=True, NORM_ADV=norm, SMOOTH_L1_LOSS=smooth_l1)
    (log, _, _), = list(net.learn(experience(states, a, old, adv, values, old_values=ov.to(DEV) if given else None)))
    advs_ref = O.normalize_advantages(cpu(adv)) if norm else cpu(adv)
    losses, raw = O.learn_iteration(R.LearnState(spec, params), [cpu(s) for s in states], advs_ref, cpu(a), cpu(old), ret,
                                    R.PPOHyper(smooth_l1=smooth_l1), old_values=ov, value_clip=c, stats=True)
    ours = net.named_grads()
    worst = max(rel_err(ours[n], raw[n]) for n in raw)
    assert worst < 2e-5, worst
    for k in KEYS:
        assert abs(log[k] - losses[k]) <= 1e-5 * max(1.0, abs(losses[k])), (k, log[k], losses[k])
    assert log["ApproxKL"] == pytest.approx(losses["ApproxKL"], rel=1e-5, abs=1e-6)
    assert abs(log["ClipFrac"] - losses["ClipFrac"]) <= 1.0 / B
    assert torch.equal(adv, adv0)                                 # the caller's advantages are not written


def test_value_clip_without_old_values_is_rejected_by_the_engine():
    from ddrl4nav_b200._lib import DDRLError
    states, a, old, adv, values = batch("navimg", 8)
    net = make("navimg", TRAINING_ITER_TIME=1, VALUE_CLIP=0.5)
    with pytest.raises(DDRLError, match="ddrl_net_backward_v"):
        net.backward_only(states, adv, a, old, values)
    net.backward_only(states, adv, a, old, values, old_values=values[0] - adv)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------- 4. minibatch = full batch
@pytest.mark.parametrize("kind,given", [("pong", True), ("navimg", False), ("navlaser", False)])
def test_minibatch_step_equals_full_batch_step_with_options(deterministic, kind, given):
    B, M, iters = 40, 3, 2
    states, a, old, adv, values = batch(kind, B)
    ov = values[0] - adv + 0.3 * torch.randn(B, generator=torch.Generator(device=DEV).manual_seed(1), device=DEV) if given else None
    netA = make(kind, MINI_BATCH_NUM=M, TRAINING_ITER_TIME=iters, MINI_BATCH_SEED=5, **ALL_ON)
    netB = make(kind, TRAINING_ITER_TIME=1, **ALL_ON)
    plan = netA.minibatch_plan(B, M)
    n = 0
    for la, upd, last in netA.learn(experience(states, a, old, adv, values, old_values=ov)):
        epoch, k = divmod(n, M)
        lo, hi = plan[k]
        rows = netA.last_minibatch_perms[epoch][lo:hi]
        (lb, _, _), = list(netB.learn(experience(states, a, old, adv, values, rows, ov)))
        n += 1
        assert set(la) == set(KEYS) | set(STATS) | {"PpoBackUpTime"}
        assert [la[x] for x in KEYS + STATS] == [lb[x] for x in KEYS + STATS], (kind, n, la, lb)
        assert torch.equal(netA._flat, netB._flat), (kind, n, rel_err(netA._flat, netB._flat))
    assert n == iters * M


# ---------------------------------------------------------------------------------------------------------- 5. graph replay
@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_graph_replay_with_options_equals_stream_launches(deterministic, monkeypatch, kind, M):
    states, a, old, adv, values = batch(kind, 40)

    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make(kind, MINI_BATCH_NUM=M, TRAINING_ITER_TIME=2, MINI_BATCH_SEED=1, **ALL_ON)
        logs = [l for _ in range(2) for l, _ in run_logs(net, experience(states, a, old, adv, values))]
        return logs, net._flat.clone(), net._m.clone()

    l_graph, p_graph, m_graph = run(False)
    l_eager, p_eager, m_eager = run(True)
    assert l_graph == l_eager
    assert torch.equal(p_graph, p_eager) and torch.equal(m_graph, m_eager)


# ---------------------------------------------------------------------------------------------------------- 6. early stop
@pytest.mark.parametrize("M", [1, 3])
def test_target_kl_stops_the_learn_call(deterministic, M):
    kind, B, iters = "navimg", 40, 3
    states, a, old, adv, values = batch(kind, B)
    exp = lambda: experience(states, a, old, adv, values)
    hyper = dict(TRAINING_ITER_TIME=iters, MINI_BATCH_NUM=M, MINI_BATCH_SEED=5, NORM_ADV=True, VALUE_CLIP=1.0)
    ref = run_logs(make(kind, PPO_STATS=True, **hyper), exp())
    assert len(ref) == iters * M
    kls = [l[len(KEYS)] for l, _ in ref]
    assert all(k > 0 for k in kls)

    def check(target, want):
        got = run_logs(make(kind, TARGET_KL=target, **hyper), exp())
        assert len(got) == want, (target, len(got), want)
        for (lg, pg), (lr, pr) in zip(got, ref):
            assert lg == lr and torch.equal(pg, pr)

    check(1e-12, 1)
    check(1e9, iters * M)
    # the first step above the first step's KL ends the call; everything before it equals the run without a target
    stop = next((i for i, k in enumerate(kls) if k > kls[0]), len(kls) - 1)
    check(kls[0], stop + 1)


# ---------------------------------------------------------------------------------------------------------- 7. full size
def test_full_size_pong_with_every_option():
    B, M = 8192, 4
    states, a, old, adv, values = batch("pong", B)
    adv0 = adv.clone()
    net = make("pong", MINI_BATCH_NUM=M, **ALL_ON)
    out = list(net.learn(experience(states, a, old, adv, values)))
    assert len(out) == 10 * M and [u for _, u, _ in out] == list(range(1, 10 * M + 1))
    assert all(set(l) == set(KEYS) | set(STATS) | {"PpoBackUpTime"} for l, _, _ in out)
    assert all(np.isfinite([l[x] for x in KEYS + STATS]).all() for l, _, _ in out)
    assert all(0.0 <= l["ClipFrac"] <= 1.0 and l["ApproxKL"] > -1e-6 for l, _, _ in out)
    assert torch.isfinite(net._flat).all()
    assert torch.equal(adv, adv0)


# ---------------------------------------------------------------------------------------------------------- 8. two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


DP_TARGET_KL = 0.05


def _dp_worker(rank, world, port, q):
    import torch.distributed as tdist
    from ddrl4nav_b200 import kernels
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    kernels.set_deterministic(True)
    tdist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world, device_id=dev)
    kind, B, M = "pong", 81, 3
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=3)
    states = R.synth_states(kind, B, seed=4)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=5)
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=10 + rank, TARGET_KL=DP_TARGET_KL,
                   **ALL_ON)
    net.load_state_dict(params)
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    lo, hi = (0, 41) if rank == 0 else (41, 81)
    exp = Experience(states=[s[lo:hi].to(dev) for s in states], advs=adv[lo:hi].to(dev), actions=a[lo:hi].to(dev),
                     old_logps=old[lo:hi].to(dev), values=ret[lo:hi].to(dev)[None])
    snaps, logs, rows = [], [], []
    plan = net.minibatch_plan(hi - lo, M)
    for n, (l, _, _) in enumerate(net.learn(exp)):
        e, k = divmod(n, M)
        rows.append((net.last_minibatch_perms[e][plan[k][0]:plan[k][1]].long().cpu() + lo).numpy())
        snaps.append(net._flat.detach().cpu().numpy())
        logs.append([l[x] for x in KEYS + STATS])
    q.put((rank, rows, snaps, logs))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_steps_with_options_equal_single_gpu_steps_on_the_union():
    from ddrl4nav_b200.data import Experience
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, rows, snaps, logs = q.get(timeout=600)
        res[r] = (rows, snaps, logs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (rows0, snaps0, logs0), (rows1, snaps1, logs1) = res[0], res[1]
    assert len(snaps0) == len(snaps1) and logs0 == logs1           # the same stop step and the same global losses
    kl = len(KEYS)
    assert all(l[kl] <= DP_TARGET_KL for l in logs0[:-1])
    assert len(logs0) == 6 or logs0[-1][kl] > DP_TARGET_KL
    for s0, s1 in zip(snaps0, snaps1):
        assert np.array_equal(s0, s1)
    kind = "pong"
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=3)
    states = R.synth_states(kind, 81, seed=4)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=5)
    ref = make(kind, seed=3, TRAINING_ITER_TIME=1, **ALL_ON)
    for n, (r0, r1) in enumerate(zip(rows0, rows1)):
        r = torch.from_numpy(np.concatenate([r0, r1]))
        exp = Experience(states=[s[r].to(DEV) for s in states], advs=adv[r].to(DEV), actions=a[r].to(DEV),
                         old_logps=old[r].to(DEV), values=ret[r].to(DEV)[None])
        (l, _, _), = list(ref.learn(exp))
        for x, want in zip(KEYS + STATS, logs0[n]):
            assert abs(l[x] - want) <= 2e-5 * max(1.0, abs(l[x])), (n, x, want, l[x])
        d = np.abs(snaps0[n] - ref._flat.cpu().numpy())
        assert (d > 3e-4).mean() < 1e-3, n
        ref._flat.copy_(torch.from_numpy(snaps0[n]).to(DEV))
        ref._weights_changed()
