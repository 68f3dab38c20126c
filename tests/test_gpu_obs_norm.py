"""Running observation normalisation (NORM_OBS) on the GPU: with the option off the learner is the default path, launch for
launch and bit for bit; the moments, merge and normalise kernels against float64 torch / the restatement (tests/obs_norm_ref.py);
a normalising learner against an option-off learner fed the normalised batch; the on-policy update rule; checkpoint and weight
blob; extra critics and graph replay; a full-size Pong run; and two-GPU parity."""
import copy
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import obs_norm_ref as N
from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")
# per kind: the NORM_OBS value the equivalence tests use and the slots it resolves to
SLOTS = {"pong": (True, (0,)), "navlaser": ((0, 1), (0, 1)), "navimg": (True, (0, 1)), "mlp": (True, (0,))}


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
        net.load_state_dict(R.init_params(R.SPECS[kind], seed=seed), strict=True)
    else:
        torch.manual_seed(seed)
        net.load_state_dict(make_net(kind, device=None).state_dict(), strict=True)
    return net.to(DEV)


def batch(kind, B, seed=9):
    """(states, actions, old log-probs, advantages, values [1, B]) on the device; the vector slots get offsets and scales far
    from (0, 1) so that the statistics matter."""
    g = torch.Generator().manual_seed(seed)
    if kind == "mlp":
        states = [torch.randn(B, 4, generator=g) * torch.tensor([1.0, 30.0, 0.05, 4.0]) + torch.tensor([0.0, 100.0, -3.0, 1.0])]
        a = torch.randint(0, 2, (B,), generator=g).float()
        old = -0.69 + 0.15 * torch.randn(B, generator=g)
        adv, ret = torch.randn(B, generator=g), torch.randn(B, generator=g)
    else:
        spec = R.SPECS[kind]
        states = R.synth_states(kind, B, seed=seed)
        if len(states) > 1:
            states[1] = states[1] * 7.0 + 3.0
        a, old, adv, ret = R.synth_learn_batch(spec, R.init_params(spec, seed=11), states, seed=seed)
    return [s.to(DEV) for s in states], a.to(DEV), old.to(DEV), adv.to(DEV), ret.to(DEV)[None]


def experience(states, a, old, adv, values):
    from ddrl4nav_b200.data import Experience
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values)


def rms_state(net):
    rms = net.obs_rms
    return {s: [t.detach().cpu().numpy().copy() for t in rms.state(s)] for s in rms.slots}


def normalized(net, states):
    """states with net's NORM_OBS slots normalised in torch with the net's CURRENT applied form."""
    net._ensure_engine()
    rms = net.obs_rms
    rms.refresh()
    out = list(states)
    for s in rms.slots:
        m, sc = rms.applied(s)
        shape = out[s].shape
        y = (out[s].reshape(shape[0], -1) - m) * sc
        if rms.clip is not None:
            y = torch.clamp(y, -rms.clip, rms.clip)
        out[s] = y.reshape(shape)
    return out


def rel_close(a, b, tol=1e-12):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))) <= tol


def check_against_ref(net, refs, tol=1e-12):
    for s, (mean, var, count) in rms_state(net).items():
        r = refs[s]
        assert rel_close(mean, r.mean, tol) or np.max(np.abs(mean - r.mean)) < tol * max(1.0, np.max(np.abs(r.mean))), s
        assert rel_close(var, r.var, tol), s
        assert abs(count[0] - r.count) <= tol * r.count, (s, count[0], r.count)


# ---------------------------------------------------------------------------------------------------------- 1. off = default
@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_option_off_is_the_default_path(deterministic, kind, M):
    from ddrl4nav_b200 import kernels
    states, a, old, adv, values = batch(kind, 40)
    out = []
    for hyper in ({}, dict(NORM_OBS=False, NORM_OBS_CLIP=3.0)):
        net = make(kind, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=3, **hyper)
        kernels.launch_count_reset()
        logs = [[l[x] for x in KEYS] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        n = kernels.launch_count()
        out.append((logs, net._flat.clone(), n, list(net.state_dict()), net.model_bytes()))
    assert out[0][0] == out[1][0]
    assert torch.equal(out[0][1], out[1][1])
    assert out[0][2] == out[1][2]
    assert out[0][3] == out[1][3] and not any(k.startswith("obs_rms") for k in out[1][3])
    assert out[0][4] == out[1][4]


# ---------------------------------------------------------------------------------------------------------- 2. kernels
@pytest.mark.parametrize("B", [1, 7, 1024, 8192])
@pytest.mark.parametrize("D", [5, 9, 960, 3 * 960, 28224])
def test_moments_match_float64_torch(B, D):
    from ddrl4nav_b200 import kernels
    g = torch.Generator(device=DEV).manual_seed(B * 7 + D)
    base = torch.randn(B * D + 1, generator=g, device=DEV) * 3.0 + 2.0
    x = base[:B * D].view(B, D)
    shift = (torch.randn(D, generator=g, device=DEV, dtype=torch.float64) + 2.0)
    sums = kernels.obs_moments(x, shift)
    d = x.double() - shift
    want1, want2 = d.sum(0), (d * d).sum(0)
    # S1 can cancel: its error is bounded against sum |d|, S2 against itself
    assert float(((sums[:D] - want1).abs() / (d.abs().sum(0))).max()) < 1e-12
    assert float(((sums[D:] - want2).abs() / want2).max()) < 1e-12
    assert torch.equal(kernels.obs_moments(x, shift), sums)                       # two launches: the same bits
    # an offset pointer takes the scalar path; it visits every column's rows in the same order
    y = base[1:].view(B, D)
    y_aligned = y.clone()
    assert torch.equal(kernels.obs_moments(y, shift), kernels.obs_moments(y_aligned, shift))


@pytest.mark.parametrize("clip", [10.0, 0.5, None])
@pytest.mark.parametrize("B,D", [(1, 5), (7, 9), (256, 960), (33, 2880), (64, 28224)])
def test_normalize_is_bit_equal_to_torch(B, D, clip):
    from ddrl4nav_b200 import kernels
    g = torch.Generator(device=DEV).manual_seed(B + D)
    x = torch.randn(B, D, generator=g, device=DEV) * 4.0 + 1.0
    m = torch.randn(D, generator=g, device=DEV)
    s = torch.rand(D, generator=g, device=DEV) * 3.0 + 0.01
    ref = (x - m) * s
    if clip is not None:
        ref = torch.clamp(ref, -clip, clip)
    assert torch.equal(kernels.obs_normalize(x, m, s, clip), ref)
    z = x.clone()
    assert kernels.obs_normalize(z, m, s, clip, out=z) is z and torch.equal(z, ref)      # in place
    base = torch.empty(B * D + 1, device=DEV)
    u = base[1:].view(B, D)
    u.copy_(x)
    assert torch.equal(kernels.obs_normalize(u, m, s, clip), ref)                       # unaligned: the scalar path


@pytest.mark.parametrize("D", [5, 2880, 28224])
def test_rms_update_matches_the_restatement(D):
    from ddrl4nav_b200 import kernels
    g = torch.Generator(device=DEV).manual_seed(D)
    ref = N.RunningMeanStd(D)
    mean = torch.zeros(D, dtype=torch.float64, device=DEV)
    var = torch.ones(D, dtype=torch.float64, device=DEV)
    count = torch.full((1,), 1e-4, dtype=torch.float64, device=DEV)
    m32, s32 = torch.empty(D, device=DEV), torch.empty(D, device=DEV)
    kernels.obs_rms_update(mean, var, count, None, 0, m32, s32)                 # n = 0: the applied form only
    assert torch.all(m32 == 0) and torch.equal(s32, torch.full((D,), float(np.float32(1 / np.sqrt(1 + 1e-8))), device=DEV))
    assert float(count) == 1e-4
    for rows, loc, sc in ((300, 5.0, 2.0), (17, -1.0, 0.1), (1, 0.0, 1.0)):
        x = torch.randn(rows, D, generator=g, device=DEV) * sc + loc
        sums = kernels.obs_moments(x, mean)
        kernels.obs_rms_update(mean, var, count, sums, rows, m32, s32)
        ref.update(x.cpu().numpy())
        assert rel_close(mean.cpu().numpy(), ref.mean) and rel_close(var.cpu().numpy(), ref.var)
        assert abs(float(count) - ref.count) <= 1e-12 * ref.count
        rm, rs = N.applied(mean.cpu().numpy(), var.cpu().numpy())
        assert np.array_equal(m32.cpu().numpy(), rm) and np.array_equal(s32.cpu().numpy(), rs)


# ---------------------------------------------------------------------------------------------------------- 3. equivalence
def _equivalence(kind, M, options=None, calls=2):
    """Net A normalises (NORM_OBS) and learns on raw X; net B (option off, same initial weights) learns on X normalised with the
    statistics A held at the start of each call.  Every step: the same losses and parameters, bit for bit."""
    norm_obs, slots = SLOTS[kind]
    hyper = dict(TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=4, **(options or {}))
    netA = make(kind, NORM_OBS=norm_obs, **hyper)
    netB = make(kind, **hyper)
    keys = KEYS + (("ApproxKL", "ClipFrac") if options and options.get("PPO_STATS") else ())
    for call in range(calls):
        states, a, old, adv, values = batch(kind, 40, seed=20 + call)
        raw = [s.clone() for s in states]
        netA._ensure_engine()
        assert netA.obs_rms.slots == slots
        x_hat = normalized(netA, states)
        n = 0
        for (la, _, _), (lb, _, _) in zip(netA.learn(experience(states, a, old, adv, values)),
                                          netB.learn(experience(x_hat, a, old, adv, values))):
            n += 1
            assert [la[k] for k in keys] == [lb[k] for k in keys], (kind, M, call, n)
            assert torch.equal(netA._flat, netB._flat), (kind, M, call, n)
        assert n == 2 * M
        assert all(torch.equal(r, s) for r, s in zip(raw, states))      # the caller's states are not written
    return netA


@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("kind", ["pong", "navlaser", "navimg", "mlp"])
def test_learner_equals_option_off_learner_on_normalised_states(deterministic, kind, M):
    _equivalence(kind, M)


def test_equivalence_with_the_ppo_options(deterministic):
    _equivalence("navlaser", 3, dict(NORM_ADV=True, VALUE_CLIP=1.0, PPO_STATS=True))


# ---------------------------------------------------------------------------------------------------------- 4. update rule
@pytest.mark.parametrize("M", [1, 3])
def test_statistics_follow_the_restatement_and_fold_before_the_final_yield(M):
    kind = "navlaser"
    net = make(kind, NORM_OBS=(0, 1), TRAINING_ITER_TIME=3, MINI_BATCH_NUM=M, MINI_BATCH_SEED=1)
    net._ensure_engine()
    refs = {s: N.RunningMeanStd(net.obs_rms.dims[s]) for s in (0, 1)}
    for call in range(2):
        states, a, old, adv, values = batch(kind, 50, seed=30 + call)
        counts = [float(net.obs_rms.count_0) for _ in net.learn(experience(states, a, old, adv, values))]
        for s in (0, 1):
            refs[s].update(states[s].cpu().numpy())
        assert counts[:-1] == [1e-4 + 50 * call] * (3 * M - 1)        # unchanged until the final step's yield
        assert counts[-1] == pytest.approx(1e-4 + 50 * (call + 1), rel=1e-15)
        check_against_ref(net, refs)


def test_target_kl_folds_once_on_the_stopping_step():
    kind = "navimg"
    net = make(kind, NORM_OBS=True, TRAINING_ITER_TIME=4, TARGET_KL=1e-12)
    states, a, old, adv, values = batch(kind, 40)
    logs = list(net.learn(experience(states, a, old, adv, values)))
    assert len(logs) == 1
    refs = {s: N.RunningMeanStd(net.obs_rms.dims[s]) for s in (0, 1)}
    for s in (0, 1):
        refs[s].update(states[s].cpu().numpy())
    check_against_ref(net, refs)


@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_act_after_learning_uses_the_new_statistics(kind):
    norm_obs, _ = SLOTS[kind]
    net = make(kind, NORM_OBS=norm_obs, TRAINING_ITER_TIME=1)
    off = make(kind, TRAINING_ITER_TIME=1)
    states, a, old, adv, values = batch(kind, 40)
    applied = lambda: [m.clone() for s in net.obs_rms.slots for m in net.obs_rms.applied(s)]
    normalized(net, states)                                   # builds the engine and the initial applied form
    before = applied()
    list(net.learn(experience(states, a, old, adv, values)))
    off.load_state_dict({k: v for k, v in net.state_dict().items() if not k.startswith("obs_rms.")}, strict=True)
    assert not any(torch.equal(x, y) for x, y in zip(before, applied()))
    q, *_ = batch(kind, 64, seed=99)
    A = net.actor.actor_linear.out_features
    draw = torch.rand(64, device=DEV) if kind == "pong" else torch.randn(64, A, device=DEV)
    for got, want in zip(net.act(q, draw=draw), off.act(normalized(net, q), draw=draw)):
        assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------------- 5. state
def _learned(kind="navlaser"):
    norm_obs, _ = SLOTS[kind]
    net = make(kind, NORM_OBS=norm_obs, TRAINING_ITER_TIME=1, NORM_OBS_CLIP=5.0)
    for call in range(2):
        states, a, old, adv, values = batch(kind, 40, seed=40 + call)
        list(net.learn(experience(states, a, old, adv, values)))
    return net


def _act_bits(net, kind="navlaser", seed=5):
    q, *_ = batch(kind, 32, seed=seed)
    draw = torch.randn(32, net.actor.actor_linear.out_features, generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)
    return net.act(q, draw=draw)


def test_state_dict_round_trip_gives_identical_act_bits():
    net = _learned()
    sd = net.state_dict()
    assert {k for k in sd if k.startswith("obs_rms.")} == {"obs_rms.%s_%d" % (w, s) for w in ("mean", "var", "count") for s in (0, 1)}
    assert all(sd[k].dtype == torch.float64 for k in sd if k.startswith("obs_rms."))
    fresh = make("navlaser", NORM_OBS=(0, 1), NORM_OBS_CLIP=5.0)
    fresh.load_state_dict(sd, strict=True)
    for x, y in zip(_act_bits(net), _act_bits(fresh)):
        assert torch.equal(x, y)
    for s in (0, 1):
        for x, y in zip(net.obs_rms.state(s) + net.obs_rms.applied(s), fresh.obs_rms.state(s) + fresh.obs_rms.applied(s)):
            assert torch.equal(x, y)


def test_blob_carries_the_applied_form_bit_exactly():
    from ddrl4nav_b200._lib import DDRLError
    net = _learned()
    blob = net.model_bytes()
    plain = make("navlaser").model_bytes()
    # per slot: mean32 [D] and scale32 [D] records (>I ndim, >I D, 4 D bytes) and the count record [1]
    assert len(blob) - len(plain) == sum(2 * (8 + 4 * d) + 12 for d in (960, 5))
    fresh = make("navlaser", NORM_OBS=(0, 1), NORM_OBS_CLIP=5.0)
    fresh.load_model_bytes(blob)
    for s in (0, 1):
        for x, y in zip(net.obs_rms.applied(s), fresh.obs_rms.applied(s)):
            assert torch.equal(x, y)
        assert float(fresh.obs_rms.state(s)[2]) == float(np.float32(float(net.obs_rms.state(s)[2])))
    for x, y in zip(_act_bits(net), _act_bits(fresh)):
        assert torch.equal(x, y)
    with pytest.raises(DDRLError, match="NORM_OBS"):
        make("navlaser", NORM_OBS=(0, 1)).load_model_bytes(plain)
    with pytest.raises(DDRLError, match="NORM_OBS"):
        make("navlaser", NORM_OBS=(0,)).load_model_bytes(plain)


def test_out_of_range_slot_is_rejected_when_the_engine_is_built():
    from ddrl4nav_b200._lib import DDRLError
    net = make("navimg", NORM_OBS=(1, 2))
    states, *_ = batch("navimg", 4)
    with pytest.raises(DDRLError, match="NORM_OBS slot"):
        net.act(states)


# ---------------------------------------------------------------------------------------------------------- 6. critics and paths
@pytest.mark.parametrize("kind", ["navimg", "pong"])       # shared mode, unshared mode (extra critic on its own engine)
def test_added_gail_critic_sees_normalised_inputs(deterministic, kind):
    from ddrl4nav_b200.runner import make_net
    norm_obs, _ = SLOTS[kind]
    nets = [make(kind, NORM_OBS=norm_obs, TRAINING_ITER_TIME=2), make(kind, TRAINING_ITER_TIME=2)]
    torch.manual_seed(3)
    c = make_net(kind, device=None).critic
    for net in nets:
        net.add_critic(copy.deepcopy(c).to(DEV))
        net.gail_critic = True
    on, off = nets
    states, a, old, adv, values = batch(kind, 40)
    values = torch.cat([values, values * 0.5 + 0.1])
    q, *_ = batch(kind, 24, seed=77)
    got, want = on.act(q, play_mode=True), off.act(normalized(on, q), play_mode=True)
    assert got[2].shape[0] == 2 and all(torch.equal(x, y) for x, y in zip(got, want))
    x_hat = normalized(on, states)
    for (la, _, _), (lb, _, _) in zip(on.learn(experience(states, a, old, adv, values)),
                                      off.learn(experience(x_hat, a, old, adv, values))):
        assert [la[k] for k in KEYS] == [lb[k] for k in KEYS]
        assert torch.equal(on._flat, off._flat)


@pytest.mark.parametrize("M", [1, 3])
def test_no_graph_gives_the_same_bits(deterministic, monkeypatch, M):
    kind = "pong"
    states, a, old, adv, values = batch(kind, 40)

    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make(kind, NORM_OBS=True, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=2)
        logs = [[l[x] for x in KEYS] for _ in range(2) for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        return logs, net._flat.clone(), rms_state(net), _act_bits_pong(net)

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])
    assert all(np.array_equal(x, y) for s in g[2] for x, y in zip(g[2][s], e[2][s]))
    assert all(torch.equal(x, y) for x, y in zip(g[3], e[3]))


def _act_bits_pong(net):
    q, *_ = batch("pong", 16, seed=3)
    return net.act(q, draw=torch.rand(16, generator=torch.Generator(device=DEV).manual_seed(3), device=DEV))


# ---------------------------------------------------------------------------------------------------------- 7. full size
def test_full_size_pong():
    B = 8192
    states, a, old, adv, values = batch("pong", B)
    net = make("pong", NORM_OBS=True)
    out = list(net.learn(experience(states, a, old, adv, values)))
    assert len(out) == 10
    assert all(np.isfinite([l[x] for x in KEYS]).all() for l, _, _ in out)
    assert torch.isfinite(net._flat).all()
    ref = N.RunningMeanStd(4 * 84 * 84)
    ref.update(states[0].cpu().numpy())
    check_against_ref(net, {0: ref})


# ---------------------------------------------------------------------------------------------------------- 8. two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, overlap, q):
    import os
    import torch.distributed as tdist
    from ddrl4nav_b200 import kernels
    if overlap:
        os.environ["DDRL_DP_OVERLAP"] = "1"
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    kernels.set_deterministic(True)
    tdist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world, device_id=dev)
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net
    kind, B = "navlaser", 81
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, NORM_OBS=(0, 1))
    net.load_state_dict(R.init_params(R.SPECS[kind], seed=11))
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    states, a, old, adv, values = batch(kind, B)
    lo, hi = (0, 41) if rank == 0 else (41, 81)
    exp = Experience(states=[s[lo:hi].to(dev) for s in states], advs=adv[lo:hi].to(dev), actions=a[lo:hi].to(dev),
                     old_logps=old[lo:hi].to(dev), values=values[:, lo:hi].to(dev))
    logs = []
    for call in range(2):
        logs += [[l[x] for x in KEYS] for l, _, _ in net.learn(exp)]
    q.put((rank, logs, net._flat.cpu().numpy(), {s: [t.cpu().numpy() for t in net.obs_rms.state(s) + net.obs_rms.applied(s)]
                                                 for s in (0, 1)}))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("overlap", [False, True])
def test_two_gpu_statistics_are_identical_and_equal_the_union(overlap):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, overlap, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, logs, flat, stats = q.get(timeout=600)
        res[r] = (logs, flat, stats)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (l0, f0, s0), (l1, f1, s1) = res[0], res[1]
    assert l0 == l1 and np.array_equal(f0, f1)
    for s in (0, 1):
        assert all(np.array_equal(x, y) for x, y in zip(s0[s], s1[s]))
    # one GPU on the union of the rows: the same statistics to fp64 rounding, and the same losses to fp32 rounding
    states, a, old, adv, values = batch("navlaser", 81)
    ref = make("navlaser", NORM_OBS=(0, 1), TRAINING_ITER_TIME=2)
    logs = []
    for call in range(2):
        logs += [[l[x] for x in KEYS] for l, _, _ in ref.learn(experience(states, a, old, adv, values))]
    for s in (0, 1):
        mean, var, count = [t.cpu().numpy() for t in ref.obs_rms.state(s)]
        assert np.max(np.abs(s0[s][0] - mean)) <= 1e-12 * max(1.0, np.max(np.abs(mean)))
        assert rel_close(s0[s][1], var) and abs(s0[s][2][0] - count[0]) <= 1e-12 * count[0]
    for x, y in zip(l0, logs):
        assert np.allclose(x, y, rtol=2e-5, atol=1e-6)
