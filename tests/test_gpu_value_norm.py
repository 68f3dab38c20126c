"""Value-target normalisation (NORM_VALUE, PopArt) on the GPU: with the option off the learner is the default path, launch for
launch and bit for bit; the update kernel against the float64 restatement (tests/value_norm_ref.py) and torch; a normalising
learner against an option-off learner given its rescaled parameters and the normalised targets; the values act returns and
their preservation across the rescale; checkpoint and weight blob; the TARGET_KL stop and graph replay; a full-size Pong run;
and two-GPU parity."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import value_norm_ref as V
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


def batch(kind, B, seed=9, loc=500.0, scale=80.0):
    """(states, actions, old log-probs, advantages, values [1, B]) on the device; the return targets are loc + scale * N(0, 1),
    far from the unit scale the critic starts at."""
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
    ret = loc + scale * torch.randn(B, generator=g)
    return [s.to(DEV) for s in states], a.to(DEV), old.to(DEV), adv.to(DEV), ret.to(DEV)[None]


def experience(states, a, old, adv, values, old_values=None):
    from ddrl4nav_b200.data import Experience
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values, old_values=old_values)


def learn_calls(net, kind, calls, B=40, seed=40):
    for call in range(calls):
        list(net.learn(experience(*batch(kind, B, seed=seed + call))))
    return net


def rel_close(a, b, tol=1e-12):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))) <= tol


def stats(net):
    return [t.detach().cpu().clone() for t in net.value_rms.state()] + [net.value_rms.applied32.detach().cpu().clone()]


# ---------------------------------------------------------------------------------------------------------- 1. off = default
@pytest.mark.parametrize("M", [1, 3])
@pytest.mark.parametrize("kind", ["pong", "mlp"])
def test_option_off_is_the_default_path(deterministic, kind, M):
    from ddrl4nav_b200 import kernels
    data = batch(kind, 40)
    out = []
    for hyper in ({}, dict(NORM_VALUE=False)):
        net = make(kind, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=3, **hyper)
        kernels.launch_count_reset()
        logs = [[l[x] for x in KEYS] for l, _, _ in net.learn(experience(*data))]
        n = kernels.launch_count()
        values = net.act(data[0], play_mode=True)[2]
        out.append((logs, net._flat.clone(), n, list(net.state_dict()), net.model_bytes(), values))
    assert out[0][0] == out[1][0]
    assert torch.equal(out[0][1], out[1][1])
    assert out[0][2] == out[1][2]
    assert out[0][3] == out[1][3] and not any(k.startswith("value_rms") for k in out[1][3])
    assert out[0][4] == out[1][4]
    assert torch.equal(out[0][5], out[1][5])


# ---------------------------------------------------------------------------------------------------------- 2. update kernel
def test_update_kernel_matches_the_restatement_and_torch_float64():
    from ddrl4nav_b200 import kernels
    ref = V.ValueRMS()
    mean = torch.zeros(1, dtype=torch.float64, device=DEV)
    var = torch.ones(1, dtype=torch.float64, device=DEV)
    count = torch.full((1,), 1e-4, dtype=torch.float64, device=DEV)
    applied = torch.empty(3, device=DEV)
    kernels.value_norm_update(mean, var, count, None, 0, applied)             # n = 0: the applied form only
    assert applied.cpu().numpy().tolist() == V.applied(0.0, 1.0).tolist() and float(count) == 1e-4
    g = torch.Generator(device=DEV).manual_seed(0)
    w = torch.randn(512, generator=g, device=DEV) * 0.05
    b = torch.full((1,), 0.3, device=DEV)
    for rows, loc, sc in ((8192, 500.0, 80.0), (37, -3.0, 0.01), (1, 0.0, 1.0), (1024, 1e4, 1e3), (300, 500.0, 80.0)):
        x = torch.randn(rows, generator=g, device=DEV) * sc + loc
        m0, v0, w0, b0 = mean.cpu(), var.cpu(), w.cpu().double(), b.cpu().double()
        sums = kernels.obs_moments(x, mean)
        kernels.value_norm_update(mean, var, count, sums, rows, applied, w, b)
        ref.update(x.cpu().numpy()[:, None])
        assert rel_close(mean.cpu().numpy(), ref.mean) and rel_close(var.cpu().numpy(), ref.var)
        assert abs(float(count) - ref.count) <= 1e-12 * ref.count
        # the applied form and the head from the kernel's float64 state, in torch float64 on the host (correctly rounded)
        m1, v1 = mean.cpu(), var.cpu()
        s0, s1 = torch.sqrt(v0 + 1e-8), torch.sqrt(v1 + 1e-8)
        assert torch.equal(applied.cpu(), torch.cat([m1, 1.0 / s1, s1]).float())
        assert torch.equal(w.cpu(), (w0 * s0 / s1).float())
        assert torch.equal(b.cpu(), ((s0 * b0 + m0 - m1) / s1).float())


# ---------------------------------------------------------------------------------------------------------- 3. equivalence
def _equivalence(kind, M, clip, calls=2):
    """Net A normalises its value targets and learns on raw returns; net B (option off) is given, at the start of every call,
    A's parameters right after A's start-of-call update, and learns on the targets (and old values) normalised in torch with
    A's new applied form.  Every step: the same losses, gradients and parameters, bit for bit."""
    hyper = dict(TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=4, **({"VALUE_CLIP": 0.5} if clip else {}))
    A = make(kind, NORM_VALUE=True, **hyper)
    B = make(kind, **hyper)
    B._ensure_engine()
    begin = type(A)._value_norm_begin
    for call in range(calls):
        states, a, old, adv, values = batch(kind, 40, seed=20 + call)
        ret_b, ov_b = torch.empty_like(values), torch.empty_like(adv)

        def hooked(data, n):
            begin(A, data, n)
            ap = A.value_rms.applied32
            ret_b.copy_((values - ap[0]) * ap[1])
            ov_b.copy_(((values[0] - adv) - ap[0]) * ap[1])        # A's VALUE_CLIP fallback: values[0] - advs
            with torch.no_grad():
                B._flat.copy_(A._flat)

        A._value_norm_begin = hooked
        n = 0
        for (la, _, _), (lb, _, _) in zip(A.learn(experience(states, a, old, adv, values)),
                                          B.learn(experience(states, a, old, adv, ret_b, ov_b if clip else None))):
            n += 1
            assert [la[k] for k in KEYS] == [lb[k] for k in KEYS], (kind, M, clip, call, n)
            assert torch.equal(A.flat_grads(), B.flat_grads()), (kind, M, clip, call, n)
            assert torch.equal(A._flat, B._flat), (kind, M, clip, call, n)
        del A._value_norm_begin
        assert n == 2 * M


@pytest.mark.parametrize("clip", [False, True])
@pytest.mark.parametrize("M", [1, 4])
@pytest.mark.parametrize("kind", ["pong", "navlaser", "navimg", "mlp"])
def test_learner_equals_option_off_learner_on_normalised_targets(deterministic, kind, M, clip):
    _equivalence(kind, M, clip)


# ---------------------------------------------------------------------------------------------------------- 4. acting
@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_act_returns_the_denormalised_values(kind):
    net = learn_calls(make(kind, NORM_VALUE=True, TRAINING_ITER_TIME=1), kind, 1)
    off = make(kind)
    off.load_state_dict({k: v for k, v in net.state_dict().items() if not k.startswith("value_rms.")}, strict=True)
    q = batch(kind, 64, seed=99)[0]
    got, want = net.act(q, play_mode=True), off.act(q, play_mode=True)
    ap = net.value_rms.applied32
    assert float(ap[0]) > 100.0                                     # the statistics moved away from (0, 1)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert torch.equal(got[2], want[2] * ap[2] + ap[0])              # a multiply and an add, each rounded on its own
    (_, _), vals = net((q), play_mode=True)
    assert torch.equal(vals[0].view(-1), got[2].view(-1))


@pytest.mark.parametrize("M", [1, 4])
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_act_values_are_preserved_across_the_rescale(kind, M):
    """With every learning rate 0 the only change a learn call makes is the PopArt rescale, so act's values must stay.  They
    agree up to fp32 rounding of the rescaled head and of the forward sums: a few ulps (2^-24) of the largest term
    |mean| + sigma * (|b'| + sum_j |w'_j h_j|) that is summed and cancelled; 1e-6 of it is a bound with margin."""
    net = make(kind, NORM_VALUE=True, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, LEARNING_RATE=0.0, ACTOR_LEARNING_RATE=0.0,
               CRITIC_LEARNING_RATE=0.0)
    q = batch(kind, 64, seed=98)[0]
    before = net.act(q, play_mode=True)[2].view(-1).double()
    for call, (loc, scale) in enumerate(((500.0, 80.0), (-30.0, 2.0), (1e3, 300.0))):
        list(net.learn(experience(*batch(kind, 40, seed=60 + call, loc=loc, scale=scale))))
        after = net.act(q, play_mode=True)[2].view(-1).double()
        ap = net.value_rms.applied32.double()
        head = net.critic.critic_linear
        feat = net.encode(q, tower=0 if net.prenet is not None else 1).double()
        big = ap[0].abs() + ap[2] * (head.bias.double().abs() + (feat.abs() @ head.weight.double().abs().view(-1)))
        assert torch.all((after - before).abs() <= 1e-6 * big), (call, float((after - before).abs().max()))
        before = after


# ---------------------------------------------------------------------------------------------------------- 5. state
def test_state_dict_round_trip_restores_the_exact_statistics():
    net = learn_calls(make("navlaser", NORM_VALUE=True, TRAINING_ITER_TIME=1), "navlaser", 2)
    sd = net.state_dict()
    assert [k for k in sd if k.startswith("value_rms.")] == ["value_rms.mean", "value_rms.var", "value_rms.count"]
    fresh = make("navlaser", NORM_VALUE=True)
    fresh.load_state_dict(sd, strict=True)
    q = batch("navlaser", 32, seed=5)[0]
    for x, y in zip(net.act(q, play_mode=True), fresh.act(q, play_mode=True)):
        assert torch.equal(x, y)
    assert all(torch.equal(x, y) for x, y in zip(stats(net), stats(fresh)))


def _tail_record(net, blob):
    wb, used = net._decode_wb(memoryview(blob)[len(blob) - 24:])
    assert used == 24
    return wb


@pytest.mark.parametrize("norm_obs", [False, (0, 1)])
def test_blob_gives_a_predictor_the_learner_bits(norm_obs):
    from ddrl4nav_b200._lib import DDRLError
    obs = dict(NORM_OBS=norm_obs) if norm_obs else {}
    net = learn_calls(make("navlaser", NORM_VALUE=True, TRAINING_ITER_TIME=1, **obs), "navlaser", 2)
    blob = net.model_bytes()
    before = make("navlaser", **obs)
    if norm_obs:
        learn_calls(before, "navlaser", 2)          # the same NORM_OBS records the learner wrote, in the same place
    obs_only = before.model_bytes()
    # the NORM_VALUE record comes last: >I 1 | >I 4 | {mean32, scale32, sigma32, count} fp32
    assert len(blob) - len(obs_only) == 24
    assert blob[len(obs_only):len(obs_only) + 8] == b"\x00\x00\x00\x01\x00\x00\x00\x04"
    rec = _tail_record(net, blob)
    ap = net.value_rms.applied32.cpu().numpy()
    assert rec[:3].tolist() == ap.tolist() and rec[3] == np.float32(float(net.value_rms.count))
    fresh = make("navlaser", NORM_VALUE=True, **obs)
    fresh.load_model_bytes(blob)
    assert torch.equal(fresh.value_rms.applied32, net.value_rms.applied32)
    q = batch("navlaser", 32, seed=5)[0]
    for x, y in zip(net.act(q, play_mode=True), fresh.act(q, play_mode=True)):
        assert torch.equal(x, y)
    with pytest.raises(DDRLError, match="NORM_VALUE"):
        make("navlaser", NORM_VALUE=True, **obs).load_model_bytes(obs_only)


# ---------------------------------------------------------------------------------------------------------- 6. call paths
@pytest.mark.parametrize("M", [1, 4])
def test_statistics_move_once_per_call_and_follow_the_restatement(M):
    net = make("navimg", NORM_VALUE=True, TRAINING_ITER_TIME=3, MINI_BATCH_NUM=M)
    ref = V.ValueRMS()
    for call in range(2):
        data = batch("navimg", 50, seed=30 + call)
        counts = [float(net.value_rms.count) for _ in net.learn(experience(*data))]
        ref.update(data[4][0].cpu().numpy()[:, None])
        assert counts == [counts[0]] * (3 * M)                        # merged once, at the start, before the first step
        assert counts[0] == pytest.approx(1e-4 + 50 * (call + 1), rel=1e-15)
        assert rel_close(net.value_rms.mean.cpu().numpy(), ref.mean) and rel_close(net.value_rms.var.cpu().numpy(), ref.var)


def test_target_kl_stop_moves_the_statistics_once():
    net = make("navimg", NORM_VALUE=True, TRAINING_ITER_TIME=4, TARGET_KL=1e-12)
    data = batch("navimg", 40)
    assert len(list(net.learn(experience(*data)))) == 1
    ref = V.ValueRMS()
    ref.update(data[4][0].cpu().numpy()[:, None])
    assert float(net.value_rms.count) == 1e-4 + 40
    assert rel_close(net.value_rms.mean.cpu().numpy(), ref.mean) and rel_close(net.value_rms.var.cpu().numpy(), ref.var)


@pytest.mark.parametrize("M", [1, 4])
def test_no_graph_gives_the_same_bits(deterministic, monkeypatch, M):
    data = batch("pong", 40)

    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make("pong", NORM_VALUE=True, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=2, VALUE_CLIP=0.3)
        logs = [[l[x] for x in KEYS] for call in range(3) for l, _, _ in net.learn(experience(*batch("pong", 40, seed=call)))]
        return logs, net._flat.clone(), stats(net), net.act(data[0], play_mode=True)

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])
    assert all(torch.equal(x, y) for x, y in zip(g[2], e[2]))
    assert all(torch.equal(x, y) for x, y in zip(g[3], e[3]))


# ---------------------------------------------------------------------------------------------------------- 7. full size
def test_full_size_pong():
    """Returns of 500 +- 80: raw, the value loss would be ~1.3e5.  Normalised, the first step's VLoss is the distance of the
    preserved initial outputs (~0 in reward units, so ~ -500 / 80 normalised units) from the normalised targets, ~20, which
    the float64 prediction from act's values before the call must match; every later VLoss stays in normalised units."""
    B = 8192
    data = batch("pong", B)
    R = data[4][0].double()
    raw = float(0.5 * (R ** 2).mean())
    net = make("pong", NORM_VALUE=True)
    for call in range(2):
        v0 = net.act(data[0], play_mode=True)[2].view(-1).double()
        out = list(net.learn(experience(*data)))
        assert len(out) == 10
        assert all(np.isfinite([l[x] for x in KEYS]).all() for l, _, _ in out)
        ap = net.value_rms.applied32.double()
        pred = float(0.5 * (((R - ap[0]) * ap[1] - (v0 - ap[0]) * ap[1]) ** 2).mean())
        assert out[0][0]["VLoss"] == pytest.approx(pred, rel=1e-3), (call, out[0][0]["VLoss"], pred)
        assert all(l["VLoss"] < 1e-2 * raw for l, _, _ in out), ([l["VLoss"] for l, _, _ in out], raw)
    assert torch.isfinite(net._flat).all()
    ref = V.ValueRMS()
    for _ in range(2):
        ref.update(data[4][0].cpu().numpy()[:, None])
    assert rel_close(net.value_rms.mean.cpu().numpy(), ref.mean) and rel_close(net.value_rms.var.cpu().numpy(), ref.var, 1e-9)


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
    kind, B = "navlaser", 81
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, NORM_OBS=(0, 1), NORM_VALUE=True)
    net.load_state_dict(R.init_params(R.SPECS[kind], seed=11), strict=False)
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    f64 = []
    real = tdist.all_reduce

    def counting(t, *args, **kwargs):
        if t.dtype == torch.float64:
            f64.append(t.numel())
        return real(t, *args, **kwargs)

    tdist.all_reduce = counting
    states, a, old, adv, values = batch(kind, B)
    lo, hi = (0, 41) if rank == 0 else (41, 81)
    exp = Experience(states=[s[lo:hi].to(dev) for s in states], advs=adv[lo:hi].to(dev), actions=a[lo:hi].to(dev),
                     old_logps=old[lo:hi].to(dev), values=values[:, lo:hi].to(dev))
    logs = []
    for call in range(2):
        logs += [[l[x] for x in KEYS] for l, _, _ in net.learn(exp)]
    tdist.all_reduce = real
    q.put((rank, logs, net._flat.cpu().numpy(), [t.cpu().numpy() for t in stats(net)], f64))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_replicas_are_identical_with_one_collective_per_call():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, logs, flat, st, f64 = q.get(timeout=600)
        res[r] = (logs, flat, st, f64)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (l0, f0, s0, c0), (l1, f1, s1, c1) = res[0], res[1]
    assert l0 == l1 and np.array_equal(f0, f1)
    assert all(np.array_equal(x, y) for x, y in zip(s0, s1))
    # one float64 all-reduce per learn call: the observation sums of both slots and the two value sums
    assert c0 == c1 == [2 * (960 + 5) + 2] * 2
    ref = V.ValueRMS()
    for _ in range(2):
        ref.update(batch("navlaser", 81)[4][0].cpu().numpy()[:, None])
    assert rel_close(s0[0], ref.mean) and rel_close(s0[1], ref.var) and abs(s0[2][0] - ref.count) <= 1e-12 * ref.count
