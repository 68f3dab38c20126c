"""Minibatch PPO epochs (MINI_BATCH_NUM = M > 1) on the GPU: the multi-tensor row gather kernel, the minibatch backward
entry point with its graph replay, and the learner built on them.  A minibatch step must be exactly the full-batch step of
the default path on the same rows (deterministic mode, bit for bit); the gradient of a minibatch must match the oracle."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")


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


def experience(states, a, old, adv, values, rows=None):
    from ddrl4nav_b200.data import Experience
    if rows is not None:
        r = rows.long()
        states = [s.index_select(0, r) for s in states]
        a, old, adv, values = a.index_select(0, r), old.index_select(0, r), adv.index_select(0, r), values.index_select(1, r)
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values)


# ---------------------------------------------------------------------------------------------------------- gather kernel
def test_gather_rows_equals_index_select():
    from ddrl4nav_b200 import kernels
    g = torch.Generator(device=DEV).manual_seed(3)
    for n_rows in (0, 1, 7, 8192):
        S = 300
        rows = torch.randint(0, S, (n_rows,), generator=g, device=DEV, dtype=torch.int32)
        if n_rows > 2:
            rows[1] = rows[0]                                 # repeated indices
        pairs, refs = [], []
        for width_bytes in (4, 20, 36, 9216, 112896):
            w = width_bytes // 4
            src = torch.randn(S, w, generator=g, device=DEV)
            dst = torch.full((max(n_rows, 1) + 3, w), -1.0, device=DEV)
            pairs.append((src, dst))
            refs.append(src.index_select(0, rows.long()))
        # 4-byte path: bases 4 bytes off a 16-byte boundary, odd strides (views into wider buffers)
        big = torch.randn(S + 1, 37, generator=g, device=DEV)
        dbig = torch.zeros(max(n_rows, 1), 41, device=DEV)
        pairs.append((big[1:, 1:33], dbig[:, 3:35]))
        refs.append(big[1:, 1:33].index_select(0, rows.long()))
        # int32 / byte payloads with 4-byte multiples
        ints = torch.randint(-2 ** 31, 2 ** 31 - 1, (S, 3), generator=g, device=DEV, dtype=torch.int32)
        dints = torch.zeros(max(n_rows, 1), 3, dtype=torch.int32, device=DEV)
        pairs.append((ints, dints))
        refs.append(ints.index_select(0, rows.long()))
        assert len(pairs) == 7
        kernels.launch_count_reset()
        kernels.gather_rows(rows, pairs)
        assert kernels.launch_count() == (1 if n_rows else 0)
        for (src, dst), ref in zip(pairs, refs):
            assert torch.equal(dst[:n_rows], ref), (n_rows, tuple(src.shape))
        if n_rows:
            assert float(pairs[0][1][n_rows:].max()) == -1.0         # rows past n_rows untouched


def test_gather_rows_clamps_out_of_range_indices():
    from ddrl4nav_b200 import kernels
    src = torch.arange(5 * 8, dtype=torch.float32, device=DEV).view(5, 8)
    dst = torch.zeros(4, 8, device=DEV)
    kernels.gather_rows(torch.tensor([-7, 4, 5, 1 << 30], dtype=torch.int32, device=DEV), [(src, dst)])
    assert torch.equal(dst, src[[0, 4, 4, 4]])


def test_gather_rows_rejects_bad_arguments():
    from ddrl4nav_b200 import _lib
    from ddrl4nav_b200._lib import GatherJob, current_stream
    lib = _lib.load()
    src = torch.zeros(8, 16, device=DEV)
    dst = torch.zeros(8, 16, device=DEV)
    rows = torch.zeros(4, dtype=torch.int32, device=DEV)
    good = lambda **kw: GatherJob(**{**dict(src=src.data_ptr(), dst=dst.data_ptr(), row_bytes=64, src_stride=64,
                                            dst_stride=64, src_rows=8), **kw})
    run = lambda jobs, n=4, r=rows.data_ptr(): lib.ddrl_gather_rows(r, n, (GatherJob * max(len(jobs), 1))(*jobs),
                                                                     len(jobs), current_stream())
    assert run([good()]) == 0
    E = -1
    assert run([good(src=None)]) == E
    assert run([good(dst=None)]) == E
    assert run([good(row_bytes=62)]) == E
    assert run([good(row_bytes=0)]) == E
    assert run([good(src_stride=66)]) == E
    assert run([good(src=src.data_ptr() + 2)]) == E
    assert run([good(src_rows=0)]) == E
    assert run([]) == E
    assert run([good()] * 13) == E
    assert run([good()] * 12) == 0
    assert run([good()], r=None) == E
    assert run([good()], n=-1) == E
    assert lib.ddrl_gather_rows(rows.data_ptr(), 4, None, 1, current_stream()) == E
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------- learner
def _stepwise_against_full_batch(kind, B, M, iters, extra=None):
    """Net A learns with M minibatches; net B (same weights) takes one default full-batch step per chunk of A's
    permutations.  Every step: same parameters and losses, bit for bit."""
    from ddrl4nav_b200.runner import make_net
    states, a, old, adv, values = batch(kind, B)
    netA = make(kind, MINI_BATCH_NUM=M, TRAINING_ITER_TIME=iters, MINI_BATCH_SEED=5)
    netB = make(kind, TRAINING_ITER_TIME=1)
    extras = []
    if extra:
        spec = R.SPECS[kind]
        ret2, extra_params = R.synth_extra_critic(R.init_params(spec, seed=11), values[0].cpu())
        values = ret2.to(DEV)
        for net in (netA, netB):
            c = make_net(kind, device=None).critic
            c.load_state_dict(extra_params, strict=True)
            c = c.to(DEV)
            net.add_critic(c)
            net.gail_critic = True
            extras.append(c)
    plan = netA.minibatch_plan(B, M)
    n = 0
    for (la, upd, last), in zip(netA.learn(experience(states, a, old, adv, values))):
        epoch, k = divmod(n, M)
        lo, hi = plan[k]
        rows = netA.last_minibatch_perms[epoch][lo:hi]
        (lb, _, _), = list(netB.learn(experience(states, a, old, adv, values, rows)))
        n += 1
        assert upd == n and last is True and set(la) == set(KEYS) | {"PpoBackUpTime"}
        assert [la[x] for x in KEYS] == [lb[x] for x in KEYS], (kind, n, la, lb)
        assert torch.equal(netA._flat, netB._flat), (kind, n, rel_err(netA._flat, netB._flat))
        for ca, cb in zip(extras[:1], extras[1:]):
            for pa, pb in zip(ca.parameters(), cb.parameters()):
                assert torch.equal(pa.grad, pb.grad), (kind, n)
    assert n == iters * M and netA.update_time == n
    perms = netA.last_minibatch_perms
    assert len(perms) == iters and all(p.dtype == torch.int32 and p.is_cuda for p in perms)
    for p in perms:
        assert torch.equal(torch.sort(p.long()).values.cpu(), torch.arange(B))
    return netA


@pytest.mark.parametrize("kind", ["pong", "navimg", "navlaser"])
def test_minibatch_step_equals_full_batch_step_on_its_rows(deterministic, kind):
    net = _stepwise_against_full_batch(kind, 40, 3, 2)
    assert net._mb["states"][0].shape[0] == 14


@pytest.mark.parametrize("kind", ["navimg", "pong"])
def test_minibatch_with_added_gail_critic(deterministic, kind):
    _stepwise_against_full_batch(kind, 40, 2, 2, extra=True)


@pytest.mark.parametrize("kind", ["pong", "navimg", "navlaser"])
def test_minibatch_graph_replay_equals_stream_launches(deterministic, monkeypatch, kind):
    from ddrl4nav_b200 import kernels
    states, a, old, adv, values = batch(kind, 40)

    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make(kind, MINI_BATCH_NUM=3, TRAINING_ITER_TIME=2, MINI_BATCH_SEED=1)
        kernels.launch_count_reset()
        losses = [[l[x] for x in KEYS] for _ in range(2) for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        return losses, net._flat.clone(), net._m.clone(), kernels.launch_count()

    l_graph, p_graph, m_graph, n_graph = run(False)
    l_eager, p_eager, m_eager, n_eager = run(True)
    assert l_graph == l_eager
    assert torch.equal(p_graph, p_eager) and torch.equal(m_graph, m_eager)
    # 12 minibatch passes with chunk sizes 14 / 13 / 13: the first pass of each size runs on the stream, the other 10 replay
    # a graph.  Replayed kernel nodes count like stream launches; a replayed backward is a chain of segments, each ending
    # with the un-permutation of its own layers' gradients (towers - 0 extra launches per pass vs the stream's single one)
    towers = 1 if R.SPECS[kind].shared else 2
    assert n_graph == n_eager + towers * 10, (n_graph, n_eager)


def test_first_minibatch_gradient_matches_oracle():
    kind, B = "pong", 40
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=11)
    states, a, old, adv, values = batch(kind, B)
    net = make(kind, MINI_BATCH_NUM=3, TRAINING_ITER_TIME=1, MINI_BATCH_SEED=2)
    next(net.learn(experience(states, a, old, adv, values)))
    rows = net.last_minibatch_perms[0][:14].long().cpu()
    st = R.LearnState(spec, params)
    losses, raw, _ = R.learn_iteration(st, [s.cpu()[rows] for s in states], adv.cpu()[rows], a.cpu()[rows], old.cpu()[rows],
                                       values[0].cpu()[rows], R.PPOHyper(), apply_update=False)
    ours = net.named_grads()
    worst = max(rel_err(ours[n], raw[n]) for n in raw)
    assert worst < 2e-5, worst
    # the loss sums of the step are over the chunk's 14 rows, scaled by 1/14
    sums = net._grads[net._P:net._P + 3].cpu().numpy()
    assert np.allclose(sums, [losses["ActorLoss"], losses["VLoss"], losses["EntLoss"]], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_one_minibatch_is_the_default_path(deterministic, kind):
    from ddrl4nav_b200 import kernels
    states, a, old, adv, values = batch(kind, 24)
    out = []
    for hyper in ({}, {"MINI_BATCH_NUM": 1}):
        net = make(kind, TRAINING_ITER_TIME=3, **hyper)
        kernels.launch_count_reset()
        losses = [[l[x] for x in KEYS] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        out.append((losses, net._flat.clone(), kernels.launch_count(), net._mb, net.last_minibatch_perms))
    assert out[0][0] == out[1][0] and torch.equal(out[0][1], out[1][1])
    assert out[0][2] == out[1][2]
    assert out[1][3] is None and out[1][4] == []


def test_micro_batched_minibatch_equals_single_shot(monkeypatch):
    states, a, old, adv, values = batch("pong", 40)
    grads = []
    for env in (None, "4"):
        if env:
            monkeypatch.setenv("DDRL_MICRO_BATCH", env)
        net = make("pong", MINI_BATCH_NUM=3, TRAINING_ITER_TIME=1, MINI_BATCH_SEED=4)
        steps = net.learn(experience(states, a, old, adv, values))
        next(steps)
        grads.append(net.flat_grads().clone())
        list(steps)                                           # the remaining (micro-batched) steps run too
    assert net._h is not None
    assert rel_err(grads[1], grads[0]) < 5e-6


def test_full_size_pong_minibatch_learn():
    B, M = 8192, 4
    states, a, old, adv, values = batch("pong", B)
    net = make("pong", MINI_BATCH_NUM=M)
    out = list(net.learn(experience(states, a, old, adv, values)))
    assert len(out) == 10 * M and [u for _, u, _ in out] == list(range(1, 10 * M + 1))
    assert all(np.isfinite([l[x] for x in KEYS]).all() for l, _, _ in out)
    assert all(set(l) == set(KEYS) | {"PpoBackUpTime"} and last is True for l, _, last in out)
    assert [t.shape[0] for t in net._mb["states"]] == [B // M] and net._mb["values"].numel() == B // M
    assert torch.isfinite(net._flat).all()


# ---------------------------------------------------------------------------------------------------------- two ranks
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
    kind, B, M = "pong", 81, 3
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=3)
    states = R.synth_states(kind, B, seed=4)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=5)
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, MINI_BATCH_NUM=M, MINI_BATCH_SEED=10 + rank)
    net.load_state_dict(params)
    net = net.to(dev)
    net.enable_data_parallel()
    net.broadcast_parameters(0)
    lo, hi = (0, 41) if rank == 0 else (41, 81)               # unequal shards: 41 / 40 rows
    exp = Experience(states=[s[lo:hi].to(dev) for s in states], advs=adv[lo:hi].to(dev), actions=a[lo:hi].to(dev),
                     old_logps=old[lo:hi].to(dev), values=ret[lo:hi].to(dev)[None])
    snaps, logs, rows = [], [], []
    plan = net.minibatch_plan(hi - lo, M)
    for n, (l, _, _) in enumerate(net.learn(exp)):
        e, k = divmod(n, M)
        rows.append((net.last_minibatch_perms[e][plan[k][0]:plan[k][1]].long().cpu() + lo).numpy())
        snaps.append(net._flat.detach().cpu().numpy())
        logs.append([l[x] for x in KEYS])
    q.put((rank, rows, snaps, logs))
    tdist.barrier()
    tdist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_minibatch_steps_equal_single_gpu_steps_on_the_union():
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
    for s0, s1 in zip(snaps0, snaps1):
        assert np.array_equal(s0, s1)                         # replicas bit-identical after every step
    # single GPU: one default step per global minibatch (the union of both ranks' chunk-k rows)
    kind = "pong"
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=3)
    states = R.synth_states(kind, 81, seed=4)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=5)
    ref = make(kind, seed=3, TRAINING_ITER_TIME=1)
    for n, (r0, r1) in enumerate(zip(rows0, rows1)):
        assert len(r0) == (14, 14, 13)[n % 3] and len(r1) == (14, 13, 13)[n % 3]
        r = torch.from_numpy(np.concatenate([r0, r1]))
        exp = Experience(states=[s[r].to(DEV) for s in states], advs=adv[r].to(DEV), actions=a[r].to(DEV),
                         old_logps=old[r].to(DEV), values=ret[r].to(DEV)[None])
        (l, _, _), = list(ref.learn(exp))
        # every step starts from the replicas' parameters (copied into ref below): the data-parallel tolerance of one step
        for x, want in zip(KEYS, logs0[n]):
            assert abs(l[x] - want) <= 2e-5 * max(1.0, abs(l[x])), (n, x, want, l[x])
        d = np.abs(snaps0[n] - ref._flat.cpu().numpy())
        assert (d > 3e-4).mean() < 1e-3, n                    # Adam step-1 sign flips on noise-level grads only
        ref._flat.copy_(torch.from_numpy(snaps0[n]).to(DEV))
        ref._weights_changed()
