"""Invalid-action masking (ACTION_MASK) on the GPU: the masked head kernel (all-ones bits, inverse CDF on its own q, the
first-allowed fallback, play mode, rows that allow nothing), log-prob bit equality of the head, pre-pass and loss kernels, the
fused loss against the float64 restatement (tests/action_mask_ref.py) with every option, whole-net gradients against the oracle,
learn() (all-ones bits against the option off, graph replay, the mask pointer in the graph key), the Forward module with a u8
mask slot, the weight blob, and two-GPU parity."""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import action_mask_ref as M
from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")
U_TOP = 1.0 - 2.0 ** -24                     # the largest fp32 below 1


@pytest.fixture
def deterministic():
    from ddrl4nav_b200 import kernels
    was = kernels.set_deterministic(True)
    yield
    kernels.set_deterministic(was)


def _logits_u(B, A, seed):
    g = torch.Generator().manual_seed(seed)
    logits = 3 * torch.randn(B, A, generator=g)
    logits[:8] = torch.round(logits[:8])     # ties
    u = torch.rand(B, generator=g)
    u[:4] = torch.tensor([0.0, U_TOP, 0.5, 1e-7])
    return logits, u, g


# ---------------------------------------------------------------------------------------------------------- 1. head kernel
@pytest.mark.parametrize("A", [2, 6, 28, 64])
def test_head_all_ones_mask_gives_the_unmasked_bits(A):
    from ddrl4nav_b200 import kernels
    logits, u, _ = _logits_u(3000, A, A)
    ones = torch.ones(3000, A, dtype=torch.uint8, device=DEV)
    for draw in (u.to(DEV), None):
        want = kernels.categorical_head(logits.to(DEV), draw)
        got = kernels.categorical_head_m(logits.to(DEV), draw, ones)
        for w, g in zip(want, got):
            assert torch.equal(w, g)


@pytest.mark.parametrize("A", [2, 6, 28, 64])
def test_head_samples_the_masked_distribution(A):
    from ddrl4nav_b200 import kernels
    B = 3000
    logits, u, _ = _logits_u(B, A, 100 + A)
    mask = M.random_mask(B, A, seed=A, empty_rows=3)
    a, lp, q = kernels.categorical_head_m(logits.to(DEV), u.to(DEV), mask.to(DEV))
    a, lp, q = a.cpu(), lp.cpu(), q.cpu()
    eff = M.effective_mask(mask)
    assert (q[~eff] == 0).all()
    want = M.sample_on_q(q.numpy(), u.numpy(), mask)
    assert np.array_equal(a.numpy().astype(np.int64), want)
    assert bool(eff[torch.arange(B), a.long()].all())                                  # never a masked action
    ref = M.masked_probs(logits.double(), mask)
    assert torch.allclose(q.double(), ref / ref.sum(-1, keepdim=True), rtol=1e-5, atol=1e-7)
    assert torch.allclose(lp.double(), M.log_prob(logits, mask, a), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("A", [6, 28])
def test_head_falls_back_to_the_first_allowed_action(A):
    """u set to the fp32 sum of each row's own masked q: no prefix sum exceeds it, so every row takes its first allowed action
    (which is not 0 where action 0 is masked)."""
    from ddrl4nav_b200 import kernels
    B = 512
    logits, _, g = _logits_u(B, A, 7)
    mask = M.random_mask(B, A, seed=8, p_allowed=0.5)
    mask[:, 0] = 0
    mask[:, -1] = 1
    _, _, q = kernels.categorical_head_m(logits.to(DEV), torch.zeros(B, device=DEV), mask.to(DEV))
    top = np.cumsum(q.cpu().numpy(), axis=1, dtype=np.float32)[:, -1]
    a, lp, _ = kernels.categorical_head_m(logits.to(DEV), torch.from_numpy(top).to(DEV), mask.to(DEV))
    first = M.first_allowed(mask)
    assert (first > 0).all() and np.array_equal(a.cpu().numpy().astype(np.int64), first)
    assert bool(M.effective_mask(mask)[torch.arange(B), a.cpu().long()].all())
    assert torch.equal(lp, kernels.logp_actions_categorical_m(logits.to(DEV), a, mask.to(DEV)))


@pytest.mark.parametrize("A", [6, 28])
def test_head_play_mode_and_rows_that_allow_nothing(A):
    from ddrl4nav_b200 import kernels
    B = 1000
    logits, u, _ = _logits_u(B, A, 9)
    mask = M.random_mask(B, A, seed=10, empty_rows=50)
    a, lp, p = kernels.categorical_head_m(logits.to(DEV), None, mask.to(DEV))
    a, p = a.cpu(), p.cpu()
    assert (lp == 0).all()
    eff = M.effective_mask(mask)
    want = np.argmax(np.where(eff.numpy(), p.numpy(), -1.0), axis=1)                  # first max over the allowed entries
    assert np.array_equal(a.numpy().astype(np.int64), want) and bool(eff[torch.arange(B), a.long()].all())
    ones = torch.ones(50, A, dtype=torch.uint8, device=DEV)
    for draw in (u[:50].to(DEV), None):
        zero_rows = kernels.categorical_head_m(logits[:50].to(DEV), draw, mask[:50].to(DEV))
        one_rows = kernels.categorical_head_m(logits[:50].to(DEV), draw, ones)
        for z, o in zip(zero_rows, one_rows):
            assert torch.equal(z, o)


# ---------------------------------------------------------------------------------------------------------- 2. log-prob bits
@pytest.mark.parametrize("A", [2, 6, 28, 64])
def test_act_prepass_and_loss_log_probs_are_equal_bits(A):
    """The head kernel's log-prob of the action it emitted, ddrl_logp_actions_categorical_m's, and the loss kernel's (ppo_clip 0
    with old = prox = that log-prob counts any r != 1 in ClipFrac) are the same bits."""
    from ddrl4nav_b200 import kernels
    B = 2000
    logits, u, g = _logits_u(B, A, 20 + A)
    mask = M.random_mask(B, A, seed=A + 1).to(DEV)
    d = lambda t: t.to(DEV)
    a, lp_act, _ = kernels.categorical_head_m(d(logits), d(u), mask)
    assert torch.equal(lp_act, kernels.logp_actions_categorical_m(d(logits), a, mask))
    v, ret, adv = (torch.randn(B, generator=g).to(DEV) for _ in range(3))
    hp = kernels.make_hparams(ppo_clip=0.0, ppo_stats=True)
    _, _, sums = kernels.ppo_loss_categorical_m(d(logits), a, lp_act, adv, ret, v, hp, True, mask=mask)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0
    _, _, sums = kernels.ppo_loss_categorical_m(d(logits), a, lp_act - 0.3, adv, ret, v, hp, True, mask=mask, prox_logp=lp_act)
    assert sums[3].item() == 0.0 and sums[4].item() == 0.0


# ---------------------------------------------------------------------------------------------------------- 3. loss kernel
OPTIONS = ["none", "dual_clip", "VALUE_CLIP", "value_norm", "prox", "prox_is_clip", "all"]


@pytest.mark.parametrize("opt", OPTIONS)
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("A", [6, 28])
def test_loss_kernel_matches_the_restatement(A, shared, opt):
    from ddrl4nav_b200 import kernels
    B = 777
    logits, _, g = _logits_u(B, A, A + 10 * shared + 100 * OPTIONS.index(opt))
    logits = logits.double() / 2
    mask = M.random_mask(B, A, seed=A + 3)
    eff = M.effective_mask(mask)
    a = torch.multinomial(M.masked_probs(logits, mask), 1, generator=g).squeeze(-1).float()
    for r in [r for r in range(B) if not eff[r].all()][:4]:                           # corrupt rows: a masked taken action
        a[r] = float(torch.nonzero(~eff[r])[0])
    lp = M.log_prob(logits, mask, a)
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
    d = lambda t: t.to(DEV)
    dl, dv, sums = kernels.ppo_loss_categorical_m(d(logits.float()), d(a), d(old), d(adv), d(ret), d(v), hp, shared,
                                                  mask=d(mask), **kw)
    ref, rdl, rdv = M.loss_and_grads(logits.float(), mask, a, old, adv, ret, v, hyper, shared, **ref_kw)
    s = sums.cpu().double().tolist()
    for i, k in enumerate(("actor", "v", "entropy", "ApproxKL")):
        assert s[i] == pytest.approx(ref[k], rel=1e-5, abs=1e-7), k
    assert s[4] == pytest.approx(ref["ClipFrac"], abs=2.0 / B)
    if "prox" in ref_kw:
        assert s[5] == pytest.approx(ref["BehaviourKL"], rel=2e-5)
    for got, want in ((dl, rdl), (dv, rdv)):
        got = got.cpu().double()
        assert torch.allclose(got, want, rtol=0, atol=1e-5 * float(want.abs().max())), float((got - want).abs().max())
    assert (dl.cpu()[~eff] == 0).all()


# ---------------------------------------------------------------------------------------------------------- 4. whole net
def make(kind, seed=11, **hyper):
    from ddrl4nav_b200.runner import make_net
    net = make_net(kind, device=None, **hyper)
    net.load_state_dict(R.init_params(R.SPECS[kind], seed=seed), strict=False)
    return net.to(DEV)


def batch(kind, B, seed=9, net=None, mask=None):
    """(states + [mask], actions, old log-probs, advantages, values [1, B]) on the device; actions sampled by `net` (or a masked
    seed-11 net), old log-probs its log-probs plus N(0, 0.15) noise.  mask: u8 [B, A], random by default."""
    g = torch.Generator().manual_seed(seed)
    A = R.SPECS[kind].act_dim
    states = [s.to(DEV) for s in R.synth_states(kind, B, seed=seed)]
    mask = (M.random_mask(B, A, seed=seed + 1) if mask is None else mask).to(DEV)
    net = net or make(kind, ACTION_MASK=True)
    u = torch.rand(B, generator=g).to(DEV)
    a, lp, _ = net.act(states + [mask], draw=u)
    old = lp + 0.15 * torch.randn(B, generator=g).to(DEV)
    adv, ret = torch.randn(B, generator=g).to(DEV), torch.randn(B, generator=g).to(DEV)
    return states + [mask.float()], a, old, adv, ret[None]


def experience(states, a, old, adv, values):
    from ddrl4nav_b200.data import Experience
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=values)


@pytest.mark.parametrize("kind,B", [("pong", 5), ("navimg", 6), ("navped", 4), ("navimg", 33)])
def test_net_gradients_match_the_oracle(kind, B):
    net = make(kind, ACTION_MASK=True)
    states, a, old, adv, values = batch(kind, B, net=net)
    assert bool(M.effective_mask(states[-1].cpu())[torch.arange(B), a.cpu().long()].all())
    net.backward_only(states, adv, a, old, values)
    grads = {n: g.detach().cpu().double() for n, g in net.named_grads().items()}
    losses, raw = M.net_grads(kind, R.init_params(R.SPECS[kind], seed=11), [s.cpu() for s in states[:-1]], states[-1].cpu(),
                              a.cpu(), old.cpu(), adv.cpu(), values[0].cpu())
    for n in raw:
        err = float((grads[n] - raw[n]).abs().max())
        assert err <= 2e-5 * float(raw[n].abs().max()), (n, err)
    sums = net._grads[net._P:net._P + 3].cpu().numpy()
    assert np.allclose(sums, [losses["ActorLoss"], losses["VLoss"], losses["EntLoss"]], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------- 5. learn()
@pytest.mark.parametrize("opts", [dict(), dict(MINI_BATCH_NUM=4, MINI_BATCH_SEED=3), dict(DECOUPLED_PPO=True, PPO_STATS=True)])
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_all_ones_mask_learns_the_option_off_bits(deterministic, kind, opts):
    B = 48
    A = R.SPECS[kind].act_dim
    states, a, old, adv, values = batch(kind, B, mask=torch.ones(B, A, dtype=torch.uint8))
    on = make(kind, ACTION_MASK=True, TRAINING_ITER_TIME=3, **opts)
    off = make(kind, TRAINING_ITER_TIME=3, **opts)
    assert torch.equal(on.act(states, draw=torch.full((B,), 0.4, device=DEV))[1],
                       off.act(states[:-1], draw=torch.full((B,), 0.4, device=DEV))[1])
    keys = KEYS + (("ApproxKL", "ClipFrac", "BehaviourKL") if opts.get("PPO_STATS") else ())
    lo = [[l[k] for k in keys] for l, _, _ in on.learn(experience(states, a, old, adv, values))]
    lf = [[l[k] for k in keys] for l, _, _ in off.learn(experience(states[:-1], a, old, adv, values))]
    assert lo == lf and torch.equal(on._flat, off._flat)


@pytest.mark.parametrize("M_", [1, 4])
def test_learn_with_every_option(M_):
    net = make("navimg", ACTION_MASK=True, MINI_BATCH_NUM=M_, MINI_BATCH_SEED=1, NORM_ADV=True, VALUE_CLIP=0.2, PPO_STATS=True,
               TARGET_KL=10.0, NORM_OBS=True, NORM_VALUE=True, DECOUPLED_PPO=True, DECOUPLED_IS_CLIP=2.0, DUEL_PPO_CLIP=2.0)
    states, a, old, adv, values = batch("navimg", 96)
    net._ensure_engine()
    assert net.obs_rms.slots == (0, 1)                          # NORM_OBS=True leaves the mask slot out
    before = net._flat.clone()
    logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, values))]
    assert len(logs) == 10 * M_ and logs[0]["ApproxKL"] == 0.0
    assert all(np.isfinite([l[k] for k in KEYS + ("ApproxKL", "ClipFrac", "BehaviourKL")]).all() for l in logs)
    assert not torch.equal(before, net._flat) and torch.isfinite(net._flat).all()
    a2, lp2, _ = net.act(states, draw=torch.rand(96, device=DEV))
    assert bool(M.effective_mask(states[-1].cpu())[torch.arange(96), a2.cpu().long()].all()) and torch.isfinite(lp2).all()


def test_extra_critics_with_the_mask():
    from ddrl4nav_b200.nn import Critic
    net = make("navimg", ACTION_MASK=True, TRAINING_ITER_TIME=2, VALUE_CLIP=0.2, DECOUPLED_PPO=True, MINI_BATCH_NUM=2)
    for _ in range(2):
        net.add_critic(Critic(device=DEV, last_input_dim=512).to(DEV))
    net.gail_critic = True
    states, a, old, adv, values = batch("navimg", 64)
    v3 = torch.cat([values, values * 0.5, values * 2], 0)
    logs = [l for l, _, _ in net.learn(experience(states, a, old, adv, v3))]
    assert len(logs) == 4 and all(np.isfinite([l[k] for k in KEYS]).all() for l in logs)
    assert net.act(states)[2].shape == (3, 64, 1)


@pytest.mark.parametrize("M_", [1, 4])
def test_graph_replay_equals_stream_launches(deterministic, monkeypatch, M_):
    """Two learn calls on the same tensors, the mask contents rewritten in place (same address) between them: the graphs read
    the new mask when they replay."""
    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make("navimg", ACTION_MASK=True, TRAINING_ITER_TIME=3, MINI_BATCH_NUM=M_, MINI_BATCH_SEED=2, PPO_STATS=True,
                   DECOUPLED_PPO=True)
        states, a, old, adv, values = batch("navimg", 40)
        logs = [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac")] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        states[-1].copy_(M.random_mask(40, 28, seed=77).to(DEV))
        logs += [[l[k] for k in KEYS + ("ApproxKL", "ClipFrac")] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        return logs, net._flat.clone()

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])


def test_graph_key_holds_the_mask_pointer(deterministic, monkeypatch):
    """navped reads its mask from obs[3], beyond the three encoder slots: a mask at a new address with every other pointer
    unchanged must not replay the graph captured on the old one."""
    def run(no_graph):
        if no_graph:
            monkeypatch.setenv("DDRL_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("DDRL_NO_GRAPH", raising=False)
        net = make("navped", ACTION_MASK=True, TRAINING_ITER_TIME=3)
        states, a, old, adv, values = batch("navped", 24)
        logs = [[l[k] for k in KEYS] for l, _, _ in net.learn(experience(states, a, old, adv, values))]
        other = M.random_mask(24, 28, seed=123, p_allowed=0.3).to(DEV).float()          # new address; the old mask stays alive
        assert other.data_ptr() != states[-1].data_ptr()
        logs += [[l[k] for k in KEYS] for l, _, _ in net.learn(experience(states[:-1] + [other], a, old, adv, values))]
        return logs, net._flat.clone()

    g, e = run(False), run(True)
    assert g[0] == e[0] and torch.equal(g[1], e[1])


# ---------------------------------------------------------------------------------------------------------- 6. Forward module
def test_forward_module_with_a_u8_mask_slot():
    from ddrl4nav_b200.server import ForwardModule, encode_forward_replies
    net = make("navimg", ACTION_MASK=True)
    B_env, n_env = 60, 10
    B = B_env * n_env
    states = [s.numpy() for s in R.synth_states("navimg", B, seed=4)]
    mask = M.random_mask(B, 28, seed=5, p_allowed=0.3).numpy()
    mask[:, 0] = 0
    host = states + [mask]
    draw = torch.rand(B, generator=torch.Generator().manual_seed(6)).to(DEV)
    a, lp, v = net.act([torch.from_numpy(s).float().to(DEV) for s in host], draw=draw)
    assert bool(M.effective_mask(torch.from_numpy(mask))[torch.arange(B), a.cpu().long()].all())
    want = [a.cpu().numpy(), lp.cpu().numpy(), v.cpu().numpy()]
    payload = b"".join(R.easybytes_encode_forward_states("10.1.2.3", 100 + j, [s[j * B_env:(j + 1) * B_env] for s in host])
                       for j in range(n_env))
    for chunk in (96 << 20, 1 << 20):                            # one call, and streamed in chunks
        fm = ForwardModule(net, device=DEV, chunk_bytes=chunk)
        got = fm.step(host, draw=draw)
        assert all(np.array_equal(x, y.reshape(x.shape)) for x, y in zip(got, want))
        ids, g2 = fm.step_bytes(payload, draw=draw)
        assert all(np.array_equal(x, y.reshape(x.shape)) for x, y in zip(g2, want))
        _, replies = fm.step_bytes_replies(payload, B_env, draw=draw)
        assert replies == encode_forward_replies(want, [B_env] * n_env)
    # forward(): the Categorical gives masked actions probability 0
    (pi, log_p), _ = net.forward([torch.from_numpy(s).to(DEV) for s in host], act=a)
    eff = M.effective_mask(torch.from_numpy(mask)).to(DEV)
    assert (pi.probs[~eff] == 0).all() and torch.allclose(log_p, lp, rtol=1e-4, atol=1e-4)
    assert bool(eff.gather(1, torch.multinomial(pi.probs, 1)).all())


def test_weight_blob_and_predictor():
    from oracle.ref_shim import _FakeRedis
    from ddrl4nav_b200.runner import make_net
    net, plain = make("navped", ACTION_MASK=True), make("navped")
    assert list(net.state_dict()) == list(plain.state_dict()) and net.model_bytes() == plain.model_bytes()
    mid = _FakeRedis()
    net.nn2redis(mid.pipeline(), "upd")
    pred = make_net("navped", device=DEV, ACTION_MASK=True)
    pred.updatenn_by_redis(mid, net.model_key)
    states, *_ = batch("navped", 16, net=net)
    draw = torch.rand(16, device=DEV)
    for x, y in zip(net.act(states, draw=draw), pred.act(states, draw=draw)):
        assert torch.equal(x, y)


def test_engine_refuses_the_switch_after_a_pass():
    from ddrl4nav_b200 import _lib
    net = make("navimg", ACTION_MASK=True)
    states, *_ = batch("navimg", 4, net=net)
    assert _lib.load().ddrl_net_set_action_mask(net._h, 0) == -3          # DDRL_E_STATE


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
    kind, B = "navimg", 81
    net = make_net(kind, device=None, TRAINING_ITER_TIME=2, PPO_STATS=True, DECOUPLED_PPO=True, ACTION_MASK=True)
    net.load_state_dict(R.init_params(R.SPECS[kind], seed=11))
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
