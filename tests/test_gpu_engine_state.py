"""The engine after parameter updates.  The engine never computes from the parameters directly: after every Adam step, weight
load or out-of-band edit it rebuilds derived copies of them (K-major repacks, space-to-depth packs, data-gradient class packs,
the fused first conv's bias copy, tf32 / fp16 splits and their transposed twins, weight amax slots), from step 2 on inside the
captured optimiser graph; and it keeps other state across calls (staged observations and their amax slots, graphs keyed on
pointers, a workspace that may regrow).  A stale copy is present on both sides of a self-consistency check and moves a
gradient by ~1e-3 only, so the learner is held against three references instead:

  1. a fresh twin: a net of the same kind built from the learner's state_dict, which prepares everything from scratch --
     act() bit-equal; backward_only() bit-equal on tc3 in deterministic mode, within 5e-6 of each tensor's max elsewhere;
  2. the float64 oracle at the learner's current parameters (engine_state_ref.grads_match_oracle: 2e-5 of each tensor's max,
     activation ties explained exactly);
  3. a float64 clip + Adam step from the engine's own p, m, v and raw gradient at every yield of learn()
     (engine_state_ref.clip_adam_step), with the engine's step number.
Batches stay at B <= 40 so that the oracle runs in seconds."""
import copy
from types import SimpleNamespace

import pytest
import torch

import action_mask_ref as AM
import beta_ref as BR
import engine_state_ref as ES
import multi_discrete_ref as MD
import value_norm_ref as VN
from oracle import restate as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")
ENGINES = ["simt", "tc", "tc2", "tc3"]
TWIN_BOUND = 5e-6        # engine vs engine, non-deterministic split-K order: the graph-replay test's run-to-run bound, per tensor
BASE = {"navimg_md": "navimg", "navlaser_beta": "navlaser"}        # kinds whose observations are those of another kind
MD_SPEC = R.NetSpec("nav", 1, 11, "multi_categorical", True)       # navimg_md: 4 x 7 branches on the shared nav encoder


@pytest.fixture
def deterministic():
    from ddrl4nav_b200 import kernels
    was = kernels.set_deterministic(True)
    yield
    kernels.set_deterministic(was)


def make(kind, engine, seed=11, **hyper):
    from ddrl4nav_b200.runner import make_net
    torch.manual_seed(seed)                 # the option kinds keep make_net's default init
    net = make_net(kind, device=None, gemm_mode=engine, **hyper)
    if kind in R.SPECS:
        missing, unexpected = net.load_state_dict(R.init_params(R.SPECS[kind], seed=seed), strict=False)
        assert not unexpected and all(k.startswith(("obs_rms.", "value_rms.")) for k in missing), (missing, unexpected)
    return net.to(DEV)


def batch(net, kind, B, seed, scale=1.0, mask=None):
    """(states, actions, old log-probs, advantages, returns [1, B]) on the device: the observations of R.synth_states (times
    `scale`), actions drawn by the net itself, old = logp + N(0, 0.15), adv and returns N(0, 1).  mask: ACTION_MASK's slot."""
    states = [s.to(DEV) * scale for s in R.synth_states(BASE.get(kind, kind), B, seed=seed)]
    if mask is not None:
        states.append(mask.to(DEV, torch.float32))
    torch.manual_seed(seed)
    a, lp, _ = net.act(states)
    g = torch.Generator(device=DEV).manual_seed(seed)
    old = lp + 0.15 * torch.randn(B, device=DEV, generator=g)
    return states, a.clone(), old, torch.randn(B, device=DEV, generator=g), torch.randn(1, B, device=DEV, generator=g)


def experience(bt):
    from ddrl4nav_b200.data import Experience
    states, a, old, adv, ret = bt
    return Experience(states=list(states), advs=adv, actions=a, old_logps=old, values=ret)


def params_of(net):
    return {n: p.detach().cpu().clone() for n, p in net.named_parameters()}


def learn_checked(net, bt, adam=True, on_first=None):
    """Runs net.learn over the batch.  adam: reference 3 at every yield -- one float64 clip + Adam step from p, m, v before the
    step and the raw gradient still in the gradient buffer, at the engine's step number.  on_first(grads, params before the
    call): called at the first yield.  Returns the loss rows."""
    net._ensure_engine()
    names = [n for n, _ in net.named_parameters()]
    lr = ES.element_lrs(SimpleNamespace(shared=net.prenet is not None), names, [p.numel() for _, p in net.named_parameters()])
    p, m, v = net._flat.clone(), net._m.clone(), net._v.clone()
    before = params_of(net)
    out = []
    for i, (log, _, _) in enumerate(net.learn(experience(bt))):
        out.append([log[k] for k in KEYS])
        if adam:
            ref = ES.clip_adam_step(p, net._grads[:net._P], m, v, net._adam_step, lr)
            bad = ES.adam_mismatch(p, (net._flat, net._m, net._v), ref[:3])
            assert not bad, ("Adam step", net._adam_step, bad)
        if i == 0 and on_first is not None:
            on_first(net.named_grads(), before)
        p, m, v = net._flat.clone(), net._m.clone(), net._v.clone()
    return out


def twin_of(net, kind, engine, **hyper):
    """Reference 1: a fresh net of the same kind, engine and options holding the learner's state (parameters, statistics) and
    copies of its extra critics."""
    from ddrl4nav_b200.runner import make_net
    twin = make_net(kind, device=None, gemm_mode=engine, **hyper)
    twin.load_state_dict(net.state_dict(), strict=True)
    twin = twin.to(DEV)
    for c in net._critics[1:]:
        twin.add_critic(copy.deepcopy(c))
    twin.gail_critic = net.gail_critic
    return twin


def check_twin(net, twin, bt, exact, label):
    """act (play mode) bit-equal; backward_only on `bt` bit-equal (exact) or within TWIN_BOUND of each tensor's max.  The twin
    first runs one backward on the rows, so that both take the training lowering.  Returns the worst relative difference."""
    states, a, old, adv, ret = bt
    twin.backward_only(states, adv, a, old, ret)
    x = net.act(states, play_mode=True, want_pi=True)
    y = twin.act(states, play_mode=True, want_pi=True)
    for what, u, w in zip(("actions", "logps", "values", "pi"), x, y):
        if exact:
            assert torch.equal(u, w), (label, what, float((u - w).abs().max()))
        elif what == "actions":                    # a greedy action may flip on a near-tie of two probabilities
            assert (u != w).float().mean() <= 1.0 / u.shape[0], (label, what)
        else:                                      # split-K forward launches: not bit-reproducible run to run
            assert float((u - w).abs().max()) <= TWIN_BOUND * max(float(w.abs().max()), 1e-30), (label, what)
    extra = lambda m: [p for c in m._critics[1:] for p in c.parameters()]
    for p in extra(net) + extra(twin):
        p.grad = None                              # the extra critics' gradients accumulate in .grad: take this pass alone
    net.backward_only(states, adv, a, old, ret)
    gn = net._grads.clone()
    twin.backward_only(states, adv, a, old, ret)
    gt = twin._grads.clone()
    for p, q in zip(extra(net), extra(twin)):
        assert (p.grad is None) == (q.grad is None), label
        if p.grad is not None:
            if exact:
                assert torch.equal(p.grad, q.grad), (label, "extra critic")
            else:
                assert float((p.grad - q.grad).abs().max()) < TWIN_BOUND * max(float(q.grad.abs().max()), 1e-30), label
    P = net._P
    worst = 0.0
    for (n, p), o in zip(net.named_parameters(), net._offsets):
        u, w = gn[o:o + p.numel()], gt[o:o + p.numel()]
        if exact:
            assert torch.equal(u, w), (label, n, int((u != w).sum()), float((u - w).abs().max()), float(w.abs().max()))
        else:
            err = float((u - w).abs().max()) / max(float(w.abs().max()), 1e-30)
            worst = max(worst, err)
            assert err < TWIN_BOUND, (label, n, err)
    if exact:
        assert torch.equal(gn[P:], gt[P:]), (label, "loss sums", gn[P:P + 3], gt[P:P + 3])
    else:
        assert torch.allclose(gn[P:P + 3], gt[P:P + 3], rtol=1e-5, atol=1e-7), (label, gn[P:P + 3], gt[P:P + 3])
    return worst


def check_oracle(net, kind, bt, label, params=None, grads=None, mask=None):
    """Reference 2: the float64 oracle at the learner's current parameters (or `params`, with the engine gradients `grads`)
    on the batch `bt`.  ACTION_MASK: the masked restatement (mask: the slot's u8 rows); NORM_VALUE: critic 0 learns the
    targets normalised with the applied statistics.  Returns the worst error / max|g|."""
    states, a, old, adv, ret = bt
    if grads is None:
        net.backward_only(states, adv, a, old, ret)
        grads = net.named_grads()
    params = params or params_of(net)
    cpu = lambda t: t.detach().cpu()
    st, a, old, adv, ret = [cpu(s) for s in states], cpu(a), cpu(old).double(), cpu(adv).double(), cpu(ret)[0].double()
    if net.value_rms is not None:
        ret = VN.normalize(ret.float(), net.value_rms.applied32.cpu()).double()
    if kind in R.SPECS and mask is None:
        oracle = ES.learn_oracle(R.SPECS[kind], params, st, adv, a, old, ret)
    else:
        if kind == "navlaser_beta":
            low, high = (torch.tensor(x, dtype=torch.float64) for x in (net.actor.action_low, net.actor.action_high))
            fn = lambda: BR.net_grads(kind, params, st, a.double(), old, adv, ret, low, high)
        elif kind == "navimg_md":
            fn = lambda: MD.net_grads(MD_SPEC, params, st, None, a.double(), net.actor.nvec, old, adv, ret)
        else:
            fn = lambda: AM.net_grads(kind, params, st[:-1], mask, a.double(), old, adv, ret)
        oracle = lambda flips=None: ES.oracle_pass(fn, flips)
    return ES.grads_match_oracle(grads, oracle, label=label)[0]


# ------------------------------------------------------------------------------------------- 1. steps within one learn call
SIZES = {"pong": 12, "navimg": 10, "navlaser": 6, "navped": 8, "navlaser3": 6}


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("kind", list(SIZES))
def test_steps_of_one_call_match_adam_twin_and_oracle(request, engine, kind):
    if engine == "tc3":
        request.getfixturevalue("deterministic")
    B = SIZES[kind]
    net = make(kind, engine, TRAINING_ITER_TIME=3)
    learn_checked(net, batch(net, kind, B, seed=1))
    assert net._adam_step == 3
    probe = batch(net, kind, B, seed=2)
    t = check_twin(net, twin_of(net, kind, engine, TRAINING_ITER_TIME=3), probe, engine == "tc3", (kind, engine))
    o = check_oracle(net, kind, probe, "%s %s" % (kind, engine))
    print("%s %s: twin %.2e (bound %.0e), oracle %.2e (bound %.0e)" % (kind, engine, t, TWIN_BOUND, o, ES.GRAD_BOUND))


@pytest.mark.parametrize("env", ["DDRL_PREP_LAUNCHES", "DDRL_NO_GRAPH"])
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_steps_of_one_call_other_preparation_paths(monkeypatch, deterministic, env, kind):
    """tc3 with the per-layer preparation on side streams (DDRL_PREP_LAUNCHES=1) and with stream launches only
    (DDRL_NO_GRAPH=1)."""
    monkeypatch.setenv(env, "1")
    B = SIZES[kind]
    net = make(kind, "tc3", TRAINING_ITER_TIME=3)
    learn_checked(net, batch(net, kind, B, seed=1))
    probe = batch(net, kind, B, seed=2)
    check_twin(net, twin_of(net, kind, "tc3", TRAINING_ITER_TIME=3), probe, True, (kind, env))
    check_oracle(net, kind, probe, "%s %s" % (kind, env))


# ------------------------------------------------------------------------------------------- 2. across learn calls
@pytest.mark.parametrize("kind", ["pong", "navimg", "navlaser"])
def test_learn_calls_with_new_magnitudes_and_sizes(deterministic, kind):
    """Four calls: B rows; the same B with observations 16x larger, written into the buffers of the first call; another B (new
    graph keys, workspace regrowth); B again.  The Adam step numbers continue across the calls (reference 3), and the first
    gradient of every call matches the oracle at the parameters the call started from.
    The tc3 split scale is a power of two, 2^(13 - floor(log2 amax)): data up to 4x the amax the scale was taken from still fit
    fp16, so only a larger step shows a stale amax.  navlaser's image conv (K = 147) reads the observations' im2col matrix
    with the persistent amax slot that every restaging must refresh: its occupancy maps have amax 1 (scale 2^13), so a slot
    kept from the first call overflows the fp16 split of the second (its 16.0 cells scale to 2^17).  (Pong's space-to-depth
    staging and navimg's thin first conv write or need no such slot.)  navlaser runs fewer rows: its sparse maps hold more max-pool near-ties."""
    B, B2 = (12, 20) if kind == "navlaser" else (24, 33)
    net = make(kind, "tc3", TRAINING_ITER_TIME=2)
    bufs = {}
    flat = lambda b: list(b[0]) + list(b[1:])
    for call, (rows, scale) in enumerate([(B, 1.0), (B, 16.0), (B2, 1.0), (B, 1.0)]):
        bt = batch(net, kind, rows, seed=10 + call, scale=scale)
        if rows in bufs:            # new contents at the addresses of an earlier call, as a reused staging buffer holds them
            for dst, src in zip(flat(bufs[rows]), flat(bt)):
                dst.copy_(src)
            bt = bufs[rows]
        else:
            bufs[rows] = bt

        def first(grads, before, bt=bt, call=call):
            check_oracle(net, kind, bt, "%s call %d" % (kind, call), params=before, grads=grads)
        learn_checked(net, bt, on_first=first)
        assert net._adam_step == 2 * (call + 1)
    probe = batch(net, kind, B, seed=20)
    check_twin(net, twin_of(net, kind, "tc3", TRAINING_ITER_TIME=2), probe, True, kind)
    check_oracle(net, kind, probe, kind + " across calls")


# ------------------------------------------------------------------------------------------- 3. minibatch learner
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_minibatch_steps_match_adam_and_twin(deterministic, kind):
    hyper = dict(TRAINING_ITER_TIME=2, MINI_BATCH_NUM=3, MINI_BATCH_SEED=5)
    net = make(kind, "tc3", **hyper)
    for call in range(2):
        learn_checked(net, batch(net, kind, 20, seed=30 + call))
    assert net._adam_step == 12
    check_twin(net, twin_of(net, kind, "tc3", **hyper), batch(net, kind, 20, seed=32), True, kind)


# ------------------------------------------------------------------------------------------- 4. calls between the yields
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_calls_between_yields_change_nothing(deterministic, kind):
    """act on a larger batch (the workspace regrows), encode, net_log_prob and a backward on other rows between the yields of
    one learn generator: losses, parameters and both Adam moments stay bit-equal to those of an uninterrupted learner."""
    from ddrl4nav_b200 import kernels
    B = 16
    runs = []
    for interrupt in (False, True):
        net = make(kind, "tc3", TRAINING_ITER_TIME=5)
        bt = batch(net, kind, B, seed=40)
        other = batch(net, kind, 40, seed=41)
        losses = []
        for i, (log, _, _) in enumerate(net.learn(experience(bt))):
            losses.append([log[k] for k in KEYS])
            if interrupt and i < 4:
                states, a, old, adv, ret = other
                [lambda: net.backward_only([x[:B + 3] for x in states], adv[:B + 3], a[:B + 3], old[:B + 3], ret[:, :B + 3]),
                 lambda: net.act(states), lambda: net.encode(states), lambda: kernels.net_log_prob(net, states, a)][i]()
        runs.append((losses, net._flat.clone(), net._m.clone(), net._v.clone()))
    assert runs[0][0] == runs[1][0]
    for what, x, y in zip(("params", "m", "v"), runs[0][1:], runs[1][1:]):
        assert torch.equal(x, y), (what, int((x != y).sum()))


# ------------------------------------------------------------------------------------------- 5. out-of-band edits
EDITS = ["load_state_dict", "load_model_bytes", "actor.pre.conv1.weight", "critic.pre.conv1.bias", "actor.pre.conv2.weight",
         "critic.pre.linear.weight", "critic.critic_linear.weight", "extra_critic"]


@pytest.mark.parametrize("edit", EDITS)
def test_out_of_band_edit_after_graphs_exist(deterministic, edit):
    """After a learn call (its graphs captured): an edit -- a state_dict / model blob of other parameters, or an in-place
    torch.no_grad() edit of one tensor: the first conv's weight and its bias (fused, space-to-depth and bias copies), the strided
    conv2 (data-gradient class and fused packs), an fc weight (transposed fp16 twin), the critic head (read from the flat
    buffer), an extra critic's weight (outside the flat buffer) -- then two more iterations on the same batch (same graph
    keys).  References 1 and 2 must hold."""
    kind = "navimg" if edit == "extra_critic" else "pong"
    net = make(kind, "tc3", TRAINING_ITER_TIME=2)
    if edit == "extra_critic":
        from ddrl4nav_b200.runner import make_net
        torch.manual_seed(3)
        net.add_critic(make_net(kind, device=None).critic.to(DEV))
    bt = batch(net, kind, 20, seed=50)
    learn_checked(net, bt, adam=edit != "extra_critic")
    other = make(kind, "tc3", seed=99)
    if edit == "load_state_dict":
        net.load_state_dict(other.state_dict())
    elif edit == "load_model_bytes":
        net.load_model_bytes(other.model_bytes())
    else:
        p = net._critics[1].critic_linear.weight if edit == "extra_critic" else dict(net.named_parameters())[edit]
        with torch.no_grad():
            p.mul_(-0.8)
    learn_checked(net, bt, adam=edit != "extra_critic")
    probe = batch(net, kind, 20, seed=51)
    check_twin(net, twin_of(net, kind, "tc3", TRAINING_ITER_TIME=2), probe, True, edit)
    check_oracle(net, kind, probe, edit)


# ------------------------------------------------------------------------------------------- 6. options and actors
OPTIONS = [("pong", {"NORM_VALUE": True}), ("navimg", {"NORM_OBS": True}), ("pong", {"DECOUPLED_PPO": True}),
           ("navimg_md", {}), ("navlaser_beta", {}), ("navped", {"ACTION_MASK": True}), ("navimg", {"gail_critic": True})]


@pytest.mark.parametrize("kind,opt", OPTIONS, ids=["norm_value", "norm_obs", "decoupled", "navimg_md", "navlaser_beta",
                                                   "action_mask", "gail_critic"])
def test_options_after_two_learn_calls(deterministic, kind, opt):
    """Reference 1 after two learn calls (the extra critic's gradients too), and reference 2 where a restatement exists.  NORM_VALUE rescales the critic
    head in the flat buffer at the start of every call without a re-preparation (the engine reads the head from there only);
    DECOUPLED_PPO's proximal log-probs at the start of the second call are the twin's net_log_prob, bit for bit."""
    from ddrl4nav_b200 import kernels
    hyper = dict(opt, TRAINING_ITER_TIME=2)
    gail = hyper.pop("gail_critic", False)
    net = make(kind, "tc3", **hyper)
    if gail:
        from ddrl4nav_b200.runner import make_net
        torch.manual_seed(3)
        net.add_critic(make_net(kind, device=None).critic.to(DEV))
        net.gail_critic = True
    B = 16
    mask = AM.random_mask(B, 28, seed=5) if hyper.get("ACTION_MASK") else None

    def bt_of(seed):
        bt = batch(net, kind, B, seed=seed, mask=mask)
        if gail:                                   # returns [V = 2, B]: the extra critic learns the second row
            bt = bt[:4] + (torch.cat([bt[4], 0.5 * bt[4] + 0.25], 0),)
        return bt
    learn_checked(net, bt_of(60), adam=False)
    bt = bt_of(61)
    if hyper.get("DECOUPLED_PPO"):
        twin = twin_of(net, kind, "tc3", **hyper)
        prox = kernels.net_log_prob(twin, bt[0], bt[1]).clone()
        seen = []
        for _ in net.learn(experience(bt)):
            seen.append(net.last_prox_logps.clone())
        assert torch.equal(seen[0], prox)
    else:
        learn_checked(net, bt, adam=False)
    probe = bt_of(62)
    check_twin(net, twin_of(net, kind, "tc3", **hyper), probe, True, (kind, opt))
    if kind in ("navimg_md", "navlaser_beta") or hyper.get("ACTION_MASK") or hyper.get("NORM_VALUE"):
        check_oracle(net, kind, probe, "%s %s" % (kind, opt), mask=mask)


# ------------------------------------------------------------------------------------------- 7. predictor refresh
@pytest.mark.parametrize("kind", ["pong", "navimg"])
def test_predictor_refresh_from_the_learner_blob(kind):
    """A predictor (inference only: Pong takes the space-to-depth lowering) acts on old weights, then loads the learner's blob:
    its outputs are bit-equal to those of a fresh predictor loaded from the same blob, and within 1e-5 of the learner's."""
    states = [s.to(DEV) for s in R.synth_states(kind, 24, seed=70)]
    pred = make(kind, "tc3", seed=3)
    before = pred.act(states, play_mode=True, want_pi=True)
    learner = make(kind, "tc3", TRAINING_ITER_TIME=2)
    learn_checked(learner, batch(learner, kind, 24, seed=71))
    blob = learner.model_bytes()
    pred.load_model_bytes(blob)
    fresh = make(kind, "tc3", seed=5)
    fresh.load_model_bytes(blob)
    x = pred.act(states, play_mode=True, want_pi=True)
    y = fresh.act(states, play_mode=True, want_pi=True)
    for u, w in zip(x, y):
        assert torch.equal(u, w)
    assert not torch.equal(x[2], before[2])
    z = learner.act(states, play_mode=True, want_pi=True)
    for u, w in zip(x[2:], z[2:]):
        assert float((u - w).abs().max()) <= 1e-5 * float(w.abs().max())
