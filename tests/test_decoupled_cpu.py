"""Decoupled PPO (DECOUPLED_PPO, DECOUPLED_IS_CLIP) without a GPU: constructor validation, no hyper-parameter bytes, self-checks
of the float64 restatement the GPU tests compare against (tests/decoupled_ref.py), and the gradient all-reduce of a
data-parallel learner, which carries one more float of the loss tail (the behaviour KL) over a gloo world of two ranks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import decoupled_ref as D
import ppo_options_ref as O
from oracle import restate as R


def _net(kind="mlp", **hyper):
    from ddrl4nav_b200.runner import make_net
    return make_net(kind, device=None, **hyper)


@pytest.mark.parametrize("bad", [1, 0, "yes", None, 1.0])
def test_decoupled_ppo_must_be_a_flag(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="DECOUPLED_PPO"):
        _net(DECOUPLED_PPO=bad)


@pytest.mark.parametrize("bad", [0, 0.0, -1.0, True, "2", float("nan"), float("inf"), [1.0]])
def test_is_clip_must_be_a_finite_number_above_zero(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="DECOUPLED_IS_CLIP"):
        _net(DECOUPLED_PPO=True, DECOUPLED_IS_CLIP=bad)


def test_is_clip_needs_the_option():
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="DECOUPLED_IS_CLIP needs DECOUPLED_PPO"):
        _net(DECOUPLED_IS_CLIP=1.0)


def test_defaults_are_off_and_add_no_hparam_or_state_bytes():
    from ddrl4nav_b200._lib import PPOHparams
    plain, off, on = _net(), _net(DECOUPLED_PPO=False), _net(DECOUPLED_PPO=np.bool_(True), DECOUPLED_IS_CLIP=2)
    assert (plain.decoupled, plain.decoupled_is_clip, plain.last_prox_logps) == (False, None, None)
    assert on.decoupled is True and on.decoupled_is_clip == 2.0 and type(on.decoupled_is_clip) is float
    assert bytes(plain.hp) == bytes(off.hp) == bytes(on.hp)
    assert len(PPOHparams._fields_) == 15
    assert list(on.state_dict()) == list(plain.state_dict())
    on.load_state_dict(plain.state_dict(), strict=True)
    assert on.model_bytes() == plain.model_bytes()


# ---------------------------------------------------------------------------------------------------------- restatement
def _setup(kind, B=24):
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=11)
    states = R.synth_states(kind, B, seed=5)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=9)
    return spec, params, states, a, old, adv, ret


@pytest.mark.parametrize("kind", ["pong", "navlaser"])
def test_reduces_to_plain_ppo_when_prox_equals_old(kind):
    spec, params, states, a, old, adv, ret = _setup(kind)
    hp = R.PPOHyper()
    out = R.ppo_forward(spec, params, states, a)
    head = out["probs"].log() if spec.dist == "categorical" else out["mu"]
    v = out["values"].squeeze()
    got, dh, dv, dls = D.loss_and_grads(spec.dist, head, a, old, old, adv, ret, v, hp, spec.shared,
                                        log_std=out.get("log_std"))
    # plain PPO on the same head, in float64 autograd
    h = head.detach().double().clone().requires_grad_(True)
    vv = v.detach().double().clone().requires_grad_(True)
    ls = out["log_std"].detach().double().clone().requires_grad_(True) if spec.dist == "gaussian" else None
    o = {"values": vv.unsqueeze(-1)}
    if spec.dist == "categorical":
        o["probs"] = torch.softmax(h, -1)
        o["logp"] = R.categorical_log_prob(o["probs"], a)
    else:
        o["mu"], o["log_std"] = h, ls
        o["logp"] = R.gaussian_log_prob(h, ls, a.double())
    actor, vl, ent, total, st = O.ppo_losses(spec, o, adv.double(), old.double(), ret.double(), hp, stats=True)
    if spec.shared:
        total.backward()
    else:
        actor.backward()
        vl.backward()
    assert got["actor"] == pytest.approx(float(actor), rel=1e-12, abs=1e-14)
    assert got["v"] == pytest.approx(float(vl), rel=1e-12) and got["entropy"] == pytest.approx(float(ent), rel=1e-12)
    assert got["ApproxKL"] == pytest.approx(st["ApproxKL"], rel=1e-9) and got["ClipFrac"] == pytest.approx(st["ClipFrac"], abs=1e-7)
    assert got["BehaviourKL"] == 0.0
    assert torch.allclose(dh, h.grad, rtol=1e-12, atol=1e-15) and torch.allclose(dv, vv.grad, rtol=1e-12, atol=1e-15)
    if ls is not None:
        assert torch.allclose(dls, ls.grad, rtol=1e-12, atol=1e-15)


def _ratios_and_advs(n=4000, seed=3):
    g = torch.Generator().manual_seed(seed)
    r = torch.exp(0.5 * torch.randn(n, generator=g, dtype=torch.float64))
    r[:8] = torch.tensor([0.8, 1.2, 1.0, 0.5, 2.0, 3.5, 0.8, 1.2], dtype=torch.float64)     # clip edges and the dual clip
    adv = torch.randn(n, generator=g, dtype=torch.float64)
    adv[:8] = torch.tensor([1.0, 1.0, -1.0, -2.0, -1.0, -1.0, -1.0, -1.0], dtype=torch.float64)
    return r, adv


@pytest.mark.parametrize("w", [0.125, 0.5, 1.0, 2.0, 8.0])
def test_weight_moves_into_the_advantage_for_positive_w(w):
    r, adv = _ratios_and_advs()
    # w > 0 keeps the sign of A and scales both branches of min / max: term(r, w A) == w term(r, A) (exact for powers of two)
    assert torch.equal(D.term(r, w * adv, 0.2, 3.0), w * D.term(r, adv, 0.2, 3.0))
    wv = torch.full_like(r, w) * torch.exp(0.1 * torch.sin(torch.arange(r.numel(), dtype=torch.float64)))
    assert torch.allclose(D.term(r, wv * adv, 0.2, 3.0), wv * D.term(r, adv, 0.2, 3.0), rtol=1e-14, atol=0)
    # ... and so do their gradients with respect to r
    r1 = r.clone().requires_grad_(True)
    r2 = r.clone().requires_grad_(True)
    D.term(r1, wv * adv, 0.2, 3.0).sum().backward()
    (wv * D.term(r2, adv, 0.2, 3.0)).sum().backward()
    assert torch.allclose(r1.grad, r2.grad, rtol=1e-14, atol=0)


def test_truncation_caps_the_weight_and_leaves_the_behaviour_kl():
    g = torch.Generator().manual_seed(1)
    old = torch.randn(500, generator=g, dtype=torch.float64)
    prox = old + 0.8 * torch.randn(500, generator=g, dtype=torch.float64)
    w = D.behaviour_weight(prox, old)
    wc = D.behaviour_weight(prox, old, 1.5)
    assert (w > 1.5).any() and (w < 1.5).any()
    assert torch.equal(wc, torch.clamp(w, max=1.5)) and float(wc.max()) == 1.5
    assert torch.equal(D.behaviour_weight(prox, old, 1e30), w)
    rho = torch.exp(prox - old)
    assert D.behaviour_kl(prox, old) == pytest.approx(float(torch.mean((rho - 1) - torch.log(rho))), rel=1e-12)
    assert D.behaviour_kl(prox, old) > 0
    logp = prox + 0.1 * torch.randn(500, generator=g, dtype=torch.float64)
    adv = torch.randn(500, generator=g, dtype=torch.float64)
    r = torch.exp(logp - prox)
    assert float(D.actor_loss(logp, prox, old, adv, is_clip=1.5)) == pytest.approx(
        float(-torch.mean(wc * D.term(r, adv, 0.2, 3.0))), rel=1e-12)


# ---------------------------------------------------------------------------------------------------------- two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch.distributed as tdist
    from ddrl4nav_b200.runner import make_net
    torch.set_num_threads(1)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    res = []
    for hyper in (dict(PPO_STATS=True), dict(PPO_STATS=True, DECOUPLED_PPO=True), dict(DECOUPLED_PPO=True)):
        net = make_net("mlp", device=None, **hyper)
        net.enable_data_parallel(collective="nccl")
        P = 16
        net._P = P
        net._grads = torch.arange(P + 8, dtype=torch.float32) + 100 * (rank + 1)
        net._allreduce_grads()
        res.append(net._grads.numpy().copy())
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), np.stack(res))
    tdist.barrier()
    tdist.destroy_process_group()


def test_two_rank_tail_carries_the_behaviour_kl(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    P = 16
    base = np.arange(P + 8, dtype=np.float32)
    for rank in range(2):
        got = np.load(os.path.join(str(tmp_path), "rank%d.npy" % rank))
        for row, tail in zip(got, (5, 6, 4)):
            want = base + 100 * (rank + 1)
            want[:P + tail] = 2 * base[:P + tail] + 300
            assert row.tolist() == want.tolist(), tail
