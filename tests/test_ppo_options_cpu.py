"""PPO training options of the learner (NORM_ADV, VALUE_CLIP, PPO_STATS, TARGET_KL) without a GPU: constructor validation, the
hyper-parameter struct the engine receives, self-checks of the CPU restatement the GPU tests compare against, the optional
old_values slot of Experience, and the advantage-moment all-reduce over a gloo world of two ranks (dist.global_moments)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import ppo_options_ref as O
from oracle import restate as R


def _net(kind="navimg", **hyper):
    from ddrl4nav_b200.runner import make_net
    return make_net(kind, device=None, **hyper)


@pytest.mark.parametrize("key", ["NORM_ADV", "PPO_STATS"])
@pytest.mark.parametrize("bad", [1, 0, "yes", None, 1.0])
def test_flag_options_must_be_bool(key, bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match=key):
        _net(**{key: bad})


@pytest.mark.parametrize("key", ["VALUE_CLIP", "TARGET_KL"])
@pytest.mark.parametrize("bad", [0, 0.0, -0.1, True, False, "0.2", float("nan"), float("inf"), [0.2]])
def test_positive_options_must_be_finite_numbers_above_zero(key, bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match=key):
        _net(**{key: bad})


def test_defaults_are_off_and_leave_the_hparams_unchanged():
    net = _net()
    assert (net.norm_adv, net.value_clip, net.ppo_stats, net.target_kl) == (False, None, False, None)
    off = _net(NORM_ADV=False, VALUE_CLIP=None, PPO_STATS=False, TARGET_KL=None)
    assert bytes(net.hp) == bytes(off.hp)
    assert net.hp.value_clip == 0.0 and net.hp.ppo_stats == 0


def test_accepted_values_reach_the_hparams():
    net = _net(NORM_ADV=np.bool_(True), VALUE_CLIP=np.float32(0.5), PPO_STATS=True)
    assert net.norm_adv is True and net.value_clip == 0.5 and type(net.value_clip) is float
    assert net.hp.value_clip == 0.5 and net.hp.ppo_stats == 1
    assert _net(VALUE_CLIP=2).value_clip == 2.0


def test_target_kl_implies_stats():
    net = _net(TARGET_KL=0.02)
    assert net.target_kl == 0.02 and net.ppo_stats is True and net.hp.ppo_stats == 1


def test_hparams_struct_appends_the_new_fields():
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200._lib import PPOHparams
    names = [f[0] for f in PPOHparams._fields_]
    assert names[-2:] == ["value_clip", "ppo_stats"] and len(names) == 15
    hp = kernels.make_hparams()
    assert hp.value_clip == 0.0 and hp.ppo_stats == 0
    # a struct built positionally from the 13 reference fields keeps the options off
    old = PPOHparams(*[getattr(hp, n) for n in names[:13]])
    assert bytes(old) == bytes(hp)


def test_experience_carries_old_values_when_every_chunk_has_them():
    from ddrl4nav_b200.data import Experience
    mk = lambda B, ov: Experience(states=[np.zeros((B, 3), np.float32)], advs=np.ones(B, np.float32),
                                  actions=np.zeros(B, np.float32), old_logps=np.zeros(B, np.float32),
                                  values=np.zeros((1, B), np.float32), old_values=ov)
    e = Experience.batch_data([mk(2, np.array([1, 2], np.float32)), mk(3, np.array([3, 4, 5], np.float32))])
    assert e.old_values.tolist() == [1, 2, 3, 4, 5]
    assert Experience.batch_data([mk(2, None), mk(3, None)]).old_values is None
    e.to_tensor(device="cpu")
    assert torch.is_tensor(e.old_values) and e.old_values.dtype == torch.float32


# ---------------------------------------------------------------------------------------------------------- CPU restatement
def _setup(kind="pong", B=24, smooth_l1=False):
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=11)
    states = R.synth_states(kind, B, seed=5)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=9)
    return spec, params, states, a, old, adv, ret, R.PPOHyper(smooth_l1=smooth_l1)


@pytest.mark.parametrize("smooth_l1", [False, True])
def test_huge_value_clip_equals_the_unclipped_loss(smooth_l1):
    spec, params, states, a, old, adv, ret, hp = _setup(smooth_l1=smooth_l1)
    ov = ret - adv
    l0, g0 = O.learn_iteration(R.LearnState(spec, params), states, adv, a, old, ret, hp)
    l1, g1 = O.learn_iteration(R.LearnState(spec, params), states, adv, a, old, ret, hp, old_values=ov, value_clip=1e30)
    ref, _, _ = R.learn_iteration(R.LearnState(spec, params), states, adv, a, old, ret, hp, apply_update=False)
    assert l0 == ref
    assert l1["VLoss"] == pytest.approx(l0["VLoss"], rel=1e-6)
    for k in g0:
        assert torch.allclose(g0[k], g1[k], rtol=1e-5, atol=1e-8), k


def test_value_clip_changes_the_loss_and_the_stats_are_plain_means():
    spec, params, states, a, old, adv, ret, hp = _setup()
    ov = ret - adv
    l0, _ = O.learn_iteration(R.LearnState(spec, params), states, adv, a, old, ret, hp, stats=True)
    l1, _ = O.learn_iteration(R.LearnState(spec, params), states, adv, a, old, ret, hp, old_values=ov, value_clip=0.1, stats=True)
    assert l1["VLoss"] > l0["VLoss"]                  # the max of the two losses can only add
    with torch.no_grad():
        lp = R.ppo_forward(spec, params, states, a)["logp"]
    r = torch.exp(lp - old)
    assert l0["ApproxKL"] == pytest.approx(float(((r - 1) - torch.log(r)).mean()), rel=1e-5)
    assert l0["ApproxKL"] > 0
    assert l0["ClipFrac"] == pytest.approx(float(((r - 1).abs() > 0.2).double().mean()), abs=1e-7)
    assert 0 < l0["ClipFrac"] < 1


@pytest.mark.parametrize("n", [1, 2, 13, 1000])
def test_normalize_advantages(n):
    a = torch.randn(n, generator=torch.Generator().manual_seed(n)) * 3 + 1
    out = O.normalize_advantages(a)
    if n == 1:
        assert torch.equal(out, a)
    else:
        assert torch.equal(out, (a - a.mean()) / (a.std() + 1e-8))
        assert abs(float(out.mean())) < 1e-5 and abs(float(out.std()) - 1) < 1e-5


# ---------------------------------------------------------------------------------------------------------- two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch.distributed as tdist
    from ddrl4nav_b200 import dist
    torch.set_num_threads(1)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    a = torch.arange(rank * 5, rank * 5 + 5 - rank, dtype=torch.float32)     # 5 rows on rank 0, 4 on rank 1
    m3 = torch.tensor([a.numel(), float(a.double().sum()), float((a.double() ** 2).sum())], dtype=torch.float64)
    out = dist.global_moments(m3)
    assert out is m3
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), m3.numpy())
    tdist.barrier()
    tdist.destroy_process_group()


def test_two_rank_global_moments(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    allrows = np.concatenate([np.arange(0, 5), np.arange(5, 9)]).astype(np.float64)
    for rank in range(2):
        m3 = np.load(os.path.join(str(tmp_path), "rank%d.npy" % rank))
        assert m3.tolist() == [9.0, allrows.sum(), (allrows ** 2).sum()]


def test_single_process_global_moments_need_no_collective():
    from ddrl4nav_b200 import dist
    m3 = torch.tensor([3.0, 1.0, 2.0], dtype=torch.float64)
    assert dist.global_moments(m3) is m3 and m3.tolist() == [3.0, 1.0, 2.0]
