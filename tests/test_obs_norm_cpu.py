"""Running observation normalisation (NORM_OBS, NORM_OBS_CLIP) without a GPU: constructor validation, the state_dict buffers a
checkpoint brings along before the engine is built, self-checks of the float64 restatement the GPU tests compare against
(tests/obs_norm_ref.py), and the all-reduce of the moment sums over a gloo world of two ranks (dist.global_obs_sums)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import obs_norm_ref as N


def _net(kind="navlaser", **hyper):
    from ddrl4nav_b200.runner import make_net
    return make_net(kind, device=None, **hyper)


@pytest.mark.parametrize("bad", [1, 0, "yes", None, 1.0, [], (), [0, 0], (1, 0, 1), [0.0], [True], [-1], [0, "1"], {0: 1}])
def test_norm_obs_rejects_anything_but_a_flag_or_distinct_slots(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="NORM_OBS"):
        _net(NORM_OBS=bad)


@pytest.mark.parametrize("bad", [0, 0.0, -1.0, True, False, "10", float("nan"), float("inf"), [10.0]])
def test_norm_obs_clip_must_be_a_positive_number_or_none(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="NORM_OBS_CLIP"):
        _net(NORM_OBS=True, NORM_OBS_CLIP=bad)


def test_accepted_values():
    assert _net().obs_rms is None and _net(NORM_OBS=False).obs_rms is None
    on = _net(NORM_OBS=np.bool_(True))
    assert on.obs_rms.wanted is None and on.obs_rms.clip == 10.0
    assert _net(NORM_OBS=[1, np.int64(0)], NORM_OBS_CLIP=5).obs_rms.wanted == (0, 1)
    assert _net(NORM_OBS=(2,), NORM_OBS_CLIP=None).obs_rms.clip is None
    assert type(_net(NORM_OBS=True, NORM_OBS_CLIP=np.float32(3)).obs_rms.clip) is float


def test_option_off_adds_no_state_and_no_blob_bytes():
    off, plain = _net("mlp", NORM_OBS=False, NORM_OBS_CLIP=4.0), _net("mlp")
    assert list(off.state_dict()) == list(plain.state_dict())
    assert [n for n, _ in off.named_parameters()] == [n for n, _ in plain.named_parameters()]
    off.load_state_dict(plain.state_dict(), strict=True)
    assert off.model_bytes() == plain.model_bytes()


def test_checkpoint_buffers_load_before_the_engine_is_built():
    """A fresh option-on net has no statistics yet (their sizes come from the engine); a checkpoint creates them, keeps the
    float64 bits, and leaves the parameter table alone."""
    net = _net(NORM_OBS=(0, 1))
    params = dict(_net().state_dict())
    assert set(net.state_dict()) == set(params)
    stats = {"obs_rms.mean_1": torch.arange(5, dtype=torch.float64) / 3, "obs_rms.var_1": torch.full((5,), 2.5, dtype=torch.float64),
             "obs_rms.count_1": torch.tensor([1e-4 + 77], dtype=torch.float64)}
    net.load_state_dict({**params, **stats}, strict=True)
    sd = net.state_dict()
    for k, v in stats.items():
        assert sd[k].dtype == torch.float64 and torch.equal(sd[k], v)
    assert [n for n, _ in net.named_parameters()] == [n for n, _ in _net().named_parameters()]
    # statistics of a slot the net does not normalise are not taken silently
    with pytest.raises(RuntimeError, match="obs_rms.mean_2"):
        _net(NORM_OBS=(0, 1)).load_state_dict({**params, "obs_rms.mean_2": torch.zeros(3)}, strict=True)


# ---------------------------------------------------------------------------------------------------------- restatement
def test_two_merges_equal_the_concatenated_batch():
    rng = np.random.default_rng(0)
    a = rng.normal(3.0, 2.0, (37, 11))
    b = rng.normal(-1.0, 0.5, (50, 11))
    r = N.RunningMeanStd(11)
    r.update(a)
    r.update(b)
    one = N.RunningMeanStd(11)
    one.update(np.concatenate([a, b]))
    assert r.count == one.count == 87 + 1e-4
    np.testing.assert_allclose(r.mean, one.mean, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(r.var, one.var, rtol=1e-13)
    # gym's start (count 1e-4, mean 0, var 1) is a prior worth 1e-4 rows: after a batch the statistics are the batch's
    x = np.concatenate([a, b])
    np.testing.assert_allclose(one.mean, x.mean(0), rtol=1e-5)
    np.testing.assert_allclose(one.var, x.var(0), rtol=1e-4)


def test_shifted_sums_equal_the_direct_form():
    rng = np.random.default_rng(1)
    x = rng.normal(1e3, 1e-2, (64, 7))                       # a large offset: the shift keeps the sums well conditioned
    direct, shifted = N.RunningMeanStd(7), N.RunningMeanStd(7)
    direct.update(x[:20])
    shifted.update(x[:20])
    direct.update(x[20:])
    s1, s2 = N.shifted_sums(x[20:], shifted.mean)
    shifted.update_from_sums(s1, s2, 44, shifted.mean)
    np.testing.assert_allclose(shifted.mean, direct.mean, rtol=1e-14)
    np.testing.assert_allclose(shifted.var, direct.var, rtol=1e-9)
    assert shifted.count == direct.count


def test_applied_form_and_normalisation():
    mean, var = np.array([0.5, -2.0, 0.0]), np.array([4.0, 0.25, 0.0])
    m32, s32 = N.applied(mean, var)
    assert m32.dtype == s32.dtype == np.float32
    assert s32.tolist() == [np.float32(1 / np.sqrt(4.0 + 1e-8)), np.float32(1 / np.sqrt(0.25 + 1e-8)), np.float32(1e4)]
    x = np.array([[2.5, -2.0, 1.0]], np.float32)
    y = N.normalize(x, m32, s32, 10.0)
    assert y.dtype == np.float32 and y[0, 1] == 0 and y[0, 2] == 10.0 and abs(y[0, 0] - 1.0) < 1e-6
    assert N.normalize(x, m32, s32, None)[0, 2] == np.float32(1e4)


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
    sums = torch.arange(6, dtype=torch.float64) * (rank + 1) + 0.25       # two slots' {S1, S2} concatenated
    out = dist.global_obs_sums(sums)
    assert out is sums
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), sums.numpy())
    tdist.barrier()
    tdist.destroy_process_group()


def test_two_rank_global_obs_sums(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    want = (np.arange(6) * 3 + 0.5).tolist()
    for rank in range(2):
        assert np.load(os.path.join(str(tmp_path), "rank%d.npy" % rank)).tolist() == want


def test_single_process_global_obs_sums_need_no_collective():
    from ddrl4nav_b200 import dist
    s = torch.tensor([1.0, 2.0], dtype=torch.float64)
    assert dist.global_obs_sums(s) is s and s.tolist() == [1.0, 2.0]
