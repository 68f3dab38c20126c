"""Value-target normalisation (NORM_VALUE) without a GPU: constructor validation, no state and no hyper-parameter bytes with the
option off, the state_dict keys with it on, self-checks of the float64 restatement the GPU tests compare against
(tests/value_norm_ref.py), and the all-reduce of the observation and value moment sums in ONE buffer over a gloo world of two
ranks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import value_norm_ref as V


def _net(kind="navlaser", **hyper):
    from ddrl4nav_b200.runner import make_net
    return make_net(kind, device=None, **hyper)


@pytest.mark.parametrize("bad", [1, 0, "yes", None, 1.0, [], (True,)])
def test_norm_value_must_be_a_flag(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="NORM_VALUE"):
        _net(NORM_VALUE=bad)


def test_option_off_adds_no_state_no_blob_bytes_and_no_hparam_bytes():
    off, plain, on = _net("mlp", NORM_VALUE=False), _net("mlp"), _net("mlp", NORM_VALUE=np.bool_(True))
    assert off.value_rms is None and plain.value_rms is None and on.value_rms is not None
    assert list(off.state_dict()) == list(plain.state_dict())
    off.load_state_dict(plain.state_dict(), strict=True)
    assert off.model_bytes() == plain.model_bytes()
    assert bytes(on.hp) == bytes(off.hp) == bytes(plain.hp)
    # the option adds three float64 buffers, not parameters
    extra = [k for k in on.state_dict() if k not in plain.state_dict()]
    assert extra == ["value_rms.mean", "value_rms.var", "value_rms.count"]
    assert all(on.state_dict()[k].dtype == torch.float64 and on.state_dict()[k].shape == (1,) for k in extra)
    assert [n for n, _ in on.named_parameters()] == [n for n, _ in plain.named_parameters()]
    st = on.state_dict()
    assert float(st["value_rms.mean"]) == 0.0 and float(st["value_rms.var"]) == 1.0 and float(st["value_rms.count"]) == 1e-4


def test_checkpoint_restores_the_statistics_before_the_engine_is_built():
    src = _net(NORM_VALUE=True, NORM_OBS=(0, 1))
    sd = dict(src.state_dict())
    sd["value_rms.mean"] = torch.tensor([512.25], dtype=torch.float64)
    sd["value_rms.var"] = torch.tensor([6400.5], dtype=torch.float64)
    sd["value_rms.count"] = torch.tensor([1e-4 + 4096], dtype=torch.float64)
    dst = _net(NORM_VALUE=True)
    dst.load_state_dict({k: v for k, v in sd.items() if not k.startswith("obs_rms.")}, strict=True)
    for k in ("mean", "var", "count"):
        assert torch.equal(dst.state_dict()["value_rms." + k], sd["value_rms." + k])


# ---------------------------------------------------------------------------------------------------------- restatement
def test_rescaled_head_preserves_the_unnormalised_outputs():
    rng = np.random.default_rng(0)
    r = V.ValueRMS()
    r.update(rng.normal(500.0, 80.0, (300, 1)))
    w, b = rng.normal(0, 0.05, 512), 0.3
    x = rng.normal(0, 1, (64, 512))
    old = (r.mean[0], r.var[0])
    out_old = r.sigma() * (x @ w + b) + r.mean[0]
    r.update(rng.normal(-40.0, 3.0, (500, 1)))
    w2, b2 = V.rescale_head(w, b, old, (r.mean[0], r.var[0]))
    out_new = r.sigma() * (x @ w2 + b2) + r.mean[0]
    np.testing.assert_allclose(out_new, out_old, rtol=1e-12, atol=1e-12 * np.abs(out_old).max())
    assert abs(r.sigma() - 1.0) > 0.5                     # the statistics did move


def test_applied_form_and_the_normalised_value_loss():
    a = V.applied(500.0, 6400.0)
    assert a.dtype == np.float32 and a.tolist() == [500.0, np.float32(1 / np.sqrt(6400.0 + 1e-8)), np.float32(np.sqrt(6400.0 + 1e-8))]
    R = torch.tensor([580.0, 420.0, 500.0])
    assert torch.allclose(V.normalize(R, a), torch.tensor([1.0, -1.0, 0.0]), atol=1e-6)
    assert torch.allclose(V.denormalize(V.normalize(R, a), a), R, rtol=1e-6)
    v = torch.tensor([0.5, -1.0, 2.0], dtype=torch.float64)
    assert float(V.value_loss(v, R, a)) == pytest.approx((0.25 + 0.0 + 4.0) / 6, rel=1e-6)
    # clipped around the normalised old values: 500, 420, 740 -> 0, -1, 3; the clipped values 0.5, -1, 2.5; per row the max
    clipped = V.value_loss(v, R, a, old_values=torch.tensor([500.0, 420.0, 740.0]), value_clip=0.5)
    assert float(clipped) == pytest.approx((0.125 + 0.0 + 3.125) / 3, rel=1e-6)
    # the clip width is in normalised units: old values of 0 (= 500) clip v = -1 to -0.5 and v = 2 to 0.5
    clipped = V.value_loss(v, R, a, old_values=torch.full((3,), 500.0), value_clip=0.5)
    assert float(clipped) == pytest.approx((0.125 + 0.125 + 2.0) / 3, rel=1e-6)


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
    from ddrl4nav_b200.nn.obs_rms import ObsRMS, ValueRMS, share_sums
    torch.set_num_threads(1)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    obs, val = ObsRMS((0, 1), None), ValueRMS()
    obs.bind(2, lambda s: (3, 2)[s], "cpu")
    val.bind("cpu")
    buf = share_sums(obs, val)
    assert buf.numel() == 2 * (3 + 2) + 2 and obs.sums.numel() == 10 and val.sums.numel() == 2
    obs.sums.copy_(torch.arange(10, dtype=torch.float64) * (rank + 1) + 0.25)
    val.sums.copy_(torch.tensor([100.0, 7.5], dtype=torch.float64) * (rank + 1))
    assert dist.global_obs_sums(buf) is buf                  # ONE collective for both
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), np.concatenate([obs.sums.numpy(), val.sums.numpy()]))
    tdist.barrier()
    tdist.destroy_process_group()


def test_two_rank_observation_and_value_sums_reduce_in_one_buffer(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    want = (np.arange(10) * 3 + 0.5).tolist() + [300.0, 22.5]
    for rank in range(2):
        assert np.load(os.path.join(str(tmp_path), "rank%d.npy" % rank)).tolist() == want
