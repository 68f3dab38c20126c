"""Host logic of the minibatch learner (PPO MINI_BATCH_NUM > 1) that needs no GPU: constructor validation, the error for
more minibatches than rows (raised before the engine is touched), the chunk plan, and the per-chunk B_global all-reduce
over a gloo world of two ranks (dist.global_chunk_rows), including the empty-global-chunk error every rank raises."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import restate as R


def _net(**hyper):
    from ddrl4nav_b200.runner import make_net
    return make_net("navimg", device=None, **hyper)


@pytest.mark.parametrize("bad", [0, -2, 1.5, 2.0, "4", True, None])
def test_mini_batch_num_must_be_a_positive_integer(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="MINI_BATCH_NUM"):
        _net(MINI_BATCH_NUM=bad)


@pytest.mark.parametrize("bad", [1.0, "7", False])
def test_mini_batch_seed_must_be_an_integer_or_none(bad):
    from ddrl4nav_b200._lib import DDRLError
    with pytest.raises(DDRLError, match="MINI_BATCH_SEED"):
        _net(MINI_BATCH_NUM=2, MINI_BATCH_SEED=bad)


def test_defaults_and_accepted_values():
    assert _net().mini_batch_num == 1
    net = _net(MINI_BATCH_NUM=np.int64(4), MINI_BATCH_SEED=7)
    assert net.mini_batch_num == 4 and type(net.mini_batch_num) is int
    assert net.last_minibatch_perms == []


def test_more_minibatches_than_rows_fails_before_the_engine():
    from ddrl4nav_b200._lib import DDRLError
    from ddrl4nav_b200.data import Experience
    B = 5
    states = R.synth_states("navimg", B, seed=1)
    exp = Experience(states=states, advs=torch.zeros(B), actions=torch.zeros(B), old_logps=torch.zeros(B),
                     values=torch.zeros(1, B))
    net = _net(MINI_BATCH_NUM=6)             # parameters on the CPU: touching the engine would fail differently
    with pytest.raises(DDRLError, match="MINI_BATCH_NUM=6 exceeds the 5 rows"):
        next(net.learn(exp))


def test_chunk_plan():
    from ddrl4nav_b200.nn import PPO
    assert PPO.minibatch_plan(40, 3) == [(0, 14), (14, 27), (27, 40)]
    assert PPO.minibatch_plan(8192, 4) == [(0, 2048), (2048, 4096), (4096, 6144), (6144, 8192)]
    for b in (1, 2, 7, 41, 1000):
        for m in range(1, min(b, 9) + 1):
            plan = PPO.minibatch_plan(b, m)
            assert len(plan) == m and plan[0][0] == 0 and plan[-1][1] == b
            assert all(plan[k][1] == plan[k + 1][0] for k in range(m - 1))
            sizes = [hi - lo for lo, hi in plan]
            assert min(sizes) >= 1 and max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch.distributed as tdist
    from ddrl4nav_b200 import dist
    from ddrl4nav_b200._lib import DDRLError
    from ddrl4nav_b200.nn import PPO
    torch.set_num_threads(1)
    tdist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    res = {}
    # unequal shards (41 / 40 rows), M = 3: chunk k of the global step = chunk k of both ranks
    b_local = (41, 40)[rank]
    sizes = [hi - lo for lo, hi in PPO.minibatch_plan(b_local, 3)]
    res["sums"] = dist.global_chunk_rows(sizes, "cpu")
    # rank 0 has 2 rows and rank 1 none: chunk 2 is empty everywhere -> both ranks raise; chunk 1 is empty on rank 1 only
    sizes = [1, 1, 0] if rank == 0 else [0, 0, 0]
    try:
        dist.global_chunk_rows(sizes, "cpu")
        res["raised"] = False
    except DDRLError as e:
        res["raised"] = "empty global chunk" in str(e)
    res["partial"] = dist.global_chunk_rows([1, 0] if rank == 0 else [1, 1], "cpu")
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), np.array([res["sums"], res["partial"] + [0], [int(res["raised"])] * 3]))
    tdist.barrier()
    tdist.destroy_process_group()


def test_two_rank_chunk_row_sums(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for rank in range(2):
        r = np.load(os.path.join(str(tmp_path), "rank%d.npy" % rank))
        assert r[0].tolist() == [14 + 14, 14 + 13, 13 + 13]
        assert r[1].tolist() == [2, 1, 0]
        assert r[2].tolist() == [1, 1, 1]


def test_single_process_chunk_row_sums_need_no_collective():
    from ddrl4nav_b200 import dist
    from ddrl4nav_b200._lib import DDRLError
    assert dist.global_chunk_rows([3, 2], "cpu") == [3, 2]
    with pytest.raises(DDRLError):
        dist.global_chunk_rows([1, 0], "cpu")
