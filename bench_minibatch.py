"""Cost of minibatch PPO epochs (MINI_BATCH_NUM = M, a non-reference learner option) against the full-batch learner.

One JSON line per configuration (Pong at 8192 rows with M in {1, 2, 4, 8}; nav-laser at 1024 and nav-image at 2048 rows
with M in {1, 4}; TRAINING_ITER_TIME = 10 epochs per learn call, inputs resident in HBM):
  ms_per_learn / ms_per_step     device time of one learn call (10 x M optimiser steps) and of one optimiser step
  value                          learner sample-iterations/s = rows x epochs / time (the unit of bench.py's `value`)
  steps_per_s                    optimiser steps/s
  gather                         the minibatch row gather kernel alone (CUDA events over repeated launches on one
                                 minibatch): ms, GB/s with bytes = 2 x bytes gathered, and its fraction of the HBM
                                 figure bench.py's GAE line uses
  launches_per_learn             ddrl_launch_count() per learn call, with graphs and with DDRL_NO_GRAPH=1 (replayed graph
                                 nodes count like stream launches), and the learn-call time with DDRL_NO_GRAPH=1
The GPU's name and power limit are read in the same run.  --gpus N runs the data-parallel learner over N ranks
(torchrun), timed as bench.py times it (the slowest rank).  Writes nothing to the tree."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

CONFIGS = [("pong", 8192, m) for m in (1, 2, 4, 8)] + [("navlaser", 1024, m) for m in (1, 4)] + [("navimg", 2048, m) for m in (1, 4)]
EPOCHS = 10


def gpu_info(index):
    info = {"name": torch.cuda.get_device_name(index), "power_limit_w": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as e:  # noqa: BLE001
        info["power_limit_error"] = str(e)
    return info


def run_config(kind, B, m, args, dev, rank, world, dist, peaks):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net

    torch.manual_seed(1000 + rank)
    net = make_net(kind, device=dev, TRAINING_ITER_TIME=EPOCHS, MINI_BATCH_NUM=m, MINI_BATCH_SEED=rank)
    if dist is not None:
        net.enable_data_parallel()
        net.broadcast_parameters(0)
    states_h, adv_h, ret_h = bench.synth_batch_host(kind, B, seed=100 + rank)
    states_d = [s.to(dev) for s in states_h]
    with torch.no_grad():
        acts_d, logp_d, _ = net.act(states_d)
    exp = Experience(states=states_d, advs=adv_h.to(dev), actions=acts_d, old_logps=logp_d + 0.15 * torch.randn(B, device=dev),
                     values=ret_h.to(dev)[None])

    def learn():
        for _ in net.learn(exp):
            pass

    for _ in range(args.warmup):
        learn()
    kernels.launch_count_reset()
    sec = bench.timed(learn, args.steps, 0, dist) / args.steps
    launches = kernels.launch_count() / args.steps
    os.environ["DDRL_NO_GRAPH"] = "1"
    try:
        learn()
        kernels.launch_count_reset()
        sec_ng = bench.timed(learn, 1, 0, dist)
        launches_ng = kernels.launch_count()
    finally:
        del os.environ["DDRL_NO_GRAPH"]
    line = {"workload": kind, "rows_per_gpu": B, "n_gpus": world, "mini_batch_num": m, "epochs": EPOCHS,
            "optimizer_steps_per_learn": EPOCHS * m, "learn_calls_timed": args.steps,
            "ms_per_learn": round(sec * 1e3, 3), "ms_per_step": round(sec * 1e3 / (EPOCHS * m), 4),
            "value": round(world * B * EPOCHS / sec, 1), "unit": "learner sample-iterations/s",
            "steps_per_s": round(EPOCHS * m / sec, 1),
            "launches_per_learn": {"graphs": launches, "no_graph": launches_ng},
            "ms_per_learn_no_graph": round(sec_ng * 1e3, 3)}
    if m > 1:
        # the gather of one minibatch, on the sources and buffers the learner used
        src = net._minibatch_sources(exp)
        rows = net.last_minibatch_perms[-1][:B // m]
        for _ in range(3):
            net._gather_minibatch(src, rows)
        reps = 50
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            net._gather_minibatch(src, rows)
        e1.record()
        torch.cuda.synchronize()
        g_sec = e0.elapsed_time(e1) / 1e3 / reps
        row_bytes = sum(t[0].numel() * 4 for t in src["states"]) + 4 * (src["actions"][0].numel() + 2 + src["values"].shape[0])
        moved = 2.0 * row_bytes * rows.numel()
        gbs = moved / g_sec / 1e9
        line["gather"] = {"ms": round(g_sec * 1e3, 4), "rows": rows.numel(), "bytes": int(moved), "gb_per_s": round(gbs, 1),
                          "hbm_peak_gb_per_s": peaks["hbm"], "hbm_peak_src": peaks["src"], "frac_of_hbm": round(gbs / peaks["hbm"], 3),
                          "ms_per_learn": round(g_sec * 1e3 * EPOCHS * m, 3)}
    del net
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed learn calls per configuration")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default=None, help="workload name: run only its configurations")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world and world == 1 and args.gpus > 1:
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
        sys.exit(subprocess.call(cmd))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod
    peaks = bench.load_peaks()
    gpu = gpu_info(local)
    for kind, B, m in CONFIGS:
        if args.only and kind != args.only:
            continue
        line = run_config(kind, B, m, args, dev, rank, world, dist, peaks)
        line["gpu"] = gpu
        if rank == 0:
            print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
