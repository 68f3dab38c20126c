"""Cost of the learner's PPO training options (NORM_ADV + VALUE_CLIP + PPO_STATS, non-reference) against the default learner.

One JSON line per configuration: Pong at 8192 rows, MINI_BATCH_NUM M in {1, 4}, TRAINING_ITER_TIME = 10, inputs resident in
HBM, every option off vs NORM_ADV + VALUE_CLIP (= 1.0, old values from the values[0] - advs fallback) + PPO_STATS:
  ms_per_learn / ms_per_step     device time of one learn call (10 x M optimiser steps) and of one optimiser step
  value                          learner sample-iterations/s = rows x epochs / time (the unit of bench.py's `value`)
  launches_per_learn             ddrl_launch_count() per learn call
Then one line per row count for the advantage normaliser alone (adv_normalize_kernel with m3 = NULL, in place, CUDA events
over repeated launches).  The configurations run interleaved (off, on, off, on, ...) and each is reported as the median of
--repeats rounds, so that drift of the shared machine falls on both arms.  The GPU's name and power limit are read in the
same run.  Writes nothing to the tree."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from bench_minibatch import gpu_info  # noqa: E402

EPOCHS = 10
OPTIONS = dict(NORM_ADV=True, VALUE_CLIP=1.0, PPO_STATS=True)


def make_learner(kind, B, m, options, dev):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net

    torch.manual_seed(1000)
    net = make_net(kind, device=dev, TRAINING_ITER_TIME=EPOCHS, MINI_BATCH_NUM=m, MINI_BATCH_SEED=0, **(OPTIONS if options else {}))
    states_h, adv_h, ret_h = bench.synth_batch_host(kind, B, seed=100)
    states_d = [s.to(dev) for s in states_h]
    with torch.no_grad():
        acts_d, logp_d, _ = net.act(states_d)
    exp = Experience(states=states_d, advs=adv_h.to(dev), actions=acts_d, old_logps=logp_d + 0.15 * torch.randn(B, device=dev),
                     values=ret_h.to(dev)[None])

    def learn():
        n = 0
        for _ in net.learn(exp):
            n += 1
        return n

    def measure(steps):
        kernels.launch_count_reset()
        sec = bench.timed(learn, steps, 0, None) / steps
        return sec, kernels.launch_count() / steps

    return learn, measure


def time_normaliser(n, dev, reps=2000):
    from ddrl4nav_b200 import kernels
    a = torch.randn(n, device=dev)
    for _ in range(10):
        kernels.adv_normalize(a, out=a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        kernels.adv_normalize(a, out=a)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps            # ms per launch, back to back (includes the launch gap)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3, help="timed learn calls per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3, help="interleaved rounds per configuration")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_ppo_options.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    kind, B = "pong", 8192
    for m in (1, 4):
        arms = {}
        for options in (False, True):
            learn, timer = make_learner(kind, B, m, options, dev)
            for _ in range(args.warmup):
                steps = learn()
            arms[options] = (timer, steps, [])
        for _ in range(args.repeats):
            for options in (False, True):
                timer, _, runs = arms[options]
                runs.append(timer(args.steps))
        base = None
        for options in (False, True):
            _, steps, runs = arms[options]
            sec = statistics.median(r[0] for r in runs)
            base = sec if base is None else base
            line = {"workload": kind, "rows_per_gpu": B, "mini_batch_num": m, "epochs": EPOCHS,
                    "options": OPTIONS if options else "off", "optimizer_steps_per_learn": steps,
                    "learn_calls_timed": args.steps * args.repeats, "ms_per_learn": round(sec * 1e3, 3),
                    "ms_per_learn_rounds": [round(r[0] * 1e3, 3) for r in runs],
                    "ms_per_step": round(sec * 1e3 / steps, 4), "value": round(B * EPOCHS / sec, 1),
                    "unit": "learner sample-iterations/s", "launches_per_learn": runs[-1][1],
                    "vs_off": round(sec / base - 1.0, 4), "gpu": gpu}
            print(json.dumps(line), flush=True)
        del arms
        torch.cuda.empty_cache()
    for n in (2048, 8192, 65536):
        ms = time_normaliser(n, dev)
        print(json.dumps({"kernel": "adv_normalize_kernel", "rows": n, "us_per_launch": round(ms * 1e3, 2),
                          "note": "one block, local moments (m3 = NULL), in place; back-to-back launches", "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
