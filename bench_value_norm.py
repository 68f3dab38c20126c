"""Cost of value-target normalisation (NORM_VALUE, non-reference, PopArt) against the default learner and Forward module.

One JSON line per measurement, inputs resident in HBM:
  learn   ms per learn call (TRAINING_ITER_TIME = 10, full batch), option off vs on, for Pong at 8192 rows, navlaser at 1024
          rows and mlp at 4096 rows; launches_per_learn = ddrl_launch_count() per call
  act     ms per act() call on Pong at B = 256 and 4096, option off vs on
  kernel  the update kernel alone (merge, applied form and the rescale of a 512-wide head), CUDA events over back-to-back
          launches: it is one block on a few hundred bytes, so its time is launch latency, not bandwidth
Off and on run interleaved (off, on, off, on, ...) and each is reported as the median of --repeats rounds, so that drift of the
shared machine falls on both arms.  The GPU's name and power limit are read in the same run.  Writes nothing to the tree."""
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
LEARN = (("pong", 8192), ("navlaser", 1024), ("mlp", 4096))


def synth(kind, B, seed):
    if kind == "mlp":
        g = torch.Generator().manual_seed(seed)
        return [torch.randn(B, 4, generator=g) * 5.0 + 2.0], torch.randn(B, generator=g), torch.randn(B, generator=g)
    return bench.synth_batch_host(kind, B, seed=seed)


def returns(B, seed):
    """Return targets at a scale the critic does not start at (500 +- 80): what the option is for."""
    return 500.0 + 80.0 * torch.randn(B, generator=torch.Generator().manual_seed(seed))


def make_learner(kind, B, norm_value, dev):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net

    torch.manual_seed(1000)
    net = make_net(kind, device=dev, TRAINING_ITER_TIME=EPOCHS, **({"NORM_VALUE": True} if norm_value else {}))
    states_h, adv_h, _ = synth(kind, B, 100)
    ret_h = returns(B, 101)
    states_d = [s.to(dev) for s in states_h]
    with torch.no_grad():
        acts_d, logp_d, _ = net.act(states_d)
    exp = Experience(states=states_d, advs=adv_h.to(dev), actions=acts_d, old_logps=logp_d + 0.15 * torch.randn(B, device=dev),
                     values=ret_h.to(dev)[None])

    def learn():
        for _ in net.learn(exp):
            pass

    def measure(steps):
        kernels.launch_count_reset()
        sec = bench.timed(learn, steps, 0, None) / steps
        return sec, kernels.launch_count() / steps

    return learn, measure


def make_actor(B, norm_value, dev):
    from ddrl4nav_b200.runner import make_net
    torch.manual_seed(1000)
    net = make_net("pong", device=dev, **({"NORM_VALUE": True} if norm_value else {}))
    states = [s.to(dev) for s in synth("pong", B, 7)[0]]
    draw = torch.rand(B, device=dev)

    def act():
        net.act(states, draw=draw)

    return act, lambda steps: (bench.timed(act, steps, 0, None) / steps, None)


def interleaved(arms, steps, repeats):
    """arms: {label: (warm-up fn, timer)} -> {label: [(sec, launches)] per round}"""
    runs = {k: [] for k in arms}
    for _ in range(repeats):
        for k, (_, timer) in arms.items():
            runs[k].append(timer(steps))
    return runs


def kernel_times(dev, reps):
    from ddrl4nav_b200 import kernels
    B, F = 8192, 512
    x = returns(B, 5).to(dev)
    mean = torch.zeros(1, dtype=torch.float64, device=dev)
    var = torch.ones(1, dtype=torch.float64, device=dev)
    count = torch.full((1,), 1e-4, dtype=torch.float64, device=dev)
    sums = kernels.obs_moments(x, mean)
    ws = torch.empty(kernels.obs_moments_ws_bytes(B, 1), dtype=torch.uint8, device=dev)
    applied = torch.empty(3, device=dev)
    w, b = torch.randn(F, device=dev) * 0.05, torch.zeros(1, device=dev)
    jobs = {
        "obs_moments of the returns (D = 1, 2 passes)": lambda: kernels.obs_moments(x, mean, sums, ws),
        "value_norm_update (merge + applied form + head rescale)": lambda: kernels.value_norm_update(mean, var, count, sums, B,
                                                                                                     applied, w, b),
    }
    res = []
    for name, fn in jobs.items():
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res.append((name, e0.elapsed_time(e1) / reps))
    return res, (B, F)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3, help="timed learn calls per round (act: 100x as many calls)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5, help="interleaved rounds per configuration")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_value_norm.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    for kind, B in LEARN:
        arms = {}
        for on in (False, True):
            learn, timer = make_learner(kind, B, on, dev)
            for _ in range(args.warmup):
                learn()
            arms[on] = (learn, timer)
        runs = interleaved(arms, args.steps, args.repeats)
        base = statistics.median(r[0] for r in runs[False])
        for on in (False, True):
            sec = statistics.median(r[0] for r in runs[on])
            print(json.dumps({"measure": "learn", "workload": kind, "rows": B, "epochs": EPOCHS,
                              "norm_value": on,
                              "ms_per_learn": round(sec * 1e3, 3), "ms_per_learn_rounds": [round(r[0] * 1e3, 3) for r in runs[on]],
                              "launches_per_learn": runs[on][-1][1], "vs_off": round(sec / base - 1.0, 4), "gpu": gpu}), flush=True)
        del arms
        torch.cuda.empty_cache()
    for B in (256, 4096):
        arms = {}
        for on in (False, True):
            act, timer = make_actor(B, on, dev)
            for _ in range(20):
                act()
            arms[on] = (act, timer)
        runs = interleaved(arms, 100 * args.steps, args.repeats)
        base = statistics.median(r[0] for r in runs[False])
        for on in (False, True):
            sec = statistics.median(r[0] for r in runs[on])
            print(json.dumps({"measure": "act", "workload": "pong", "rows": B, "norm_value": on, "ms_per_act": round(sec * 1e3, 4),
                              "ms_per_act_rounds": [round(r[0] * 1e3, 4) for r in runs[on]], "vs_off": round(sec / base - 1.0, 4),
                              "gpu": gpu}), flush=True)
        del arms
        torch.cuda.empty_cache()
    res, (B, F) = kernel_times(dev, 200)
    for name, ms in res:
        print(json.dumps({"measure": "kernel", "kernel": name, "rows": B, "head_width": F, "us_per_launch": round(ms * 1e3, 2),
                          "note": "back-to-back launches", "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
