"""Cost of running observation normalisation (NORM_OBS, non-reference) against the default learner and Forward module.

One JSON line per measurement, inputs resident in HBM:
  learn   ms per learn call (TRAINING_ITER_TIME = 10, full batch), option off vs on, for Pong (slot 0) at 8192 rows, navlaser
          (slots 0 and 1) at 1024 rows and mlp at 4096 rows; launches_per_learn = ddrl_launch_count() per call
  act     ms per act() call on Pong at B = 256 and 4096, option off vs on
  kernel  the moments (both passes), normalise and merge kernels alone at Pong size (8192 x 28224 fp32 = 925 MB, larger than
          the 126 MB L2), CUDA events over back-to-back launches; GB/s = the bytes each must move / its time
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
LEARN = (("pong", 8192, True), ("navlaser", 1024, (0, 1)), ("mlp", 4096, True))


def synth(kind, B, seed):
    if kind == "mlp":
        g = torch.Generator().manual_seed(seed)
        return [torch.randn(B, 4, generator=g) * 5.0 + 2.0], torch.randn(B, generator=g), torch.randn(B, generator=g)
    return bench.synth_batch_host(kind, B, seed=seed)


def make_learner(kind, B, norm_obs, dev):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net

    torch.manual_seed(1000)
    net = make_net(kind, device=dev, TRAINING_ITER_TIME=EPOCHS, **({"NORM_OBS": norm_obs} if norm_obs else {}))
    states_h, adv_h, ret_h = synth(kind, B, 100)
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


def make_actor(B, norm_obs, dev):
    from ddrl4nav_b200.runner import make_net
    torch.manual_seed(1000)
    net = make_net("pong", device=dev, **({"NORM_OBS": True} if norm_obs else {}))
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
    B, D = 8192, 4 * 84 * 84
    x = torch.rand(B, D, device=dev)
    out = torch.empty_like(x)
    shift = torch.full((D,), 0.5, dtype=torch.float64, device=dev)
    sums = torch.empty(2 * D, dtype=torch.float64, device=dev)
    ws = torch.empty(kernels.obs_moments_ws_bytes(B, D), dtype=torch.uint8, device=dev)
    mean = torch.zeros(D, dtype=torch.float64, device=dev)
    var = torch.ones(D, dtype=torch.float64, device=dev)
    count = torch.full((1,), 1e-4, dtype=torch.float64, device=dev)
    m32, s32 = torch.zeros(D, device=dev), torch.ones(D, device=dev)
    jobs = {
        "obs_moments (2 passes)": (lambda: kernels.obs_moments(x, shift, sums, ws), 4.0 * B * D + ws.numel() * 2 + 16.0 * D),
        "obs_normalize": (lambda: kernels.obs_normalize(x, m32, s32, 10.0, out), 8.0 * B * D),
        "obs_rms_update": (lambda: kernels.obs_rms_update(mean, var, count, sums, B, m32, s32), 8.0 * 6 * D),
    }
    res = []
    for name, (fn, nbytes) in jobs.items():
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res.append((name, ms, nbytes / (ms * 1e-3) / 1e9))
    return res, (B, D)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3, help="timed learn calls per round (act: 100x as many calls)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5, help="interleaved rounds per configuration")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_obs_norm.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    for kind, B, norm_obs in LEARN:
        arms = {}
        for on in (False, True):
            learn, timer = make_learner(kind, B, norm_obs if on else False, dev)
            for _ in range(args.warmup):
                learn()
            arms[on] = (learn, timer)
        runs = interleaved(arms, args.steps, args.repeats)
        base = statistics.median(r[0] for r in runs[False])
        for on in (False, True):
            sec = statistics.median(r[0] for r in runs[on])
            print(json.dumps({"measure": "learn", "workload": kind, "rows": B, "epochs": EPOCHS,
                              "norm_obs": (list(norm_obs) if isinstance(norm_obs, tuple) else norm_obs) if on else False,
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
            print(json.dumps({"measure": "act", "workload": "pong", "rows": B, "norm_obs": on, "ms_per_act": round(sec * 1e3, 4),
                              "ms_per_act_rounds": [round(r[0] * 1e3, 4) for r in runs[on]], "vs_off": round(sec / base - 1.0, 4),
                              "gpu": gpu}), flush=True)
        del arms
        torch.cuda.empty_cache()
    res, (B, D) = kernel_times(dev, 50)
    for name, ms, gbs in res:
        print(json.dumps({"measure": "kernel", "kernel": name, "rows": B, "elems_per_row": D, "us_per_launch": round(ms * 1e3, 2),
                          "GB_per_s": round(gbs, 1), "note": "back-to-back launches, inputs larger than L2", "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
