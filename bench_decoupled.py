"""Cost of the decoupled PPO objective (DECOUPLED_PPO, non-reference) against the default learner, and what it does to a stale batch.

One JSON line per measurement, inputs resident in HBM:
  learn    ms per learn call (TRAINING_ITER_TIME = 10) and launches per call (ddrl_launch_count()), option off vs on, for
           Pong at 8192 rows with MINI_BATCH_NUM 1 and 4, navlaser (the Gaussian actor) at 1024 rows and mlp at 4096 rows
  prepass  the pre-pass alone (ddrl_net_log_prob: the training forward + the log-prob kernel) on Pong at 8192 rows, CUDA events
           over back-to-back calls
  stale    not a speed number: a Pong batch sampled by the policy theta_0 is learned by a net that has taken 10 and 50 optimiser
           steps since (on other batches); the first step's ApproxKL and ClipFrac of that learn call, option off vs on, and
           the BehaviourKL the option reports
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
LEARN = (("pong", 8192, 1), ("pong", 8192, 4), ("navlaser", 1024, 1), ("mlp", 4096, 1))


def synth(kind, B, seed):
    if kind == "mlp":
        g = torch.Generator().manual_seed(seed)
        return [torch.randn(B, 4, generator=g) * 5.0 + 2.0], torch.randn(B, generator=g), torch.randn(B, generator=g)
    return bench.synth_batch_host(kind, B, seed=seed)


def experience(net, kind, B, seed, dev):
    """A batch acted by `net`, with its log-probs made stale by N(0, 0.15) noise."""
    from ddrl4nav_b200.data import Experience
    states_h, adv_h, ret_h = synth(kind, B, seed)
    states_d = [s.to(dev) for s in states_h]
    with torch.no_grad():
        acts_d, logp_d, _ = net.act(states_d)
    g = torch.Generator(device=dev).manual_seed(seed)
    return Experience(states=states_d, advs=adv_h.to(dev), actions=acts_d,
                      old_logps=logp_d + 0.15 * torch.randn(B, device=dev, generator=g), values=ret_h.to(dev)[None])


def make_learner(kind, B, m, on, dev):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.runner import make_net

    torch.manual_seed(1000)
    net = make_net(kind, device=dev, TRAINING_ITER_TIME=EPOCHS, MINI_BATCH_NUM=m, MINI_BATCH_SEED=1,
                   **({"DECOUPLED_PPO": True} if on else {}))
    exp = experience(net, kind, B, 100, dev)

    def learn():
        for _ in net.learn(exp):
            pass

    def measure(steps):
        kernels.launch_count_reset()
        sec = bench.timed(learn, steps, 0, None) / steps
        return sec, kernels.launch_count() / steps

    return learn, measure, net, exp


def interleaved(arms, steps, repeats):
    """arms: {label: (warm-up fn, timer)} -> {label: [(sec, launches)] per round}"""
    runs = {k: [] for k in arms}
    for _ in range(repeats):
        for k, (_, timer) in arms.items():
            runs[k].append(timer(steps))
    return runs


def prepass_time(net, exp, reps):
    from ddrl4nav_b200 import kernels
    out = torch.empty(len(exp.states[0]), device=exp.actions.device)
    fn = lambda: kernels.net_log_prob(net, exp.states, exp.actions, out=out)
    for _ in range(5):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def stale(dev, B, lags):
    """First-step statistics of a learn call on a batch sampled `lag` optimiser steps before the learner's weights."""
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.runner import make_net
    torch.manual_seed(2000)
    src = make_net("pong", device=dev, TRAINING_ITER_TIME=EPOCHS)
    exp = experience(src, "pong", B, 300, dev)
    exp.old_logps = kernels.net_log_prob(src, exp.states, exp.actions).clone()       # exactly theta_0's log-probs
    res, done = [], 0
    for lag in lags:
        call = 0
        while done < lag:
            for _ in src.learn(experience(src, "pong", B, 400 + call, dev)):
                done += 1
            call += 1
        row = {"lag_steps": done}
        for on in (False, True):
            net = make_net("pong", device=dev, TRAINING_ITER_TIME=1, PPO_STATS=True, **({"DECOUPLED_PPO": True} if on else {}))
            net.load_state_dict(src.state_dict())
            (log, _, _), = net.learn(exp)
            row["on" if on else "off"] = {k: log[k] for k in ("ApproxKL", "ClipFrac", "BehaviourKL") if k in log}
        res.append(row)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3, help="timed learn calls per round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=5, help="interleaved rounds per configuration")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_decoupled.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    for kind, B, m in LEARN:
        arms, keep = {}, {}
        for on in (False, True):
            learn, timer, net, exp = make_learner(kind, B, m, on, dev)
            for _ in range(args.warmup):
                learn()
            arms[on] = (learn, timer)
            keep[on] = (net, exp)
        runs = interleaved(arms, args.steps, args.repeats)
        base = statistics.median(r[0] for r in runs[False])
        for on in (False, True):
            sec = statistics.median(r[0] for r in runs[on])
            print(json.dumps({"measure": "learn", "workload": kind, "rows": B, "minibatches": m, "epochs": EPOCHS,
                              "decoupled": on, "ms_per_learn": round(sec * 1e3, 3),
                              "ms_per_learn_rounds": [round(r[0] * 1e3, 3) for r in runs[on]],
                              "launches_per_learn": runs[on][-1][1], "vs_off": round(sec / base - 1.0, 4), "gpu": gpu}), flush=True)
        if kind == "pong" and m == 1:
            ms = prepass_time(*keep[True], 50)
            print(json.dumps({"measure": "prepass", "workload": kind, "rows": B, "ms_per_call": round(ms, 3),
                              "note": "ddrl_net_log_prob alone, back-to-back calls", "gpu": gpu}), flush=True)
        del arms, keep
        torch.cuda.empty_cache()
    for row in stale(dev, 2048, (10, 50)):
        print(json.dumps({"measure": "stale", "workload": "pong", "rows": 2048, **row,
                          "note": "first step of the learn call; illustrates the objective, not a speed number", "gpu": gpu}),
              flush=True)


if __name__ == "__main__":
    main()
