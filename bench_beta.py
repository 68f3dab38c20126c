"""Cost of the Beta actor (BetaActor, non-reference) against the Gaussian actor of the C2 nav-laser configuration.

One JSON line per measurement, inputs resident in HBM:
  act     ms per PPO.act call (sampling, log-prob, values) of navlaser vs navlaser_beta at B = 256 and 4096: CUDA events over
          back-to-back calls
  kernel  the head kernel (ddrl_gaussian_head vs ddrl_beta_head, sampling) and the fused loss kernel (ddrl_ppo_loss_gaussian_dc vs
          ddrl_ppo_loss_beta, unshared, PPO_STATS) alone at B = 8192, A = 2: 100 back-to-back launches captured in a CUDA graph,
          CUDA events around its replays (so that the host's launch cost does not hide the kernel's time)
  learn   ms per learn call (TRAINING_ITER_TIME = 10) of navlaser vs navlaser_beta at 1024 rows, and launches per call
Gaussian and Beta run interleaved (gaussian, beta, gaussian, beta, ...) and each is reported as the median of --repeats rounds,
so that drift of the shared machine falls on both arms.  The GPU's name and power limit are read in the same run.  Writes
nothing to the tree."""
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

KINDS = ("navlaser", "navlaser_beta")
EPOCHS = 10


def event_ms(fn, reps):
    """ms per call of `fn` over `reps` back-to-back calls, CUDA events around the whole window."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def interleaved(arms, reps, repeats, warmup=5):
    """arms: {label: fn} -> {label: [ms per call, one per round]}"""
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    runs = {k: [] for k in arms}
    for _ in range(repeats):
        for k, fn in arms.items():
            runs[k].append(event_ms(fn, reps))
    return runs


def graphed(fn, n=100):
    """A callable replaying n back-to-back calls of `fn` captured in one CUDA graph."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n):
            fn()
    return g.replay


def report(measure, runs, gpu, **extra):
    base = statistics.median(runs[KINDS[0]]) if KINDS[0] in runs else None
    for k, r in runs.items():
        ms = statistics.median(r)
        row = {"measure": measure, "arm": k, **extra, "ms": round(ms, 4), "ms_rounds": [round(x, 4) for x in r]}
        if base:
            row["vs_gaussian"] = round(ms / base - 1.0, 4)
        print(json.dumps({**row, "gpu": gpu}), flush=True)


def make(kind, dev, **hyper):
    from ddrl4nav_b200.runner import make_net
    torch.manual_seed(1000)
    return make_net(kind, device=dev, **hyper)


def act_bench(dev, B, args, gpu):
    arms = {}
    for kind in KINDS:
        net = make(kind, dev)
        states = [s.to(dev) for s in bench.synth_batch_host("navlaser", B, seed=1)[0]]
        g = torch.Generator(device=dev).manual_seed(2)
        draw = (torch.randn if kind == "navlaser" else torch.rand)(B, 2, device=dev, generator=g)
        arms[kind] = (lambda n, s, d: (lambda: n.act(s, draw=d)))(net, states, draw)
    report("act", interleaved(arms, args.reps, args.repeats), gpu, rows=B)


def kernel_bench(dev, args, gpu):
    from ddrl4nav_b200 import kernels
    B, A = 8192, 2
    g = torch.Generator(device=dev).manual_seed(3)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    mu, log_std, eps = r(B, A), torch.full((A,), -0.5, device=dev), r(B, A)
    head, u = r(B, 2 * A), torch.rand(B, A, device=dev, generator=g)
    low, high = torch.full((A,), -1.0, device=dev), torch.full((A,), 1.0, device=dev)
    ga, glp = kernels.gaussian_head(mu, log_std, eps)
    ba, blp, _ = kernels.beta_head(head, low, high, u, want_conc=False)
    old, adv, ret, v = r(B), r(B), r(B), r(B)
    hp = kernels.make_hparams(ppo_stats=True)
    heads = {"navlaser": lambda: kernels.gaussian_head(mu, log_std, eps),
             "navlaser_beta": lambda: kernels.beta_head(head, low, high, u, want_conc=False)}
    per_launch = lambda runs: {k: [ms / 100 for ms in r] for k, r in runs.items()}
    runs = interleaved({k: graphed(fn) for k, fn in heads.items()}, args.kernel_reps, args.repeats)
    report("kernel", per_launch(runs), gpu, kernel="head (sampling)", rows=B, act_dim=A)
    losses = {"navlaser": lambda: kernels.ppo_loss_gaussian_dc(mu, log_std, ga, glp + 0.1, adv, ret, v, hp, False),
              "navlaser_beta": lambda: kernels.ppo_loss_beta(head, low, high, ba, blp + 0.1, adv, ret, v, hp, False)}
    runs = interleaved({k: graphed(fn) for k, fn in losses.items()}, args.kernel_reps, args.repeats)
    report("kernel", per_launch(runs), gpu, kernel="ppo loss (unshared, PPO_STATS)", rows=B, act_dim=A)


def learn_bench(dev, args, gpu):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    B = 1024
    arms, launches = {}, {}
    for kind in KINDS:
        net = make(kind, dev, TRAINING_ITER_TIME=EPOCHS)
        states_h, adv_h, ret_h = bench.synth_batch_host("navlaser", B, seed=100)
        states = [s.to(dev) for s in states_h]
        a, lp, _ = net.act(states)
        exp = Experience(states=states, advs=adv_h.to(dev), actions=a, old_logps=lp + 0.1, values=ret_h.to(dev)[None])
        learn = (lambda n, e: (lambda: [None for _ in n.learn(e)]))(net, exp)
        learn()
        kernels.launch_count_reset()
        learn()
        launches[kind] = kernels.launch_count()
        arms[kind] = learn
    runs = interleaved(arms, args.steps, args.repeats, warmup=args.warmup)
    report("learn", runs, gpu, rows=B, epochs=EPOCHS, launches_per_learn=launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200, help="act calls per timed window")
    ap.add_argument("--kernel-reps", dest="kernel_reps", type=int, default=20, help="graph replays (100 launches each) per timed window")
    ap.add_argument("--steps", type=int, default=5, help="learn calls per timed window")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=7, help="interleaved rounds per measurement")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_beta.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    for B in (256, 4096):
        act_bench(dev, B, args, gpu)
    kernel_bench(dev, args, gpu)
    learn_bench(dev, args, gpu)


if __name__ == "__main__":
    main()
