"""Cost of the MultiDiscrete actor (MultiCategoricalActor, non-reference) against the flat categorical actor it factors.

One JSON line per measurement, inputs resident in HBM:
  act     ms per PPO.act call (sampling, log-prob, values): navimg (a flat Categorical over the 28 (v, w) commands) against
          navimg_md (4 speeds x 7 turn rates, head width 11) at B = 256 and 4096; CUDA events over back-to-back calls
  kernel  the head kernel (ddrl_categorical_head vs ddrl_multi_categorical_head, sampling) and the fused loss kernel
          (ddrl_ppo_loss_categorical_m vs ddrl_ppo_loss_multi_categorical, shared, PPO_STATS) alone at B = 8192: 100 back-to-back
          launches captured in a CUDA graph, CUDA events around its replays.  Three arms: the flat head of width 28, the (4, 7)
          head of width 11 (what a user switching navimg to navimg_md runs), and a (4, 7, 17) head of width 28 (the branch loop
          at the flat head's width)
  learn   ms per learn call (TRAINING_ITER_TIME = 10) of navimg against navimg_md at 2048 rows, and launches per call
The arms run interleaved (flat, md, flat, md, ...) and each is reported as the median of --repeats rounds, so that drift of the
shared machine falls on all of them.  The GPU's name and power limit are read in the same run.  Writes nothing to the tree."""
import argparse
import sys

import torch

import bench
import bench_action_mask as ba
import bench_beta as bb
from bench_minibatch import gpu_info

EPOCHS = 10
NVEC = (4, 7)


def report(measure, runs, gpu, **extra):
    import json
    import statistics
    base = statistics.median(runs["flat"])
    for k, r in runs.items():
        ms = statistics.median(r)
        row = {"measure": measure, "arm": k, **extra, "ms": round(ms, 4), "ms_rounds": [round(x, 4) for x in r],
               "vs_flat": round(ms / base - 1.0, 4)}
        print(json.dumps({**row, "gpu": gpu}), flush=True)


def act_bench(dev, B, args, gpu):
    states = [s.to(dev) for s in bench.synth_batch_host("navimg", B, seed=1)[0]]
    g = torch.Generator(device=dev).manual_seed(2)
    draws = {"flat": torch.rand(B, device=dev, generator=g), "md": torch.rand(B, len(NVEC), device=dev, generator=g)}
    arms = {}
    for arm, kind in (("flat", "navimg"), ("md", "navimg_md")):
        net = bb.make(kind, dev)
        arms[arm] = (lambda n, d: (lambda: n.act(states, draw=d)))(net, draws[arm])
    report("act", bb.interleaved(arms, args.reps, args.repeats), gpu, rows=B, nvec={"flat": [28], "md": list(NVEC)})


def kernel_bench(dev, args, gpu):
    from ddrl4nav_b200 import kernels
    B = 8192
    g = torch.Generator(device=dev).manual_seed(3)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    nvecs = {"flat": (28,), "md": NVEC, "md_w28": (4, 7, 17)}
    logits = {k: 2 * r(B, sum(n)) for k, n in nvecs.items()}
    u = {k: torch.rand(B, len(n), device=dev, generator=g) for k, n in nvecs.items()}
    mask = {k: ba.mask_of(B, sum(n), dev).float() for k, n in nvecs.items()}
    adv, ret, v = r(B), r(B), r(B)
    hp = kernels.make_hparams(ppo_stats=True)
    per_launch = lambda runs: {k: [ms / 100 for ms in r] for k, r in runs.items()}
    for masked in (False, True):
        m = lambda k: mask[k] if masked else None
        heads = {"flat": lambda: kernels.categorical_head_m(logits["flat"], u["flat"].view(B), m("flat"), want_probs=False)}
        for k in ("md", "md_w28"):
            heads[k] = (lambda k: lambda: kernels.multi_categorical_head(logits[k], nvecs[k], u[k], m(k), want_probs=False))(k)
        runs = bb.interleaved({k: bb.graphed(fn) for k, fn in heads.items()}, args.kernel_reps, args.repeats)
        report("kernel", per_launch(runs), gpu, kernel="head (sampling)", masked=masked, rows=B, nvec=nvecs)
        losses = {}
        for k, n in nvecs.items():
            a, lp, _ = kernels.multi_categorical_head(logits[k], n, u[k], m(k), want_probs=False)
            lp = lp + 0.1
            if k == "flat":
                losses[k] = (lambda a, lp: lambda: kernels.ppo_loss_categorical_m(logits["flat"], a.view(B), lp, adv, ret,
                                                                                  v, hp, True, mask=m("flat")))(a, lp)
            else:
                losses[k] = (lambda k, a, lp: lambda: kernels.ppo_loss_multi_categorical(logits[k], nvecs[k], a, lp, adv, ret,
                                                                                         v, hp, True, mask=m(k)))(k, a, lp)
        runs = bb.interleaved({k: bb.graphed(fn) for k, fn in losses.items()}, args.kernel_reps, args.repeats)
        report("kernel", per_launch(runs), gpu, kernel="ppo loss (shared, PPO_STATS)", masked=masked, rows=B, nvec=nvecs)


def learn_bench(dev, args, gpu):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    B = 2048
    states_h, adv_h, ret_h = bench.synth_batch_host("navimg", B, seed=100)
    states = [s.to(dev) for s in states_h]
    arms, launches = {}, {}
    for arm, kind in (("flat", "navimg"), ("md", "navimg_md")):
        net = bb.make(kind, dev, TRAINING_ITER_TIME=EPOCHS)
        a, lp, _ = net.act(states)
        exp = Experience(states=states, advs=adv_h.to(dev), actions=a, old_logps=lp + 0.1, values=ret_h.to(dev)[None])
        learn = (lambda n, e: (lambda: [None for _ in n.learn(e)]))(net, exp)
        learn()
        kernels.launch_count_reset()
        learn()
        launches[arm] = kernels.launch_count()
        arms[arm] = learn
    report("learn", bb.interleaved(arms, args.steps, args.repeats, warmup=args.warmup), gpu, rows=B, epochs=EPOCHS,
           launches_per_learn=launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200, help="act calls per timed window")
    ap.add_argument("--kernel-reps", dest="kernel_reps", type=int, default=20, help="graph replays (100 launches each) per timed window")
    ap.add_argument("--steps", type=int, default=5, help="learn calls per timed window")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=7, help="interleaved rounds per measurement")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_multi_discrete.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    for B in (256, 4096):
        act_bench(dev, B, args, gpu)
    kernel_bench(dev, args, gpu)
    learn_bench(dev, args, gpu)


if __name__ == "__main__":
    main()
