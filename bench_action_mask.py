"""Cost of invalid-action masking (ACTION_MASK, non-reference) on the categorical actor.

One JSON line per measurement, inputs resident in HBM, masks u8 0/1 with ~70 % of the actions allowed:
  act     ms per PPO.act call (sampling, log-prob, values) without and with the mask: navimg (A = 28) at B = 256 and 4096, pong
          (A = 6) at B = 4096; CUDA events over back-to-back calls
  kernel  the head kernel (ddrl_categorical_head vs ddrl_categorical_head_m, sampling) and the fused loss kernel
          (ddrl_ppo_loss_categorical_dc vs ddrl_ppo_loss_categorical_m, shared, PPO_STATS) alone at B = 8192, A = 28: 100
          back-to-back launches captured in a CUDA graph, CUDA events around its replays
  learn   ms per learn call (TRAINING_ITER_TIME = 10) of navimg at 2048 rows without and with the mask, and launches per call
The two arms run interleaved (off, mask, off, mask, ...) and each is reported as the median of --repeats rounds, so that drift
of the shared machine falls on both.  The GPU's name and power limit are read in the same run.  Writes nothing to the tree."""
import argparse
import sys

import torch

import bench
import bench_beta as bb
from bench_minibatch import gpu_info

ARMS = ("off", "mask")
EPOCHS = 10


def report(measure, runs, gpu, **extra):
    import json
    import statistics
    base = statistics.median(runs["off"])
    for k, r in runs.items():
        ms = statistics.median(r)
        row = {"measure": measure, "arm": k, **extra, "ms": round(ms, 4), "ms_rounds": [round(x, 4) for x in r],
               "vs_off": round(ms / base - 1.0, 4)}
        print(json.dumps({**row, "gpu": gpu}), flush=True)


def mask_of(B, A, dev, seed=5):
    g = torch.Generator(device=dev).manual_seed(seed)
    return (torch.rand(B, A, device=dev, generator=g) < 0.7).to(torch.uint8)


def act_bench(dev, kind, B, args, gpu):
    A = {"navimg": 28, "pong": 6}[kind]
    states = [s.to(dev) for s in bench.synth_batch_host(kind, B, seed=1)[0]]
    draw = torch.rand(B, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    mask = mask_of(B, A, dev).float()
    arms = {}
    for arm in ARMS:
        net = bb.make(kind, dev, ACTION_MASK=arm == "mask")
        st = states + [mask] if arm == "mask" else states
        arms[arm] = (lambda n, s: (lambda: n.act(s, draw=draw)))(net, st)
    report("act", bb.interleaved(arms, args.reps, args.repeats), gpu, kind=kind, rows=B, act_dim=A)


def kernel_bench(dev, args, gpu):
    from ddrl4nav_b200 import kernels
    B, A = 8192, 28
    g = torch.Generator(device=dev).manual_seed(3)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    logits, u = 2 * r(B, A), torch.rand(B, device=dev, generator=g)
    mask = mask_of(B, A, dev).float()
    a, lp, _ = kernels.categorical_head_m(logits, u, mask, want_probs=False)
    adv, ret, v = r(B), r(B), r(B)
    hp = kernels.make_hparams(ppo_stats=True)
    per_launch = lambda runs: {k: [ms / 100 for ms in r] for k, r in runs.items()}
    heads = {"off": lambda: kernels.categorical_head(logits, u, want_probs=False),
             "mask": lambda: kernels.categorical_head_m(logits, u, mask, want_probs=False)}
    runs = bb.interleaved({k: bb.graphed(fn) for k, fn in heads.items()}, args.kernel_reps, args.repeats)
    report("kernel", per_launch(runs), gpu, kernel="head (sampling)", rows=B, act_dim=A)
    losses = {"off": lambda: kernels.ppo_loss_categorical_dc(logits, a, lp + 0.1, adv, ret, v, hp, True),
              "mask": lambda: kernels.ppo_loss_categorical_m(logits, a, lp + 0.1, adv, ret, v, hp, True, mask=mask)}
    runs = bb.interleaved({k: bb.graphed(fn) for k, fn in losses.items()}, args.kernel_reps, args.repeats)
    report("kernel", per_launch(runs), gpu, kernel="ppo loss (shared, PPO_STATS)", rows=B, act_dim=A)


def learn_bench(dev, args, gpu):
    from ddrl4nav_b200 import kernels
    from ddrl4nav_b200.data import Experience
    kind, B, A = "navimg", 2048, 28
    states_h, adv_h, ret_h = bench.synth_batch_host(kind, B, seed=100)
    states = [s.to(dev) for s in states_h]
    mask = mask_of(B, A, dev).float()
    arms, launches = {}, {}
    for arm in ARMS:
        net = bb.make(kind, dev, TRAINING_ITER_TIME=EPOCHS, ACTION_MASK=arm == "mask")
        st = states + [mask] if arm == "mask" else states
        a, lp, _ = net.act(st)
        exp = Experience(states=st, advs=adv_h.to(dev), actions=a, old_logps=lp + 0.1, values=ret_h.to(dev)[None])
        learn = (lambda n, e: (lambda: [None for _ in n.learn(e)]))(net, exp)
        learn()
        kernels.launch_count_reset()
        learn()
        launches[arm] = kernels.launch_count()
        arms[arm] = learn
    report("learn", bb.interleaved(arms, args.steps, args.repeats, warmup=args.warmup), gpu, kind=kind, rows=B, epochs=EPOCHS,
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
        sys.exit("bench_action_mask.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    gpu = gpu_info(0)
    for kind, B in (("navimg", 256), ("navimg", 4096), ("pong", 4096)):
        act_bench(dev, kind, B, args, gpu)
    kernel_bench(dev, args, gpu)
    learn_bench(dev, args, gpu)


if __name__ == "__main__":
    main()
