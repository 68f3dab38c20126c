#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the DDRL4NAV actor-learner hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload pong|navlaser|navimg|navlaser3] [--impl reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one Backward-module learn call on one batch = TRAINING_ITER_TIME (10) full-batch PPO
iterations (forward + fused loss + backward + [NCCL all-reduce] + fused clip+Adam), exactly what
BackwardTrainThread does per batch (USTC_lab/server/backward.py:182-189, nn/ppo.py:77-142).
value   = learner sample-iterations/s over all ranks, inputs resident in HBM (metric of BASELINE.json).
e2e     = the same through the public API (BackwardModule.train_on) from PINNED HOST buffers: H2D of the
          batch and D2H of the losses inside the timed region, every step.
extra   = Forward-module actions/s (PPO.act), GAE elements/s, per-kernel-class device time.
--impl reference = the reference's CPU path (oracle port, torch CPU, all host threads), rank 0 only.
--dump-outputs DIR = after the K timed learn calls, rank 0 writes what the last one handed its caller: DIR/losses.npy (float64
          [iterations, 4]: PpoTotalLoss, ActorLoss, VLoss, EntLoss) and DIR/param.<name>.npy (float32, every parameter after
          the call).  Inputs, initial weights and sampling draws are seeded, and the whole run uses the engine's deterministic
          mode (DESIGN.md section 3; config.deterministic in the JSON line): the default mode adds block partials with
          unordered atomics, and Adam amplifies their last-bit differences from iteration to iteration (weights 1e-2 apart
          after 5 learn calls), so only deterministic mode writes the same files every run.  Two builds that add in a
          different order still differ in the last bits, which Adam amplifies the same way: compare them with a tolerance.
          The whole run, timings included, is of deterministic mode, which covers the tc3 engine only (--gemm-mode tc3) and
          is slower (Pong: 67 vs 48 ms per step on one B200 at a 1000 W power limit); time the default mode without
          --dump-outputs.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "PPO learner samples/s & batched policy actions/s at 1/2/4/8 B200"

# per-GPU batch of the named BASELINE.json configs (weak scaling: fixed per GPU)
WORKLOADS = {
    # C4 = "8xB200 data-parallel learner: Pong PPO batch 64k, minibatch sharded" -> 8192 rows per GPU
    "pong": dict(batch=8192, fwd_batch=32768, cpu_batch=1024, ref_batch=8192, desc="Pong PPO learner, NatureCNN 4x84x84, unshared towers, "
                 "6-way categorical (BASELINE C1/C4: 64k batch at 8 GPUs = 8192 rows/GPU)",
                 flops_fwd=37.37e6, flops_learn=99.0e6, obs_bytes=112896),
    # C2 = "robot-nav PPO: laser-scan + goal/vel vector, Gaussian policy" (reference shapes: 1x960 + 5 + 3x48x48)
    "navlaser": dict(batch=1024, fwd_batch=4096, cpu_batch=128, ref_batch=256, desc="robot-nav PPO learner, NavPreNet1D laser 1x960 + vec5 + "
                     "ped-map 3x48x48, unshared towers, 2-d Gaussian (BASELINE C2)",
                     flops_fwd=545.3e6, flops_learn=1562.6e6, obs_bytes=31508),
    # NOT a reference configuration (SURVEY 8d asks for it beside C2, labelled): BASELINE's "3 x 960" laser wording -- the same
    # stack with Conv1d(3, 32, 5, 2); 3-frame laser stacking is an env option only, no shipped encoder consumes it
    "navlaser3": dict(batch=1024, fwd_batch=4096, cpu_batch=128, ref_batch=256, desc="NON-REFERENCE variant of C2: NavPreNet1D with a "
                      "3x960 laser (Conv1d(3,32,5,2)) + vec5 + ped-map 3x48x48, unshared towers, 2-d Gaussian",
                      flops_fwd=545.9e6, flops_learn=1563.8e6, obs_bytes=39188),
    # C5 = "nav image-env PPO (1x48x48 egocentric map), shared encoder, 28-way categorical"
    "navimg": dict(batch=2048, fwd_batch=8192, cpu_batch=256, ref_batch=1024, desc="nav image-env PPO learner, NavPreNet 1x48x48 + vec9, shared "
                   "encoder, 28-way categorical (BASELINE C5)",
                   flops_fwd=183.0e6, flops_learn=546.4e6, obs_bytes=9252),
}
ITERS = 10          # TRAINING_ITER_TIME, config/config_nn.py:45


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        pk = dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor_sustained=d["bf16_tflops_sustained"], src="measured")
    else:
        pk = dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, src="fallback")
    # tcgen05 issue-rate ceilings measured by this repo (scratch/mma_bench.cu -> profiles/tf32_peak.json): what a 3-product
    # split engine can reach at best is a third of the kind::tf32 / kind::f16 rate
    pk["tf32_issue"], pk["f16_issue"] = 1116.4, 2232.7
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "tf32_peak.json")))
        rates = {(m["kind"], m["N"], m["a"]): m["chip_tflops_sustained"] for m in t["tcgen05"]["mma"]}
        pk["tf32_issue"], pk["f16_issue"] = rates[("tf32", 128, "tmem")], rates[("f16", 128, "tmem")]
    except Exception:  # noqa: BLE001
        pass
    return pk


class ClockSampler:
    """Samples SM clock + throttle reasons during the timed region (pynvml, 100 ms period)."""

    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self.index = index
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = str(e)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture of this same workload (profiles/ncu_traffic.json; null when there is no capture for it)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(p))
        return d[workload][kernel]["bytes_per_launch"]
    except Exception:  # noqa: BLE001
        return None


def synth_states(kind, B, seed):
    """Synthetic observations of the named shapes (SURVEY 8d): Pong frames U[0,1) [B,4,84,84]; nav-laser scan U[0,1)
    [B,1,960] + N(0,1) vector [B,5] + sparse pedestrian map [B,3,48,48] (3 % occupied cells carrying U(-.5,.5)
    velocities); nav-image map U[0,1) [B,1,48,48] + N(0,1) vector [B,9].  (The product arm generates its own inputs:
    nothing under oracle/ is imported outside the cpu_baseline / --impl reference legs.)"""
    g = torch.Generator().manual_seed(seed)
    if kind == "pong":
        return [torch.rand(B, 4, 84, 84, generator=g)]
    if kind in ("navlaser", "navlaser3"):
        laser = torch.rand(B, 3 if kind == "navlaser3" else 1, 960, generator=g)
        vec = torch.randn(B, 5, generator=g)
        occ = (torch.rand(B, 1, 48, 48, generator=g) < 0.03).float()
        vel = (torch.rand(B, 2, 48, 48, generator=g) - 0.5) * occ
        return [laser, vec, torch.cat([occ, vel], dim=1)]
    if kind == "navimg":
        return [torch.rand(B, 1, 48, 48, generator=g), torch.randn(B, 9, generator=g)]
    raise ValueError(kind)


def synth_batch_host(kind, B, seed):
    """Synthetic rollouts of the named observation shape (SURVEY 8d), as host fp32 tensors."""
    states = synth_states(kind, B, seed=seed)
    g = torch.Generator().manual_seed(seed + 17)
    adv = torch.randn(B, generator=g)
    ret = torch.randn(B, generator=g)
    return states, adv, ret


def wl_dist(kind):
    """True for the categorical (1-D action) workloads."""
    return kind not in ("navlaser", "navlaser3")


def encode_forward_payload(arrays, per_env):
    """Forward payload in the reference's wire format (data/easybytes.py:62-75,141-148): one message per env process of
    `per_env` rows: [length >Q][ip 4 x >H][process_env_id >I][blocks: type >h | count >I | ndim >I | shape >I.. | raw]."""
    import struct
    code = {np.dtype(np.uint8): 1, np.dtype(np.float16): 2, np.dtype(np.float32): 3, np.dtype(np.float64): 4}
    B = len(arrays[0])
    out = []
    for j, r0 in enumerate(range(0, B, per_env)):
        body = b""
        for a in arrays:
            sl = np.ascontiguousarray(a[r0:r0 + per_env])
            body += struct.pack(">hII", code[sl.dtype], sl.size, sl.ndim) + struct.pack(">" + "I" * sl.ndim, *sl.shape) + sl.tobytes()
        out.append(struct.pack(">Q", len(body)) + struct.pack(">HHHH", 10, 0, 0, 1) + struct.pack(">I", j) + body)
    return b"".join(out)


def timed(fn, steps, warmup, dist=None):
    """W warm-up + K timed calls bracketed by barrier + synchronize; device time by CUDA events on the current
    stream; returns max-over-ranks seconds."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sec = e0.elapsed_time(e1) / 1e3
    if dist is not None:
        t = torch.tensor([sec], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    return sec


def run_ours(args):
    import ctypes as C
    from ddrl4nav_b200 import _lib, kernels
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net
    from ddrl4nav_b200.server import BackwardModule, ForwardModule

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # the initial weights, the actions sampled for the batch and the old log-prob noise come from torch's global generators
    torch.manual_seed(1000 + rank)
    if args.dump_outputs:
        kernels.set_deterministic(True)
    # host threads and the pinned buffers they allocate next to the GPU's PCIe root (ddrl4nav_b200.dist.bind_host_to_device);
    # DDRL_NO_NUMA_BIND=1 leaves the placement to the scheduler
    from ddrl4nav_b200.dist import bind_host_to_device
    host_bind = None if os.environ.get("DDRL_NO_NUMA_BIND") == "1" else bind_host_to_device(local)
    dist = None
    saved_stdout = None
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: NCCL writes its version banner to fd 1 from C (at NCCL_DEBUG=VERSION and
        # above), so fd 1 points at stderr until the line is printed
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod
    wl = WORKLOADS[args.workload]
    B = args.batch or wl["batch"]
    peaks = load_peaks()
    lib = _lib.load()

    net = make_net(args.workload, device=dev, gemm_mode=args.gemm_mode, TRAINING_ITER_TIME=ITERS)
    collective = "none (1 GPU)"
    if dist is not None:
        net.enable_data_parallel()
        net.broadcast_parameters(0)
        collective = ("own peer-memory all-reduce kernel (NVSwitch multicast)" if net._peer and net._peer["mc"] else
                      "own peer-memory all-reduce kernel (peer loads/stores)" if net._peer else "NCCL all_reduce")
        if os.environ.get("DDRL_DP_OVERLAP") == "1":
            collective = "NCCL all_reduce per backward segment, under the backward"
    # ---- synthetic rollout shard of this rank (different rows per rank), host + device copies
    states_h, adv_h, ret_h = synth_batch_host(args.workload, B, seed=100 + rank)
    states_d = [s.to(dev) for s in states_h]
    with torch.no_grad():
        acts_d, logp_d, _ = net.act(states_d)                 # actions sampled from the net (SURVEY 8d)
    old_d = logp_d + 0.15 * torch.randn(B, device=dev)
    exp_dev = Experience(states=states_d, advs=adv_h.to(dev), actions=acts_d, old_logps=old_d, values=ret_h.to(dev)[None])
    pin = lambda t: t.contiguous().pin_memory()
    host_fields = dict(states=[pin(s) for s in states_h], advs=pin(adv_h), actions=pin(acts_d.cpu()),
                       old_logps=pin(old_d.cpu()), values=pin(ret_h[None]))
    h2d_bytes = sum(t.numel() * 4 for t in host_fields["states"]) + sum(
        host_fields[k].numel() * 4 for k in ("advs", "actions", "old_logps", "values"))

    # ---- headline: K learn calls, inputs resident in HBM
    last_losses = {}
    step_losses = []                    # the loss dicts of the latest learn call, one per iteration

    def step_resident():
        step_losses.clear()
        for loss, upd, last in net.learn(exp_dev):
            last_losses.update(loss)
            step_losses.append(loss)

    if args.profile_step:
        for _ in range(args.warmup):
            step_resident()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return

    sampler = ClockSampler(local)
    kernels.launch_count_reset()
    for _ in range(args.warmup):
        step_resident()
    kernels.launch_count_reset()
    sampler.start()
    sec = timed(step_resident, args.steps, 0, dist)
    launches = kernels.launch_count()
    clocks = sampler.stop()
    value = world * B * ITERS * args.steps / sec
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_losses, net)

    # ---- e2e: same metric through BackwardModule.train_on from pinned host buffers (H2D + D2H per step)
    bm = BackwardModule(net, device=dev)

    def host_exp():
        return Experience(states=list(host_fields["states"]), advs=host_fields["advs"], actions=host_fields["actions"],
                          old_logps=host_fields["old_logps"], values=host_fields["values"])

    pending = [None]

    def step_e2e():
        # every step copies ONE batch host->device inside the timed region: the NEXT step's batch, on the copy stream,
        # while this step's batch trains (BackwardModule.prefetch = the reference's concurrent BackwardGetDataThread);
        # the first batch was copied by the warm-up step, the last prefetched one is never trained on: K copies, K steps
        cur = pending[0]
        if cur is None:
            cur = host_exp()
        nxt = host_exp()
        bm.prefetch(nxt)
        logs = bm.train_on(cur)                            # 10 iterations; 16-byte D2H of the losses each
        pending[0] = nxt
        return logs

    sec_e2e = timed(step_e2e, max(2, args.steps // 2), 2, dist)     # 2 warm-up steps: the first also fills the prefetch pipeline
    e2e_value = world * B * ITERS * max(2, args.steps // 2) / sec_e2e
    pending[0] = None

    # ---- per-kernel-class device time of ONE learn call (separate pass: events after every launch)
    prof = {}
    torch.cuda.synchronize()
    lib.ddrl_prof_start(C.c_void_p(torch.cuda.current_stream().cuda_stream))
    step_resident()
    buf = C.create_string_buffer(1 << 16)
    lib.ddrl_prof_stop(buf, len(buf))
    for line in buf.value.decode().splitlines():
        name, ms, n, work = line.split()
        prof[name] = dict(ms=float(ms), launches=int(n), work=float(work))
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    gemm_names = [k for k in prof if "gemm" in k or "tc2" in k or "tc3" in k or "conv_tc" in k]
    dom = max(prof, key=lambda k: prof[k]["ms"])
    if dom in gemm_names:
        # achieved = ALGORITHMIC flops of the launches of the dominant kernel (the launchers declare 2*M*N*K of the
        # convolution / GEMM they implement, not of the zero-padded tiles they issue) / their CUDA-event time
        ach = prof[dom]["work"] / (prof[dom]["ms"] / 1e3) / 1e12
        split = {"tc3": ("f16", peaks["f16_issue"]), "tc2": ("tf32", peaks["tf32_issue"]), "tc": ("tf32", peaks["tf32_issue"])}.get(args.gemm_mode)
        roof = dict(bound="tensor", kernel=dom, achieved=round(ach, 2), peak=peaks["tensor_sustained"], unit="TFLOP/s",
                    frac=round(ach / peaks["tensor_sustained"], 4), traffic=ncu_traffic(args.workload, dom),
                    peak_note="frac: of the bf16 cuBLAS sustained rate (%s, MEASURED_PEAKS.json).  The engine computes fp32 results "
                              "as THREE kind::%s products: its ceiling is a third of the tcgen05 kind::%s issue rate measured by "
                              "scratch/mma_bench.cu (profiles/tf32_peak.json), reported as frac_split3" % (
                                  peaks["src"], split[0] if split else "-", split[0] if split else "-"),
                    share_of_step=round(prof[dom]["ms"] / tot_ms, 3), avg_launch_ms=round(prof[dom]["ms"] / prof[dom]["launches"], 4))
        if split:
            roof["split3_peak"] = round(split[1] / 3.0, 1)
            roof["frac_split3"] = round(ach / (split[1] / 3.0), 4)
        all_tc_ms = sum(prof[k]["ms"] for k in gemm_names)
        roof["all_gemm_kernels"] = dict(share_of_step=round(all_tc_ms / tot_ms, 3),
                                        achieved=round(sum(prof[k]["work"] for k in gemm_names) / (all_tc_ms / 1e3) / 1e12, 2))
    else:
        ach = prof[dom]["work"] / (prof[dom]["ms"] / 1e3) / 1e9
        roof = dict(bound="hbm", kernel=dom, achieved=round(ach, 1), peak=peaks["hbm"], unit="GB/s",
                    frac=round(ach / peaks["hbm"], 4), traffic=None, share_of_step=round(prof[dom]["ms"] / tot_ms, 3),
                    avg_launch_ms=round(prof[dom]["ms"] / prof[dom]["launches"], 4))
    kernel_shares = {k: round(v["ms"] / tot_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    # ---- Forward module: actions/s (resident) and e2e (ForwardModule.step from host arrays)
    Bf = args.fwd_batch or wl["fwd_batch"]
    fstates_h, _, _ = synth_batch_host(args.workload, Bf, seed=200 + rank)
    fstates_d = [s.to(dev) for s in fstates_h]
    # the Forward module is its own process with its own net object in the reference (predictor vs trainer managers): an
    # inference-only engine instance (no training workspace) with the learner's current weights
    fnet = make_net(args.workload, device=dev, gemm_mode=args.gemm_mode)
    fnet.load_state_dict(net.state_dict())
    sec_f = timed(lambda: fnet.act(fstates_d), 5, 3, dist)
    fwd_value = world * Bf * 5 / sec_f
    fm = ForwardModule(fnet, device=dev)
    f_np = [s.numpy() for s in fstates_h]
    sec_fe = timed(lambda: fm.step(f_np), 3, 2, dist)
    fwd_e2e = world * Bf * 3 / sec_fe
    # ... the Forward tick as the reference runs it (server/forward.py:117-181): a Redis payload of env-process messages in,
    # reply bytes out -- ForwardModule.step_bytes_replies from a PINNED payload: H2D of the wire bytes (streamed in chunks),
    # decode + net + sampling + reply encode on the device, D2H of the replies, all inside the timed region.  Wire dtypes:
    # the reference's Pong wrapper emits float64 frames (warputils.py:300); uint8 frames are what the emulator produces.
    fwd_wire = {}
    per_env = 64
    wires = (("u8", np.uint8), ("f64", np.float64), ("f32", np.float32)) if args.workload == "pong" else (("f32", np.float32),)
    if args.profile_forward:
        # one Forward tick (first wire dtype) and one GAE scan between cudaProfilerStart/Stop, for the ncu metric passes
        # over the HBM-bound kernels (decode, heads, sampling, reply encode, GAE)
        arrs = [(a * 255).astype(np.uint8) if (i == 0 and wires[0][1] is np.uint8) else a for i, a in enumerate(f_np)]
        payload = torch.frombuffer(bytearray(encode_forward_payload(arrs, per_env)), dtype=torch.uint8).pin_memory()
        gv, gr = torch.randn(2049, 1, 16384, device=dev), torch.randn(2048, 1, 16384, device=dev)
        gd = (torch.rand(2048, 1, 16384, device=dev) < 0.02).to(torch.uint8)
        for _ in range(2):
            fm.step_bytes_replies(payload, per_env)
            kernels.gae(gv, gr, gd, [0.99], 0.95)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        fm.step_bytes_replies(payload, per_env)
        kernels.gae(gv, gr, gd, [0.99], 0.95)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return
    for tag, dt in wires:
        rows_w = Bf // 4 if dt is np.float64 else Bf          # float64 frames are 8 bytes per pixel: a quarter batch bounds the payload
        arrs = [(a[:rows_w] * 255).astype(np.uint8) if (i == 0 and dt is np.uint8) else (a[:rows_w].astype(dt) if i == 0 else a[:rows_w])
                for i, a in enumerate(f_np)]
        payload = torch.frombuffer(bytearray(encode_forward_payload(arrs, per_env)), dtype=torch.uint8).pin_memory()
        sec_w = timed(lambda: fm.step_bytes_replies(payload, per_env), 3, 4, dist)
        fwd_wire[tag] = {"value": round(world * rows_w * 3 / sec_w, 1), "rows_per_gpu": rows_w, "h2d_bytes_per_step": int(payload.numel()),
                         "d2h_bytes_per_step": int(lib.ddrl_easybytes_reply_bytes(per_env, 0 if wl_dist(args.workload) else 2, 1)) * (rows_w // per_env)}
        del payload, arrs
    # ... and the batch grid of SURVEY 8(d): resident actions/s and per-call latency at B = 256 / 4096 / Bf (the live
    # predictor runs at a few hundred rows per tick, server/forward.py:117-131)
    fwd_grid = {}
    for bq in (256, 4096):
        if bq >= Bf:
            continue
        sq = [s[:bq].contiguous() for s in fstates_d]
        sec_q = timed(lambda: fnet.act(sq), 20, 5, dist)
        arrs_q = [(a[:bq] * 255).astype(np.uint8) if (i == 0 and args.workload == "pong") else a[:bq] for i, a in enumerate(f_np)]
        pay_q = torch.frombuffer(bytearray(encode_forward_payload(arrs_q, per_env)), dtype=torch.uint8).pin_memory()
        sec_qe = timed(lambda: fm.step_bytes_replies(pay_q, per_env), 10, 3, dist)
        fwd_grid[str(bq)] = {"actions_per_s": round(world * bq * 20 / sec_q, 1), "latency_ms": round(sec_q / 20 * 1e3, 4),
                             "e2e_actions_per_s": round(world * bq * 10 / sec_qe, 1), "e2e_latency_ms": round(sec_qe / 10 * 1e3, 4),
                             "e2e_wire": "u8" if args.workload == "pong" else "f32", "e2e_h2d_bytes": int(pay_q.numel())}

    # ---- GAE: BASELINE C3 corner 64k envs x T=2048 (2.28 GB algorithmic traffic), columns sharded over ranks
    T, N = 2048, 65536
    gv = torch.randn(T + 1, 1, N, device=dev)
    gr = torch.randn(T, 1, N, device=dev)
    gd = (torch.rand(T, 1, N, device=dev) < 0.02).to(torch.uint8)
    sec_g = timed(lambda: kernels.gae(gv, gr, gd, [0.99], 0.95), 10, 3, dist)
    gae_elems = world * T * N * 10 / sec_g
    gae_gbs = 17.0 * T * N * 10 / sec_g / 1e9          # per GPU
    del gv, gr, gd

    # ---- the other named single-GPU configurations (BASELINE configs[1] / [4]), short runs, N=1 only
    others = {}
    if not args.no_others:
        # every rank runs its shard of the other named configurations too (BASELINE configs[1] and [4]: the nav learner /
        # "inference sharded over 8 GPUs"), so the scaling runs carry them
        del net, fnet, exp_dev, states_d, fstates_d, bm, fm
        torch.cuda.empty_cache()
        for other in [w for w in ("navlaser", "navimg", "pong") if w != args.workload]:
            others[other] = quick_workload(other, args.gemm_mode, dev, dist, world, rank)
            torch.cuda.empty_cache()
        # BASELINE configs[3] as a STRONG-scaling point: the 64k-row Pong batch split over the ranks (N = 1 runs all 65536
        # rows, micro-batched through the 8192-row workspace)
        others["pong_64k_strong"] = dict(quick_workload("pong", args.gemm_mode, dev, dist, world, rank, rows=65536 // world, forward=False),
                                         scaling="strong")
        torch.cuda.empty_cache()

    # ---- CPU baseline beside it (rank 0 only, N=1 only): the oracle port on the host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        if host_bind is not None:
            os.sched_setaffinity(0, host_bind[0])         # the CPU leg runs on every core the process was given
        cpu = cpu_reference(args.workload, wl["cpu_batch"], iters=2, warm=1)

    if dist is not None:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": "learner sample-iterations/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(sec / args.steps * 1e3, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"simt": "f32", "tc3": "f32 (three tcgen05 kind::f16 products of scaled fp16 hi/lo splits, fp32 accumulate)"}.get(
                args.gemm_mode, "f32 (3xTF32 tcgen05 GEMMs, fp32 accumulate)"),
            "data": "synthetic",
            "config": {"workload": wl["desc"], "rows_per_gpu": B, "global_batch": B * world, "iters_per_step": ITERS,
                       "parallelism": "dp%d" % world, "gemm_mode": args.gemm_mode, "collective": collective,
                       "deterministic": bool(args.dump_outputs),
                       "l2": "inputs larger than L2 (%.0f MB observations per GPU)" % (B * wl["obs_bytes"] / 1e6),
                       "host_affinity": ("CPUs of NUMA node %d (the GPU's)" % host_bind[1]) if host_bind is not None else "unchanged"},
            "e2e": {"value": round(e2e_value, 1), "unit": "learner sample-iterations/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 16 * ITERS},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "kernel_time_shares": kernel_shares,
            "learner_tflops": round(value * wl["flops_learn"] / 1e12, 2),
            "forward": {"value": round(fwd_value, 1), "unit": "actions/s", "rows_per_gpu": Bf,
                        "e2e": round(fwd_e2e, 1), "e2e_note": "ForwardModule.step from pageable fp32 numpy arrays",
                        "e2e_wire": fwd_wire, "batch_grid": fwd_grid,
                        "tflops": round(fwd_value * wl["flops_fwd"] / 1e12, 2)},
            "gae": {"value": round(gae_elems, 1), "unit": "(t*env) elements/s", "shape": "T=2048 x N=65536 per GPU",
                    "roofline": {"bound": "hbm", "achieved": round(gae_gbs, 1), "peak": peaks["hbm"], "unit": "GB/s",
                                 "frac": round(gae_gbs / peaks["hbm"], 4)}},
            "losses_last": {k: round(float(v), 6) for k, v in last_losses.items() if k != "PpoBackUpTime"},
        }
        if others:
            line["other_workloads"] = others
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


LOSS_KEYS = ("PpoTotalLoss", "ActorLoss", "VLoss", "EntLoss")
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, step_losses, net):
    """What one learn call hands its caller: the per-iteration losses and the parameters it leaves behind (PpoBackUpTime,
    a wall-clock time, is left out)."""
    arrays = {"losses": np.array([[l[k] for k in LOSS_KEYS] for l in step_losses], dtype=np.float64)}
    for name, p in net.named_parameters():
        arrays["param." + name] = p.detach().float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, "outputs of %d bytes exceed the %d-byte dump budget" % (total, DUMP_LIMIT)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def quick_workload(kind, gemm_mode, dev, dist, world=1, rank=0, rows=None, forward=True):
    """Learner sample-iterations/s (3 warm-up + 2 timed learn calls, inputs resident) and Forward actions/s of another
    named configuration, same definitions as the headline numbers (whole-job aggregates over `world` ranks: rows
    sharded, one gradient all-reduce per iteration; inference shards env rows with no collective)."""
    from ddrl4nav_b200.data import Experience
    from ddrl4nav_b200.runner import make_net
    wl = WORKLOADS[kind]
    B, Bf = rows or wl["batch"], wl["fwd_batch"]
    net = make_net(kind, device=dev, gemm_mode=gemm_mode, TRAINING_ITER_TIME=ITERS)
    if dist is not None:
        net.enable_data_parallel()
        net.broadcast_parameters(0)
    states_h, adv_h, ret_h = synth_batch_host(kind, B, seed=100 + rank)
    states_d = [s.to(dev) for s in states_h]
    with torch.no_grad():
        acts_d, logp_d, _ = net.act(states_d)
    old_d = logp_d + 0.15 * torch.randn(B, device=dev)
    exp = Experience(states=states_d, advs=adv_h.to(dev), actions=acts_d, old_logps=old_d, values=ret_h.to(dev)[None])

    def step():
        for _ in net.learn(exp):
            pass
    sec = timed(step, 2, 3 if rows is None else 1, dist)
    if not forward:
        return {"workload": wl["desc"], "rows_per_gpu": B, "global_batch": B * world, "n_gpus": world,
                "value": round(world * B * ITERS * 2 / sec, 1), "unit": "learner sample-iterations/s",
                "ms_per_step": round(sec / 2 * 1e3, 3)}
    fstates_d = [s.to(dev) for s in synth_batch_host(kind, Bf, seed=200 + rank)[0]]
    fnet = make_net(kind, device=dev, gemm_mode=gemm_mode)          # inference-only engine instance (predictor process)
    fnet.load_state_dict(net.state_dict())
    del net, exp
    torch.cuda.empty_cache()
    sec_f = timed(lambda: fnet.act(fstates_d), 5, 3, dist)
    return {"workload": wl["desc"], "rows_per_gpu": B, "n_gpus": world, "value": round(world * B * ITERS * 2 / sec, 1),
            "unit": "learner sample-iterations/s", "ms_per_step": round(sec / 2 * 1e3, 3),
            "learner_tflops": round(world * B * ITERS * 2 / sec * wl["flops_learn"] / 1e12, 2),
            "forward_actions_per_s": round(world * Bf * 5 / sec_f, 1), "forward_rows_per_gpu": Bf}


def _reference_learner(kind, B):
    """One full-batch PPO iteration on the host cores as a callable, plus what ran it.
    kind "reference": the UNMODIFIED reference (`USTC_lab.nn.PPO.learn`, nn/ppo.py:77-142, one iteration per call) imported
    from /root/reference or from the snapshot build() leaves in oracle/_ref/ (oracle/snapshot_ref.py);
    kind "port": the oracle restatement of the same torch op sequence, when neither exists."""
    from oracle import restate as R
    torch.set_num_threads(os.cpu_count() or 1)
    spec = R.SPECS[kind]
    params = R.init_params(spec, seed=1)
    states = R.synth_states(kind, B, seed=2)
    a, old, adv, ret = R.synth_learn_batch(spec, params, states, seed=3)
    try:
        from oracle import ref_shim
        if not ref_shim.reference_available():
            raise RuntimeError("no reference tree")
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):            # the reference's config prints the env name on import
            net, _, _ = ref_shim.make_ref_net(kind)
        from USTC_lab.data import Experience as RefExperience
        net.load_state_dict({k: params[k] for k in net.state_dict()})
        net.training_iter_time = 1
        exp = RefExperience(states=states, advs=adv, actions=a, old_logps=old, values=ret.unsqueeze(0))

        def step():
            for _ in net.learn(exp):
                pass
        return step, "reference", "USTC_lab.nn.PPO.learn (unmodified reference, %s)" % (
            "mounted tree" if ref_shim.REFERENCE_ROOT != ref_shim.SNAPSHOT_ROOT else "oracle/_ref snapshot")
    except Exception as e:                      # noqa: BLE001 -- any import problem falls back to the port, and says so
        why = "%s: %s" % (type(e).__name__, e)
    st = R.LearnState(spec, params)
    hp = R.PPOHyper()
    return (lambda: R.learn_iteration(st, states, adv, a, old, ret, hp)), "port", "oracle/restate.py port (reference not importable: %s)" % why[:120]


def cpu_reference(kind, B, iters, warm):
    """The reference's CPU path for the learner step on all host cores (the real `PPO.learn` when the reference or its
    snapshot is importable, else the oracle port).  Returns the cpu_baseline object."""
    step, how, what = _reference_learner(kind, B)
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(iters):
        step()
    dt = time.perf_counter() - t0
    return {"value": round(B * iters / dt, 1), "unit": "learner sample-iterations/s", "cores": torch.get_num_threads(),
            "kind": how, "sample": "%d full-batch iterations of B=%d (%s), %s, torch %s CPU" % (iters, B, kind, what, torch.__version__)}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the learner step, rank 0 only.  Each step is ONE
    full-batch iteration (a tenth of the 10-iteration learn call) at the product arm's rows per GPU."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    B = args.batch or wl["ref_batch"]
    step, how, what = _reference_learner(args.workload, B)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = B * args.steps / dt
    sample = "each step = ONE full-batch iteration of B=%d rows (a tenth of the %d-row x %d-iteration learn call); %s" % (
        B, wl["batch"], ITERS, what)
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": "learner sample-iterations/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "rows_per_gpu": B, "global_batch": B, "iters_per_step": 1, "device": "cpu"},
            "cpu_baseline": {"value": round(value, 1), "unit": "learner sample-iterations/s", "cores": torch.get_num_threads(),
                             "kind": how, "sample": sample},
            "e2e": {"value": round(value, 1), "unit": "learner sample-iterations/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("DDRL_BENCH_WORKLOAD", "pong"), choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gemm-mode", dest="gemm_mode", default=os.environ.get("DDRL_GEMM_MODE", "tc3"),
                    choices=["simt", "tc", "tc2", "tc3"])
    ap.add_argument("--batch", type=int, default=0, help="rows per GPU (default: the workload's)")
    ap.add_argument("--fwd-batch", dest="fwd_batch", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-others", dest="no_others", action="store_true", help="skip the short runs of the other named workloads")
    ap.add_argument("--profile-step", action="store_true",
                    help="warm up, then run ONE learn step between cudaProfilerStart/Stop and exit (for ncu --profile-from-start off)")
    ap.add_argument("--profile-forward", dest="profile_forward", action="store_true",
                    help="run ONE Forward tick (wire bytes in, replies out) and one GAE scan between cudaProfilerStart/Stop and exit")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="run in deterministic mode and write the losses and parameters of the last timed learn call as "
                         "DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the product arm (--impl ours)")
    if args.dump_outputs and (args.profile_step or args.profile_forward):
        ap.error("--dump-outputs needs the timed steps, which --profile-step / --profile-forward skip")
    if args.dump_outputs and args.gemm_mode != "tc3":
        ap.error("--dump-outputs runs in deterministic mode, which covers the tc3 engine only (--gemm-mode tc3)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "navlaser3":
        # non-reference variant: the reference has no encoder for it, so there is no CPU arm to put beside it
        args.no_cpu = True
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "unavailable": "navlaser3 is a non-reference variant (no reference encoder takes a 3x960 laser)"}), flush=True)
            return 0
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            # convenience: re-launch under torchrun
            import subprocess
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
                   "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
            sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
