"""TEST INFRASTRUCTURE ONLY -- CPU restatement (oracle) of DDRL4NAV's actor-learner hot path.

This file restates, in plain functional PyTorch / NumPy on the CPU, what the reference
computes on the path SURVEY.md section 8(a) lists.  It exists so that the CUDA path in
``ddrl4nav_b200/`` can be checked on a GPU box where ``/root/reference`` is not mounted.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it; the product package never does.

Pinning status: the reference ships no tests, golden vectors or seeds (SURVEY.md section 4),
so the oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF run in the build container:
``tests/golden/make_golden.py`` imports the unmodified reference (``oracle/ref_shim.py``),
runs it on seeded inputs and commits the vectors under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks every function below against them (bit-for-bit where
the arithmetic is the same torch/numpy call sequence).

The arithmetic of this path lives in third-party dependencies the reference does not pin
(``requirements.txt`` lists numpy unpinned and omits torch; README suggests torch 1.10.2):
PyTorch (conv/linear/softmax/distributions/autograd/clip_grad_norm_/Adam) and NumPy (GAE).
The container's torch 2.11.0 / numpy 2.3.5 are therefore the de-facto definition.

Parameters are passed as a flat ``dict`` keyed by the reference's own ``state_dict()`` names
(``actor.pre.conv1.weight`` ...), so a reference checkpoint can be fed in unchanged.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
F32_EPS = float(torch.finfo(torch.float32).eps)     # 1.1920929e-07
F32_MIN = float(torch.finfo(torch.float32).min)


@dataclass(frozen=True)
class NetSpec:
    """What ``runner/utils.py:59-170`` (create_net) decides for one task."""
    arch: str            # 'atari' | 'nav' | 'navped' | 'nav1d' | 'mlp'
    in_ch: int           # AtariPreNet num_inputs / Nav* image_channel / MLP input_dim
    act_dim: int         # ACTION_OUTPUT_DIM
    dist: str            # 'categorical' | 'gaussian'
    shared: bool         # SHARE_CNN_NET
    feat: int = 512      # AC_INPUT_DIM (MLPPreNet: last_output_dim)
    laser_ch: int = 1    # nav1d: Conv1d(laser_ch, 32, 5, 2); the reference has 1 (nn/nav_encoder.py:87)


SPECS = {
    "pong": NetSpec("atari", 4, 6, "categorical", False),       # BASELINE config C1
    "navlaser": NetSpec("nav1d", 3, 2, "gaussian", False),      # C2
    # NOT a reference configuration: the "3 x 960" laser wording of BASELINE (3-frame laser stacking is an env option,
    # envs/cfg/old_cfg/image_ped_circle.yaml:25; no shipped encoder consumes it).  Same stack with Conv1d(3, 32, 5, 2)
    "navlaser3": NetSpec("nav1d", 3, 2, "gaussian", False, 512, 3),
    "navimg": NetSpec("nav", 1, 28, "categorical", True),       # C5
    "navped": NetSpec("navped", 4, 28, "categorical", True),    # C5 "+ scan" variant: NavPedPreNet, cat(map, ped-map)
}


@dataclass
class PPOHyper:
    """``config/config_nn.py:27-57`` defaults."""
    ppo_clip: float = 0.2
    dual_clip: float = 3.0
    v_coef: float = 1.0
    ent_coef: float = 0.05
    max_grad_norm: float = 0.5
    clip_grad: bool = True
    lr: float = 2e-4
    lr_actor: float = 5e-5
    lr_critic: float = 1e-3
    smooth_l1: bool = False
    iters: int = 10


# --------------------------------------------------------------------------------------
# parameter tables (names / shapes / order = reference named_parameters(), SURVEY App. C)
# --------------------------------------------------------------------------------------
def encoder_param_shapes(arch: str, in_ch: int, feat: int = 512, laser_ch: int = 1) -> List[Tuple[str, Tuple[int, ...]]]:
    if arch == "atari":      # nn/atari_encoder.py:12-23
        return [("conv1.weight", (32, in_ch, 8, 8)), ("conv1.bias", (32,)),
                ("conv2.weight", (64, 32, 4, 4)), ("conv2.bias", (64,)),
                ("conv3.weight", (64, 64, 3, 3)), ("conv3.bias", (64,)),
                ("linear.weight", (512, 3136)), ("linear.bias", (512,))]
    if arch in ("nav", "navped"):   # nn/nav_encoder.py:13-26, 47-62
        return [("conv1.weight", (64, in_ch, 3, 3)), ("conv1.bias", (64,)),
                ("conv2.weight", (128, 64, 3, 3)), ("conv2.bias", (128,)),
                ("conv3.weight", (256, 128, 3, 3)), ("conv3.bias", (256,)),
                ("fc0.0.weight", (512, 9216)), ("fc0.0.bias", (512,)),
                ("fc1.0.weight", (512, 521)), ("fc1.0.bias", (512,)),
                ("fc2.weight", (512, 512)), ("fc2.bias", (512,))]
    if arch == "nav1d":      # nn/nav_encoder.py:83-97
        return [("conv1.weight", (64, in_ch, 7, 7)), ("conv1.bias", (64,)),
                ("conv2.weight", (128, 64, 5, 5)), ("conv2.bias", (128,)),
                ("conv3.weight", (256, 128, 3, 3)), ("conv3.bias", (256,)),
                ("conv1d1.weight", (32, laser_ch, 5)), ("conv1d1.bias", (32,)),
                ("conv1d2.weight", (32, 32, 3)), ("conv1d2.bias", (32,)),
                ("fc_1d.0.weight", (256, 7616)), ("fc_1d.0.bias", (256,)),
                ("fc0.0.weight", (512, 6400)), ("fc0.0.bias", (512,)),
                ("fc1.0.weight", (512, 773)), ("fc1.0.bias", (512,)),
                ("fc2.weight", (512, 512)), ("fc2.bias", (512,))]
    if arch == "mlp":        # nn/mlp_encoder.py:13-18
        return [("fc0.0.weight", (feat, in_ch)), ("fc0.0.bias", (feat,))]
    raise ValueError(arch)


def param_table(spec: NetSpec) -> List[Tuple[str, Tuple[int, ...]]]:
    """Full ``named_parameters()`` order of ``PPO`` (``nn/ppo.py:26-30``: prenet, actor, critic;
    ``nn/actor.py:12-16,52-56``: parameters before sub-modules, ``pre`` before ``actor_linear``;
    ``nn/critic.py:8-12``: ``critic_linear`` before ``pre``)."""
    enc = encoder_param_shapes(spec.arch, spec.in_ch, spec.feat, spec.laser_ch)
    out: List[Tuple[str, Tuple[int, ...]]] = []
    if spec.shared:
        out += [("prenet." + n, s) for n, s in enc]
    if spec.dist == "gaussian":
        out.append(("actor.log_std", (spec.act_dim,)))
    if not spec.shared:
        out += [("actor.pre." + n, s) for n, s in enc]
    out += [("actor.actor_linear.weight", (spec.act_dim, spec.feat)), ("actor.actor_linear.bias", (spec.act_dim,))]
    out += [("critic.critic_linear.weight", (1, spec.feat)), ("critic.critic_linear.bias", (1,))]
    if not spec.shared:
        out += [("critic.pre." + n, s) for n, s in enc]
    return out


def init_params(spec: NetSpec, seed: int = 0) -> Dict[str, Tensor]:
    """PyTorch default init of the reference modules (Conv/Linear.reset_parameters:
    kaiming-uniform a=sqrt(5) == U(+-1/sqrt(fan_in)) for weight and bias; log_std=-0.5,
    ``nn/actor.py:55``).  Same distribution as the reference, NOT the same RNG stream."""
    g = torch.Generator().manual_seed(seed)
    params: Dict[str, Tensor] = {}
    table = param_table(spec)
    fan_in = {}
    for name, shape in table:
        if name.endswith(".weight"):
            fan_in[name[:-7]] = int(np.prod(shape[1:]))
    for name, shape in table:
        if name.endswith("log_std"):
            params[name] = torch.full(shape, -0.5, dtype=torch.float32)
            continue
        base = name.rsplit(".", 1)[0]
        bound = 1.0 / math.sqrt(fan_in[base])
        params[name] = (torch.rand(shape, generator=g, dtype=torch.float32) * 2 - 1) * bound
    return params


# --------------------------------------------------------------------------------------
# encoders
# --------------------------------------------------------------------------------------
def _lin(p, pre, name, x):
    return F.linear(x, p[pre + name + ".weight"], p[pre + name + ".bias"])


# Activation ties.  relu / leaky_relu are not differentiable at 0; the reference takes slope 0 (relu) / 0.01 (leaky) at
# exactly 0 (SURVEY App. A.2), but a pre-activation that is zero only to within fp32 rounding (|z| ~ 1e-8) lands on
# either side depending on the summation order of whoever computes it -- torch CPU, torch CUDA and the kernels here
# all differ there.  TIE_HOOK lets the parity tests (a) record every pre-activation and (b) re-run the backward with
# the branch of chosen tie elements flipped, so that "equal up to measure-zero ties" can be asserted exactly.
TIE_HOOK = None      # callable(layer_name, z, a, slope_neg) -> a'   (test infrastructure only)
# The same holds for the 2 x 2 max pools of the nav encoders: two activations of one window that agree to fp32 rounding may
# rank either way.  POOL_HOOK replaces the pool so that the tests can record those windows and route the gradient of chosen
# ones to the runner-up.
POOL_HOOK = None     # callable(layer_name, a) -> max_pool2d(a, 2, stride=2)   (test infrastructure only)


def _act(name, z, slope):
    a = F.leaky_relu(z, slope) if slope else F.relu(z)
    return TIE_HOOK(name, z, a, slope) if TIE_HOOK is not None else a


class TieRecorder:
    """Records pre-activations; optionally flips the backward slope of given flat indices per layer (forward value kept)."""

    def __init__(self, flips=None):
        self.z = {}
        self.flips = flips or {}

    def __call__(self, name, z, a, slope):
        self.z[name] = z.detach()
        idx = self.flips.get(name)
        if idx is None or len(idx) == 0:
            return a
        zf = z.reshape(-1)
        sel = torch.zeros_like(zf)
        sel[torch.as_tensor(idx, dtype=torch.long)] = 1.0
        cur = torch.where(zf.detach() > 0, torch.ones_like(zf), torch.full_like(zf, slope))
        new = torch.where(zf.detach() > 0, torch.full_like(zf, slope), torch.ones_like(zf))
        # zero-valued term whose gradient replaces slope `cur` by slope `new` on the selected elements
        return a + (sel * (new - cur) * (zf - zf.detach())).reshape(a.shape)


def _conv_relu_pool(p, pre, name, x, pad):
    # nn/nav_encoder.py:29-31,100-102: max_pool2d(relu(conv(x)), 2, stride=2)
    z = F.conv2d(x, p[pre + name + ".weight"], p[pre + name + ".bias"], padding=pad)
    a = _act(pre + name, z, 0.0)
    return POOL_HOOK(pre + name, a) if POOL_HOOK is not None else F.max_pool2d(a, 2, stride=2)


def encoder_forward(arch: str, p: Dict[str, Tensor], pre: str, states: Sequence[Tensor]) -> Tensor:
    if arch == "atari":
        # nn/atari_encoder.py:25-32 -- leaky_relu(0.01) x3, C-major flatten, linear WITHOUT activation
        x = _act(pre + "conv1", F.conv2d(states[0], p[pre + "conv1.weight"], p[pre + "conv1.bias"], stride=4), 0.01)
        x = _act(pre + "conv2", F.conv2d(x, p[pre + "conv2.weight"], p[pre + "conv2.bias"], stride=2), 0.01)
        x = _act(pre + "conv3", F.conv2d(x, p[pre + "conv3.weight"], p[pre + "conv3.bias"], stride=1), 0.01)
        return _lin(p, pre, "linear", x.reshape(x.shape[0], -1))
    if arch in ("nav", "navped"):
        # nn/nav_encoder.py:28-43 (NavPreNet) / :64-79 (NavPedPreNet: image = cat(state[0], state[2]))
        img = states[0] if arch == "nav" else torch.cat([states[0], states[2]], dim=1)
        x = _conv_relu_pool(p, pre, "conv1", img, 1)
        x = _conv_relu_pool(p, pre, "conv2", x, 1)
        x = _conv_relu_pool(p, pre, "conv3", x, 1)
        x = _act(pre + "fc0", _lin(p, pre, "fc0.0", x.reshape(x.shape[0], -1)), 0.0)
        x = torch.cat((x, states[1]), dim=1)
        x = _act(pre + "fc1", _lin(p, pre, "fc1.0", x), 0.0)
        return _lin(p, pre, "fc2", x)
    if arch == "nav1d":
        # nn/nav_encoder.py:99-128 -- laser: conv1d,conv1d (NO activation between), fc_1d+relu
        l = F.conv1d(states[0], p[pre + "conv1d1.weight"], p[pre + "conv1d1.bias"], stride=2)
        l = F.conv1d(l, p[pre + "conv1d2.weight"], p[pre + "conv1d2.bias"], stride=2)
        l = _act(pre + "fc_1d", _lin(p, pre, "fc_1d.0", l.reshape(l.shape[0], -1)), 0.0)
        x = _conv_relu_pool(p, pre, "conv1", states[2], 1)
        x = _conv_relu_pool(p, pre, "conv2", x, 1)
        x = _conv_relu_pool(p, pre, "conv3", x, 1)
        x = _act(pre + "fc0", _lin(p, pre, "fc0.0", x.reshape(x.shape[0], -1)), 0.0)
        x = torch.cat((l, x, states[1]), dim=1)
        x = _act(pre + "fc1", _lin(p, pre, "fc1.0", x), 0.0)
        return _lin(p, pre, "fc2", x)
    if arch == "mlp":
        return _act(pre + "fc0", _lin(p, pre, "fc0.0", states[0]), 0.0)    # nn/mlp_encoder.py:21-27
    raise ValueError(arch)


# --------------------------------------------------------------------------------------
# heads, distributions (nn/actor.py, nn/critic.py, nn/ppo.py:72-75)
# --------------------------------------------------------------------------------------
def categorical_normalise(probs: Tensor) -> Tuple[Tensor, Tensor]:
    """torch/distributions/categorical.py:70 + utils.py probs_to_logits: p/sum(p), log(clamp(p,eps,1-eps))."""
    q = probs / probs.sum(-1, keepdim=True)
    return q, torch.log(q.clamp(min=F32_EPS, max=1 - F32_EPS))


def categorical_log_prob(probs: Tensor, act: Tensor) -> Tensor:
    _, logits = categorical_normalise(probs)
    return logits.gather(-1, act.long().unsqueeze(-1)).squeeze(-1)     # nn/actor.py:100-101


def categorical_entropy(probs: Tensor) -> Tensor:
    q, logits = categorical_normalise(probs)
    return -(logits.clamp(min=F32_MIN) * q).sum(-1)                    # categorical.py:151-155


def gaussian_log_prob(mu: Tensor, log_std: Tensor, act: Tensor) -> Tensor:
    # nn/actor.py:63-70 ; torch/distributions/normal.py:87-102
    std = torch.exp(log_std)
    var = std ** 2
    lp = -((act - mu) ** 2) / (2 * var) - torch.log(std) - math.log(math.sqrt(2 * math.pi))
    return lp.sum(-1)


def gaussian_entropy(mu: Tensor, log_std: Tensor) -> Tensor:
    # normal.py:114-115: 0.5 + 0.5*log(2*pi) + log(scale), broadcast to mu's shape
    return (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(torch.exp(log_std))).expand_as(mu)


def ppo_forward(spec: NetSpec, p: Dict[str, Tensor], states: Sequence[Tensor], act: Optional[Tensor] = None):
    """``PPO.forward`` (nn/ppo.py:72-75).  Returns dict with probs|mu, log_std, logp (if act), values [B,1]."""
    if spec.shared:
        h_a = h_c = encoder_forward(spec.arch, p, "prenet.", states)
    else:
        h_a = encoder_forward(spec.arch, p, "actor.pre.", states)
        h_c = encoder_forward(spec.arch, p, "critic.pre.", states)
    out = {}
    head = _lin(p, "", "actor.actor_linear", h_a)
    if spec.dist == "categorical":
        out["probs"] = F.softmax(head, dim=-1)                         # nn/actor.py:91-94
        if act is not None:
            out["logp"] = categorical_log_prob(out["probs"], act)
    else:
        out["mu"] = head
        out["log_std"] = p["actor.log_std"]
        if act is not None:
            out["logp"] = gaussian_log_prob(head, p["actor.log_std"], act)
    out["values"] = _lin(p, "", "critic.critic_linear", h_c)           # [B,1], nn/critic.py:21
    return out


# --------------------------------------------------------------------------------------
# sampling (uniform-draw contract: server/utils.py:20-47; play mode: server/forward.py:139-144)
# --------------------------------------------------------------------------------------
def sample_categorical(probs: np.ndarray, u: np.ndarray) -> np.ndarray:
    """``random_choice_prob_index`` with the uniforms supplied: (cumsum(p,1) > u[:,None]).argmax(1).
    Sequential fp32 prefix sum; all-False row -> 0."""
    probs = np.asarray(probs)
    return (probs.cumsum(axis=1) > np.asarray(u)[:, None]).argmax(axis=1)


def argmax_first(probs: np.ndarray) -> np.ndarray:
    return np.argmax(np.asarray(probs), axis=1)


def sample_gaussian(mu: Tensor, log_std: Tensor, eps: Tensor) -> Tensor:
    """torch.normal(mu, std) with the N(0,1) draw supplied: mu + std*eps (mul then add, no FMA)."""
    return mu + torch.exp(log_std) * eps


def forward_body(spec: NetSpec, p: Dict[str, Tensor], states: Sequence[Tensor], draw: Optional[Tensor],
                 play_mode: bool = False):
    """Compute body of ``ForwardThread.run`` (server/forward.py:128-146) with the random draw supplied.

    draw: categorical -> uniforms [B]; gaussian -> N(0,1) [B,A]; ignored in play mode.
    Returns (actions fp32 [B] or [B,A], logps fp32 [B], values fp32 [V=1,B,1])."""
    with torch.no_grad():
        out = ppo_forward(spec, p, states)
        B = out["values"].shape[0]
        if spec.dist == "categorical":
            if play_mode:
                a = torch.argmax(out["probs"], dim=1).to(torch.float32)
                logp = torch.zeros(B, dtype=torch.float32)
            else:
                a = torch.from_numpy(sample_categorical(out["probs"].numpy(), draw.numpy())).to(torch.float32)
                logp = categorical_log_prob(out["probs"], a)
        else:
            if play_mode:
                a = out["mu"]
                logp = torch.zeros(B, dtype=torch.float32)
            else:
                a = sample_gaussian(out["mu"], out["log_std"], draw)
                logp = gaussian_log_prob(out["mu"], out["log_std"], a)
        return a, logp, out["values"].unsqueeze(0)


# --------------------------------------------------------------------------------------
# GAE (agent/agent.py:124-140)
# --------------------------------------------------------------------------------------
def gae(values: np.ndarray, dones: np.ndarray, rewards: np.ndarray, gamma: np.ndarray, lam: float):
    """values [T+1,V,N] f32, dones [T+1,V,N] u8 (row T unused), rewards [T+1,R,N] f32 (row T unused),
    gamma [V,1] f32 (``self.discounts``), lam python float (``self.landa``).
    Returns (returns [T,V,N] f32, advs [T,N] f32).  Same numpy op sequence as the reference loop."""
    T = values.shape[0] - 1
    g = np.zeros_like(rewards[0], dtype=np.float32)
    nv = values[T]
    rets = np.empty((T,) + values.shape[1:], dtype=np.float32)
    advs = np.empty((T, values.shape[2]), dtype=np.float32)
    for t in reversed(range(T)):
        g *= (1 - dones[t])
        g = gamma * lam * g + (gamma * nv * (1 - dones[t]) - values[t] + rewards[t])
        nv = values[t]
        rets[t] = values[t] + g
        advs[t] = g[0] * 1.0
    return rets, advs


def gae_tempo(values: np.ndarray, dones: np.ndarray, rewards: np.ndarray, durations: np.ndarray,
              gamma_base: float, lam: float):
    """``_accumulate_tempo_rewards`` (agent/agent.py:142-160): per-step discount gamma**duration[t]
    taken from a float64 logspace table (agent.py:119), so the recurrence runs in float64 there.
    durations [T+1] int."""
    table = np.logspace(0, 100, 101, base=gamma_base)
    T = values.shape[0] - 1
    g = np.zeros_like(rewards[0], dtype=np.float32)
    nv = values[T]
    rets, advs = [None] * T, [None] * T
    for t in reversed(range(T)):
        g *= (1 - dones[t])
        td = table[durations[t]]
        g = td * lam * g + (td * nv * (1 - dones[t]) - values[t] + rewards[t])
        nv = values[t]
        rets[t] = values[t] + g
        advs[t] = g[0] * 1.0
    return np.stack(rets), np.stack(advs)


# --------------------------------------------------------------------------------------
# PPO loss / learn (nn/ppo.py:77-142)
# --------------------------------------------------------------------------------------
def ppo_losses(spec: NetSpec, out: dict, advs: Tensor, old_logps: Tensor, returns: Tensor, hp: PPOHyper):
    """Returns (actor_loss, v_loss, entropy, total).  ``returns`` = data.values[0,:] (SURVEY App. D)."""
    ratio = torch.exp(out["logp"] - old_logps)
    surr = torch.min(ratio * advs, torch.clamp(ratio, 1.0 - hp.ppo_clip, 1.0 + hp.ppo_clip) * advs)
    actor_loss = -torch.mean(torch.where(advs > 0, surr, torch.max(surr, hp.dual_clip * advs)))
    v = out["values"].squeeze()
    if hp.smooth_l1:
        v_loss = F.smooth_l1_loss(returns, v)            # nn/ppo.py:54-55 (input=returns, target=v)
    else:
        v_loss = torch.mean((returns - v) ** 2) / 2      # nn/ppo.py:57
    if spec.dist == "categorical":
        ent = torch.mean(categorical_entropy(out["probs"]))
    else:
        ent = torch.mean(gaussian_entropy(out["mu"], out["log_std"]))
    total = actor_loss + v_loss * hp.v_coef - ent * hp.ent_coef
    return actor_loss, v_loss, ent, total


def param_groups(spec: NetSpec, names: Sequence[str]):
    """Which Adam (and LR) owns each parameter: nn/ppo.py:40-42,110-129."""
    if spec.shared:
        return {n: "all" for n in names}
    return {n: ("actor" if n.startswith("actor.") else "critic") for n in names}


def clip_grad_norm(grads: Dict[str, Tensor], max_norm: float) -> float:
    """torch/nn/utils/clip_grad.py: norm of per-tensor norms, coef=min(1, max/(total+1e-6)), always multiplied."""
    total = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(g, 2.0) for g in grads.values()]), 2.0)
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    for g in grads.values():
        g.mul_(coef)
    return float(total)


def adam_step(p: Tensor, g: Tensor, m: Tensor, v: Tensor, step: int, lr: float,
              b1: float = 0.9, b2: float = 0.999, eps: float = 1e-8):
    """torch/optim/adam.py single-tensor path, capturable=False (SURVEY App. A.2). In place; step>=1."""
    m.lerp_(g, 1 - b1)
    v.mul_(b2).addcmul_(g, g, value=1 - b2)
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    step_size = lr / bc1
    denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
    p.addcdiv_(m, denom, value=-step_size)


class LearnState:
    """Parameters + the two (or one) Adam states of ``PPO`` (nn/ppo.py:40-42)."""

    def __init__(self, spec: NetSpec, params: Dict[str, Tensor]):
        self.spec = spec
        self.params = {k: v.clone().requires_grad_(True) for k, v in params.items()}
        self.m = {k: torch.zeros_like(v) for k, v in params.items()}
        self.v = {k: torch.zeros_like(v) for k, v in params.items()}
        self.step = 0


def learn_iteration(st: LearnState, states: Sequence[Tensor], advs: Tensor, actions: Tensor, old_logps: Tensor,
                    returns: Tensor, hp: PPOHyper, apply_update: bool = True):
    """One pass of the ``for _ in range(training_iter_time)`` loop (nn/ppo.py:79-142).

    Returns (losses dict, raw grads dict (before clipping), total grad norm)."""
    spec = st.spec
    for q in st.params.values():
        q.grad = None
    out = ppo_forward(spec, st.params, states, actions)
    actor_loss, v_loss, ent, total = ppo_losses(spec, out, advs, old_logps, returns, hp)
    if spec.shared:
        total.backward()                                  # nn/ppo.py:111-112
    else:
        actor_loss.backward()                             # nn/ppo.py:122-123 (entropy gets NO gradient)
        v_loss.backward()
    grads = {k: (q.grad.detach().clone() if q.grad is not None else torch.zeros_like(q)) for k, q in st.params.items()}
    raw = {k: g.clone() for k, g in grads.items()}
    # clip over every parameter that HAS a grad (clip_grad_norm_ skips grad=None parameters)
    live = {k: g for k, g in grads.items() if st.params[k].grad is not None}
    norm = clip_grad_norm(live, hp.max_grad_norm) if hp.clip_grad else float("nan")
    if apply_update:
        st.step += 1
        groups = param_groups(spec, list(st.params))
        lrs = {"all": hp.lr, "actor": hp.lr_actor, "critic": hp.lr_critic}
        with torch.no_grad():
            for k, q in st.params.items():
                if q.grad is None:
                    continue                              # Adam skips parameters without grad
                adam_step(q, grads[k], st.m[k], st.v[k], st.step, lrs[groups[k]])
    losses = {"PpoTotalLoss": float(total.detach()), "ActorLoss": float(actor_loss.detach()), "VLoss": float(v_loss.detach()),
              "EntLoss": float(ent.detach())}
    return losses, raw, norm


# --------------------------------------------------------------------------------------
# synthetic workloads (SURVEY section 8d) -- shared by tests and bench so both arms see the same data
# --------------------------------------------------------------------------------------
def synth_states(kind: str, B: int, seed: int = 0) -> List[Tensor]:
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
    if kind == "navped":
        img = torch.rand(B, 1, 48, 48, generator=g)
        vec = torch.randn(B, 9, generator=g)
        occ = (torch.rand(B, 1, 48, 48, generator=g) < 0.03).float()
        vel = (torch.rand(B, 2, 48, 48, generator=g) - 0.5) * occ
        return [img, vec, torch.cat([occ, vel], dim=1)]
    raise ValueError(kind)


def synth_learn_batch(spec: NetSpec, params: Dict[str, Tensor], states: Sequence[Tensor], seed: int = 0):
    """actions sampled from the net, old_logp = logp + N(0,0.15), adv, ret ~ N(0,1) (SURVEY 8d)."""
    g = torch.Generator().manual_seed(seed + 1)
    B = states[0].shape[0]
    draw = torch.rand(B, generator=g) if spec.dist == "categorical" else torch.randn(B, spec.act_dim, generator=g)
    a, logp, _ = forward_body(spec, params, states, draw)
    old = logp + 0.15 * torch.randn(B, generator=g)
    adv = torch.randn(B, generator=g)
    ret = torch.randn(B, generator=g)
    return a, old, adv, ret


def synth_extra_critic(params: Dict[str, Tensor], ret: Tensor, seed: int = 77):
    """Second critic the way runner/utils.py:162 makes it (copy.deepcopy(critic)) with re-seeded weights so that its values
    differ, and the [V=2, B] returns matrix a V > 1 learner reads (nn/ppo.py:95-104).  Returns (ret2, extra) with `extra`
    keyed by the critic's own parameter names (critic_linear.*, pre.*) in registration order."""
    g = torch.Generator().manual_seed(seed)
    ret2 = torch.stack([ret, ret * 0.5 + 0.25 * torch.randn(ret.shape[0], generator=g)])
    extra = {}
    for n, p in params.items():
        if n.startswith("critic."):
            extra[n[len("critic."):]] = p.detach().clone() + 0.05 * torch.randn(p.shape, generator=g)
    return ret2, extra


# =========================================================================================
# EasyBytes wire format (SURVEY 8f row f2) -- USTC_lab/data/easybytes.py
# =========================================================================================
EASYBYTES_TYPES = {1: (1, np.uint8), 2: (2, np.float16), 3: (4, np.float32), 4: (8, np.float64)}   # easybytes.py:21-26


def easybytes_decode_data(buf: bytes) -> List[np.ndarray]:
    """easybytes.py:47-61: repeated blocks [type >h][count >I][ndim >I][shape >I x ndim][count*size raw bytes]."""
    import struct
    out, i = [], 0
    while i < len(buf):
        code = struct.unpack(">h", buf[i:i + 2])[0]
        size, dt = EASYBYTES_TYPES[code]
        count, ndim = struct.unpack(">II", buf[i + 2:i + 10])
        shape = struct.unpack(">" + "I" * ndim, buf[i + 10:i + 10 + 4 * ndim])
        i += 10 + 4 * ndim
        out.append(np.frombuffer(buf[i:i + count * size], dtype=dt).reshape(*shape))
        i += count * size
    return out


def easybytes_decode_forward_states(buf: bytes) -> Tuple[List[str], List[np.ndarray]]:
    """easybytes.py:114-139: messages [length >Q][ip 4 x >H][process_env_id >I][decode_data payload of `length` bytes];
    state slot i of the batch = concatenation over messages (axis 0) of their i-th array."""
    import struct
    ids, per_msg, i = [], [], 0
    while i < len(buf):
        length = struct.unpack(">Q", buf[i:i + 8])[0]
        ip = struct.unpack(">HHHH", buf[i + 8:i + 16])
        env_id = struct.unpack(">I", buf[i + 16:i + 20])[0]
        per_msg.append(easybytes_decode_data(buf[i + 20:i + 20 + length]))
        ids.append(".".join(str(x) for x in ip) + "_" + str(env_id))
        i += 20 + length
    slots = [np.concatenate([m[k] for m in per_msg], axis=0) for k in range(len(per_msg[0]))]
    return ids, slots


def easybytes_forward_states_fp32(buf: bytes) -> Tuple[List[str], List[np.ndarray]]:
    """decode_forward_states followed by the fp32 conversion of the Forward thread (server/forward.py:128-131,
    torch.tensor(state, dtype=float32)): what the device decoder must reproduce bit for bit."""
    ids, slots = easybytes_decode_forward_states(buf)
    return ids, [s.astype(np.float32) for s in slots]


def easybytes_decode_backward_data(buf: bytes):
    """easybytes.py:163-171: [len >Q][states blocks][len >Q][advs, actions, old_logps, values blocks][marshal dict]."""
    import marshal
    import struct
    n0 = struct.unpack(">Q", buf[:8])[0]
    states = easybytes_decode_data(buf[8:8 + n0])
    n1 = struct.unpack(">Q", buf[8 + n0:16 + n0])[0]
    other = easybytes_decode_data(buf[16 + n0:16 + n0 + n1])
    return states, other, marshal.loads(buf[16 + n0 + n1:])


_EASYBYTES_CODE = {np.dtype(np.uint8): 1, np.dtype(np.float16): 2, np.dtype(np.float32): 3, np.dtype(np.float64): 4}


def easybytes_encode_data(arrays: Sequence[np.ndarray]) -> bytes:
    """easybytes.py:62-75: per array [type >h][count >I][ndim >I][shape >I x ndim][raw bytes]."""
    import struct
    out = b""
    for a in arrays:
        a = np.asarray(a)
        out += struct.pack(">h", _EASYBYTES_CODE[a.dtype]) + struct.pack(">II", int(a.size), a.ndim)
        out += struct.pack(">" + "I" * a.ndim, *a.shape) + a.tobytes()
    return out


def easybytes_encode_forward_states(ip: str, process_env_id: int, arrays: Sequence[np.ndarray]) -> bytes:
    """easybytes.py:28-33,141-148: [length >Q][ip 4 x >H][process_env_id >I][blocks]; length counts the blocks only."""
    import struct
    body = easybytes_encode_data(arrays)
    return struct.pack(">Q", len(body)) + struct.pack(">HHHH", *[int(x) for x in ip.split(".")]) + struct.pack(">I", process_env_id) + body


def easybytes_encode_backward_data(states: Sequence[np.ndarray], other4: Sequence[np.ndarray], logger: dict) -> bytes:
    """easybytes.py:150-161."""
    import marshal
    import struct
    s, o = easybytes_encode_data(states), easybytes_encode_data(other4)
    return struct.pack(">Q", len(s)) + s + struct.pack(">Q", len(o)) + o + marshal.dumps(logger)


def easybytes_encode_forward_return_data(arrays: Sequence[np.ndarray], env_batch_nums: Sequence[int]) -> List[bytes]:
    """easybytes.py:77-109: env process j gets rows [i0, i1) of every array -- columns [i0, i1) of array 2 (values [V, B, 1])."""
    out, i0 = [], 0
    for nb in env_batch_nums:
        out.append(easybytes_encode_data([a[:, i0:i0 + nb] if k == 2 else a[i0:i0 + nb] for k, a in enumerate(arrays)]))
        i0 += nb
    return out
