"""TEST INFRASTRUCTURE ONLY -- float64 CPU restatement of the Beta actor (ddrl4nav_b200.nn.BetaActor), in plain torch / scipy
on top of oracle.restate:

  head [B, 2A] -> alpha = 1 + softplus(head[:, :A]), beta = 1 + softplus(head[:, A:])     (F.softplus, threshold 20)
  sample        x = betaincinv(alpha, beta, u), clamped into [1e-6, 1 - 1e-6]; a = low + (high - low) * fp32(x)
  log-prob      sum_j Beta(alpha, beta).log_prob(clamp((a - low) / (high - low))) - log(high - low)
  entropy       Beta(alpha, beta).entropy() + log(high - low) per element; EntLoss is its mean over [B, A]

The PPO loss is the one of the other actors with every option (dual clip, VALUE_CLIP, NORM_VALUE's normalised targets,
DECOUPLED_PPO's proximal ratio and behaviour weight); gradients come from autograd."""
from typing import Optional

import numpy as np
import scipy.special as sp
import torch
import torch.nn.functional as F
from torch.distributions.beta import Beta

import decoupled_ref as D
from oracle import restate as R

Tensor = torch.Tensor
EPS = 1e-6

# oracle specs of the Beta kinds of runner.make_net: act_dim is the head width 2A (alpha | beta), the parameter table is then
# oracle.restate's without log_std
SPECS = {
    "navlaser_beta": R.NetSpec("nav1d", 3, 4, "beta", False),
    "navimg_beta": R.NetSpec("nav", 1, 4, "beta", True),
}
STATES_OF = {"navlaser_beta": "navlaser", "navimg_beta": "navimg"}


def concentrations(head: Tensor):
    """(alpha, beta) [B, A] of a head [B, 2A], in the head's dtype."""
    A = head.shape[-1] // 2
    c = 1.0 + F.softplus(head)
    return c[..., :A], c[..., A:]


def sample(head: Tensor, low: Tensor, high: Tensor, u: Tensor) -> Tensor:
    """fp32 actions [B, A] for the uniforms u [B, A]: the fp32 concentrations, scipy's fp64 inverse, the clamp, then low + (high -
    low) * fp32(x) with the multiply and the add rounded separately."""
    al, be = concentrations(head.float())
    x = sp.betaincinv(al.double().numpy(), be.double().numpy(), u.double().numpy())
    x = np.clip(x, EPS, 1 - EPS).astype(np.float32)
    lo, w = low.float().numpy(), (high.float() - low.float()).numpy()
    return torch.from_numpy(lo + (w * x).astype(np.float32))


def mean_action(head: Tensor, low: Tensor, high: Tensor) -> Tensor:
    al, be = concentrations(head.float())
    return low.float() + (high.float() - low.float()) * (al / (al + be))


def log_prob(head: Tensor, low: Tensor, high: Tensor, a: Tensor) -> Tensor:
    """[B] in float64 (differentiable in head)."""
    al, be = concentrations(head.double())
    lo, w = low.double(), (high.double() - low.double())
    x = torch.clamp((a.double() - lo) / w, EPS, 1 - EPS)
    return (Beta(al, be).log_prob(x) - torch.log(w)).sum(-1)


def entropy(head: Tensor, low: Tensor, high: Tensor) -> Tensor:
    """[B, A] in float64 (differentiable in head)."""
    al, be = concentrations(head.double())
    return Beta(al, be).entropy() + torch.log(high.double() - low.double())


def losses(logp: Tensor, ent: Tensor, v: Tensor, old: Tensor, adv: Tensor, returns: Tensor, hp: R.PPOHyper,
           old_values: Optional[Tensor] = None, value_clip: Optional[float] = None, value_norm=None,
           prox: Optional[Tensor] = None, is_clip: Optional[float] = None):
    """(actor, v, entropy, stats dict) of the fused loss from the per-row log-probs [B], entropies [B, A] and values [B].
    value_norm = (mean32, scale32) normalises the targets and the old values in fp32 first."""
    returns = returns.float()
    if value_norm is not None:
        m, s = (torch.tensor(t, dtype=torch.float32) for t in value_norm)
        returns = (returns - m) * s
        old_values = None if old_values is None else (old_values.float() - m) * s
    returns = returns.double()
    centre = old.double() if prox is None else prox.double()
    w = torch.ones_like(centre) if prox is None else D.behaviour_weight(prox.double(), old.double(), is_clip)
    log_ratio = logp - centre
    ratio = torch.exp(log_ratio)
    actor = -torch.mean(w * D.term(ratio, adv.double(), hp.ppo_clip, hp.dual_clip))
    rows = (lambda x: F.smooth_l1_loss(returns, x, reduction="none")) if hp.smooth_l1 else (lambda x: (returns - x) ** 2 / 2)
    if value_clip is None:
        vl = torch.mean(rows(v))
    else:
        ov = old_values.double()
        vl = torch.mean(torch.max(rows(v), rows(ov + torch.clamp(v - ov, -value_clip, value_clip))))
    ent_mean = torch.mean(ent)
    with torch.no_grad():
        stats = {"ApproxKL": float(torch.mean((ratio - 1) - log_ratio)),
                 "ClipFrac": float(torch.mean(((ratio - 1).abs() > hp.ppo_clip).double()))}
        if prox is not None:
            stats["BehaviourKL"] = D.behaviour_kl(prox, old)
    return actor, vl, ent_mean, stats


def loss_and_grads(head: Tensor, low: Tensor, high: Tensor, actions: Tensor, old: Tensor, adv: Tensor, returns: Tensor, v: Tensor,
                   hp: R.PPOHyper, shared: bool, **options):
    """The fused Beta loss kernel restated: ({actor, v, entropy, ApproxKL, ClipFrac[, BehaviourKL]}, d/d head, d/d v).  Shared:
    gradients of actor + v_coef * v - ent_coef * entropy; unshared: the head's from the actor loss only, v's from the value
    loss only."""
    head = head.detach().double().clone().requires_grad_(True)
    v = v.detach().double().clone().requires_grad_(True)
    a, vl, ent, stats = losses(log_prob(head, low, high, actions), entropy(head, low, high), v, old, adv, returns, hp, **options)
    if shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    out = {"actor": float(a.detach()), "v": float(vl.detach()), "entropy": float(ent.detach()), **stats}
    zero = lambda t: t.grad if t.grad is not None else torch.zeros_like(t)
    return out, zero(head), zero(v)


def net_grads(kind: str, params, states, actions: Tensor, old: Tensor, adv: Tensor, returns: Tensor, low: Tensor, high: Tensor,
              hp: R.PPOHyper = None):
    """Whole-net losses {ActorLoss, VLoss, EntLoss} and raw parameter gradients of one PPO step of a Beta kind, in float64, the
    encoders from oracle.restate.encoder_forward."""
    hp = hp or R.PPOHyper()
    spec = SPECS[kind]
    p = {k: v.detach().double().clone().requires_grad_(True) for k, v in params.items()}
    st = [s.double() for s in states]
    if spec.shared:
        fa = fc = R.encoder_forward(spec.arch, p, "prenet.", st)
    else:
        fa = R.encoder_forward(spec.arch, p, "actor.pre.", st)
        fc = R.encoder_forward(spec.arch, p, "critic.pre.", st)
    head = F.linear(fa, p["actor.actor_linear.weight"], p["actor.actor_linear.bias"])
    v = F.linear(fc, p["critic.critic_linear.weight"], p["critic.critic_linear.bias"]).squeeze(-1)
    a, vl, ent, _ = losses(log_prob(head, low, high, actions), entropy(head, low, high), v, old, adv, returns, hp)
    if spec.shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    grads = {k: (q.grad if q.grad is not None else torch.zeros_like(q)) for k, q in p.items()}
    return {"ActorLoss": float(a.detach()), "VLoss": float(vl.detach()), "EntLoss": float(ent.detach())}, grads
