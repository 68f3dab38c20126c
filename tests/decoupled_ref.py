"""TEST INFRASTRUCTURE ONLY -- float64 CPU restatement of the decoupled PPO objective of the learner (config_nn DECOUPLED_PPO,
DECOUPLED_IS_CLIP; Hilton, Cobbe & Schulman 2022), in plain torch autograd on top of oracle.restate:

  r_b = exp(logp_b - prox_b)                      clipped exactly as PPO, dual clip included
  w_b = exp(prox_b - old_b), min(w_b, c) with c   a constant: no gradient
  actor = -mean_b w_b * term(r_b, A_b)
  BehaviourKL = mean_b (rho_b - 1) - log rho_b,   rho_b = exp(prox_b - old_b) untruncated

torch.min / torch.max split ties 1/2-1/2 and clamp passes the gradient on the closed interval, as the kernels do.  With
prox == old (w == 1) the functions below are oracle.restate's PPO loss."""
from typing import Optional

import torch

from oracle import restate as R

Tensor = torch.Tensor


def term(ratio: Tensor, adv: Tensor, ppo_clip: float, dual_clip: float) -> Tensor:
    """Per-row dual-clip surrogate of oracle.restate.ppo_losses (before the mean and the sign)."""
    surr = torch.min(ratio * adv, torch.clamp(ratio, 1.0 - ppo_clip, 1.0 + ppo_clip) * adv)
    return torch.where(adv > 0, surr, torch.max(surr, dual_clip * adv))


def behaviour_weight(prox: Tensor, old: Tensor, is_clip: Optional[float] = None) -> Tensor:
    w = torch.exp(prox - old).detach()
    return w if is_clip is None else torch.clamp(w, max=is_clip)


def behaviour_kl(prox: Tensor, old: Tensor) -> float:
    log_rho = (prox - old).double()
    return float(torch.mean((torch.exp(log_rho) - 1) - log_rho))


def actor_loss(logp: Tensor, prox: Tensor, old: Tensor, adv: Tensor, ppo_clip: float = 0.2, dual_clip: float = 3.0,
               is_clip: Optional[float] = None) -> Tensor:
    w = behaviour_weight(prox, old, is_clip)
    return -torch.mean(w * term(torch.exp(logp - prox), adv, ppo_clip, dual_clip))


def loss_and_grads(dist: str, head: Tensor, actions: Tensor, old: Tensor, prox: Tensor, adv: Tensor, returns: Tensor, v: Tensor,
                   hp: R.PPOHyper, shared: bool, is_clip: Optional[float] = None, log_std: Optional[Tensor] = None):
    """The fused loss kernel restated in float64: returns ({actor, v, entropy, ApproxKL, ClipFrac, BehaviourKL}, d/d head
    (logits | mu), d/d v, d/d log_std | None).  Shared: gradients of actor + v_coef * v - ent_coef * entropy; unshared: the
    head's from the actor loss only and v's from the value loss only."""
    f64 = lambda t: t.detach().double().clone().requires_grad_(True)
    head, v = f64(head), f64(v)
    ls = f64(log_std) if log_std is not None else None
    old, prox, adv, returns = (t.detach().double() for t in (old, prox, adv, returns))
    if dist == "categorical":
        probs = torch.softmax(head, -1)
        logp = R.categorical_log_prob(probs, actions)
        ent = torch.mean(R.categorical_entropy(probs))
    else:
        logp = R.gaussian_log_prob(head, ls, actions.double())
        ent = torch.mean(R.gaussian_entropy(head, ls))
    a = actor_loss(logp, prox, old, adv, hp.ppo_clip, hp.dual_clip, is_clip)
    vl = torch.mean((returns - v) ** 2) / 2
    if shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    with torch.no_grad():
        log_ratio = logp - prox
        r = torch.exp(log_ratio)
        out = {"actor": float(a), "v": float(vl), "entropy": float(ent), "ApproxKL": float(torch.mean((r - 1) - log_ratio)),
               "ClipFrac": float(torch.mean(((r - 1).abs() > hp.ppo_clip).double())), "BehaviourKL": behaviour_kl(prox, old)}
    zero = lambda t: t.grad if t.grad is not None else torch.zeros_like(t)
    return out, zero(head), zero(v), (zero(ls) if ls is not None else None)
