"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the non-reference PPO training options of the learner (config_nn NORM_ADV,
VALUE_CLIP, PPO_STATS), in plain torch autograd on top of oracle.restate, with the cleanrl / SB3 formulas:

  advantage normalisation   (a - mean) / (std + 1e-8), unbiased std; one row is left unchanged
  clipped value loss        v_c = v_old + clamp(v - v_old, -c, c); loss = mean(max(vloss(R, v), vloss(R, v_c)))
  statistics                ApproxKL = mean((r - 1) - log r), ClipFrac = mean(|r - 1| > PPO_CLIP)

With every option off the functions below are oracle.restate's ppo_losses / learn_iteration."""
from typing import Optional, Sequence

import torch
import torch.nn.functional as F

from oracle import restate as R

Tensor = torch.Tensor


def normalize_advantages(a: Tensor) -> Tensor:
    if a.numel() <= 1:
        return a.clone()
    return (a - a.mean()) / (a.std() + 1e-8)


def ppo_losses(spec: R.NetSpec, out: dict, advs: Tensor, old_logps: Tensor, returns: Tensor, hp: R.PPOHyper,
               old_values: Optional[Tensor] = None, value_clip: Optional[float] = None, stats: bool = False):
    """(actor_loss, v_loss, entropy, total) as oracle.restate.ppo_losses, plus a dict {ApproxKL, ClipFrac} when stats."""
    actor_loss, v_loss, ent, total = R.ppo_losses(spec, out, advs, old_logps, returns, hp)
    if value_clip is not None:
        if old_values is None:
            raise ValueError("value_clip needs old_values")
        v = out["values"].squeeze()
        rows = (lambda x: F.smooth_l1_loss(returns, x, reduction="none")) if hp.smooth_l1 else (lambda x: (returns - x) ** 2 / 2)
        v_clipped = old_values + torch.clamp(v - old_values, -value_clip, value_clip)
        v_loss = torch.mean(torch.max(rows(v), rows(v_clipped)))
        total = actor_loss + v_loss * hp.v_coef - ent * hp.ent_coef
    if not stats:
        return actor_loss, v_loss, ent, total
    with torch.no_grad():
        log_ratio = out["logp"] - old_logps
        ratio = torch.exp(log_ratio)
        extra = {"ApproxKL": float(torch.mean((ratio - 1) - log_ratio)),
                 "ClipFrac": float(torch.mean(((ratio - 1).abs() > hp.ppo_clip).float()))}
    return actor_loss, v_loss, ent, total, extra


def learn_iteration(st: R.LearnState, states: Sequence[Tensor], advs: Tensor, actions: Tensor, old_logps: Tensor,
                    returns: Tensor, hp: R.PPOHyper, old_values: Optional[Tensor] = None, value_clip: Optional[float] = None,
                    stats: bool = False):
    """One optimiser step's losses and raw (pre-clip) gradients, as oracle.restate.learn_iteration(apply_update=False);
    the losses dict carries ApproxKL / ClipFrac when stats."""
    spec = st.spec
    for q in st.params.values():
        q.grad = None
    out = R.ppo_forward(spec, st.params, states, actions)
    actor_loss, v_loss, ent, total, *extra = ppo_losses(spec, out, advs, old_logps, returns, hp, old_values, value_clip, stats)
    if spec.shared:
        total.backward()
    else:
        actor_loss.backward()
        v_loss.backward()
    raw = {k: (q.grad.detach().clone() if q.grad is not None else torch.zeros_like(q)) for k, q in st.params.items()}
    losses = {"PpoTotalLoss": float(total.detach()), "ActorLoss": float(actor_loss.detach()), "VLoss": float(v_loss.detach()),
              "EntLoss": float(ent.detach())}
    for e in extra:
        losses.update(e)
    return losses, raw
