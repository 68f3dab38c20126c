"""TEST INFRASTRUCTURE ONLY -- float64 CPU restatement of invalid-action masking for the categorical actor (non-reference option
ACTION_MASK), in plain torch on top of oracle.restate:

  probs     softmax(logits.masked_fill(~m, -inf)), m = mask != 0, a row with no allowed action taken as all-ones
  log-prob  the reference chain on those probs: q = p / sum(p), log(clamp(q, eps, 1 - eps)), gathered at the action
  entropy   -(clamp(log q, min=f32 min) * q).sum(-1): masked entries add 0 * log(eps) = 0

The PPO loss is the one of the other actors with every option (tests/beta_ref.losses); gradients come from autograd through the
masked_fill, so masked logits get exactly zero gradient."""
import numpy as np
import torch
import torch.nn.functional as F

import beta_ref as BR
from oracle import restate as R

Tensor = torch.Tensor


def effective_mask(mask: Tensor) -> Tensor:
    """bool [B, A]: allowed actions, with rows that allow nothing taken as all-ones."""
    m = torch.as_tensor(mask) != 0
    return m | ~m.any(-1, keepdim=True)


def masked_probs(logits: Tensor, mask) -> Tensor:
    """softmax over the allowed entries; mask None: the plain softmax."""
    if mask is None:
        return F.softmax(logits, -1)
    return F.softmax(logits.masked_fill(~effective_mask(mask), float("-inf")), -1)


def log_prob(logits: Tensor, mask, actions: Tensor) -> Tensor:
    return R.categorical_log_prob(masked_probs(logits.double(), mask), actions)


def entropy(logits: Tensor, mask) -> Tensor:
    return R.categorical_entropy(masked_probs(logits.double(), mask))


def first_allowed(mask) -> np.ndarray:
    return np.argmax(effective_mask(mask).numpy(), axis=1)


def sample_on_q(q: np.ndarray, u: np.ndarray, mask) -> np.ndarray:
    """Inverse CDF on the (fp32) masked q with the sequential fp32 prefix sum and strict >, only allowed actions as hits; no hit
    gives the first allowed action."""
    q = np.asarray(q, np.float32)
    hit = (np.cumsum(q, axis=1, dtype=np.float32) > np.asarray(u, np.float32)[:, None]) & effective_mask(mask).numpy()
    return np.where(hit.any(1), hit.argmax(1), first_allowed(mask))


def loss_and_grads(logits: Tensor, mask, actions: Tensor, old: Tensor, adv: Tensor, returns: Tensor, v: Tensor, hp: R.PPOHyper,
                   shared: bool, **options):
    """The fused categorical loss kernel with the mask restated: ({actor, v, entropy, ApproxKL, ClipFrac[, BehaviourKL]},
    d/d logits, d/d v).  Shared: gradients of actor + v_coef * v - ent_coef * entropy; unshared: the logits' from the actor loss
    only, v's from the value loss only."""
    logits = logits.detach().double().clone().requires_grad_(True)
    v = v.detach().double().clone().requires_grad_(True)
    a, vl, ent, stats = BR.losses(log_prob(logits, mask, actions), entropy(logits, mask), v, old, adv, returns, hp, **options)
    if shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    out = {"actor": float(a.detach()), "v": float(vl.detach()), "entropy": float(ent.detach()), **stats}
    zero = lambda t: t.grad if t.grad is not None else torch.zeros_like(t)
    return out, zero(logits), zero(v)


def net_grads(kind: str, params, states, mask, actions: Tensor, old: Tensor, adv: Tensor, returns: Tensor, hp: R.PPOHyper = None):
    """Whole-net losses {ActorLoss, VLoss, EntLoss} and raw parameter gradients of one PPO step of a categorical kind with the
    mask, in float64, the encoders from oracle.restate.encoder_forward."""
    hp = hp or R.PPOHyper()
    spec = R.SPECS[kind]
    p = {k: t.detach().double().clone().requires_grad_(True) for k, t in params.items()}
    st = [s.double() for s in states]
    if spec.shared:
        fa = fc = R.encoder_forward(spec.arch, p, "prenet.", st)
    else:
        fa = R.encoder_forward(spec.arch, p, "actor.pre.", st)
        fc = R.encoder_forward(spec.arch, p, "critic.pre.", st)
    logits = F.linear(fa, p["actor.actor_linear.weight"], p["actor.actor_linear.bias"])
    v = F.linear(fc, p["critic.critic_linear.weight"], p["critic.critic_linear.bias"]).squeeze(-1)
    a, vl, ent, _ = BR.losses(log_prob(logits, mask, actions), entropy(logits, mask), v, old, adv, returns, hp)
    if spec.shared:
        (a + vl * hp.v_coef - ent * hp.ent_coef).backward()
    else:
        a.backward()
        vl.backward()
    grads = {k: (q.grad if q.grad is not None else torch.zeros_like(q)) for k, q in p.items()}
    return {"ActorLoss": float(a.detach()), "VLoss": float(vl.detach()), "EntLoss": float(ent.detach())}, grads


def random_mask(B: int, A: int, seed: int, p_allowed: float = 0.6, empty_rows: int = 2) -> Tensor:
    """u8 [B, A] with ~p_allowed of the actions allowed and the first `empty_rows` rows allowing nothing."""
    g = torch.Generator().manual_seed(seed)
    m = (torch.rand(B, A, generator=g) < p_allowed).to(torch.uint8)
    m[:empty_rows] = 0
    return m
