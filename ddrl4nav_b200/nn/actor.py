"""Actor heads -- USTC_lab/nn/actor.py:10-101.

`pre` is registered before `actor_linear`, and GaussionActor's `log_std` is a direct Parameter
(so it precedes everything in named_parameters()), exactly as in the reference.  BetaActor is this library's own
(non-reference) head for bounded continuous actions, and MultiCategoricalActor its own head for MultiDiscrete actions."""
import numpy as np
import torch
from torch import nn
from torch.distributions.beta import Beta
from torch.distributions.categorical import Categorical
from torch.distributions.normal import Normal
from torch.distributions.transformed_distribution import TransformedDistribution
from torch.distributions.transforms import AffineTransform

from .._lib import DDRLError


class Actor(nn.Module):
    DIST = None

    def __init__(self, **kwargs):
        nn.Module.__init__(self)           # not super(): with the reference's class in the MRO its __init__ must not run
        self.pre = kwargs["pre"]
        self.device = kwargs["device"]

    def _distribution(self, x, play_mode=False):
        raise NotImplementedError

    def _log_prob_from_distribution(self, pi, act):
        raise NotImplementedError

    def log_prob_from_distribution(self, pi, act):
        return self._log_prob_from_distribution(pi, act)

    def _head(self, x):
        from .. import kernels
        if self.pre is not None:
            x = self.pre(x)                    # nn/actor.py:28-31: states -> features through the actor's own encoder
        return kernels.gemm(0, x, self.actor_linear.weight.detach(), self.actor_linear.bias.detach())

    def forward(self, x, act=None, play_mode=False):
        """Stand-alone call (nn/actor.py:26-40): x = states when the actor owns an encoder, features [B, last_input_dim]
        otherwise; PPO.forward is the fused path."""
        pi = self._distribution(self._head(x), play_mode)
        log_p = self._log_prob_from_distribution(pi, act) if act is not None else None
        return pi, log_p


def _reference_bases(name):
    """When the host application is the reference (its `USTC_lab.nn` is already imported), our actor classes also derive
    from the reference's class of the same name, so that the reference's own `isinstance(net.actor, GaussionActor /
    CategoricalActor)` dispatch (server/forward.py:140-142) holds without patching anything.  Our class comes first in the
    MRO and never calls the reference's __init__ / forward: only the type relation is inherited."""
    import sys
    ref = sys.modules.get("USTC_lab.nn")
    cls = getattr(ref, name, None) if ref is not None else None
    return (Actor, cls) if isinstance(cls, type) and cls is not Actor else (Actor,)


class GaussionActor(*_reference_bases("GaussionActor")):
    DIST = "gaussian"

    def __init__(self, action_output_dim=1, device="cpu", soft_max_grid=True, last_input_dim=512, pre=None,
                 nn_dtype=torch.float32):
        Actor.__init__(self, pre=pre, device=device)
        self.actor_linear = nn.Linear(last_input_dim, action_output_dim)
        self.log_std = nn.Parameter(torch.full((action_output_dim,), -0.5, dtype=nn_dtype))

    def _distribution(self, mu, play_mode=False):
        return mu if play_mode else Normal(mu, torch.exp(self.log_std.detach()))

    def _log_prob_from_distribution(self, pi, act):
        return pi.log_prob(act).sum(axis=-1)


class CategoricalActor(*_reference_bases("CategoricalActor")):
    DIST = "categorical"

    def __init__(self, action_output_dim, device="cpu", soft_max_grid=True, last_input_dim=512, pre=None,
                 nn_dtype=torch.float32):
        Actor.__init__(self, pre=pre, device=device)
        self.logits_net = None
        self.action_output_dim = action_output_dim
        self.actor_linear = nn.Linear(last_input_dim, action_output_dim)
        self.soft_max_grid = soft_max_grid

    def _distribution(self, logits, play_mode=False):
        from .. import kernels
        _, _, probs = kernels.categorical_head(logits, None)      # raw softmax (play-mode path)
        return probs if play_mode else Categorical(probs)

    def _log_prob_from_distribution(self, pi, act):
        return pi.log_prob(act)


def _bound_list(v, n, what):
    vals = list(v) if isinstance(v, (list, tuple, np.ndarray, torch.Tensor)) else [v] * n
    if len(vals) != n:
        raise DDRLError("%s must be a number or a sequence of %d numbers (got %r)" % (what, n, v))
    out = []
    for x in vals:
        x = x.item() if isinstance(x, (np.generic, torch.Tensor)) else x
        if isinstance(x, bool) or not isinstance(x, (int, float)) or not abs(x) <= float(np.finfo(np.float32).max):
            raise DDRLError("%s must hold finite fp32 numbers (got %r)" % (what, v))
        out.append(float(np.float32(x)))
    return tuple(out)


class BetaActor(Actor):
    """Beta policy on [low_j, high_j] per action dimension (Chou, Maturana & Scherer, ICML 2017): actor_linear is
    Linear(F, 2A), columns [0, A) give alpha = 1 + softplus(.) and columns [A, 2A) beta = 1 + softplus(.).  Every sample lies
    inside the bounds, so no action is ever clipped.  low / high (numbers or length-A sequences, finite, low < high) are
    configuration: they are not parameters, not in the state_dict and not in the weight blob, so a predictor must be built
    with the learner's bounds.

    Not derived from a reference class: the reference's ForwardThread only knows Gaussian and Categorical actors; a Beta net
    is served by PPO.act, ForwardModule and server.threads.ForwardThread, which do not dispatch on the actor type."""
    DIST = "beta"

    def __init__(self, action_output_dim=1, device="cpu", soft_max_grid=True, last_input_dim=512, pre=None,
                 nn_dtype=torch.float32, low=-1.0, high=1.0):
        Actor.__init__(self, pre=pre, device=device)
        if isinstance(action_output_dim, bool) or not isinstance(action_output_dim, (int, np.integer)) or action_output_dim < 1:
            raise DDRLError("BetaActor needs action_output_dim >= 1 (got %r)" % (action_output_dim,))
        self.action_output_dim = int(action_output_dim)
        self.action_low = _bound_list(low, self.action_output_dim, "low")
        self.action_high = _bound_list(high, self.action_output_dim, "high")
        if not all(lo < hi for lo, hi in zip(self.action_low, self.action_high)):
            raise DDRLError("BetaActor needs low < high in every dimension (got low=%r, high=%r)" % (low, high))
        self.actor_linear = nn.Linear(last_input_dim, 2 * self.action_output_dim)

    def bounds(self, device):
        """(low [A], high [A]) fp32 tensors on `device`."""
        f = lambda v: torch.tensor(v, dtype=torch.float32, device=device)
        return f(self.action_low), f(self.action_high)

    def distribution(self, conc):
        """Beta(alpha, beta) mapped onto [low, high], from the concentrations alpha | beta [B, 2A] of the head kernel."""
        low, high = self.bounds(conc.device)
        A = self.action_output_dim
        return TransformedDistribution(Beta(conc[:, :A], conc[:, A:]), AffineTransform(low, high - low))

    def _distribution(self, head, play_mode=False):
        from .. import kernels
        low, high = self.bounds(head.device)
        mean, _, conc = kernels.beta_head(head, low, high, None)
        return mean if play_mode else self.distribution(conc)

    def _log_prob_from_distribution(self, pi, act):
        return pi.log_prob(act).sum(axis=-1)


MAX_BRANCHES = 8           # kCatMaxBranches (csrc/categorical.cuh)
MAX_HEAD_WIDTH = 64        # kCatMaxA


def branch_sizes(nvec):
    """Validated MultiDiscrete branch sizes: a sequence of 1..8 integers >= 1 whose sum is <= 64 -> tuple of ints."""
    ok = isinstance(nvec, (list, tuple, np.ndarray, torch.Tensor)) and 1 <= len(nvec) <= MAX_BRANCHES
    vals = []
    if ok:
        for n in nvec:
            n = n.item() if isinstance(n, (np.generic, torch.Tensor)) else n
            if isinstance(n, (bool, np.bool_)) or not isinstance(n, (int, np.integer)) or n < 1:
                ok = False
                break
            vals.append(int(n))
    if not ok or sum(vals) > MAX_HEAD_WIDTH:
        raise DDRLError("nvec must be a sequence of 1..%d integers >= 1 with a sum <= %d (got %r)" % (MAX_BRANCHES, MAX_HEAD_WIDTH,
                                                                                                  nvec))
    return tuple(vals)


class MultiCategorical:
    """The product of independent Categoricals, one per branch, over per-branch probabilities [B, sum n] (gym's MultiDiscrete):
    sample() -> [..., B, K], log_prob(actions [B, K]) and entropy() summed over the branches in branch order."""

    def __init__(self, probs, nvec):
        self.nvec = tuple(nvec)
        self.probs = probs
        self.dists = [Categorical(p) for p in torch.split(probs, list(self.nvec), dim=-1)]

    def sample(self, sample_shape=torch.Size()):
        return torch.stack([d.sample(sample_shape) for d in self.dists], dim=-1)

    def log_prob(self, actions):
        out = self.dists[0].log_prob(actions[..., 0])
        for i, d in enumerate(self.dists[1:], 1):
            out = out + d.log_prob(actions[..., i])
        return out

    def entropy(self):
        out = self.dists[0].entropy()
        for d in self.dists[1:]:
            out = out + d.entropy()
        return out


class MultiCategoricalActor(Actor):
    """MultiDiscrete policy: K independent categorical branches of nvec = (n_1, ..., n_K) actions (1 <= K <= 8, sum n_i <= 64)
    over one head.  actor_linear is Linear(F, sum n_i); columns [o_i, o_i + n_i), o_i = n_1 + ... + n_{i-1}, hold branch i's
    logits.  Actions are [B, K] (fp32 holding integers); the log-prob and the entropy are the sums over the branches.
    nvec = (A,) is the CategoricalActor, with actions [B, 1].

    nvec is configuration, like BetaActor's bounds: no parameter, no state_dict key, no weight-blob byte, so a predictor must be
    built with the learner's nvec.  A different sum n_i is caught by the parameter shapes; a different split with the same sum
    cannot be detected.  action_output_dim, when given, must equal sum n_i.

    Not derived from a reference class: the reference's ForwardThread only knows Gaussian and Categorical actors; a MultiDiscrete
    net is served by PPO.act, ForwardModule and server.threads.ForwardThread, which do not dispatch on the actor type."""
    DIST = "multi_categorical"

    def __init__(self, nvec, device="cpu", last_input_dim=512, pre=None, action_output_dim=None, soft_max_grid=True,
                 nn_dtype=torch.float32):
        Actor.__init__(self, pre=pre, device=device)
        self.nvec = branch_sizes(nvec)
        if action_output_dim is not None and action_output_dim != sum(self.nvec):
            raise DDRLError("MultiCategoricalActor: action_output_dim %r differs from sum(nvec) = %d" % (action_output_dim,
                                                                                                       sum(self.nvec)))
        self.action_output_dim = sum(self.nvec)
        self.actor_linear = nn.Linear(last_input_dim, self.action_output_dim)

    def _distribution(self, logits, play_mode=False):
        from .. import kernels
        _, _, probs = kernels.multi_categorical_head(logits, self.nvec, None)    # per-branch softmax (play-mode path)
        return probs if play_mode else MultiCategorical(probs, self.nvec)

    def _log_prob_from_distribution(self, pi, act):
        return pi.log_prob(act)
