"""Experience -- the batch container handed to ``PPO.learn`` (USTC_lab/data/experience.py:23-62).

Field names, ``get_xrapv`` order and ``to_tensor`` semantics are the boundary data contract
(SURVEY 2 #4); ``values`` holds RETURNS [V, B] by the time it reaches the learner (App. D).

``old_values`` (non-reference, optional) holds the rollout's value predictions of critic 0 [B] for the clipped value loss
(config_nn.VALUE_CLIP); without it the learner uses values[0] - advs."""
from typing import List

import numpy as np
import torch


class Experience:
    __slots__ = ["states", "actions", "old_logps", "rewards", "dones", "advs", "values", "durations", "is_clean", "old_values"]

    def __init__(self, states, advs=None, actions=None, old_logps=None, values=None, rewards=None, dones=None,
                 durations=None, is_clean=None, old_values=None):
        self.states = states
        self.advs = advs
        self.actions = actions
        self.old_logps = old_logps
        self.values = values
        self.rewards = rewards
        self.dones = dones
        self.durations = durations
        self.is_clean = is_clean
        self.old_values = old_values

    def __len__(self):
        return len(self.states[0])

    def get_xrapv(self):
        return [self.states, self.advs, self.actions, self.old_logps, self.values]

    def to_tensor(self, dtype=torch.float32, device="cuda", non_blocking=True):
        """fp32 device copies of all five fields, and of old_values when present (reference: experience.py:56-62, one
        blocking torch.tensor() each).  Host arrays are staged through pinned memory so the H2D copies are asynchronous."""
        def move(x):
            if torch.is_tensor(x):
                return x.to(device=device, dtype=dtype, non_blocking=non_blocking)
            t = torch.from_numpy(np.ascontiguousarray(x))
            if torch.cuda.is_available() and str(device).startswith("cuda"):
                t = t.pin_memory()
            return t.to(device=device, dtype=dtype, non_blocking=non_blocking)
        self.states = [move(s) for s in self.states]
        self.advs, self.actions, self.old_logps, self.values = map(move, (self.advs, self.actions, self.old_logps, self.values))
        if self.old_values is not None:
            self.old_values = move(self.old_values)

    @classmethod
    def batch_data(cls, exps: List["Experience"]) -> "Experience":
        """Concatenate per-env chunks into one training batch (experience.py:116-148, clean=True path).  old_values are
        carried when every chunk has them."""
        n_slots = len(exps[0].states)
        states = [np.concatenate([e.states[i] for e in exps], axis=0) for i in range(n_slots)]
        cat = lambda f, ax: np.concatenate([getattr(e, f) for e in exps], axis=ax)
        old_values = cat("old_values", 0) if all(e.old_values is not None for e in exps) else None
        return cls(states=states, advs=cat("advs", 0), actions=cat("actions", 0), old_logps=cat("old_logps", 0),
                   values=cat("values", 1), old_values=old_values)
