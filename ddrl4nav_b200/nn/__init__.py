"""Mirror of ``USTC_lab.nn`` for the hot path: same class names and constructor signatures
(USTC_lab/nn/__init__.py:8-43).  RND / GAIL / Discriminator stay with the reference (out of scope)."""
from .utils import mlp, merge
from .base import Basenn, PreNet
from .critic import Critic
from .actor import BetaActor, CategoricalActor, Actor, GaussionActor, MultiCategorical, MultiCategoricalActor
from .ppo import PPO
from .nav_encoder import NavPreNet, NavPedPreNet, NavPreNet1D
from .atari_encoder import AtariPreNet
from .mlp_encoder import MLPPreNet

NETWORK_MAP = {"ppo": PPO}

__all__ = ["PPO", "NavPreNet", "Basenn", "PreNet", "NETWORK_MAP", "CategoricalActor", "GaussionActor", "BetaActor", "Critic",
           "MultiCategoricalActor", "MultiCategorical",
           "AtariPreNet", "MLPPreNet", "Actor", "mlp", "merge", "NavPedPreNet", "NavPreNet1D"]
