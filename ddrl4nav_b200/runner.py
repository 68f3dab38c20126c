"""Net factory -- the decisions of ``create_net`` (USTC_lab/runner/utils.py:59-170) for the hot path:
which encoder family per task type and whether actor/critic share it.  ``create_net(configs)``
takes the reference's ``configs`` dict unchanged; ``make_net(kind)`` is the short form used by
tests and bench for the three BASELINE configurations."""
from types import SimpleNamespace

import torch

from ._lib import DDRLError
from .nn import (PPO, AtariPreNet, BetaActor, CategoricalActor, Critic, GaussionActor, MLPPreNet, MultiCategoricalActor, NavPedPreNet,
                 NavPreNet, NavPreNet1D)


def _bounds_kwargs(actor_cls, config_nn):
    """BetaActor's action interval from the optional config_nn.ACTION_LOW / ACTION_HIGH (numbers or length-A sequences;
    BetaActor validates them), and MultiCategoricalActor's branch sizes from config_nn.ACTION_NVEC (required; the actor
    validates them).  Other actors take neither."""
    if actor_cls is MultiCategoricalActor:
        nvec = getattr(config_nn, "ACTION_NVEC", None)
        if nvec is None:
            raise DDRLError("MultiCategoricalActor needs config_nn.ACTION_NVEC (the branch sizes)")
        return {"nvec": nvec}
    if actor_cls is not BetaActor:
        return {}
    kw = {}
    for key, arg in (("ACTION_LOW", "low"), ("ACTION_HIGH", "high")):
        v = getattr(config_nn, key, None)
        if v is not None:
            kw[arg] = v
    return kw


def create_net(configs):
    config, config_nn, config_env = configs["config"], configs["config_nn"], configs["config_env"]
    dev = getattr(config_nn, "DEVICE", "cuda")
    feat = config_nn.AC_INPUT_DIM
    actor_cls = config_nn.ACTOR_CLASS
    if isinstance(actor_cls, type) and actor_cls.__module__.startswith("USTC_lab"):     # reference class -> ours
        actor_cls = GaussionActor if actor_cls.__name__ == "GaussionActor" else CategoricalActor

    def heads(pre_a, pre_c):
        actor = actor_cls(action_output_dim=config_nn.ACTION_OUTPUT_DIM, device=dev, soft_max_grid=config_nn.SOFT_MAX_GRID,
                          last_input_dim=feat, nn_dtype=config_nn.MODULE_TENSOR_DTYPE, pre=pre_a,
                          **_bounds_kwargs(actor_cls, config_nn))
        return actor, Critic(device=dev, last_input_dim=feat, pre=pre_c)

    share = config_nn.SHARE_CNN_NET
    task = config.TASK_TYPE
    if task in ("mujoco", "classical"):
        mk = lambda: MLPPreNet(config_env.get("input_dim", 4), feat)
    elif task in ("robot_nav", "gazebo_env", "real_env"):
        if share:
            if config_env["ped_sim"]["total"] > 0:
                mk = lambda: NavPedPreNet(image_channel=config_env["image_batch"] + 3, last_output_dim=feat)
            else:
                mk = lambda: NavPreNet(image_channel=config_env["image_batch"], last_output_dim=feat)
        else:
            mk = lambda: NavPreNet1D(image_channel=3, last_output_dim=feat)
    elif task == "atari":
        mk = lambda: AtariPreNet(config_env["int_frame_stack"], last_output_dim=feat, device=dev)
    else:
        raise ValueError("unknown TASK_TYPE %r" % task)
    if getattr(config, "USE_RND", False) or config_nn.NETWORK_TYPE != "ppo":
        raise NotImplementedError("RND / GAIL are outside the B200 hot path; use the reference's create_net")
    if share:
        actor, critic = heads(None, None)
        prenet = mk()
    else:
        actor, critic = heads(mk(), mk())
        prenet = None
    return PPO(actor, critic, prenet, None, config, config_nn).to(dev)


_KINDS = {
    #  kind: (encoder factory, distribution, act_dim, shared)
    "pong": (lambda: AtariPreNet(4, 512), "categorical", 6, False),                 # BASELINE C1 / C4
    "navlaser": (lambda: NavPreNet1D(image_channel=3), "gaussian", 2, False),       # C2
    "navlaser3": (lambda: NavPreNet1D(image_channel=3, laser_channel=3), "gaussian", 2, False),   # NON-reference 3 x 960 laser
    "navimg": (lambda: NavPreNet(image_channel=1), "categorical", 28, True),        # C5
    "navped": (lambda: NavPedPreNet(image_channel=4), "categorical", 28, True),
    "mlp": (lambda: MLPPreNet(4, 128), "categorical", 2, False),
    # NON-reference Beta actor on [ACTION_LOW, ACTION_HIGH] (default [-1, 1]) per dimension: C2's encoder, and C5's
    "navlaser_beta": (lambda: NavPreNet1D(image_channel=3), "beta", 2, False),
    "navimg_beta": (lambda: NavPreNet(image_channel=1), "beta", 2, True),
    # NON-reference MultiDiscrete actor (act_dim: the default branch sizes, ACTION_NVEC overrides them): C5's 28 (v, w) commands
    # as 4 speeds x 7 turn rates on the shared encoder, and a 5 x 9 grid on C2's unshared one
    "navimg_md": (lambda: NavPreNet(image_channel=1), "multi_categorical", (4, 7), True),
    "navlaser_md": (lambda: NavPreNet1D(image_channel=3), "multi_categorical", (5, 9), False),
}


def make_net(kind: str, device="cuda", gemm_mode=None, **hyper):
    """PPO net of one of the named configurations with the reference's default hyper-parameters
    (config/config_nn.py:27-57); `hyper` overrides ConfigNN attribute names (e.g. TRAINING_ITER_TIME=1, ACTION_LOW /
    ACTION_HIGH for the Beta kinds, or ACTION_NVEC for the MultiDiscrete kinds)."""
    mk, dist, act_dim, shared = _KINDS[kind]
    if dist == "multi_categorical":
        hyper.setdefault("ACTION_NVEC", act_dim)
        act_dim = None
    cfg_nn = dict(SHARE_CNN_NET=shared, PPO_CLIP=0.2, DUEL_PPO_CLIP=3, V_LOSS_THETA=1.0, ENTROPY_LOSS_THETA=0.05,
                  CLIP_GRID=True, CLIP_GRID_NUM=0.5, SMOOTH_L1_LOSS=False, LEARNING_RATE=2e-4, ACTOR_LEARNING_RATE=5e-5,
                  CRITIC_LEARNING_RATE=1e-3, TRAINING_ITER_TIME=10)
    cfg_nn.update(hyper)
    if gemm_mode is not None:
        cfg_nn["GEMM_MODE"] = gemm_mode
    config_nn = SimpleNamespace(**cfg_nn)
    config = SimpleNamespace(DEVICE=device, TASK_NAME="t-127.0.0.1", MODULE_KEY="MODEL")
    feat = 128 if kind == "mlp" else 512
    actor_cls = {"gaussian": GaussionActor, "beta": BetaActor, "multi_categorical": MultiCategoricalActor}.get(dist, CategoricalActor)
    bounds = _bounds_kwargs(actor_cls, config_nn)
    if shared:
        actor = actor_cls(action_output_dim=act_dim, device=device, last_input_dim=feat, **bounds)
        critic = Critic(device=device, last_input_dim=feat)
        prenet = mk()
    else:
        actor = actor_cls(action_output_dim=act_dim, device=device, last_input_dim=feat, pre=mk(), **bounds)
        critic = Critic(device=device, last_input_dim=feat, pre=mk())
        prenet = None
    net = PPO(actor, critic, prenet, None, config, config_nn)
    return net.to(device) if device is not None else net
