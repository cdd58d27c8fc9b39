"""xuanpolicy_b200 — B200-native (sm_100a) on-policy PPO hot path behind XuanCe's Python API.

Drop-in classes (same names / signatures as the reference, see each module's docstring for file:line):
    DummyVecEnv_Gym      vec_env.py   <- xuance/environment/gym/gym_vec_env.py:148-231
    DummyOnPolicyBuffer  buffer.py    <- xuance/common/memory_tools.py:143-245
    PPOCLIP_Learner      learner.py   <- xuance/torch/learners/policy_gradient/ppoclip_learner.py:4-65
    A2C / PG / PPOKL / PPG_Learner   learner.py <- xuance/torch/learners/policy_gradient/{a2c,pg,ppokl,ppg}_learner.py
    PPOCLIP_Agent        agent.py     <- xuance/torch/agents/policy_gradient/ppoclip_agent.py:4-165 (vectorised loop)
    A2C_Agent            agent.py     <- xuance/torch/agents/policy_gradient/a2c_agent.py:6-100 (same loop, A2C surrogate)
    PG_Agent             agent.py     <- xuance/torch/agents/policy_gradient/pg_agent.py:4-96 (same loop, returns as weights)
    PPOKL_Agent          agent.py     <- xuance/torch/agents/policy_gradient/ppokl_agent.py (same loop, adaptive KL penalty)
    PPG_Agent            agent.py     <- xuance/torch/agents/policy_gradient/ppg_agent.py:4-109 (device rollout, 3 update phases)
All arithmetic on the path runs in hand-written CUDA kernels reached through the C ABI of include/xb200.h
(libxb200.so, bound with ctypes in _lib.py).  There is no CPU fallback: importing works anywhere, but
constructing any of the classes without the library or without a CUDA device raises.
"""
from ._lib import XB200Error, load as load_library  # noqa: F401
from .spaces import Box, Discrete  # noqa: F401
from .vec_env import (AlreadySteppingError, DummyVecEnv_Gym, EnvFn, NotSteppingError, make_env_fns,  # noqa: F401
                      make_spaces)
from .buffer import DummyOnPolicyBuffer  # noqa: F401
from .learner import A2C_Learner, PG_Learner, PPG_Learner, PPOCLIP_Learner, PPOKL_Learner  # noqa: F401
from .policies import (CategoricalActor, CategoricalActorCritic, CategoricalPPGActorCritic, GaussianActorCritic,  # noqa: F401
                       GaussianActor, GaussianPPGActorCritic, MLPRepresentation, make_policy)

__version__ = "0.1.0"


def __getattr__(name):
    if name in ("PPOCLIP_Agent", "A2C_Agent", "PG_Agent", "PPOKL_Agent", "PPG_Agent"):
        from . import agent
        return getattr(agent, name)
    raise AttributeError(name)
