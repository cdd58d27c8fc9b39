"""Default PPO-Clip hyper-parameters for the classic-control tasks, as a Namespace shaped like the one the
reference builds from YAML (xuance/common/common_tools.py:32-83).  Values restate
xuance/configs/ppo/classic_control/CartPole-v1.yaml and Pendulum-v1.yaml (identical except env_id/policy);
`use_obsnorm` / `use_rewnorm` default to False here because the BASELINE configs are measured without them (the yaml
default is True); the device-side normalisers (SURVEY.md §8 f1, csrc/normalize.cu) run when they are switched on,
single GPU and env-sharded."""
from argparse import Namespace

_COMMON = dict(
    agent="PPO_Clip", env_name="Classic Control", vectorize="B200_Gym", representation="Basic_MLP", runner="DRL",
    representation_hidden_size=[128], actor_hidden_size=[128], critic_hidden_size=[128], activation="LeakyReLU",
    seed=1, parallels=10, running_steps=300000, n_steps=256, n_epoch=8, n_minibatch=8, learning_rate=0.0004,
    use_grad_clip=True, vf_coef=0.25, ent_coef=0.01, target_kl=0.001, clip_range=0.2, clip_grad_norm=0.5, gamma=0.98,
    use_gae=True, gae_lambda=0.95, use_advnorm=True, use_obsnorm=False, use_rewnorm=False, obsnorm_range=5,
    rewnorm_range=5, render=False, device="cuda", model_dir="./models/ppo/", log_dir="./logs/ppo/",
)


def ppo_config(env_id, **overrides):
    """`policy`: "Gaussian_AC" for an env with a Box action (Pendulum-v1, MountainCarContinuous-v0), "Categorical_AC"
    otherwise (ids without a device kernel included)."""
    from .vec_env import SPECS, continuous_actions
    cfg = dict(_COMMON)
    cfg["env_id"] = env_id
    cfg["policy"] = "Gaussian_AC" if env_id in SPECS and continuous_actions(env_id) else "Categorical_AC"
    cfg.update(overrides)
    return Namespace(**cfg)


def build_ppo(env_id, device="cuda", process_group=None, policy_seed=None, agent_class=None, **overrides):
    """Envs + policy + Adam + LinearLR + agent, wired like Runner_DRL.__init__ (xuance/torch/runners/runner_drl.py:15-74).
    `agent_class`: PPOCLIP_Agent (default) or A2C_Agent."""
    import torch

    from .agent import PPOCLIP_Agent
    from .policies import make_policy
    from .vec_env import DummyVecEnv_Gym, make_env_fns
    cfg = ppo_config(env_id, device=device, **overrides)
    torch.manual_seed(cfg.seed if policy_seed is None else policy_seed)   # replicated policy: same init on every rank
    envs = DummyVecEnv_Gym(make_env_fns(env_id, cfg.seed, cfg.parallels), device=device, native=True)
    envs.reset()                                                          # runner_basic.py:12
    policy = make_policy(envs.observation_space, envs.action_space, hidden=tuple(cfg.representation_hidden_size),
                         device=device)
    optimizer = torch.optim.Adam(policy.parameters(), cfg.learning_rate, eps=1e-5)      # runner_drl.py:71
    scheduler = torch.optim.lr_scheduler.LinearLR(optimizer, start_factor=1.0, end_factor=0.0,
                                                  total_iters=int(cfg.running_steps))    # runner_drl.py:72-73
    agent = (agent_class or PPOCLIP_Agent)(cfg, envs, policy, optimizer, scheduler, device, process_group=process_group)
    return agent


# xuance/configs/pg/classic_control/*.yaml and xuance/configs/ppg/classic_control/*.yaml (activation: the yamls say ReLU)
_PG = dict(_COMMON, agent="PG", n_steps=128, n_epoch=1, n_minibatch=1, clip_grad=0.5, use_gae=False, use_advnorm=False,
           use_obsnorm=True, use_rewnorm=True, activation="ReLU", model_dir="./models/pg/", log_dir="./logs/pg/")
_PPG = dict(_COMMON, agent="PPG", n_steps=256, n_epoch=1, n_minibatch=1, policy_nepoch=4, value_nepoch=8, aux_nepoch=8,
            kl_beta=1.0, use_obsnorm=True, use_rewnorm=True, activation="ReLU", model_dir="./models/ppg/",
            log_dir="./logs/ppg/")


def _build(defaults, env_id, agent_name, policy_builder, device, overrides, agent_class=None, process_group=None,
           policy_seed=None):
    import torch
    from torch import nn

    from . import agent as agents
    from .policies import MLPRepresentation
    from .vec_env import DummyVecEnv_Gym, make_env_fns
    cfg = dict(defaults, env_id=env_id, device=device)
    cfg.update(overrides)
    cfg = Namespace(**cfg)
    torch.manual_seed(cfg.seed if policy_seed is None else policy_seed)
    envs = DummyVecEnv_Gym(make_env_fns(env_id, cfg.seed, cfg.parallels), device=device, native=True)
    envs.reset()
    act = {"ReLU": nn.ReLU, "LeakyReLU": nn.LeakyReLU}[cfg.activation]
    rep = MLPRepresentation(envs.observation_space.shape, list(cfg.representation_hidden_size), activation=act, device=device)
    policy = policy_builder(cfg, envs, rep, act)
    optimizer = torch.optim.Adam(policy.parameters(), cfg.learning_rate, eps=1e-5)
    scheduler = torch.optim.lr_scheduler.LinearLR(optimizer, start_factor=1.0, end_factor=0.0, total_iters=int(cfg.running_steps))
    return (agent_class or getattr(agents, agent_name))(cfg, envs, policy, optimizer, scheduler, device, process_group=process_group)


def build_pg(env_id, device="cuda", agent_class=None, process_group=None, policy_seed=None, **overrides):
    """PG_Agent wired like Runner_DRL does for the pg yamls (Categorical_Actor / Gaussian_Actor policy).
    `process_group`: env-sharded training as in build_ppo (default: the initialised default group, if any); `policy_seed`:
    the torch seed of the policy's initialisation, as in build_ppo (default: the config seed)."""
    from .policies import CategoricalActor, GaussianActor
    from .spaces import is_discrete

    def policy(cfg, envs, rep, act):
        cls = CategoricalActor if is_discrete(envs.action_space) else GaussianActor
        return cls(envs.action_space, rep, list(cfg.actor_hidden_size), activation=act, device=device)
    return _build(_PG, env_id, "PG_Agent", policy, device, overrides, agent_class, process_group, policy_seed)


def build_ppg(env_id, device="cuda", agent_class=None, process_group=None, policy_seed=None, **overrides):
    """PPG_Agent wired like Runner_DRL does for the ppg yamls (Categorical_PPG / Gaussian_PPG policy).
    `process_group`: env-sharded training as in build_ppo (default: the initialised default group, if any); `policy_seed`:
    the torch seed of the policy's initialisation, as in build_ppo (default: the config seed)."""
    from .policies import CategoricalPPGActorCritic, GaussianPPGActorCritic
    from .spaces import is_discrete

    def policy(cfg, envs, rep, act):
        cls = CategoricalPPGActorCritic if is_discrete(envs.action_space) else GaussianPPGActorCritic
        return cls(envs.action_space, rep, list(cfg.actor_hidden_size), list(cfg.critic_hidden_size), activation=act,
                   device=device)
    return _build(_PPG, env_id, "PPG_Agent", policy, device, overrides, agent_class, process_group, policy_seed)


def build_ppokl(env_id, device="cuda", agent_class=None, process_group=None, policy_seed=None, **overrides):
    """PPOKL_Agent wired like build_ppo (envs, the actor-critic policy, Adam, LinearLR, the agent).  The reference's ppokl
    yamls are not restated here, so the defaults are the PPO classic-control ones of `_COMMON` (including its `target_kl`)
    with `agent="PPO_KL"`; every key can be overridden.  `process_group` / `policy_seed` as in build_ppo."""
    from .agent import PPOKL_Agent
    return build_ppo(env_id, device=device, process_group=process_group, policy_seed=policy_seed,
                     agent_class=agent_class or PPOKL_Agent, **dict(dict(agent="PPO_KL"), **overrides))
