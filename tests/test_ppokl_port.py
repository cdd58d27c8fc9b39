"""CPU: the restated PPOKL_Agent loop (tests/ppokl_port.PPOKLAgentPort) is PPOAgentPort's rollout with the old
distributions stored, and each of its updates is `ppokl_update` on that minibatch with the coefficient carried over;
`configs.build_ppokl` wires the documented config."""
import copy

import numpy as np
import pytest
import torch

from oracle import ref_port
from tests.ppokl_port import PPOKLAgentPort
from xuanpolicy_b200 import policies

N, T, H = 4, 8, 16


def _setup(env_id, seed=3):
    torch.manual_seed(5)
    np.random.seed(5)
    envs = ref_port.VecEnvPort(env_id, N, seed=seed, trig="cr")
    envs.reset()
    pol = policies.make_policy(envs.observation_space, envs.action_space, hidden=(H,), device="cpu")
    opt = torch.optim.Adam(pol.parameters(), 4e-4, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=1000)
    return envs, pol, opt, sched


def _first_rollout(port):
    """The buffer the first update reads (taken at the first `sample`)."""
    mem, out = port.memory, {}
    sample = mem.sample

    def hook(idx):
        if not out:
            out.update(obs=mem.observations.copy(), act=mem.actions.copy(), rew=mem.rewards.copy(), val=mem.values.copy(),
                       ret=mem.returns.copy(), adv=mem.advantages.copy(), term=mem.terminals.copy())
        return sample(idx)
    mem.sample = hook
    return out


@pytest.mark.parametrize("env_id,use_gae", [("CartPole-v1", True), ("Pendulum-v1", False)])
def test_ppokl_port_rollout_is_the_ppo_port_rollout(env_id, use_gae):
    envs, pol, opt, sched = _setup(env_id)
    kw = dict(use_gae=use_gae, use_advnorm=True, use_obsnorm=True, use_rewnorm=True)
    port = PPOKLAgentPort(envs, pol, opt, sched, T, 2, 2, 0.98, 0.95, record=True, **kw)
    mine = _first_rollout(port)
    port.train(T + 2)
    envs2, pol2, opt2, sched2 = _setup(env_id)          # same envs, same initial parameters
    ppo = ref_port.PPOAgentPort(envs2, pol2, opt2, sched2, T, 2, 2, 0.98, 0.95, action_tape=np.stack(port.recorded_actions),
                                perm_tape=port.recorded_perms, **kw)
    theirs = _first_rollout(ppo)
    ppo.train(T)
    assert set(mine) == set(theirs)
    for k in mine:
        assert np.array_equal(mine[k], theirs[k]), k
    # the stored old distributions are the parameters the actions were drawn from
    old = port.memory.auxiliary_infos["old_dist"]
    assert old.shape == (N, T, 2)
    assert np.all(np.isfinite(old))


@pytest.mark.parametrize("env_id", ["CartPole-v1", "Pendulum-v1"])
def test_ppokl_port_updates_are_ppokl_update(env_id):
    envs, pol, opt, sched = _setup(env_id)
    port = PPOKLAgentPort(envs, pol, opt, sched, T, 2, 2, 0.98, 0.95, target_kl=0.001, use_obsnorm=True)
    checked = []
    update = port.update

    def hook(obs, act, ret, adv, old):
        p = policies.make_policy(envs.observation_space, envs.action_space, hidden=(H,), device="cpu")
        p.load_state_dict(port.policy.state_dict())
        o = torch.optim.Adam(p.parameters(), 4e-4, eps=1e-5)
        o.load_state_dict(copy.deepcopy(port.optimizer.state_dict()))
        s = torch.optim.lr_scheduler.LinearLR(o, start_factor=1.0, end_factor=0.0, total_iters=1000)
        s.load_state_dict(port.scheduler.state_dict())
        st = dict(port.kl_state)
        want = ref_port.ppokl_update(p, o, s, (obs, act, ret, adv), old, st, vf_coef=0.25, ent_coef=0.01, target_kl=0.001)
        info = update(obs, act, ret, adv, old)
        for a, b in zip(p.parameters(), port.policy.parameters()):
            assert torch.equal(a, b)
        assert st == port.kl_state and info == want
        checked.append(info["kl"])
        return info
    port.update = hook
    port.train(2 * T)
    assert len(checked) == 2 * 2 * 2
    kl, used, after = zip(*port.kl_trace)
    assert used[0] == 1.0 and all(u == a for u, a in zip(used[1:], after[:-1]))
    for k, u, a in port.kl_trace:                   # the rule of ppokl_learner.py:39-43
        want = u * 2.0 if k > 0.0015 else (u / 2.0 if k < 0.0005 else u)
        assert a == float(np.clip(want, 0.1, 20))


def test_build_ppokl_config(monkeypatch):
    from xuanpolicy_b200 import configs, spaces, vec_env

    class FakeEnvs:
        def __init__(self, fns, device=None, native=False):
            self.observation_space, self.action_space = spaces.Box(-1.0, 1.0, (4,)), spaces.Discrete(2)

        def reset(self):
            pass
    monkeypatch.setattr(vec_env, "DummyVecEnv_Gym", FakeEnvs)
    monkeypatch.setattr(policies, "make_policy", lambda o, a, hidden, device: torch.nn.Linear(4, 2))
    got = {}

    def agent(cfg, envs, policy, opt, sched, device, process_group=None):
        got.update(cfg=cfg, opt=opt, sched=sched)
        return "agent"
    assert configs.build_ppokl("CartPole-v1", device="cpu", agent_class=agent, target_kl=0.02, n_steps=16) == "agent"
    cfg = got["cfg"]
    assert cfg.agent == "PPO_KL" and cfg.env_id == "CartPole-v1" and cfg.policy == "Categorical_AC"
    assert cfg.target_kl == 0.02 and cfg.n_steps == 16
    for k, v in configs._COMMON.items():
        if k not in ("agent", "target_kl", "n_steps", "device"):
            assert getattr(cfg, k) == v, k
    assert isinstance(got["opt"], torch.optim.Adam) and isinstance(got["sched"], torch.optim.lr_scheduler.LinearLR)
    assert got["sched"].total_iters == configs._COMMON["running_steps"]
    from xuanpolicy_b200.agent import PPOKL_Agent
    import xuanpolicy_b200 as xb
    assert xb.PPOKL_Agent is PPOKL_Agent
