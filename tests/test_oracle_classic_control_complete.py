"""CPU: the last two of gym 0.26.2's six classic-control ids, MountainCarContinuous-v0 and CartPole-v0, in the oracles and
the drop-in's host side.

- the C oracle and the Python restatement of Continuous_MountainCarEnv (tests/classic_control_ext.c / .py) agree bit for bit in both trig flavours over a tape
  with actions outside [-1, 1], cars stopped by the left wall, goal terminations and truncations at 999;
- known answers written out from the operation order (the first step of an episode runs on the unrounded fp64 draw, every
  later one on the float32 state; the reward's penalty takes the unclipped action);
- CartPole-v0: the same agreement, with truncation at 200;
- the spaces of the three new ids, the 4-frame port of the continuous env and the PPO config's policy choice."""
import math

import numpy as np
import pytest

from tests import classic_control_ext as ext


def _pump(obs_v, rng, n, amp=1.6):
    """Energy pumping along the velocity with Gaussian noise: actions outside [-1, 1], swings that reach the goal and the
    left wall."""
    return (np.where(obs_v > 0, amp, -amp) + 0.5 * rng.standard_normal(n)).astype(np.float32)


def _wall(obs):
    """Pumps on the left slope only: the car swings ever higher to the left and is stopped by the wall at -1.2."""
    p, v = obs[:, 0], obs[:, 1]
    return np.where(v < 0, -1.6, np.where(p < -0.75, 1.6, -1.6)).astype(np.float32)


@pytest.mark.parametrize("flavour", ["cr", "libm"])
def test_mountaincar_continuous_c_and_python_restatements_agree(flavour):
    n = 8
    ref = ext.vec_env_c("gym:MountainCarContinuous-v0", n, seed=3, flavour=flavour, n_warm_resets=2)
    envs = []
    for e in range(n):
        p = ext.make("MountainCarContinuous-v0", trig=flavour)
        p.reset(seed=3)
        ob, _ = p.reset()
        assert np.array_equal(ob, ref.obs[e])
        envs.append(p)
    assert envs[0]._max_episode_steps == 999
    rng = np.random.default_rng(11)
    n_term = n_trunc = n_wall = n_outside = 0
    obs = ref.obs.copy()
    for t in range(1100):
        a = _pump(obs[:, 1], rng, n)
        a[4:6] = _wall(obs[4:6])
        a[6:] = (0.3 * rng.standard_normal(2)).astype(np.float32)      # two cars without a plan: they truncate at 999
        n_outside += int((np.abs(a) > 1.0).sum())
        o = ref.step(a.reshape(n, 1))
        for e in range(n):
            ob, r, term, trunc, _ = envs[e].step(a[e:e + 1])
            assert np.array_equal(ob, o["obs"][e]) and np.float32(r) == o["rew"][e], (flavour, t, e)
            assert term == o["term"][e] and trunc == o["trunc"][e], (flavour, t, e)
            n_wall += int(ob[0] == np.float32(-1.2) and ob[1] == 0.0)
            n_term, n_trunc = n_term + int(term), n_trunc + int(trunc)
            if term or trunc:
                ro, _ = envs[e].reset()
                assert np.array_equal(ro, o["reset_obs"][e])
            # the fp64 state: (double)(float) after a step, the unrounded draw after a reset
            assert np.array_equal(np.asarray(envs[e].env.state, np.float64), o["state"][e]), (flavour, t, e)
        obs = np.where((o["term"] | o["trunc"])[:, None], o["reset_obs"], o["obs"])
    assert n_term > 0 and n_trunc >= 2 and n_wall > 0 and n_outside > 0, (n_term, n_trunc, n_wall, n_outside)
    assert o["ep_step"][6:].tolist() == [1100 - 999] * 2                 # the planless cars truncated once, at step 999


def _cos_cr(x):
    from oracle import gym_restated
    return gym_restated._cos_cr(x)


def test_mountaincar_continuous_known_answers():
    """The operation order written out in fp64 (every operation rounded on its own), against the C oracle ("cr")."""
    env = ext.vec_env_c("gym:MountainCarContinuous-v0", 1, seed=1, flavour="cr", n_warm_resets=2)
    draw = np.random.Generator(np.random.PCG64(np.random.SeedSequence(1)))
    draw.uniform(-0.6, -0.4)
    p64 = float(draw.uniform(-0.6, -0.4))
    assert env.state[0].tolist() == [p64, 0.0] and float(np.float32(p64)) != p64       # the state after reset is the fp64 draw
    # step 1 (action 0.5): on the UNROUNDED position
    v = 0.0 + (0.5 * 0.0015 - 0.0025 * _cos_cr(3 * p64))
    p = p64 + v
    o = env.step(np.array([[0.5]], np.float32))
    assert o["state"][0].tolist() == [float(np.float32(p)), float(np.float32(v))]
    v_rounded = 0.0 + (0.5 * 0.0015 - 0.0025 * _cos_cr(3 * float(np.float32(p64))))
    p_rounded = float(np.float32(p64)) + v_rounded                         # the rounded draw gives another answer
    assert [float(np.float32(p_rounded)), float(np.float32(v_rounded))] != o["state"][0].tolist()
    assert o["rew"][0] == np.float32(-(0.5 * 0.5) * 0.1) and not o["term"][0]
    # step 2 (action -3.0: force clipped to -1, penalty on the unclipped action): on the float32 state
    p1, v1 = (float(x) for x in o["state"][0])
    v2 = v1 + (-1.0 * 0.0015 - 0.0025 * _cos_cr(3 * p1))
    o = env.step(np.array([[-3.0]], np.float32))
    assert o["state"][0].tolist() == [float(np.float32(p1 + v2)), float(np.float32(v2))]
    assert float(o["rew"][0]) == float(np.float32(0.0 - 9.0 * 0.1)) and o["ep_score"][0] == -(0.25 * 0.1) + -(9.0 * 0.1)
    assert [float.hex(float(x)) for x in o["state"][0]] == MC_CONT_KAT
    # the goal: from (0.44, 0.02) with action 1.25, terminated on the fp64 values, reward 100 - 1.25**2 * 0.1
    env.state[0] = [0.44, 0.02]
    o = env.step(np.array([[1.25]], np.float32))
    assert o["term"][0] and o["rew"][0] == np.float32(100.0 - 1.5625 * 0.1)
    # the left wall: position clipped to -1.2 and the velocity stopped
    env.state[0] = [-1.19, -0.05]
    o = env.step(np.array([[-1.0]], np.float32))
    assert o["state"][0].tolist() == [float(np.float32(-1.2)), 0.0] and not o["term"][0]


MC_CONT_KAT = ["-0x1.a650380000000p-2", "-0x1.3d71260000000p-9"]


def test_cartpole_v0_c_and_python_restatements_agree_and_truncate_at_200():
    for fl in ("cr", "libm"):
        n = 4
        ref = ext.vec_env_c("CartPole-v0", n, seed=2, flavour=fl, n_warm_resets=2)
        envs = []
        for e in range(n):
            p = ext.make("CartPole-v0", trig=fl)
            p.reset(seed=2)
            assert np.array_equal(p.reset()[0], ref.obs[e])
            envs.append(p)
        rng = np.random.default_rng(1)
        n_trunc = n_term = 0
        obs = ref.obs.copy()
        for t in range(450):
            heur = (obs[:, 2] + 0.5 * obs[:, 3] > 0).astype(np.int64)           # balances: the episodes reach 200
            a = np.where(rng.random(n) < 0.95, heur, rng.integers(0, 2, n))
            a[3] = rng.integers(0, 2)                                            # falls over: terminates
            o = ref.step(a)
            for e in range(n):
                ob, r, term, trunc, _ = envs[e].step(a[e])
                assert np.array_equal(ob, o["obs"][e]) and r == o["rew"][e], (fl, t, e)
                assert term == o["term"][e] and trunc == o["trunc"][e], (fl, t, e)
                if trunc:
                    assert o["ep_step"][e] == 200
                n_term, n_trunc = n_term + int(term), n_trunc + int(trunc)
                if term or trunc:
                    assert np.array_equal(envs[e].reset()[0], o["reset_obs"][e])
            obs = np.where((o["term"] | o["trunc"])[:, None], o["reset_obs"], o["obs"])
        assert n_term > 0 and n_trunc > 0 and o["ep_step"].max() <= 200


def test_spaces_of_the_new_ids():
    import xuanpolicy_b200 as xb
    from xuanpolicy_b200.vec_env import SPECS, continuous_actions
    f32 = lambda x: np.asarray(x, np.float32)
    for env_id in ("gym:MountainCarContinuous-v0", "MountainCarContinuous-v0"):
        obs_space, act_space = xb.make_spaces(env_id)
        assert isinstance(act_space, xb.Box) and act_space.shape == (1,) and act_space.dtype == np.float32
        assert np.array_equal(act_space.low, f32([-1.0])) and np.array_equal(act_space.high, f32([1.0]))
        k = 1 if env_id.startswith("gym:") else 4
        assert obs_space.shape == (2 * k,) and obs_space.dtype == np.float32
        assert np.array_equal(obs_space.low, f32([-1.2, -0.07] * k)) and np.array_equal(obs_space.high, f32([0.6, 0.07] * k))
        assert continuous_actions(env_id) and SPECS[env_id]["max_steps"] == 999 and SPECS[env_id]["obs_dim"] == 2 * k
    gym_env = ext.MountainCarContinuousRestated()        # gym's own spaces (bounds as float32)
    obs_space, act_space = xb.make_spaces("gym:MountainCarContinuous-v0")
    assert np.array_equal(obs_space.low, gym_env.observation_space.low)
    assert np.array_equal(obs_space.high, gym_env.observation_space.high)
    assert np.array_equal(act_space.low, gym_env.action_space.low) and np.array_equal(act_space.high, gym_env.action_space.high)
    obs_space, act_space = xb.make_spaces("CartPole-v0")
    ref_obs, ref_act = xb.make_spaces("CartPole-v1")
    assert np.array_equal(obs_space.low, ref_obs.low) and np.array_equal(obs_space.high, ref_obs.high)
    assert isinstance(act_space, xb.Discrete) and act_space.n == 2 and not continuous_actions("CartPole-v0")
    assert SPECS["CartPole-v0"]["max_steps"] == 200 and SPECS["CartPole-v0"]["kind"] == SPECS["CartPole-v1"]["kind"]
    cp = ext.make("CartPole-v0", trig="libm")
    assert cp._max_episode_steps == 200 and np.array_equal(cp.observation_space.high, ref_obs.high)
    with pytest.raises(NotImplementedError):
        xb.make_spaces("MountainCarContinuous-v1")


def test_port_applies_the_four_frame_wrapper(monkeypatch):
    from oracle import ref_port
    ext.register(monkeypatch)
    n = 3
    port = ref_port.VecEnvPort("MountainCarContinuous-v0", n, seed=4, trig="cr")
    assert isinstance(port.envs[0], ref_port.MountainCarStackPort) and port.max_episode_length == 999
    assert port.observation_space.shape == (8,) and port.action_space.shape == (1,)
    obs, _ = port.reset()
    assert np.array_equal(obs[:, 0:2], obs[:, 6:8]) and np.array_equal(obs[:, 0:2], obs[:, 2:4])
    ref = ext.vec_env_c("MountainCarContinuous-v0", n, seed=4, flavour="cr", n_warm_resets=2)
    assert np.array_equal(obs, ref.obs)
    rng = np.random.default_rng(0)
    for t in range(20):
        a = _pump(obs[:, -1], rng, n).reshape(n, 1)
        obs, rew, term, trunc, _ = port.step(a)
        o = ref.step(a)
        assert np.array_equal(obs, o["obs"]) and np.array_equal(rew, o["rew"]), t
    bare = ref_port.VecEnvPort("gym:MountainCarContinuous-v0", n, seed=4, trig="cr")
    assert not isinstance(bare.envs[0], ref_port.MountainCarStackPort) and bare.observation_space.shape == (2,)


def test_ppo_config_policy_follows_the_action_space():
    from xuanpolicy_b200.configs import ppo_config
    for env_id in ("MountainCarContinuous-v0", "gym:MountainCarContinuous-v0", "Pendulum-v1"):
        assert ppo_config(env_id).policy == "Gaussian_AC", env_id
    for env_id in ("CartPole-v1", "CartPole-v0", "MountainCar-v0", "gym:MountainCar-v0", "Acrobot-v1", "LunarLander-v2"):
        assert ppo_config(env_id).policy == "Categorical_AC", env_id
    assert math.isclose(ppo_config("MountainCarContinuous-v0").learning_rate, 0.0004)
