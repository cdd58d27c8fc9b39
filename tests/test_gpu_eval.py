"""GPU: `test()` on native device envs (DeviceEvaluator + xb_eval_step) against the reference's evaluation loop.

The oracle replay takes the actions the device drew (the evaluator's action tape) and runs them through the C oracle with the
reference's test loop (ppoclip_agent.py:113-165) and its RunningMeanStd: the scores must be equal bit for bit and in order, and
the observation statistics within the normaliser tolerances of test_gpu_normalize.py."""
import os

import numpy as np
import pytest
import torch

import xuanpolicy_b200 as xb
from xuanpolicy_b200 import checkpoint
from xuanpolicy_b200.agent import A2C_Agent
from xuanpolicy_b200.configs import build_pg, build_ppg, build_ppo

pytestmark = pytest.mark.gpu
ENVS = ["CartPole-v1", "Pendulum-v1", "Acrobot-v1", "MountainCar-v0", "gym:MountainCar-v0"]
EVAL_SEED = 11


def _env_fn(env_id, n, native=True, seed=EVAL_SEED):
    return lambda: xb.DummyVecEnv_Gym(xb.make_env_fns(env_id, seed, n), device="cuda", native=native)


def _stats(agent):
    return agent._obs_rms[agent._rms_cur].clone(), agent._obs_rms[agent._rms_cur ^ 1].clone()


def _run(agent, env_id, n, test_episode, tape_steps=640):
    """test() with the action tape on: (scores, tape of the steps that ran, statistics before)."""
    agent._eval_tape_steps = tape_steps
    before = _stats(agent)
    scores = agent.test(_env_fn(env_id, n), test_episode)
    torch.cuda.synchronize()
    ev = agent._evaluator
    steps = int(ev.step.item())
    assert steps < tape_steps
    return scores, ev.tape[:steps].cpu().numpy(), before


def _oracle(agent, env_id, n, test_episode, tape, state0):
    """The reference's test loop over the C oracle, actions from the tape: (scores, RunningMeanStd, steps, finishers per step)."""
    from oracle import c_oracle, ref_port
    od, D = agent._obs_dim, agent.memory.obs_row
    ref = c_oracle.VecEnvC(env_id, n, seed=EVAL_SEED, flavour="cr")      # two resets: the env's construction and envs.reset()
    rms = ref_port.RunningMeanStdPort((od,))
    st = state0.cpu().numpy()
    rms.mean, rms.var, rms.count = st[:od].astype(np.float32), st[D:D + od].astype(np.float32), float(st[2 * D])
    obs, scores, finishers, t = ref.obs[:, :od].copy(), [], [], 0
    while len(scores) < test_episode:
        if agent.use_obsnorm:
            rms.update(obs)
        o = ref.step(tape[t])
        done = o["term"] | o["trunc"]
        idx = np.nonzero(done)[0]
        scores += [float(s) for s in o["ep_score"][idx]]
        finishers.append(idx)
        obs = o["obs"][:, :od].copy()
        obs[done] = o["reset_obs"][done][:, :od]
        t += 1
    return scores, rms, t, finishers


def _check_against_oracle(agent, env_id, n, test_episode):
    scores, tape, (cur0, other0) = _run(agent, env_id, n, test_episode)
    want, rms, steps, finishers = _oracle(agent, env_id, n, test_episode, tape, cur0)
    assert tape.shape[0] == steps
    assert scores == want
    assert all(isinstance(s, float) for s in scores)
    cur, other = _stats(agent)
    assert torch.equal(other, other0)
    od, D = agent._obs_dim, agent.memory.obs_row
    st = cur.cpu().numpy()
    if agent.use_obsnorm:
        assert np.allclose(st[:od], rms.mean, rtol=1e-5, atol=1e-6), (st[:od], rms.mean)
        assert np.allclose(st[D:D + od], rms.var, rtol=1e-5, atol=1e-7), (st[D:D + od], rms.var)
        assert np.isclose(st[2 * D], rms.count, rtol=1e-12)
    else:
        assert torch.equal(cur, cur0)
    return scores, finishers


@pytest.mark.parametrize("n", [16, 4096])
@pytest.mark.parametrize("use_obsnorm", [False, True])
@pytest.mark.parametrize("env_id", ENVS)
def test_ppo_scores_and_statistics_equal_the_oracle_replay(env_id, use_obsnorm, n):
    """N = 16 runs the torch forward, N = 4096 the tcgen05 forward (normalising in-kernel for 4-float rows)."""
    agent = build_ppo(env_id, parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=use_obsnorm, seed=3)
    if n >= 2048:
        assert agent.learner._fused is not None
    _check_against_oracle(agent, env_id, n, n)


@pytest.mark.parametrize("build,env_id", [(lambda e, **k: build_ppo(e, agent_class=A2C_Agent, use_obsnorm=True, **k), "Acrobot-v1"),
                                          (build_pg, "CartPole-v1"), (build_pg, "Pendulum-v1"), (build_ppg, "CartPole-v1")])
def test_other_agents_equal_the_oracle_replay(build, env_id):
    """A2C; the actor-only PG policy (two outputs); PPG's four-output policy — their host test() raised before."""
    agent = build(env_id, parallels=16, n_steps=8, seed=4)
    _check_against_oracle(agent, env_id, 64, 40)


def test_first_finishers_over_many_ctas_are_all_kept_in_env_order():
    """CartPole at N = 65 536 with test_episode = 10: the step at which the first episodes end has far more than 10 finishers,
    spread over many CTAs.  All of them are returned, in env order.  (Without observation normalisation: at 65 536 rows the
    float32 column means of the reference's RunningMeanStd drift past the normaliser bars on their own.)"""
    agent = build_ppo("CartPole-v1", parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=False, seed=5)
    scores, finishers = _check_against_oracle(agent, "CartPole-v1", 65536, 10)
    first = next(f for f in finishers if len(f))
    assert len(first) > 10 and len(np.unique(first // 128)) > 8
    assert len(scores) == len(first) and finishers[-1] is first


def _eval_state(agent):
    ev = agent._evaluator
    torch.cuda.synchronize()
    return [t.clone() for t in (ev.state, ev.rng, ev.elapsed, ev.ep_score, ev.x, ev.step, ev.count, ev.stats,
                                ev.scores[:int(ev.count.item())], agent._obs_rms[0], agent._obs_rms[1])]


@pytest.mark.parametrize("env_id", ["CartPole-v1", "Pendulum-v1"])
def test_chunk_size_and_stop_rule(env_id):
    """K = 1, 5 and 32 steps per chunk give the same scores, env state and statistics; launches after the stop change nothing."""
    runs = []
    for k in (1, 5, 32):
        agent = build_ppo(env_id, parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=True, seed=6)
        agent._eval_chunk = k
        scores = agent.test(_env_fn(env_id, 300), 100)
        runs.append((scores, _eval_state(agent)))
        before = runs[-1][1]
        with torch.no_grad():
            agent._evaluator.graph.replay()                 # a whole chunk after the stop
        for x, y in zip(before, _eval_state(agent)):
            assert torch.equal(x, y)
    for scores, st in runs[1:]:
        assert scores == runs[0][0]
        for x, y in zip(st, runs[0][1]):
            assert torch.equal(x, y)


def _train_state(agent):
    torch.cuda.synchronize()
    return {k: v.detach().clone() for k, v in agent._state_tensors().items()}


def test_reproducible_and_training_untouched():
    """Two agents of one config return the same scores.  Without observation normalisation, train -> test -> train equals
    the same training without the test, bit for bit (episode totals are atomics-summed: fp64 tolerance)."""
    kw = dict(parallels=64, n_steps=16, n_epoch=2, n_minibatch=2, shuffle="device", seed=7)
    a, b = build_ppo("CartPole-v1", **kw), build_ppo("CartPole-v1", **kw)
    a.train(32)
    b.train(32)
    ctr0 = a._ctr.clone()
    assert a.test(_env_fn("CartPole-v1", 4096), 500) == b.test(_env_fn("CartPole-v1", 4096), 500)
    assert torch.equal(a._ctr, ctr0)
    c = build_ppo("CartPole-v1", **kw)
    c.train(32)
    info_a, info_c = a.train(32), c.train(32)
    sa, sc = _train_state(a), _train_state(c)
    assert sorted(sa) == sorted(sc)
    for k in sa:
        if k == "env.ep_stats":
            assert torch.equal(sa[k][0], sc[k][0]) and torch.allclose(sa[k][1:], sc[k][1:], rtol=1e-12, atol=0)
        else:
            assert torch.equal(sa[k], sc[k]), k
    for k in info_a:
        if k.startswith("mean_episode"):
            assert np.isclose(info_a[k], info_c[k], rtol=1e-12, atol=0, equal_nan=True), k
        elif torch.is_tensor(info_a[k]):
            assert torch.equal(info_a[k], info_c[k]), k
        else:
            assert info_a[k] == info_c[k], k


def test_resume_gives_the_same_scores_and_old_checkpoints_load(tmp_path):
    kw = dict(parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=True, seed=8)
    a = build_ppo("Pendulum-v1", **kw)
    a.train(8)
    a.test(_env_fn("Pendulum-v1", 32), 8)
    a.save_checkpoint(str(tmp_path / "ck"))
    first = a.test(_env_fn("Pendulum-v1", 32), 40)
    assert a.test(_env_fn("Pendulum-v1", 32), 40) != first         # the next evaluation draws other actions
    b = build_ppo("Pendulum-v1", policy_seed=99, **kw)
    b.load_checkpoint(str(tmp_path / "ck"))
    assert b._eval_index == 1 and b.test(_env_fn("Pendulum-v1", 32), 40) == first
    # a checkpoint written before device evaluation existed: no evaluation index in its host state
    f = checkpoint.rank_file(str(tmp_path / "ck"), 0, 1)
    payload = torch.load(f, weights_only=False)
    del payload["host"]["eval_index"]
    os.makedirs(str(tmp_path / "old"))
    torch.save(payload, checkpoint.rank_file(str(tmp_path / "old"), 0, 1))
    c = build_ppo("Pendulum-v1", policy_seed=98, **kw)
    c.load_checkpoint(str(tmp_path / "old"))
    assert c._eval_index == 0


@pytest.mark.parametrize("build", [build_ppo, build_pg, build_ppg])
def test_compat_envs_take_the_host_loop(build):
    """PG_Agent.test and PPG_Agent.test on compat envs raised at their first step (the policy has two / four outputs)."""
    agent = build("CartPole-v1", parallels=16, n_steps=8, seed=9)
    scores = agent.test(_env_fn("CartPole-v1", 8, native=False), 5)
    assert len(scores) >= 5 and all(8 <= s <= 500 for s in scores)
    assert agent._evaluator is None


def test_no_episodes_requested():
    agent = build_ppo("CartPole-v1", parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=True, seed=10)
    before = _stats(agent)
    made = []

    def env_fn():
        made.append(_env_fn("CartPole-v1", 8)())
        return made[-1]
    assert agent.test(env_fn, 0) == [] and made[0].closed
    for x, y in zip(before, _stats(agent)):
        assert torch.equal(x, y)
