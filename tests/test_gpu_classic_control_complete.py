"""GPU: MountainCarContinuous-v0 (gym's bare env and the reference's 4-frame stack) and CartPole-v0 on the device.

- physics against the C oracle ("cr"), bit for bit, at ragged N, through episodes that terminate at the goal and truncate at
  999 (200 for CartPole-v0): fp64 states, observations, rewards, flags, reset observations, episode counters and ep_stats;
- the device rollout (fused sample + step + store) replayed through the C oracle;
- PPO on the stacked env at 2048 envs (tcgen05 MLP, observation and reward normalisers on) against the restated reference loop
  (oracle/ref_port.PPOAgentPort) replaying the device's actions and the same minibatch permutations;
- A2C, PG, PPG and PPO-KL: one rollout and update on the stacked env; captured graphs against eager launches;
- `test()` on the device against the reference's test loop over the C oracle; checkpoint resume; two ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import classic_control_ext as ext
from tests.helpers import gae_close

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONT = ["gym:MountainCarContinuous-v0", "MountainCarContinuous-v0"]


def _envs(env_id, n, seed=1, **kw):
    import xuanpolicy_b200 as xb
    return xb.DummyVecEnv_Gym(xb.make_env_fns(env_id, seed, n), **kw)


def _actions(env_id, obs, rng, n):
    if env_id == "CartPole-v0":
        heur = (obs[:, 2] + 0.5 * obs[:, 3] > 0).astype(np.int64)
        return np.where(rng.random(n) < 0.9, heur, rng.integers(0, 2, n))
    # energy pumping along the newest frame's velocity plus Gaussian noise (actions outside [-1, 1] too); every fourth car
    # drives without a plan and truncates at 999
    a = np.where(obs[:, -1] > 0, 1.3, -1.3) + 0.4 * rng.standard_normal(n)
    a[::4] = 0.3 * rng.standard_normal(len(a[::4]))
    return a.astype(np.float32).reshape(n, 1)


@pytest.mark.parametrize("env_id,n,steps", [("gym:MountainCarContinuous-v0", 2051, 1100), ("MountainCarContinuous-v0", 1033, 1100),
                                            ("CartPole-v0", 2051, 450)])
def test_physics_bit_exact_vs_c_oracle(env_id, n, steps):
    envs = _envs(env_id, n, 3)
    ref = ext.vec_env_c(env_id, n, seed=3, flavour="cr")
    obs, _ = envs.reset()
    assert np.array_equal(obs, ref.obs) and np.array_equal(envs.get_state(), ref.state)
    rng = np.random.default_rng(9)
    n_term = n_trunc = 0
    score_sum = len_sum = 0.0
    for t in range(steps):
        a = _actions(env_id, obs, rng, n)
        obs, rew, term, trunc, infos = envs.step(a)
        o = ref.step(a)
        assert np.array_equal(obs, o["obs"]) and np.array_equal(rew, o["rew"]) and rew.dtype == np.float32, t
        assert np.array_equal(term, o["term"]) and np.array_equal(trunc, o["trunc"]), t
        assert np.array_equal(envs.get_state(), o["state"]), t
        assert [i["episode_step"] for i in infos] == o["ep_step"].tolist(), t
        assert [i["episode_score"] for i in infos] == o["ep_score"].tolist(), t
        done = term | trunc
        if done.any():
            ro = np.stack([infos[i]["reset_obs"] for i in np.nonzero(done)[0]])
            assert np.array_equal(ro, o["reset_obs"][done]), t
            obs = obs.copy()
            obs[done] = ro
        n_term, n_trunc = n_term + int(term.sum()), n_trunc + int(trunc.sum())
        score_sum += float(o["ep_score"][done].sum())
        len_sum += float(o["ep_step"][done].sum())
    assert n_term > 0 and n_trunc > 0, (n_term, n_trunc)
    st = envs.ep_stats.cpu().numpy()
    assert st[0] == n_term + n_trunc and st[2] == len_sum and np.isclose(st[1], score_sum, rtol=1e-12)


def test_native_mode_takes_float32_actions():
    for env_id in CONT:
        nat = _envs(env_id, 16, native=True)
        obs, _ = nat.reset()
        assert obs.is_cuda and obs.shape == (16, 8 if env_id == "MountainCarContinuous-v0" else 2)
        assert nat._act.dtype == torch.float32
        o, r, d, tr, infos = nat.step(torch.full((16, 1), 2.0, device="cuda"))
        assert torch.equal(r, torch.full_like(r, -0.4)) and infos[0]["episode_step"] == 1      # -(2.0 * 2.0) * 0.1, unclipped


@pytest.mark.parametrize("env_id", CONT)
@pytest.mark.parametrize("graphs", [True, False])
def test_device_rollout_replays_bit_exact_through_the_oracle(env_id, graphs):
    """The fused rollout step's actions replayed through the C oracle: observations, rewards and flags bit for bit; GAE equal
    to the fp64 oracle's with the stored values and bootstraps; stored log-probs those of the rollout policy."""
    from oracle import c_oracle
    from xuanpolicy_b200.configs import build_ppo
    n, T = 40, 520
    agent = build_ppo(env_id, parallels=n, n_steps=T, n_epoch=1, n_minibatch=2, use_cuda_graphs=graphs, shuffle="device", seed=5)
    assert agent._fused_step and not agent.discrete
    mem = agent.memory
    ref = ext.vec_env_c(env_id, n, seed=5, flavour="cr")
    trunc_seen = 0
    for rollout in range(2):                      # 1040 steps: every env crosses step 999
        with torch.cuda.device(agent.device):
            if graphs and agent._rollout_graph is None:
                agent._capture()
            agent._rollout_graph.replay() if graphs else agent._rollout()
        torch.cuda.synchronize()
        obs, act, od = mem._obs.cpu().numpy(), mem._act.cpu().numpy(), mem.obs_dim
        for t in range(T):
            assert np.array_equal(obs[t, :, :od], ref.obs), (rollout, t)
            o = ref.step(act[t, :, :1])
            assert np.array_equal(mem._rew[t].cpu().numpy(), o["rew"]), (rollout, t)
            assert np.array_equal(mem._term[t].cpu().numpy(), o["term"].astype(np.float32))
            assert np.array_equal(mem._trunc[t].cpu().numpy(), o["trunc"].astype(np.uint8))
            done = o["term"] | o["trunc"]
            trunc_seen += int(o["trunc"].sum())
            ref.obs[done] = o["reset_obs"][done]
        adv64, ret64 = c_oracle.gae(mem._rew.cpu().numpy(), mem._val.cpu().numpy(), mem._term.cpu().numpy(),
                                    agent._boot_last.cpu().numpy(), agent.gamma, agent.gae_lam,
                                    segend=mem._trunc.cpu().numpy(), boot=mem._boot.cpu().numpy())
        assert gae_close(mem._adv.cpu().numpy(), adv64)[0] and gae_close(mem._ret.cpu().numpy(), ret64)[0]
        with torch.no_grad():
            _, dist, v = agent.policy(mem._obs.reshape(T * n, mem.obs_row)[:, :od])
            lp = dist.log_prob(mem._act.reshape(T * n, -1))
        assert torch.allclose(v.reshape(T, n), mem._val, atol=1e-5, rtol=1e-5)
        assert torch.allclose(lp.reshape(T, n), mem._logp, atol=2e-5, rtol=1e-5)
    assert trunc_seen > 0


class _DeviceRms:
    """The port's observation RunningMeanStd with the device's arithmetic (tests/test_gpu_rollout_fp64.Normaliser: fp64 batch
    moments, float32 Chan merge).  Every env starts from the same seed, so on the first step all observations are equal, the
    variance is ~6e-8 and one float32 rounding of the mean moves a normalised input by ~0.02: the installed numpy's float32
    restatement of the reference's update lands 6e-6 away from the exact mean there, the device's arithmetic on it."""

    def __init__(self, od):
        from tests.test_gpu_rollout_fp64 import Normaliser
        self._n = Normaliser(od)

    mean = property(lambda self: self._n.mean)
    var = property(lambda self: self._n.var)
    count = property(lambda self: self._n.count)
    std = property(lambda self: np.sqrt(self._n.var))

    def update(self, x):
        self._n.merge(np.asarray(x, np.float32))


def test_ppo_on_the_stack_reproduces_the_restated_loop(monkeypatch):
    """2048 envs (the tensor-core MLP; the fused rollout step with the observation and reward normalisers): the device
    agent's actions and a fixed permutation tape replayed by oracle/ref_port.PPOAgentPort on the CPU.  Bars of
    test_gpu_agent_f3.py: actions and flags exact, buffers 1e-5, returns / advantages 2e-5, parameters after every update
    phase 1e-4 relative; normaliser states 1e-5.  The port's observation normaliser runs the device's arithmetic (_DeviceRms)."""
    from oracle import ref_port
    from tests.test_gpu_agent_f3 import _compare, _hook_update_snapshots, _snap_port
    from xuanpolicy_b200 import policies
    from xuanpolicy_b200.configs import build_ppo
    env_id, n, T, n_epoch, n_mb, h, seed = "MountainCarContinuous-v0", 2048, 8, 2, 2, 128, 4
    steps = 2 * T + 3
    agent = build_ppo(env_id, parallels=n, n_steps=T, n_epoch=n_epoch, n_minibatch=n_mb, seed=seed, use_obsnorm=True,
                      use_rewnorm=True, representation_hidden_size=[h], actor_hidden_size=[h], critic_hidden_size=[h],
                      shuffle="host", use_cuda_graphs=False, running_steps=1000)
    assert agent._fused_step and agent._fused_norm and agent.learner._fused is not None and agent.memory.obs_row == 8
    rng = np.random.default_rng(2)
    perms = [rng.permutation(n * T) for _ in range(2 * n_epoch)]
    agent._feeder.get = lambda it, ep: torch.as_tensor(perms[it * n_epoch + ep], dtype=torch.int64).pin_memory()
    agent._feeder.prefetch = lambda it: None
    agent._feeder.mark_consumed = lambda it: None
    p0 = {k: v.detach().cpu().clone() for k, v in agent.policy.state_dict().items()}
    acts = []
    orig_step = agent._rollout_step

    def step(t):
        orig_step(t)
        acts.append(agent._act.cpu().numpy().reshape(n, 1).copy())
    agent._rollout_step = step
    native = _hook_update_snapshots(agent)
    agent.train(steps)
    assert len(acts) == steps and len(native) == 2
    # ---- the restated reference loop on the same draws
    cfg = agent.config
    ext.register(monkeypatch)
    envs = ref_port.VecEnvPort(env_id, n, seed=seed, trig="cr")
    envs.reset()
    pol = policies.make_policy(envs.observation_space, envs.action_space, hidden=(h,), device="cpu")
    pol.load_state_dict(p0, strict=True)
    opt = torch.optim.Adam(pol.parameters(), cfg.learning_rate, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=1000)
    port = ref_port.PPOAgentPort(envs, pol, opt, sched, T, n_epoch, n_mb, cfg.gamma, cfg.gae_lambda, vf_coef=cfg.vf_coef,
                                 ent_coef=cfg.ent_coef, clip_range=cfg.clip_range, clip_grad_norm=cfg.clip_grad_norm,
                                 use_gae=True, use_advnorm=True, use_obsnorm=True, use_rewnorm=True,
                                 action_tape=np.stack(acts), perm_tape=perms)
    port.obs_rms = _DeviceRms(8)
    ported, mem = [], port.memory
    clear = mem.clear

    def clear_and_snapshot():                       # end of an update phase
        s = _snap_port(port)
        s["params"] = {k: v.detach().clone().numpy() for k, v in pol.state_dict().items()}
        ported.append(s)
        clear()
    mem.clear = clear_and_snapshot
    port.train(steps)
    # the port snapshots its buffer after the phase, the device before it: rows are the same, parameters after the phase
    _compare(native, ported, "ppo/MountainCarContinuous-v0")
    st = agent._obs_rms[agent._rms_cur].cpu().numpy()
    port.obs_rms.update(port.envs.buf_obs)           # the fused step already merged the observations the next step acts on
    assert np.allclose(st[:8], port.obs_rms.mean, rtol=1e-5, atol=1e-6) and np.allclose(st[8:16], port.obs_rms.var, rtol=1e-5, atol=1e-7)
    assert np.isclose(st[16], port.obs_rms.count, rtol=1e-12)
    ret = agent._ret_rms.cpu().numpy()
    assert np.isclose(ret[0], float(port.ret_rms.mean), rtol=1e-5, atol=1e-7) and np.isclose(ret[1], float(port.ret_rms.var), rtol=1e-5)
    assert np.isclose(ret[2], float(port.ret_rms.count), rtol=1e-9)
    assert np.allclose(agent._returns.cpu().numpy(), port.returns, rtol=1e-5, atol=1e-6)
    assert agent.memory.ptr == 3


def _builders():
    from xuanpolicy_b200.agent import A2C_Agent
    from xuanpolicy_b200.configs import build_pg, build_ppg, build_ppo, build_ppokl
    return {"a2c": lambda e, **k: build_ppo(e, agent_class=A2C_Agent, **k), "pg": build_pg,
            "ppg": lambda e, **k: build_ppg(e, policy_nepoch=1, value_nepoch=1, aux_nepoch=1, **k),
            "ppokl": lambda e, **k: build_ppokl(e, target_kl=0.01, **k), "ppo": build_ppo}


@pytest.mark.parametrize("kind", ["a2c", "pg", "ppg", "ppokl", "ppo"])
def test_every_agent_trains_on_the_stack(kind):
    agent = _builders()[kind]("MountainCarContinuous-v0", parallels=2048, n_steps=8, n_epoch=2, n_minibatch=2, seed=3,
                              use_obsnorm=True, use_rewnorm=True, shuffle="device")
    assert agent._fused_step and not agent.discrete and agent.memory.obs_row == 8
    before = [p.detach().clone() for p in agent.policy.parameters()]
    info = agent.train(8 + 1)
    assert all(np.isfinite(float(v)) for k, v in info.items()
               if not k.startswith("mean_episode") and (torch.is_tensor(v) or isinstance(v, (int, float)))), info
    assert any(not torch.equal(a, b) for a, b in zip(before, agent.policy.parameters()))
    assert all(torch.isfinite(p).all() for p in agent.policy.parameters())
    assert torch.isfinite(agent._obs_rms[agent._rms_cur]).all() and torch.isfinite(agent.memory._ret).all()


@pytest.mark.parametrize("kind", ["ppo", "ppg", "ppokl"])
def test_graphs_equal_eager(kind):
    """The captured rollout and epochs against the same launches issued eagerly: identical buffers, statistics, env state and
    parameters (PPO-Clip: one rollout, its Gaussian update within the bars of test_gpu_agent.py's graph test)."""
    rollouts = 1 if kind == "ppo" else 3
    out = []
    for graphs in (True, False):
        kw = dict(shuffle="device") if kind != "ppg" else {}
        agent = _builders()[kind]("MountainCarContinuous-v0", parallels=1024, n_steps=16, n_epoch=2, n_minibatch=2, seed=3,
                                  use_obsnorm=True, use_rewnorm=True, use_cuda_graphs=graphs, **kw)
        agent.train(rollouts * 16)
        torch.cuda.synchronize()
        assert (agent._rollout_graph is not None) == graphs
        out.append((agent.memory._ret.clone(), agent.memory._obs.clone(), agent._obs_rms[agent._rms_cur].clone(),
                    agent._ret_rms.clone(), agent.envs._state.clone(), [p.detach().clone() for p in agent.policy.parameters()]))
    a, b = out
    for x, y in zip(a[:5], b[:5]):
        assert torch.equal(x, y)
    for x, y in zip(a[5], b[5]):
        if kind == "ppo":
            assert torch.allclose(x, y, atol=2e-5, rtol=1e-4), (x - y).abs().max()
        else:
            assert torch.equal(x, y)


@pytest.mark.parametrize("n", [64, 2048])
@pytest.mark.parametrize("use_obsnorm", [False, True])
@pytest.mark.parametrize("env_id", CONT + ["CartPole-v0"])
def test_device_test_equals_the_oracle_replay(env_id, use_obsnorm, n):
    """The check of test_gpu_eval.py: the device's action tape through the C oracle with the reference's test loop
    (ppoclip_agent.py:113-165) gives the same scores, in order, and the same observation statistics.  Episodes of an untrained
    policy last up to 999 steps here, hence the longer tape."""
    from oracle import ref_port
    from tests.test_gpu_eval import EVAL_SEED, _run, _stats
    from xuanpolicy_b200.configs import build_ppo
    agent = build_ppo(env_id, parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=use_obsnorm, seed=3)
    if n >= 2048:
        assert agent.learner._fused is not None
    scores, tape, (cur0, other0) = _run(agent, env_id, n, n, tape_steps=1100)
    od, D = agent._obs_dim, agent.memory.obs_row
    ref = ext.vec_env_c(env_id, n, seed=EVAL_SEED, flavour="cr")        # two resets: the env's construction and envs.reset()
    rms = ref_port.RunningMeanStdPort((od,))
    st0 = cur0.cpu().numpy()
    rms.mean, rms.var, rms.count = st0[:od].astype(np.float32), st0[D:D + od].astype(np.float32), float(st0[2 * D])
    obs, want, t = ref.obs[:, :od].copy(), [], 0
    while len(want) < n:
        if use_obsnorm:
            rms.update(obs)
        o = ref.step(tape[t])
        done = o["term"] | o["trunc"]
        want += [float(x) for x in o["ep_score"][np.nonzero(done)[0]]]
        obs = o["obs"][:, :od].copy()
        obs[done] = o["reset_obs"][done][:, :od]
        t += 1
    assert tape.shape[0] == t and scores == want and len(scores) >= n
    cur, other = _stats(agent)
    assert torch.equal(other, other0)
    st = cur.cpu().numpy()
    if use_obsnorm:
        assert np.allclose(st[:od], rms.mean, rtol=1e-5, atol=1e-6), (st[:od], rms.mean)
        assert np.allclose(st[D:D + od], rms.var, rtol=1e-5, atol=1e-7), (st[D:D + od], rms.var)
        assert np.isclose(st[2 * D], rms.count, rtol=1e-12)
    else:
        assert torch.equal(cur, cur0)


def test_checkpoint_resume(tmp_path):
    from xuanpolicy_b200.configs import build_ppo
    kw = dict(parallels=1024, n_steps=8, n_epoch=2, n_minibatch=2, seed=5, shuffle="device", use_obsnorm=True, use_rewnorm=True)
    a = build_ppo("MountainCarContinuous-v0", **kw)
    a.train(8 + 3)                                   # mid-rollout
    a.save_checkpoint(str(tmp_path / "ck"))
    a.train(2 * 8)
    b = build_ppo("MountainCarContinuous-v0", policy_seed=77, **kw)
    b.load_checkpoint(str(tmp_path / "ck"))
    b.train(2 * 8)
    for x, y in zip(a.policy.parameters(), b.policy.parameters()):
        assert torch.equal(x, y)
    for x, y in ((a.envs._state, b.envs._state), (a._obs_rms[a._rms_cur], b._obs_rms[b._rms_cur]), (a._ret_rms, b._ret_rms),
                 (a.memory._obs, b.memory._obs)):
        assert torch.equal(x, y)


WORKER = r'''
import os, sys, torch
sys.path.insert(0, %r)
import torch.distributed as dist
from xuanpolicy_b200 import dist as xd
from xuanpolicy_b200.configs import build_pg, build_ppg, build_ppo, build_ppokl
rank, local, world = xd.init_from_env("nccl")


def gather_equal(t):
    t = t.detach().reshape(-1).double().contiguous()
    all_ = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(all_, t)
    return all(torch.equal(all_[0], x) for x in all_)


def agent_check(build, **kw):
    a = build("MountainCarContinuous-v0", device="cuda", parallels=2048, n_steps=8, seed=3 + 10 * rank, use_obsnorm=True,
              use_rewnorm=True, n_epoch=2, n_minibatch=2, **kw)
    a.train(2 * 8 + 1)
    torch.cuda.synchronize()
    params = torch.cat([p.detach().reshape(-1) for p in a.policy.parameters()])
    norm_state = torch.cat([a._obs_rms[a._rms_cur], a._ret_rms, a._rew_std.double()])
    checks = dict(params=gather_equal(params), stats=gather_equal(norm_state), envs_differ=not gather_equal(a.envs._state),
                  fused=a._fused_norm and a._shard_norm, finite=bool(torch.isfinite(params).all()))
    bad = [k for k, v in checks.items() if not v]
    return "ok" if not bad else "BAD(%%s)" %% ",".join(bad)


res = {"PPO": agent_check(build_ppo, shuffle="device"), "PG": agent_check(build_pg),
       "PPG": agent_check(build_ppg, policy_nepoch=1, value_nepoch=1, aux_nepoch=1),
       "PPOKL": agent_check(build_ppokl, shuffle="device", target_kl=0.01)}
if rank == 0:
    for k, v in res.items():
        print("RESULT %%s %%s" %% (k, v))
dist.destroy_process_group()
''' % REPO


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_on_the_stack(tmp_path):
    """Env-sharded over peer memory, normalisers on: replicas and normaliser states bit-identical across the ranks."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29573", str(script)],
                         capture_output=True, text=True, timeout=900, env=dict(os.environ, XB_PEER_COMM="1"))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    lines = [l.split() for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert sorted(l[1] for l in lines) == ["PG", "PPG", "PPO", "PPOKL"], out.stdout[-3000:]
    assert all(l[2] == "ok" for l in lines), "\n".join(" ".join(l) for l in lines)
