"""CPU, wherever the reference is importable (installed into oracle/_ref by `python -m oracle.build_ref`, or a source tree
named by XB200_REFERENCE_ROOT; skipped elsewhere): the oracle's restatements run side by side with the LIVE reference
objects on fresh seeded inputs — not via stored goldens.

    RunningMeanStdPort   vs  xuance.common.RunningMeanStd                     statistic_tools.py:35-112
    PPOAgentPort.train   vs  PPOCLIP_Agent.train (built by xuance.get_runner)  ppoclip_agent.py:59-111
    vec_env._describe    on the reference's own `_thunk` closure               environment/__init__.py:36-90
"""
import numpy as np
import pytest
import torch

from oracle import ref_loader, ref_port

pytestmark = [pytest.mark.reference,
              pytest.mark.skipif(not ref_loader.available(), reason="the reference is not importable (python -m oracle.build_ref)")]


def test_running_mean_std_port_equals_live_reference_bit_for_bit():
    ref_loader.load()
    from xuance.common import RunningMeanStd
    rng = np.random.default_rng(5)
    for shape, dtype in (((3,), np.float32), ((4,), np.float32), ((), np.float64)):
        live, port = RunningMeanStd(shape=shape, comm=None, use_mpi=False), ref_port.RunningMeanStdPort(shape)
        for n in (8, 1, 33, 2, 1, 1, 100):
            x = (rng.standard_normal((n,) + shape) * 7 + 3).astype(dtype)
            live.update(x)
            port.update(x)
            assert np.array_equal(np.asarray(live.mean), np.asarray(port.mean))
            assert np.array_equal(np.asarray(live.var), np.asarray(port.var))
            assert live.count == port.count and np.asarray(live.mean).dtype == np.asarray(port.mean).dtype
            assert np.array_equal(np.asarray(live.std), np.asarray(port.std))


@pytest.mark.parametrize("env_id,n,T,steps", [("CartPole-v1", 6, 24, 24 * 2 + 7), ("Pendulum-v1", 3, 110, 110 * 2 + 3)])
def test_port_agent_equals_live_reference_agent(env_id, n, T, steps):
    """Same seeds, same torch / numpy RNG streams, same machine: the restated loop must take the same actions and end with
    the same buffers, statistics and parameters as the unmodified PPOCLIP_Agent."""
    from oracle import ref_agent
    from xuanpolicy_b200 import policies
    torch.set_num_threads(1)
    runner = ref_agent.build_runner(env_id, trig="libm", parallels=n, n_steps=T, seed=7, n_epoch=2, n_minibatch=3,
                                    representation_hidden_size=[16], actor_hidden_size=[16], critic_hidden_size=[16])
    live = runner.agent
    import xuance.torch.agents.policy_gradient.ppoclip_agent as mod
    mod.tqdm = lambda x: x
    envs = ref_port.VecEnvPort(env_id, n, seed=7, trig="libm")
    envs.reset()
    pol = policies.make_policy(envs.observation_space, envs.action_space, hidden=(16,), device="cpu")
    pol.load_state_dict(live.policy.state_dict(), strict=True)          # same parameter names as the reference's modules
    cfg = live.config
    opt = torch.optim.Adam(pol.parameters(), cfg.learning_rate, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=live.learner.scheduler.total_iters)
    port = ref_port.PPOAgentPort(envs, pol, opt, sched, T, 2, 3, cfg.gamma, cfg.gae_lambda, vf_coef=cfg.vf_coef,
                                 ent_coef=cfg.ent_coef, clip_range=cfg.clip_range, clip_grad_norm=cfg.clip_grad_norm,
                                 use_obsnorm=cfg.use_obsnorm, use_rewnorm=cfg.use_rewnorm, obsnorm_range=cfg.obsnorm_range,
                                 rewnorm_range=cfg.rewnorm_range)
    assert cfg.use_obsnorm and cfg.use_rewnorm                         # the yaml default
    torch.manual_seed(11); np.random.seed(11)
    live.train(steps)
    torch.manual_seed(11); np.random.seed(11)
    port.train(steps)
    lm, pm = live.memory, port.memory
    assert lm.ptr == pm.ptr and live.current_step == port.current_step
    # Discrete actions: the trajectory is reproduced exactly.  Box actions are mu + std * eps: after the first update the
    # restated learner's parameters differ from the reference's in the last bits (expression order), so does mu, and the
    # continuous trajectory follows at the 1e-7 level — compared with a tolerance.
    same = np.array_equal if env_id == "CartPole-v1" else (lambda x, y: np.allclose(x, y, rtol=1e-5, atol=1e-6))
    for name, a, b in (("obs", lm.observations, pm.observations), ("act", lm.actions, pm.actions), ("rew", lm.rewards, pm.rewards),
                       ("term", lm.terminals, pm.terminals)):
        assert same(a[:, :lm.ptr], b[:, :pm.ptr]), name
    # network outputs: the mirror modules evaluate log-softmax / the Gaussian log-density with their own expression order
    for name, a, b in (("val", lm.values, pm.values), ("logp", lm.auxiliary_infos["old_logp"], pm.auxiliary_infos["old_logp"])):
        assert np.allclose(a[:, :lm.ptr], b[:, :pm.ptr], rtol=1e-5, atol=1e-6), name
    assert same(np.asarray(live.obs_rms.mean), np.asarray(port.obs_rms.mean))
    tight = 1e-12 if env_id == "CartPole-v1" else 1e-6
    assert np.allclose(np.asarray(live.ret_rms.var), np.asarray(port.ret_rms.var), rtol=tight)
    assert np.allclose(live.returns, port.returns, rtol=tight, atol=0)
    for (k, v), (k2, v2) in zip(live.policy.state_dict().items(), pol.state_dict().items()):
        assert k == k2 and torch.allclose(v, v2, rtol=1e-5, atol=1e-6), (k, (v - v2).abs().max())


def test_describe_reads_env_id_and_seed_from_the_reference_thunk():
    """INTEGRATION.md §1b: `make_envs` hands the registered class a list of `_thunk` closures over `config`
    (environment/__init__.py:36-90); the drop-in learns env_id / seed / N from them without instantiating N envs."""
    ref_loader.load()
    from argparse import Namespace
    import xuance.environment as E
    from xuanpolicy_b200 import vec_env
    seen = {}

    class Probe:
        def __init__(self, env_fns):
            seen["fns"] = env_fns
    E.REGISTRY_VEC_ENV["XB200_Probe"] = Probe
    try:
        cfg = Namespace(env_name="Classic Control", env_id="Pendulum-v1", seed=42, parallels=5, vectorize="XB200_Probe",
                        render_mode="rgb_array")
        E.make_envs(cfg)
    finally:
        del E.REGISTRY_VEC_ENV["XB200_Probe"]
    fns = seen["fns"]
    assert len(fns) == 5 and all(vec_env._describe(fn) == ("Pendulum-v1", 42) for fn in fns)
    assert not hasattr(fns[0], "env_id") and fns[0].__closure__ is not None      # the real closure, not our EnvFn


def test_pg_port_agent_equals_live_reference_pg_agent():
    """PG_Agent.train (pg_agent.py:49-96) + PG_Learner.update (pg_learner.py:17-45), yaml defaults (ReLU, use_gae False, obs /
    reward normalisation on): same seeds -> same actions, buffers (incl. the no-GAE returns with the reward-bootstrap at a full
    buffer, :60-62), statistics and parameters."""
    from oracle import ref_agent
    from xuanpolicy_b200 import policies
    torch.set_num_threads(1)
    n, T, steps = 5, 20, 20 * 3 + 4
    runner = ref_agent.build_runner("CartPole-v1", trig="libm", method="pg", parallels=n, n_steps=T, seed=3, n_epoch=2,
                                    representation_hidden_size=[16], actor_hidden_size=[16])
    live = runner.agent
    import xuance.torch.agents.policy_gradient.pg_agent as mod
    mod.tqdm = lambda x: x
    cfg = live.config
    assert type(live).__name__ == "PG_Agent" and cfg.use_gae is False and cfg.activation == "ReLU"
    envs = ref_port.VecEnvPort("CartPole-v1", n, seed=3, trig="libm")
    envs.reset()
    rep = policies.MLPRepresentation(envs.observation_space.shape, [16], activation=torch.nn.ReLU, device="cpu")
    pol = policies.CategoricalActor(envs.action_space, rep, [16], activation=torch.nn.ReLU, device="cpu")
    pol.load_state_dict(live.policy.state_dict(), strict=True)
    opt = torch.optim.Adam(pol.parameters(), cfg.learning_rate, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=live.learner.scheduler.total_iters)
    port = ref_port.PGAgentPort(envs, pol, opt, sched, T, 2, cfg.gamma, cfg.gae_lambda, ent_coef=cfg.ent_coef, clip_grad=cfg.clip_grad,
                                use_gae=cfg.use_gae, use_advnorm=cfg.use_advnorm, use_obsnorm=cfg.use_obsnorm,
                                use_rewnorm=cfg.use_rewnorm)
    torch.manual_seed(21); np.random.seed(21)
    live.train(steps)
    torch.manual_seed(21); np.random.seed(21)
    port.train(steps)
    lm, pm = live.memory, port.memory
    assert lm.ptr == pm.ptr == 4 and live.current_step == port.current_step
    for name, a, b in (("obs", lm.observations, pm.observations), ("act", lm.actions, pm.actions), ("rew", lm.rewards, pm.rewards),
                       ("term", lm.terminals, pm.terminals), ("ret", lm.returns, pm.returns)):
        assert np.array_equal(a[:, :4], b[:, :4]) or np.allclose(a[:, :4], b[:, :4], rtol=1e-6, atol=1e-7), name
    assert np.array_equal(np.asarray(live.obs_rms.mean), np.asarray(port.obs_rms.mean))
    assert np.allclose(np.asarray(live.ret_rms.var), np.asarray(port.ret_rms.var), rtol=1e-12)
    for (k, v), (k2, v2) in zip(live.policy.state_dict().items(), pol.state_dict().items()):
        assert k == k2 and torch.allclose(v, v2, rtol=1e-5, atol=1e-6), (k, (v - v2).abs().max())


@pytest.mark.parametrize("env_id", ["CartPole-v1", "Pendulum-v1"])
def test_ppg_port_agent_equals_live_reference_ppg_agent(env_id):
    """PPG_Agent.train (ppg_agent.py:55-109) + PPG_Learner's three phase updates (ppg_learner.py:23-88), yaml defaults (obs /
    reward normalisation on, ret_rms never updated): same seeds -> same buffers, statistics and parameters after two
    rollouts of policy / critic / old-distribution refresh / auxiliary phases."""
    from oracle import ref_agent
    from xuanpolicy_b200 import policies
    torch.set_num_threads(1)
    n, T, steps = 4, 12, 12 * 2 + 3
    runner = ref_agent.build_runner(env_id, trig="libm", method="ppg", parallels=n, n_steps=T, seed=5, n_epoch=2,
                                    policy_nepoch=2, value_nepoch=2, aux_nepoch=2, representation_hidden_size=[16],
                                    actor_hidden_size=[16], critic_hidden_size=[16])
    live = runner.agent
    import xuance.torch.agents.policy_gradient.ppg_agent as mod
    mod.tqdm = lambda x: x
    cfg = live.config
    assert type(live).__name__ == "PPG_Agent" and live.batch_size == n * T // 2
    act = {"ReLU": torch.nn.ReLU, "LeakyReLU": torch.nn.LeakyReLU}[cfg.activation]
    envs = ref_port.VecEnvPort(env_id, n, seed=5, trig="libm")
    envs.reset()
    rep = policies.MLPRepresentation(envs.observation_space.shape, [16], activation=act, device="cpu")
    cls = policies.CategoricalPPGActorCritic if env_id == "CartPole-v1" else policies.GaussianPPGActorCritic
    pol = cls(envs.action_space, rep, [16], [16], activation=act, device="cpu")
    pol.load_state_dict(live.policy.state_dict(), strict=True)
    opt = torch.optim.Adam(pol.parameters(), cfg.learning_rate, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=live.learner.scheduler.total_iters)
    act_shape = () if env_id == "CartPole-v1" else envs.action_space.shape
    mem = ref_port.OldDistBufferPort(envs.observation_space.shape, act_shape, n, T, cfg.use_gae, cfg.use_advnorm, cfg.gamma,
                                     cfg.gae_lambda)
    hp = dict(ent_coef=cfg.ent_coef, clip_range=cfg.clip_range, kl_beta=cfg.kl_beta)
    upd = {ph: (lambda o, a, r, ad, old, ph=ph: ref_port.ppg_update(ph, pol, opt, sched, (o, a, r, ad), old, **hp))
           for ph in ("policy", "critic", "aux")}
    port = ref_port.PPGAgentPort(envs, pol, mem, upd["policy"], upd["critic"], upd["aux"], n_steps=T, n_minibatch=2,
                                 policy_nepoch=2, value_nepoch=2, aux_nepoch=2, use_obsnorm=cfg.use_obsnorm,
                                 use_rewnorm=cfg.use_rewnorm)
    torch.manual_seed(21); np.random.seed(21)
    live.train(steps)
    torch.manual_seed(21); np.random.seed(21)
    port.train(steps)
    lm = live.memory
    assert lm.ptr == mem.ptr == 3 and live.current_step == port.current_step
    for name, a, b in (("obs", lm.observations, mem.observations), ("act", lm.actions, mem.actions), ("rew", lm.rewards, mem.rewards),
                       ("val", lm.values, mem.values), ("term", lm.terminals, mem.terminals)):
        assert np.allclose(a[:, :3], b[:, :3], rtol=1e-4, atol=1e-5), name
    assert np.allclose(np.asarray(live.obs_rms.mean), np.asarray(port.obs_rms.mean), rtol=1e-6, atol=1e-7)
    assert float(np.asarray(live.ret_rms.count)) == float(np.asarray(port.ret_rms.count))       # never updated by PPG_Agent
    for (k, v), (k2, v2) in zip(live.policy.state_dict().items(), pol.state_dict().items()):
        assert k == k2 and torch.allclose(v, v2, rtol=1e-4, atol=2e-6), (k, (v - v2).abs().max())
