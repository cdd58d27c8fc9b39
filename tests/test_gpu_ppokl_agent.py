"""GPU: the device-loop PPOKL_Agent.

- against the restated loop (tests/ppokl_port.PPOKLAgentPort) on its recorded action and permutation tapes: actions and flags
  exact, buffers 1e-5, returns / advantages 2e-5, parameters after every update phase 1e-4 relative, the adaptive coefficient
  after every update phase equal;
- the fused rollout step's old-distribution rows, the one-launch packed loss against an fp64 restatement of `ppokl_update`,
  captured epochs against eager ones, the general path (Discrete(3) heads), checkpoints and `test()`;
- 2 ranks (skipped with fewer GPUs): replicas bit-identical with peer memory and with the NCCL fallback."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.ppokl_port import PPOKLAgentPort
from tests.test_gpu_agent_f3 import _compare, _hook_update_snapshots, _record_rollouts
from tests.test_gpu_agent_golden import _TapedAgentMixin

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _port_for(agent, env_id, h, seed, norm, record=True):
    from oracle import ref_port
    from xuanpolicy_b200 import policies
    cfg = agent.config
    envs = ref_port.VecEnvPort(env_id, agent.n_envs, seed=seed, trig="cr")
    envs.reset()
    pol = policies.make_policy(envs.observation_space, envs.action_space, hidden=(h,), device="cpu")
    pol.load_state_dict({k: v.detach().cpu() for k, v in agent.policy.state_dict().items()}, strict=True)
    opt = torch.optim.Adam(pol.parameters(), cfg.learning_rate, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=int(cfg.running_steps))
    return PPOKLAgentPort(envs, pol, opt, sched, cfg.n_steps, cfg.n_epoch, cfg.n_minibatch, cfg.gamma, cfg.gae_lambda,
                          vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef, target_kl=cfg.target_kl, use_gae=cfg.use_gae,
                          use_advnorm=cfg.use_advnorm, use_obsnorm=norm, use_rewnorm=norm, record=record)


@pytest.mark.parametrize("env_id,use_gae,norm", [("CartPole-v1", True, False), ("CartPole-v1", False, True),
                                                 ("Pendulum-v1", True, True), ("Pendulum-v1", False, False)])
def test_native_ppokl_agent_reproduces_the_restated_loop(env_id, use_gae, norm, monkeypatch):
    import xuanpolicy_b200 as xb
    from xuanpolicy_b200.configs import build_ppokl
    monkeypatch.setenv("XB_FUSED_STEP", "0")
    n, T, h, seed, target = 6, 16, 32, 4, 1e-4

    class Taped(_TapedAgentMixin, xb.PPOKL_Agent):
        pass
    agent = build_ppokl(env_id, agent_class=Taped, parallels=n, n_steps=T, n_epoch=2, n_minibatch=2, seed=seed, use_gae=use_gae,
                        representation_hidden_size=[h], actor_hidden_size=[h], critic_hidden_size=[h], use_obsnorm=norm,
                        use_rewnorm=norm, shuffle="host", use_cuda_graphs=False, running_steps=1000, target_kl=target)
    torch.manual_seed(9)
    np.random.seed(9)
    port = _port_for(agent, env_id, h, seed, norm)
    steps = 3 * T + 5
    ported = _record_rollouts(port, steps)
    assert len(ported) == 3
    # the adaptation decisions of the port must not hinge on the last bit of a KL
    for kl, _, _ in port.kl_trace:
        for edge in (1.5 * target, 0.5 * target):
            assert abs(kl - edge) > 1e-3 * edge, (kl, edge)
    agent.set_tapes(np.stack(port.recorded_actions), port.recorded_perms)
    native = _hook_update_snapshots(agent)
    coefs = []
    orig = agent._update_phase

    def update_phase():
        orig()
        coefs.append(float(agent.learner._kl_coef_dev.item()))
    agent._update_phase = update_phase
    info = agent.train(steps)
    assert set(info) >= {"actor-loss", "critic-loss", "entropy", "learning_rate", "kl", "predict_value"}
    assert "clip_ratio" not in info
    _compare(native, ported, "ppokl")
    per_phase = 2 * 2
    want = [port.kl_trace[(k + 1) * per_phase - 1][2] for k in range(3)]
    assert coefs == [float(np.float32(w)) for w in want], (coefs, want)      # (the device coefficient is float32)
    last = port.last_info
    for k in ("actor-loss", "critic-loss", "entropy", "kl", "predict_value"):
        assert np.isclose(float(info[k]), float(last[k]), rtol=2e-3, atol=2e-6), (k, info[k], last[k])
    assert agent.memory.ptr == port.memory.ptr == 5


@pytest.mark.parametrize("env_id", ["CartPole-v1", "Pendulum-v1"])
def test_fused_step_writes_the_old_distribution(env_id):
    from xuanpolicy_b200.configs import build_ppokl
    N, T = 4096, 4
    agent = build_ppokl(env_id, parallels=N, n_steps=T, n_minibatch=2, n_epoch=1, seed=2, use_cuda_graphs=False)
    assert agent._fused_step and agent.learner._fused is not None
    seen = []
    orig = agent._policy_forward

    def forward(x, norm=None, xn=None):
        dist, v = orig(x, norm, xn)
        prm = dist.get_param()
        seen.append((prm if agent.discrete else prm[0])[:N].clone())
        return dist, v
    agent._policy_forward = forward
    agent.train(T - 1)                                   # a partial rollout: the buffer rows stay in place
    rows = agent.memory._dist
    assert len(seen) == T - 1
    for t in range(T - 1):
        if agent.discrete:
            assert torch.equal(rows[t], seen[t])
        else:
            assert torch.equal(rows[t][:, 0], seen[t][:, 0])
            std = agent.policy.actor.logstd.detach().exp()
            assert torch.equal(rows[t][:, 1], std.expand(N))


def _ref_kl_loss(P, obs, buf, scal, old, gauss, kl_coef, hp):
    """fp64 restatement of `ppokl_update`'s loss (oracle/ref_port.py) on the reference module graph, with the kernel's activation
    pattern, and its log scalars."""
    from tests.test_gpu_mlp_h256 import _ref_forward
    act_out, v = _ref_forward(P, obs, buf, "actor.mu" if gauss else "actor.model")
    a, _, adv, ret = scal.double().unbind(1)
    adv = (adv - adv.mean()) / (adv.std(unbiased=False) + 1e-8)          # DummyOnPolicyBuffer.sample's normalisation
    if gauss:
        ls, mu = P["actor.logstd"][0], act_out[:, 0]
        omu, ostd = old[:, 0].double(), old[:, 1].double()
        logp = -(a - mu) ** 2 / (2 * torch.exp(2 * ls)) - ls - 0.5 * math.log(2 * math.pi)
        old_logp = -(a - omu) ** 2 / (2 * ostd ** 2) - ostd.log() - 0.5 * math.log(2 * math.pi)
        vr = (torch.exp(ls) / ostd) ** 2
        kl = 0.5 * (vr + ((mu - omu) / ostd) ** 2 - 1 - vr.log())
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + ls).expand_as(logp)
    else:
        lp, lq = torch.log_softmax(act_out, 1), torch.log_softmax(old.double(), 1)
        logp, old_logp = lp.gather(1, a.long()[:, None])[:, 0], lq.gather(1, a.long()[:, None])[:, 0]
        kl = (lp.exp() * (lp - lq)).sum(1)
        ent = -(lp.exp() * lp).sum(1)
    a_loss = -(torch.exp(logp - old_logp) * adv).mean() + kl_coef * kl.mean()
    c_loss = ((v - ret) ** 2).mean()
    info = {"actor-loss": a_loss, "critic-loss": c_loss, "entropy": ent.mean(), "kl": kl.mean(), "predict_value": v.mean()}
    return a_loss - hp["ent_coef"] * ent.mean() + hp["vf_coef"] * c_loss, {k: float(x) for k, x in info.items()}


def _adapt32(coef, kl, target):
    """ppokl_learner.py:39-43 in the device's float32."""
    c, k, t = np.float32(coef), np.float32(kl), np.float32(target)
    c = c * np.float32(2.0) if k > t * np.float32(1.5) else (c / np.float32(2.0) if k < t * np.float32(0.5) else c)
    return float(np.clip(c, np.float32(0.1), np.float32(20.0)))


@pytest.mark.parametrize("env_id,h", [("CartPole-v1", 128), ("Pendulum-v1", 128), ("CartPole-v1", 256), ("Pendulum-v1", 256)])
def test_packed_minibatch_update_against_fp64(env_id, h):
    """Two native minibatch updates of 4096 rows (the one-launch packed loss between the tensor-core forward and backward, Adam
    without clipping) against `ppokl_update` restated in fp64 on the same inputs, with the bars of tests/test_gpu_mlp_h256.py:
    every param.grad (the log-std's from the kernel's fp64 sum included) and the log scalars within 1e-4, the parameters after
    each step within 1e-5, the coefficient after each step exact.  The policy is perturbed after the rollout, so KL(new || old)
    and its gradient are far from zero; the reference uses the kernel's LeakyReLU pattern (sign words) and, like that test,
    starts each step from the parameters the native step before produced, with its own Adam moments."""
    from tests.helpers import rel_err
    from tests.test_gpu_mlp_h256 import _ref_adam_step, _sign_bits
    from xuanpolicy_b200.configs import build_ppokl
    N, T = 2048, 2
    agent = build_ppokl(env_id, parallels=N, n_steps=T, n_minibatch=1, n_epoch=1, seed=6, use_cuda_graphs=False,
                        representation_hidden_size=[h], actor_hidden_size=[h], critic_hidden_size=[h])
    L, mem, cfg = agent.learner, agent.memory, agent.config
    gauss = not agent.discrete
    with torch.no_grad():
        agent._rollout()
        g = torch.Generator(device="cuda").manual_seed(3)
        for p in agent.policy.parameters():
            p.add_(0.05 * torch.randn(p.shape, device="cuda", generator=g))
    B = N * T
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(1)).cuda()
    assert L._packed_loss_ok(mem, B)
    rows = (idx % T) * N + idx // T
    old = mem._dist.reshape(T * N, 2)[rows]
    hp = dict(vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef)
    mine = dict(agent.policy.named_parameters())
    names = list(mine)
    m = {n: torch.zeros_like(q, dtype=torch.float64) for n, q in mine.items()}
    v = {n: torch.zeros_like(q, dtype=torch.float64) for n, q in mine.items()}
    with torch.no_grad():                                      # KL ~ 3 target: the coefficient doubles at step 1
        mem.ptr, mem.size = 0, T
        prm = agent.policy(mem.sample(idx)[0])[1].get_param()
        if gauss:
            mu, std = prm[0][:, 0].double(), prm[1].double().reshape(-1)
            vr = (std / old[:, 1].double()) ** 2
            probe = (0.5 * (vr + ((mu - old[:, 0].double()) / old[:, 1].double()) ** 2 - 1 - vr.log())).mean()
        else:
            lp, lq = torch.log_softmax(prm.double(), 1), torch.log_softmax(old.double(), 1)
            probe = (lp.exp() * (lp - lq)).sum(1).mean()
    coef, target = 0.7, float(probe) / 3.0
    L.kl_coef, L.target_kl = coef, target
    L._fused.splits_fresh = False
    for t in (1, 2):
        P = {n: q.detach().double() for n, q in mine.items()}
        L.update_from_buffer(mem, idx)
        torch.cuda.synchronize()
        mb, b = L._mb[(B, mem.obs_dim)], L._fused._last[1]
        if b.get("signs") is not None:
            bits = _sign_bits(b["signs"], h).double()
            buf = dict(h1=b["h1"], ya=bits[:, :h], yc=bits[:, h:])
        else:
            buf = b
        Pg = {n: x.clone().requires_grad_(True) for n, x in P.items()}
        loss, ref_info = _ref_kl_loss(Pg, mb["obs"], buf, mb["scal"], old, gauss, float(np.float32(coef)), hp)
        ref_grads = dict(zip(names, torch.autograd.grad(loss, [Pg[n] for n in names])))
        for edge in (1.5 * target, 0.5 * target):           # no decision hinges on the last bit of the KL
            assert abs(ref_info["kl"] - edge) > 1e-3 * edge
        gerr = {n: rel_err(mine[n].grad, ref_grads[n]) for n in names}
        info = L.info(B)
        ierr = {k: abs(float(info[k]) - r) / max(1.0, abs(r)) for k, r in ref_info.items()}
        lr = cfg.learning_rate * (1.0 - (t - 1) / cfg.running_steps)
        P = _ref_adam_step(P, ref_grads, m, v, t, lr, 0.0)
        perr = {n: rel_err(mine[n].detach(), P[n]) for n in names}
        print("%s H=%d step %d: grad %.2e (%s)  info %.2e (%s)  param %.2e (%s)  kl %.3e"
              % (env_id, h, t, max(gerr.values()), max(gerr, key=gerr.get), max(ierr.values()), max(ierr, key=ierr.get),
                 max(perr.values()), max(perr, key=perr.get), ref_info["kl"]))
        for n, e in gerr.items():
            assert e < 1e-4, (t, n, e)
        for k, e in ierr.items():
            assert e < 1e-4, (t, k, e)
        for n, e in perr.items():
            assert e < 1e-5, (t, n, e)
        assert float(L._kl_used.item()) == float(np.float32(coef))
        coef = _adapt32(coef, ref_info["kl"], target)
        assert float(L._kl_coef_dev.item()) == coef, (t, float(L._kl_coef_dev.item()), coef)
        if t == 1:
            assert coef == float(np.float32(0.7) * np.float32(2.0))


@pytest.mark.parametrize("env_id", ["CartPole-v1", "Pendulum-v1"])
def test_captured_epochs_equal_eager(env_id):
    from xuanpolicy_b200.configs import build_ppokl
    out = []
    for graphs in (True, False):
        agent = build_ppokl(env_id, parallels=1024, n_steps=8, n_minibatch=2, n_epoch=2, seed=3, use_cuda_graphs=graphs,
                            shuffle="device", target_kl=0.01)
        assert agent.learner._packed_loss_ok(agent.memory, agent.batch_size) or not agent.memory.packed
        coefs = []
        for _ in range(3):
            info = agent.train(8)
            coefs.append((float(agent.learner._kl_coef_dev.item()), info["kl"]))
        out.append(([p.detach().clone() for p in agent.policy.parameters()], coefs))
    (pa, ca), (pb, cb) = out
    assert ca == cb
    for x, y in zip(pa, pb):
        assert torch.equal(x, y)
    assert len({c for c, _ in ca}) > 1 or ca[0][0] != 1.0          # the coefficient moved


@pytest.mark.parametrize("env_id", ["Acrobot-v1", "MountainCar-v0"])
def test_general_path_trains(env_id):
    from xuanpolicy_b200.configs import build_ppokl
    agent = build_ppokl(env_id, parallels=1024, n_steps=8, n_minibatch=2, n_epoch=2, seed=3, shuffle="device", target_kl=0.01)
    assert not agent.learner._packed_loss_ok(agent.memory, agent.batch_size)
    before = [p.detach().clone() for p in agent.policy.parameters()]
    for _ in range(2):
        info = agent.train(8)
    assert all(np.isfinite(info[k]) for k in ("actor-loss", "critic-loss", "entropy", "kl", "predict_value"))
    assert info["kl"] > 0.0 and float(agent.learner._kl_coef_dev.item()) != 1.0
    assert any(not torch.equal(a, b) for a, b in zip(before, agent.policy.parameters()))


@pytest.mark.parametrize("parallels", [64, 1024])
def test_checkpoint_resume_and_test(tmp_path, parallels):
    from xuanpolicy_b200.configs import build_ppokl
    from xuanpolicy_b200.vec_env import DummyVecEnv_Gym, make_env_fns
    kw = dict(parallels=parallels, n_steps=8, n_minibatch=2, n_epoch=2, seed=5, shuffle="device", target_kl=0.01,
              use_obsnorm=True, use_rewnorm=True)
    a = build_ppokl("Pendulum-v1", **kw)
    a.train(8 + 3)                                       # mid-rollout: old-distribution rows of steps 0..2 are pending
    a.save_checkpoint(str(tmp_path / "ck"))
    a.train(2 * 8)
    b = build_ppokl("Pendulum-v1", **kw)
    b.load_checkpoint(str(tmp_path / "ck"))
    b.train(2 * 8)
    for x, y in zip(a.policy.parameters(), b.policy.parameters()):
        assert torch.equal(x, y)
    assert torch.equal(a.learner._kl_coef_dev, b.learner._kl_coef_dev)
    assert torch.equal(a.learner._kl_used, b.learner._kl_used)
    assert torch.equal(a.memory._dist, b.memory._dist)
    # test() on device envs: scores back, training state untouched (apart from the observation statistics it merges)
    snap = {k: v.clone() for k, v in a._state_tensors().items() if not k.startswith("obs_rms")}
    scores = a.test(lambda: DummyVecEnv_Gym(make_env_fns("Pendulum-v1", 11, 16), device="cuda", native=True), 4)
    assert len(scores) >= 4 and all(np.isfinite(scores))
    for k, v in a._state_tensors().items():
        if k in snap:
            assert torch.equal(v, snap[k]), k


WORKER = r'''
import os, sys, torch
sys.path.insert(0, %r)
import torch.distributed as dist
from xuanpolicy_b200 import dist as xd
from xuanpolicy_b200.configs import build_ppokl
rank, local, world = xd.init_from_env("nccl")
peer_on = os.environ.get("XB_PEER_COMM", "1") != "0"


def gather_equal(t):
    t = t.detach().reshape(-1).double().contiguous()
    all_ = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(all_, t)
    return all(torch.equal(all_[0], x) for x in all_)


def agent_check(env_id, parallels, norm):
    a = build_ppokl(env_id, device="cuda", parallels=parallels, n_steps=8, n_epoch=2, n_minibatch=2, seed=3 + 10 * rank,
                    shuffle="device", target_kl=0.01, use_obsnorm=norm, use_rewnorm=norm)
    coefs = []
    for _ in range(3):
        a.train(8)
        coefs.append(a.learner._kl_coef_dev.clone())
    torch.cuda.synchronize()
    params = torch.cat([p.detach().reshape(-1) for p in a.policy.parameters()])
    checks = dict(params=gather_equal(params), kl_coef=gather_equal(torch.cat(coefs)), envs_differ=not gather_equal(a.envs._state),
                  moved=len(set(float(c) for c in coefs)) > 1 or float(coefs[0]) != 1.0)
    if norm:
        checks["stats"] = gather_equal(torch.cat([a._obs_rms[a._rms_cur], a._ret_rms, a._rew_std.double()]))
    bad = [k for k, v in checks.items() if not v]
    return "ok" if not bad else "BAD(%%s)" %% ",".join(bad)


# each rank's update on its half of a seeded rollout against the single-process update on the whole (a one-rank group); the
# target is the global KL, so a KL count or normalisation off by the world size would flip the decision (x2 or /2)
singles = [dist.new_group([r]) for r in range(world)]


def learner_check(env_id, T):
    from xuanpolicy_b200.buffer import DummyOnPolicyBuffer
    from xuanpolicy_b200.learner import PPOKL_Learner
    from xuanpolicy_b200.policies import make_policy
    from xuanpolicy_b200.vec_env import make_spaces
    obs_space, act_space = make_spaces(env_id)
    od, N, gauss = obs_space.shape[0], 64, env_id == "Pendulum-v1"
    g = torch.Generator(device="cuda").manual_seed(7)
    f = lambda *s: torch.randn(*s, device="cuda", generator=g)
    obs, rew, val = f(T, N, 4), f(T, N), f(T, N)
    obs[..., od:] = 0.0

    def policy():
        torch.manual_seed(21)
        return make_policy(obs_space, act_space, hidden=(128,), device="cuda")
    with torch.no_grad():
        _, d0, _ = policy()(obs.reshape(-1, 4)[:, :od])
        if gauss:
            mu, std = d0.get_param()
            act = (mu + std * f(T * N, 1)).reshape(T, N, 1)
            old = torch.cat([mu + 0.2 * f(T * N, 1), std.reshape(-1, 1).expand(T * N, 1) * 1.3], 1)
            vr = (std.reshape(-1, 1) / old[:, 1:]) ** 2
            kl = (0.5 * (vr + ((mu - old[:, :1]) / old[:, 1:]) ** 2 - 1 - vr.log())).mean()
        else:
            z = d0.get_param()
            act = torch.randint(0, 2, (T, N, 1), device="cuda", generator=g).float()
            old = z + 0.5 * f(T * N, 2)
            lp, lq = torch.log_softmax(z, 1), torch.log_softmax(old, 1)
            kl = (lp.exp() * (lp - lq)).sum(1).mean()
        old = old.reshape(T, N, 2)

    def make(lo, hi, group):
        pol = policy()
        L = PPOKL_Learner(pol, torch.optim.Adam(pol.parameters(), 4e-4, eps=1e-5), None, "cuda", vf_coef=0.25, ent_coef=0.01,
                          target_kl=float(kl))
        L.enable_fused_optimizer(group)
        mem = DummyOnPolicyBuffer(obs_space, act_space, {"old_dist": None}, hi - lo, T, True, True, 0.99, 0.95, device="cuda",
                                  native=True)
        for dst, src in ((mem._obs, obs), (mem._act, act), (mem._rew, rew), (mem._val, val)):
            dst.copy_(src[:, lo:hi])
        mem._term.zero_()
        mem._trunc.zero_()
        mem._dist, mem._dist_kind = old[:, lo:hi].contiguous(), "gaussian" if gauss else "categorical"
        mem.finish_rollout(val[T - 1, lo:hi].contiguous())
        return pol, L, mem
    n = N // world
    pol, L, mem = make(rank * n, (rank + 1) * n, dist.group.WORLD)
    ref, R, rmem = make(0, N, singles[rank])
    assert L.world_size == world and R.world_size == 1 and R._peer is None
    bad = []
    for step in range(2):
        L.update_from_buffer(mem, torch.randperm(n * T, generator=torch.Generator().manual_seed(step)).cuda())
        R.update_from_buffer(rmem, torch.randperm(N * T, generator=torch.Generator().manual_seed(step)).cuda())
        torch.cuda.synchronize()
        p = torch.cat([q.detach().reshape(-1) for q in pol.parameters()])
        r = torch.cat([q.detach().reshape(-1) for q in ref.parameters()])
        rel = float((p - r).abs().max() / r.abs().max())
        if rel > 1e-5:
            bad.append("step%%d:rel=%%.2e" %% (step, rel))
        if not torch.equal(L._kl_coef_dev, R._kl_coef_dev):
            bad.append("step%%d:kl_coef %%g vs %%g" %% (step, float(L._kl_coef_dev), float(R._kl_coef_dev)))
        if not gather_equal(p):
            bad.append("step%%d:ranks" %% step)
    return "ok" if not bad else "BAD(%%s)" %% ",".join(bad)


res = {}
for env_id in ("CartPole-v1", "Pendulum-v1"):
    for T in (64, 16):                      # 2048 local rows: the packed one-launch loss; 512: the general path
        res["LEARNER/%%s/%%d" %% (env_id, T)] = learner_check(env_id, T)
for env_id in ("CartPole-v1", "Pendulum-v1", "Acrobot-v1"):
    for parallels in (64, 2048):
        res["%%s/%%d" %% (env_id, parallels)] = agent_check(env_id, parallels, peer_on)
if rank == 0:
    for k, v in res.items():
        print("RESULT %%s %%s" %% (k, v))
dist.destroy_process_group()
''' % REPO


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_rank_ppokl_agent(tmp_path, peer):
    """Two ranks, each on its own envs: each rank's update on its half equals the single-process update on the whole minibatch
    (coefficient included), and over a few agent iterations parameters and the coefficient stay bit-identical across the
    ranks, over peer memory (normalisers on) and over the NCCL fallback."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, XB_PEER_COMM=peer)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29563" if peer == "1" else "29564", str(script)],
                         capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    lines = [l.split() for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert len(lines) == 10, out.stdout[-3000:]
    assert all(l[2] == "ok" for l in lines), "\n".join(" ".join(l) for l in lines)
