"""GPU, 2 ranks: env-sharded PPG (learner and agent) and env-sharded running statistics of the 6- and 8-float observation rows
(Acrobot-v1, the 4-frame MountainCar-v0).  Skipped with fewer than 2 GPUs."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import copy, os, sys, torch
sys.path.insert(0, %r)
import torch.distributed as dist
from torch import nn
from xuanpolicy_b200 import dist as xd
from xuanpolicy_b200.configs import build_ppg, build_ppo
from xuanpolicy_b200.learner import PPG_Learner
from xuanpolicy_b200.policies import CategoricalPPGActorCritic, GaussianPPGActorCritic, MLPRepresentation, OldDistBatch
from xuanpolicy_b200.vec_env import make_spaces
rank, local, world = xd.init_from_env("nccl")
peer_on = os.environ.get("XB_PEER_COMM", "1") != "0"


def gather_equal(t):
    t = t.detach().reshape(-1).double().contiguous()
    all_ = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(all_, t)
    return all(torch.equal(all_[0], x) for x in all_)


def flat(policy):
    return torch.cat([p.detach().reshape(-1) for p in policy.parameters()])


# (1) learner equivalence: each rank updates on its half of a seeded global minibatch; the single-process update of the same
#     policy copy on the whole minibatch is the reference
def learner_check(env_id):
    obs_space, act_space = make_spaces(env_id)
    torch.manual_seed(11 + rank)                    # different initialisations: the sharded learner broadcasts rank 0's
    rep = MLPRepresentation(obs_space.shape, [64], activation=nn.ReLU, device="cuda")
    cls = CategoricalPPGActorCritic if env_id == "CartPole-v1" else GaussianPPGActorCritic
    pol = cls(act_space, rep, [64], [64], activation=nn.ReLU, device="cuda")
    opt = torch.optim.Adam(pol.parameters(), 4e-4, eps=1e-5)
    kw = dict(ent_coef=0.01, clip_range=0.2, kl_beta=1.0)
    L = PPG_Learner(pol, opt, None, "cuda", process_group=dist.group.WORLD, **kw)
    ref = copy.deepcopy(pol)
    R = PPG_Learner(ref, torch.optim.Adam(ref.parameters(), 4e-4, eps=1e-5), None, "cuda", **kw)
    B, od = 2048, obs_space.shape[0]
    g = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.randn(B, od, device="cuda", generator=g)
    ret, adv = torch.randn(B, device="cuda", generator=g) * 3, torch.randn(B, device="cuda", generator=g)
    with torch.no_grad():
        _, d0, _, _ = ref(obs)
    if env_id == "CartPole-v1":
        act = torch.randint(0, 2, (B,), device="cuda", generator=g).float()
        logits = d0.get_param() + 0.1 * torch.randn(B, 2, device="cuda", generator=g)
        old = lambda s: OldDistBatch("categorical", logits[s].contiguous())
    else:
        act = torch.randn(B, 1, device="cuda", generator=g)
        mu, std = d0.get_param()
        mu = mu + 0.1 * torch.randn(B, 1, device="cuda", generator=g)
        std = std.reshape(-1, 1).expand(B, 1).contiguous()
        old = lambda s: OldDistBatch("gaussian", mu[s].contiguous(), std[s].contiguous())
    h = slice(rank * B // world, (rank + 1) * B // world)
    full = slice(0, B)
    bad = []
    for phase in ("update_policy", "update_critic", "update_auxiliary"):
        before = {id(p): {k: v.clone() if torch.is_tensor(v) else v for k, v in opt.state[p].items()} for p in pol.parameters()}
        getattr(L, phase)(obs[h], act[h], ret[h], adv[h], old(h))
        getattr(R, phase)(obs, act, ret, adv, old(full))
        torch.cuda.synchronize()
        if not gather_equal(flat(pol)):
            bad.append(phase + ":ranks")
        p, r = flat(pol), flat(ref)
        rel = float((p - r).abs().max() / r.abs().max())
        if rel > 1e-5:
            bad.append("%%s:rel=%%.2e" %% (phase, rel))
        for a, b in zip(pol.parameters(), ref.parameters()):
            if (a.grad is None) != (b.grad is None):
                bad.append(phase + ":reach")
            if a.grad is None:
                st, st0 = opt.state[a], before[id(a)]
                same = st.keys() == st0.keys() and all(torch.equal(st[k], st0[k]) if torch.is_tensor(st[k]) else st[k] == st0[k]
                                                       for k in st)
                if not same:
                    bad.append(phase + ":state")
        if phase != "update_auxiliary" and all(q.grad is not None for q in pol.parameters()):
            bad.append(phase + ":all-reached")       # the policy and critic phases each leave sub-networks untouched
    return "ok" if not bad else "BAD(%%s)" %% ",".join(bad)


# (2) the agent: params + obs_rms bit-identical, env states differ, every env of every rank merged at every step
def agent_check(build, env_id, norm, **kw):
    a = build(env_id, device="cuda", parallels=64, n_steps=16, seed=3 + 10 * rank, use_obsnorm=norm, use_rewnorm=norm, **kw)
    a.train(2 * 16)
    torch.cuda.synchronize()
    D = a.memory.obs_row
    st = a._obs_rms[a._rms_cur]
    norm_state = torch.cat([st, a._ret_rms, a._rew_std.double()])
    params = flat(a.policy)
    checks = dict(params=gather_equal(params), envs_differ=not gather_equal(a.envs._state),
                  finite=bool(torch.isfinite(params).all() and torch.isfinite(norm_state).all()))
    if norm:
        merged_steps = 2 * 16 + (1 if a._fused_norm else 0)
        checks.update(stats=gather_equal(norm_state), fused=a._fused_norm,
                      count=abs(float(st[2 * D]) - (1e-4 + merged_steps * 64 * world)) < 1e-6)
    bad = [k for k, v in checks.items() if not v]
    return "ok" if not bad else "BAD(%%s)" %% ",".join(bad)


res = {}
for env_id in ("CartPole-v1", "Pendulum-v1"):
    res["LEARNER " + env_id] = learner_check(env_id)
for env_id in ("CartPole-v1", "Pendulum-v1", "Acrobot-v1", "MountainCar-v0"):
    if peer_on:
        res["PPG " + env_id] = agent_check(build_ppg, env_id, True, n_epoch=2, policy_nepoch=1, value_nepoch=1, aux_nepoch=1)
    else:    # the NCCL fallback of the gradient / advantage-statistics exchanges (the normalisers need peer memory)
        res["PPG " + env_id] = agent_check(build_ppg, env_id, False, n_epoch=2, policy_nepoch=1, value_nepoch=1, aux_nepoch=1)
if peer_on:
    for env_id in ("Acrobot-v1", "MountainCar-v0"):
        res["PPO " + env_id] = agent_check(build_ppo, env_id, True, n_epoch=1, n_minibatch=2, shuffle="device")
if rank == 0:
    for k, v in res.items():
        print("RESULT %%s %%s" %% (k.replace(" ", "/"), v))
dist.destroy_process_group()
''' % REPO


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_rank_ppg_and_wide_rows(tmp_path, peer):
    """peer=1: gradients, advantage statistics and running statistics exchanged over NVLink peer memory; peer=0: PPG's NCCL
    fallback.  Either way every replica stays bit-identical and matches the single-process update."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, XB_PEER_COMM=peer)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29543" if peer == "1" else "29544", str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    lines = [l.split() for l in out.stdout.splitlines() if l.startswith("RESULT")]
    want = ["LEARNER/CartPole-v1", "LEARNER/Pendulum-v1", "PPG/CartPole-v1", "PPG/Pendulum-v1", "PPG/Acrobot-v1", "PPG/MountainCar-v0"]
    if peer == "1":
        want += ["PPO/Acrobot-v1", "PPO/MountainCar-v0"]
    assert sorted(l[1] for l in lines) == sorted(want), out.stdout[-3000:]
    assert all(l[2] == "ok" for l in lines), "\n".join(" ".join(l) for l in lines)
