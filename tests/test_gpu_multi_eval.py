"""GPU, 2 ranks: env-sharded `test()`.  The two ranks' test envs form one vector env; the scores both ranks return must equal the
C oracle's replay of the reference's test loop over the concatenated envs, driven by the ranks' action tapes, in (step, rank,
env) order.  Skipped with fewer than 2 GPUs."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
import numpy as np
import torch
sys.path.insert(0, %r)
import torch.distributed as dist
import xuanpolicy_b200 as xb
from xuanpolicy_b200 import dist as xd
from xuanpolicy_b200.configs import build_ppg, build_ppo
rank, local, world = xd.init_from_env("nccl")
peer_on = os.environ.get("XB_PEER_COMM", "1") != "0"
EVAL_SEED = 11


def gather(t):
    t = t.contiguous()
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return out


def same(t):
    return all(torch.equal(x, gather(t)[0]) for x in gather(t))


def env_fn(env_id, n):
    return lambda: xb.DummyVecEnv_Gym(xb.make_env_fns(env_id, EVAL_SEED, n), device="cuda", native=True)


def flat(a):
    return torch.cat([p.detach().reshape(-1) for p in a.policy.parameters()])


def oracle(a, env_id, n, test_episode, tape, state0):
    from oracle import c_oracle, ref_port
    od, D = a._obs_dim, a.memory.obs_row
    ref = c_oracle.VecEnvC(env_id, n, seed=EVAL_SEED, flavour="cr")
    rms = ref_port.RunningMeanStdPort((od,))
    st = state0.cpu().numpy()
    rms.mean, rms.var, rms.count = st[:od].astype(np.float32), st[D:D + od].astype(np.float32), float(st[2 * D])
    obs, scores, t = ref.obs[:, :od].copy(), [], 0
    while len(scores) < test_episode:
        if a.use_obsnorm:
            rms.update(obs)
        o = ref.step(tape[t])
        done = o["term"] | o["trunc"]
        scores += [float(s) for s in o["ep_score"][np.nonzero(done)[0]]]
        obs = o["obs"][:, :od].copy()
        obs[done] = o["reset_obs"][done][:, :od]
        t += 1
    return scores, rms, t


def eval_check(build, env_id, n, norm, test_episode, **kw):
    a = build(env_id, device="cuda", parallels=64, n_steps=16, seed=3, use_obsnorm=norm, **kw)
    a.train(16)
    a._eval_tape_steps = 640
    st0 = a._obs_rms[a._rms_cur].clone()
    scores = a.test(env_fn(env_id, n), test_episode)
    ev = a._evaluator
    bad = []
    if ev is None or ev.peer is None:
        return "BAD(host-loop)"
    steps = int(ev.step.item())
    tape = torch.cat(gather(ev.tape[:steps]), dim=1).cpu().numpy()        # global env r * n + e = env e of rank r
    if not same(torch.tensor([len(scores)], device="cuda")) or not same(torch.tensor(scores, dtype=torch.float64, device="cuda")):
        bad.append("ranks-scores")
    want, rms, t = oracle(a, env_id, world * n, test_episode, tape, st0)
    if scores != want or t != steps:
        bad.append("oracle")
    st = a._obs_rms[a._rms_cur]
    if not same(st):
        bad.append("ranks-stats")
    od, D = a._obs_dim, a.memory.obs_row
    h = st.cpu().numpy()
    if norm and not (np.allclose(h[:od], rms.mean, rtol=1e-5, atol=1e-6) and np.allclose(h[D:D + od], rms.var, rtol=1e-5, atol=1e-7)
                     and np.isclose(h[2 * D], rms.count, rtol=1e-12)):
        bad.append("oracle-stats")
    a.train(16)                                        # train -> test -> train: replicas stay bit-identical
    torch.cuda.synchronize()
    if not same(flat(a)) or not same(a._obs_rms[a._rms_cur]):
        bad.append("ranks-after-train")
    try:
        a.learner._peer.check()
    except RuntimeError:
        bad.append("timeout")
    return "ok" if not bad else "BAD(%%s)" %% ",".join(bad)


def mismatch_check():
    a = build_ppo("CartPole-v1", device="cuda", parallels=64, n_steps=16, seed=3, use_obsnorm=True)
    raised = []
    for n, te in ((64 if rank == 0 else 32, 50), (64, 50 if rank == 0 else 49)):
        try:
            a.test(env_fn("CartPole-v1", n), te)
            raised.append(False)
        except ValueError:
            raised.append(True)
    ok = all(raised) and a._evaluator is None and a._eval_index == 0
    ok = ok and len(a.test(env_fn("CartPole-v1", 64), 50)) >= 50         # the ranks are still in step
    return "ok" if ok else "BAD(%%s)" %% raised


def host_check():
    a = build_ppo("CartPole-v1", device="cuda", parallels=64, n_steps=16, seed=3)
    scores = a.test(env_fn("CartPole-v1", 64), 50)
    return "ok" if a._evaluator is None and len(scores) >= 50 else "BAD"


res = {}
if peer_on:
    for n in (64, 4096):
        res["PPO/CartPole-v1/%%d" %% n] = eval_check(build_ppo, "CartPole-v1", n, True, n, n_epoch=1, n_minibatch=2)
    res["PPO/Acrobot-v1"] = eval_check(build_ppo, "Acrobot-v1", 64, True, 64, n_epoch=1, n_minibatch=2)
    res["PPG/Pendulum-v1"] = eval_check(build_ppg, "Pendulum-v1", 64, True, 64, n_epoch=2, policy_nepoch=1, value_nepoch=1,
                                        aux_nepoch=1)
    res["MISMATCH"] = mismatch_check()
else:
    res["HOST"] = host_check()
if rank == 0:
    for k, v in res.items():
        print("RESULT %%s %%s" %% (k, v))
dist.destroy_process_group()
''' % REPO


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_rank_evaluation(tmp_path, peer):
    """peer=1: the device loop over both ranks' envs, exchanged over peer memory; peer=0: every rank on the host loop."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, XB_PEER_COMM=peer)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29553" if peer == "1" else "29554", str(script)],
                         capture_output=True, text=True, timeout=900, env=env, cwd=REPO)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    lines = [l.split() for l in out.stdout.splitlines() if l.startswith("RESULT")]
    want = (["PPO/CartPole-v1/64", "PPO/CartPole-v1/4096", "PPO/Acrobot-v1", "PPG/Pendulum-v1", "MISMATCH"] if peer == "1"
            else ["HOST"])
    assert sorted(l[1] for l in lines) == sorted(want), out.stdout[-3000:]
    assert all(l[2] == "ok" for l in lines), "\n".join(" ".join(l) for l in lines)
