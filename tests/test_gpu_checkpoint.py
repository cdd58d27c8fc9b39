"""GPU: training checkpoints (agent.save_checkpoint / load_checkpoint) and the reference's weights-only save_model / load_model.

Every resume case compares three runs of one config: A trains k1 then k2 steps uninterrupted; B trains k1 and saves; C, built
with another policy seed (so its state visibly comes from the file), loads B's checkpoint and trains k2.  C must end bit for
bit where A ends.  Each case first checks that a second uninterrupted run A' equals A, so a failure points at the checkpoint
and not at run-to-run nondeterminism.  Two fp64 tolerances, for sums taken with atomics that may differ in the last bits from
run to run: `ep_stats[1:]` (episode score and length totals) and the loss scalars of PPG's update kernels, and the log values
derived from them."""
import glob
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from xuanpolicy_b200 import checkpoint
from xuanpolicy_b200.agent import A2C_Agent
from xuanpolicy_b200.configs import build_pg, build_ppg, build_ppo

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_BUFFER = ("_obs", "_act", "_rew", "_val", "_term", "_trunc", "_logp", "_boot", "_dist", "_adv", "_ret")


def _state(agent):
    """(device tensors, host values) of everything a resumed run must reproduce: the checkpoint's tensors, the whole buffer
    and the host counters, the torch optimiser / scheduler state and the last log."""
    torch.cuda.synchronize()
    dev = {k: v.detach().clone() for k, v in agent._checkpoint_tensors(0).items()}
    for n in _BUFFER:
        if getattr(agent.memory, n) is not None:
            dev["memory" + n] = getattr(agent.memory, n).clone()
    return dev, checkpoint.to_cpu(agent._host_state())


def _close(a, b):
    return a == b or (isinstance(a, float) and isinstance(b, float) and abs(a - b) <= 1e-9 * max(1.0, abs(a), abs(b)))


def _assert_same(x, y, what):
    (dx, hx), (dy, hy) = x, y
    hx, hy = dict(hx), dict(hy)          # (the last log is compared on its own below)
    assert sorted(dx) == sorted(dy), what
    for k in dx:
        a, b = dx[k], dy[k]
        if k == "env.ep_stats":
            assert torch.equal(a[0], b[0]), (what, k)
            assert torch.allclose(a[1:], b[1:], rtol=1e-12, atol=0), (what, k, a, b)
        elif k == "learner.scalars":
            assert torch.allclose(a, b, rtol=1e-9, atol=1e-9), (what, k, a, b)
        else:
            assert torch.equal(a, b), (what, k, (a.double() - b.double()).abs().max())
    info_x, info_y = hx.pop("last_info"), hy.pop("last_info")
    assert sorted(info_x) == sorted(info_y), what
    for k in info_x:
        a, b = info_x[k], info_y[k]
        if torch.is_tensor(a):
            assert torch.equal(a, b), (what, "last_info", k)
        elif k.startswith("mean_episode"):
            assert np.isclose(a, b, rtol=1e-12, atol=0, equal_nan=True), (what, "last_info", k)
        else:
            assert _close(a, b), (what, "last_info", k, a, b)
    _assert_nested_equal(hx, hy, what)


def _assert_nested_equal(a, b, what):
    if torch.is_tensor(a):
        assert torch.is_tensor(b) and torch.equal(a.cpu(), b.cpu()), what
    elif isinstance(a, dict):
        assert sorted(a, key=str) == sorted(b, key=str), what
        for k in a:
            _assert_nested_equal(a[k], b[k], "%s/%s" % (what, k))
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), what
        for u, v in zip(a, b):
            _assert_nested_equal(u, v, what)
    else:
        assert a == b, (what, a, b)


def _params(agent):
    return torch.cat([p.detach().reshape(-1) for p in agent.policy.parameters()])


def _resume(tmp_path, build, k1, k2, warm=0, **kw):
    """A: train(k1); train(k2).  B: train(k1); save.  C (another policy seed; `warm` steps of its own first, which captures
    its graphs): load; train(k2).  Returns C."""
    runs = []
    for _ in range(2):
        a = build(**kw)
        a.train(k1)
        a.train(k2)
        runs.append(_state(a))
        del a
    _assert_same(runs[0], runs[1], "two uninterrupted runs")
    b = build(**kw)
    b.train(k1)
    path = str(tmp_path / "ckpt")
    b.save_checkpoint(path)
    assert os.listdir(path) == ["rank0-of-1.pt"]
    c = build(policy_seed=1234, **kw)
    if warm:
        c.train(warm)
        assert c._rollout_graph is not None
    assert not torch.equal(_params(c), _params(b))
    graph = c._rollout_graph
    c.load_checkpoint(path)
    assert torch.equal(_params(c), _params(b))
    c.train(k2)
    if warm:
        assert c._rollout_graph is graph          # resumed on the graphs captured before the load
    _assert_same(runs[0], _state(c), "resumed run")
    return c


T = 16


def test_ppo_cartpole_host_shuffle_graphs_normalisers_at_a_boundary(tmp_path):
    c = _resume(tmp_path, build_ppo, 2 * T, 2 * T, env_id="CartPole-v1", parallels=1024, n_steps=T, n_epoch=2, n_minibatch=4,
                shuffle="host", use_obsnorm=True, use_rewnorm=True, seed=3)
    assert c.learner._fused is not None and c._epoch_graphs is not None and c.batch_size >= 2048


def test_ppo_pendulum_device_shuffle_mid_rollout(tmp_path):
    c = _resume(tmp_path, build_ppo, T + T // 2, 2 * T, env_id="Pendulum-v1", parallels=1024, n_steps=T, n_epoch=2,
                n_minibatch=4, shuffle="device", seed=4)
    assert c._t == T // 2 and c.learner._fused is not None


def test_ppo_acrobot_wide_rows_folded_head_with_normalisers(tmp_path):
    c = _resume(tmp_path, build_ppo, T + T // 2, T + T // 2, env_id="Acrobot-v1", parallels=1024, n_steps=T, n_epoch=2,
                n_minibatch=4, shuffle="device", use_obsnorm=True, use_rewnorm=True, seed=5)
    assert c.memory.obs_row == 8 and c.learner._fused is not None and c.learner._fused.fold3


def test_a2c_at_a_boundary(tmp_path):
    _resume(tmp_path, build_ppo, 2 * T, T, env_id="CartPole-v1", agent_class=A2C_Agent, parallels=512, n_steps=T,
            n_epoch=1, n_minibatch=2, shuffle="device", use_obsnorm=True, use_rewnorm=True, seed=6)


def test_pg_at_a_boundary(tmp_path):
    _resume(tmp_path, build_pg, 2 * T, T, env_id="CartPole-v1", parallels=512, n_steps=T, seed=7)


@pytest.mark.parametrize("k1", [2 * T, T + T // 2])
def test_ppg_cartpole(tmp_path, k1):
    """At a boundary, and mid-rollout (the stored old-distribution rows travel with the checkpoint)."""
    c = _resume(tmp_path, build_ppg, k1, 2 * T, env_id="CartPole-v1", parallels=256, n_steps=T, n_epoch=2, policy_nepoch=1,
                value_nepoch=1, aux_nepoch=1, seed=8)
    assert c.learner.policy_iterations > 0 and c.learner._flat is None


def test_loading_into_an_agent_that_has_captured_its_graphs(tmp_path):
    _resume(tmp_path, build_ppo, 2 * T, 2 * T, warm=T, env_id="CartPole-v1", parallels=1024, n_steps=T, n_epoch=2,
            n_minibatch=4, shuffle="host", use_obsnorm=True, use_rewnorm=True, seed=3)


@pytest.mark.parametrize("field,change", [("seed", dict(seed=10)), ("env_id", dict(env_id="Acrobot-v1")),
                                          ("n_envs", dict(parallels=128))])
def test_mismatched_checkpoints_are_refused_and_leave_the_agent_untouched(tmp_path, field, change):
    kw = dict(env_id="CartPole-v1", parallels=256, n_steps=T, n_epoch=1, n_minibatch=2, shuffle="device", seed=9)
    b = build_ppo(**kw)
    b.train(T + 3)
    path = str(tmp_path / "ckpt")
    b.save_checkpoint(path)
    c = build_ppo(**dict(kw, **change))
    c.train(T)
    before = _state(c)
    with pytest.raises(ValueError, match=field):
        c.load_checkpoint(path)
    _assert_same(before, _state(c), "refused load")


def test_save_model_and_load_model_round_trip(tmp_path):
    kw = dict(env_id="Pendulum-v1", parallels=64, n_steps=T, n_epoch=1, n_minibatch=2, shuffle="device", seed=2,
              use_obsnorm=True, model_dir=str(tmp_path / "models"))
    a = build_ppo(**kw)
    a.train(2 * T)
    a.save_model("final_model.pth")
    run_dirs = glob.glob(str(tmp_path / "models" / "seed_2_*"))
    assert len(run_dirs) == 1 and sorted(os.listdir(run_dirs[0])) == ["final_model.pth", "obs_rms.npy"]
    stat = np.load(os.path.join(run_dirs[0], "obs_rms.npy"), allow_pickle=True).item()
    st = a._obs_rms[a._rms_cur].cpu().numpy()
    assert sorted(stat) == ["count", "mean", "var"] and stat["mean"].shape == (3,) and stat["count"] == st[8]
    assert np.array_equal(stat["mean"], st[:3]) and np.array_equal(stat["var"], st[4:7])
    b = build_ppo(policy_seed=77, **kw)
    assert not torch.equal(_params(a), _params(b))
    assert b.load_model(str(tmp_path / "models"), seed=2) == run_dirs[0]
    assert torch.equal(_params(a), _params(b))
    for s in b._obs_rms:
        assert torch.equal(s[:3], torch.from_numpy(stat["mean"]).cuda()) and torch.equal(s[4:7], torch.from_numpy(stat["var"]).cuda())
        assert float(s[8]) == stat["count"]
    import xuanpolicy_b200 as xb
    scores = b.test(lambda: xb.DummyVecEnv_Gym(xb.make_env_fns("Pendulum-v1", 3, 4), device="cuda", native=True), 4)
    assert len(scores) >= 4 and all(np.isfinite(scores))


def test_obs_rms_file_matches_the_reference_agent(tmp_path):
    """Where the reference is importable: its Agent.save_model writes the same obs_rms.npy structure, and our load_model reads
    the file its agent wrote."""
    from oracle import ref_agent, ref_loader
    if not ref_loader.available():
        pytest.skip("the reference is not importable (python -m oracle.build_ref)")
    runner = ref_agent.build_runner("Pendulum-v1", parallels=4, n_steps=T, seed=2, use_obsnorm=True,
                                    model_dir=str(tmp_path / "ref_models"))
    live = runner.agent
    live.obs_rms.update(np.random.default_rng(0).standard_normal((50, 3)).astype(np.float32))
    live.save_model("final_model.pth")
    ref_file = glob.glob(str(tmp_path / "ref_models" / "**" / "obs_rms.npy"), recursive=True)
    assert len(ref_file) == 1
    ref = np.load(ref_file[0], allow_pickle=True).item()
    a = build_ppo("Pendulum-v1", parallels=64, n_steps=T, seed=2, use_obsnorm=True, model_dir=str(tmp_path / "models"))
    a.train(T)
    a.save_model("final_model.pth")
    ours = np.load(glob.glob(str(tmp_path / "models" / "seed_2_*" / "obs_rms.npy"))[0], allow_pickle=True).item()
    assert sorted(ours) == sorted(ref) and all(np.shape(ours[k]) == np.shape(ref[k]) for k in ref)
    # our load_model reads the reference's file (its policy has the same parameter names)
    a.load_model(os.path.dirname(os.path.dirname(ref_file[0])), seed=2)
    st = a._obs_rms[0].cpu().numpy()
    assert np.allclose(st[:3], ref["mean"]) and np.allclose(st[4:7], ref["var"]) and np.isclose(st[8], ref["count"])


WORKER = r'''
import os, shutil, sys, torch
sys.path.insert(0, %r)
import torch.distributed as dist
from xuanpolicy_b200 import dist as xd
from xuanpolicy_b200.configs import build_ppg, build_ppo
rank, local, world = xd.init_from_env("nccl")
out = sys.argv[1]


def flat_state(a):
    """The bytes of the training state (ep_stats[1:] aside: fp64 totals summed with atomics)."""
    torch.cuda.synchronize()
    t = dict(a._checkpoint_tensors(0), **{"env.ep_stats": a.envs.ep_stats[:1]})
    t.pop("learner.scalars")       # PPG sums its loss scalars with atomics
    return torch.cat([v.detach().contiguous().reshape(-1).view(torch.uint8) for _, v in sorted(t.items())])


def replicas_equal(a):
    from xuanpolicy_b200 import checkpoint
    named = [(k, v) for k, v in sorted(a._checkpoint_tensors(0).items()) if k.startswith(checkpoint._REPLICATED)]
    return not checkpoint.differing_across_ranks(named, a.device)


def case(name, build, k1, k2, **kw):
    a = build(**kw); a.train(k1); a.train(k2); ref = flat_state(a); del a
    b = build(**kw); b.train(k1)
    path = os.path.join(out, name)
    b.save_checkpoint(path); del b
    c = build(policy_seed=99, **kw)
    c.load_checkpoint(path)
    c.train(k2)
    ok = torch.equal(ref, flat_state(c)) and replicas_equal(c)
    return "ok" if ok else "BAD"


res = {}
res["PPO"] = case("ppo", build_ppo, 24, 24, env_id="CartPole-v1", parallels=1024, n_steps=16, n_epoch=2, n_minibatch=4,
                  shuffle="host", use_obsnorm=True, use_rewnorm=True, seed=3)
res["PPG"] = case("ppg", build_ppg, 24, 32, env_id="CartPole-v1", parallels=128, n_steps=16, n_epoch=2, policy_nepoch=1,
                  value_nepoch=1, aux_nepoch=1, seed=3)
if rank == 0:
    for k, v in res.items():
        print("RESULT", k, v)
dist.destroy_process_group()
''' % REPO


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_resume_equals_the_uninterrupted_run(tmp_path):
    """Env-sharded PPO with the normalisers over peer memory, and PPG: each rank writes and reads its own file, the resumed
    run equals the uninterrupted one and the replicas stay bit-identical across the ranks."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29547", str(script), str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    lines = [l.split() for l in out.stdout.splitlines() if l.startswith("RESULT")]
    assert sorted(l[1] for l in lines) == ["PPG", "PPO"] and all(l[2] == "ok" for l in lines), out.stdout[-3000:]
    assert sorted(os.listdir(tmp_path / "ppo")) == ["rank0-of-2.pt", "rank1-of-2.pt"]
