"""bench.py --dump-outputs: what the timed path computed in its last step, as float32 / float64 .npy files within the size
budget; the same seeded inputs give the same outputs, so two builds can be compared output for output."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import bench


def _stand_in_agent(T, N, od=3):
    g = torch.Generator().manual_seed(3)
    r = lambda *s: torch.randn(*s, generator=g)
    mem = SimpleNamespace(n_envs=N, obs_dim=od, _obs=r(T, N, 4), _act=r(T, N, 1), _rew=r(T, N), _val=r(T, N),
                          _term=(r(T, N) > 1).float(), _logp=r(T, N), _adv=r(T, N), _ret=r(T, N))
    return SimpleNamespace(memory=mem, last_info={"actor-loss": 0.5, "episodes": 7}, policy=torch.nn.Linear(od, 2),
                           _obs_rms=[torch.rand(9, dtype=torch.float64), torch.rand(9, dtype=torch.float64)], _rms_cur=1,
                           _ret_rms=torch.rand(3, dtype=torch.float64))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_keeps_whole_rollout_within_budget(tmp_path):
    agent = _stand_in_agent(16, 64)
    names = bench.dump_outputs(agent, str(tmp_path))
    out = _load(str(tmp_path))
    assert sorted(out) == names
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert out["obs"].shape == (16, 64, 3) and np.array_equal(out["obs"], agent.memory._obs[..., :3].numpy())
    assert np.array_equal(out["adv"], agent.memory._adv.numpy()) and out["act"].shape == (16, 64, 1)
    assert out["info_actor_loss"] == 0.5 and out["info_episodes"] == 7.0
    assert np.array_equal(out["obs_rms"], agent._obs_rms[1].numpy()) and out["obs_rms"].dtype == np.float64
    assert np.array_equal(out["ret_rms"], agent._ret_rms.numpy()) and out["ret_rms"].dtype == np.float64
    for k, v in agent.policy.state_dict().items():
        assert np.array_equal(out["param_" + k], v.numpy()), k
    for k in ("rew", "val", "term", "logp", "ret"):
        assert np.array_equal(out[k], getattr(agent.memory, "_" + k).numpy()), k


def test_dump_samples_envs_of_a_large_rollout_with_a_fixed_seed(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    agent = _stand_in_agent(32, 4096)               # 32 x 4096 x 11 floats = 5.8 MB of rollout
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    bench.dump_outputs(agent, a)
    bench.dump_outputs(agent, b)
    out = _load(a)
    assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= (1 << 20) + 128 * len(out)   # + .npy headers
    keep = out["rew"].shape[1]
    assert 0 < keep < 4096 and all(out[k].shape[:2] == (32, keep) for k in ("obs", "act", "val", "term", "logp", "adv", "ret"))
    cols = [int(np.flatnonzero((agent.memory._rew.numpy().T == out["rew"][:, j]).all(1))[0]) for j in range(keep)]
    assert cols == sorted(set(cols))                                   # distinct envs, in env order
    assert np.array_equal(out["ret"], agent.memory._ret.numpy()[:, cols])
    assert all(np.array_equal(x, y) for x, y in zip(out.values(), _load(b).values()))


@pytest.mark.gpu
def test_two_runs_of_the_timed_path_dump_the_same_outputs(tmp_path):
    """Everything the headline path consumes is seeded: two agents built and timed alike compute the same outputs."""
    torch.cuda.set_device(0)
    flush = torch.zeros(1 << 20, dtype=torch.float32, device="cuda")
    dirs = []
    for run in range(2):
        agent, _, _ = bench.measure(bench.WORKLOADS["c2"], 1, 2, 3, flush, "device", False, True)
        dirs.append(str(tmp_path / str(run)))
        bench.dump_outputs(agent, dirs[-1])
        del agent
    a, b = _load(dirs[0]), _load(dirs[1])
    assert sorted(a) == sorted(b) and a["obs"].shape == (128, 4096, 3) and np.isfinite(a["adv"]).all()
    for k in a:
        if k == "info_mean_episode_score":      # fp64 sum of finished episodes' scores, added up by atomics in any order
            assert np.allclose(a[k], b[k], rtol=1e-12, atol=0), k
        else:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
