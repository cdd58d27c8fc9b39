"""The device rollout at the benchmark's env counts against an fp64 restatement of the policy: stored values and
log-probs, bootstrap values, and the statistics of the action draws.

Each case builds the agent the way bench.build_agent does (configs.build_ppo, one config seed, graphs on, observation and
reward normalisation on unless the case says otherwise) and trains two rollouts: rollout 1 -> update -> rollout 2 ->
update.  At the entry of every update phase the buffer, `_boot_last` and the policy parameters are snapshotted; the
parameters at that point are the ones the preceding rollout ran on, so rollout 2 checks that the weights Adam moved reach
the rollout forward (tf32 hi/lo copies re-split, Discrete(3) head re-folded: `_rollout_begin -> refresh_weights`).

The reference is the module graph of policies.py in float64 (trunk, actor and critic hidden layers with LeakyReLU(0.01),
the heads, `logstd`; Discrete(3) with its unfolded three-logit head, so the fold is checked too), loaded from the snapshot.
The raw observations, terminal ones included, come from replaying the stored actions through the C oracle (bit-exact, see
test_gpu_agent.py).  The observation normaliser is restated from them on the agent's schedule (agent.py:104-116; the fused
step merges the moments of the observations it produces into the next step's state): fp64 batch moments and the float32
Chan merge of normalize.cuh, whose state holds float32 values like the reference's arrays; then the float32 arithmetic of
norm_coeffs / norm_apply.  The reference input is then the kernel's input, which the first assertion checks against the
stored observations.

Checks, on every stored (t, env) of both rollouts:
  1. values      mem._val[t] vs V64(mem._obs[t]): rel_err <= MAX_BAR, rel_rms_err <= RMS_BAR (tests/helpers.py;
                 2 * RMS_BAR at H = 256, see rms_bar);
  2. log-probs   mem._logp[t] vs log pi64(mem._act[t] | mem._obs[t]), the head-output bar propagated: Gaussian
                 |d| <= 2e-5 + MAX_BAR * S * |z| / sigma, categorical |d| <= 2e-5 + 2 * MAX_BAR * S, rms(d) <= 1e-5, with
                 S the head-output scale of the row as rel_err defines it (max(|out|, rms(out)); categorical: of the
                 logits centred per row);
  3. bootstraps  every entry of mem._boot[0..T-2] and of _boot_last vs V64(normalised terminal obs of that step, with that
                 step's normaliser state), bars of 1;
  4. draws       Gaussian z = (a - mu64) / sigma: mean, variance and P(|z| > 2) within 5 sigma of N(0, 1); categorical:
                 sum(1[a = j] - p_j) / sqrt(sum p_j (1 - p_j)) within +-5 for every j; independence of the standardised
                 residuals (z, or the residual of action 0) between step t and t + 1, env e and e + 1, and rollout 1 and
                 rollout 2 at the same (t, e): sum(x y) / sqrt(sum x^2 y^2) within +-5.  Every seed is fixed, so these are
                 deterministic.

Measured on one NVIDIA B200 at its 1000 W power limit; rel_err / rel_rms_err for values and bootstraps, max |d| / rms(d)
for log-probs, worst of the two rollouts:
  case              values              log-probs           bootstraps
  c2                5.5e-6 / 1.5e-6     5.9e-6 / 4.9e-7     6.8e-6 / 1.6e-6
  c2_raw            4.5e-6 / 1.7e-6     8.1e-6 / 6.5e-7     4.5e-6 / 1.7e-6
  c3                3.8e-6 / 1.2e-6     1.0e-6 / 1.3e-7     4.8e-6 / 1.3e-6
  c5                1.2e-5 / 3.8e-6     8.9e-6 / 1.2e-6     1.1e-5 / 5.5e-6
  ragged            5.1e-6 / 1.4e-6     6.2e-6 / 5.8e-7     6.3e-6 / 1.5e-6
  mountaincar       5.5e-6 / 1.1e-6     7.2e-7 / 1.1e-7     7.1e-6 / 1.2e-6
  mountaincar_raw   1.8e-6 / 4.7e-7     3.1e-7 / 8.2e-8     2.0e-6 / 4.7e-7
  acrobot           3.8e-6 / 1.0e-6     7.9e-7 / 1.2e-7     3.0e-6 / 1.0e-6
The worst log-prob error is 0.11 of its bar (c5).  Every standardised draw statistic lies within +-2.3.  Wall time of the
single-GPU cases on that card: about 20 s for the file (c5 4.7 s, c2 2.3 s, every other case under 2 s); the two-rank case
was not measured (one GPU).
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.helpers import MAX_BAR, RMS_BAR, rel_err, rel_rms_err

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# id: (env_id, n_envs, hidden, n_steps, normalisers on, n_minibatch)
CASES = {
    # C2: the one-launch forward with in-kernel normalisation; rollout 2 crosses step 200, where every env truncates
    "c2": ("Pendulum-v1", 4096, 128, 128, True, 4),
    # the same without normalisers: the forward's norm_new == nullptr branch, raw observations stored
    "c2_raw": ("Pendulum-v1", 4096, 128, 128, False, 4),
    # C3 on one rank: the largest rollout grid (131 072 forward rows), the categorical softmax pair
    "c3": ("CartPole-v1", 65536, 128, 16, True, 4),
    # C5: H = 256, the multi-launch forward after xb_rms_apply
    "c5": ("Pendulum-v1", 262144, 256, 4, True, 4),
    # N % 128 = 37: one 128-row tile of the one-launch forward holds rows of both normaliser states
    "ragged": ("Pendulum-v1", 1024 + 37, 128, 201, True, 1),
    # 8-float rows, Discrete(3) on the multi-launch forward, truncations in both rollouts
    "mountaincar": ("MountainCar-v0", 1024 + 37, 128, 201, True, 1),
    # Discrete(3) on the one-launch forward: the folded head comes only from refresh_weights
    "mountaincar_raw": ("gym:MountainCar-v0", 2048, 128, 16, True, 2),
    # 6-float rows
    "acrobot": ("Acrobot-v1", 2048, 128, 32, True, 2),
}
GAMMA = {"CartPole-v1": 0.99}


def drive(env_id, n, H, T, norm, n_minibatch, seed=1):
    """Builds the agent like bench.build_agent, trains two rollouts and returns (agent, snapshots): one dict per update
    phase with the buffer, `_boot_last` and the parameters the rollout before it ran on."""
    from xuanpolicy_b200.configs import build_ppo
    h = [H]
    agent = build_ppo(env_id, device="cuda", parallels=n, n_steps=T, gamma=GAMMA.get(env_id, 0.98), gae_lambda=0.95,
                      n_epoch=1, n_minibatch=n_minibatch, representation_hidden_size=h, actor_hidden_size=h,
                      critic_hidden_size=h, shuffle="host", seed=seed, policy_seed=seed, use_obsnorm=norm, use_rewnorm=norm,
                      use_cuda_graphs=True)
    assert agent.learner._fused is not None and agent.learner._fused.H == H and agent._fused_step
    assert agent._fused_norm == norm
    snaps = []
    orig = agent._update_phase

    def update_phase():
        mem = agent.memory
        snap = {k: getattr(mem, "_" + k).clone() for k in ("obs", "act", "val", "logp", "boot", "term", "trunc")}
        snap["boot_last"] = agent._boot_last.clone()
        snap["params"] = {k: v.detach().clone() for k, v in agent.policy.state_dict().items()}
        snaps.append(snap)
        orig()
    agent._update_phase = update_phase
    agent.train(2 * T)
    torch.cuda.synchronize()
    assert len(snaps) == 2 and agent._rollout_graph is not None
    assert not torch.equal(snaps[0]["params"]["critic.model.0.weight"], snaps[1]["params"]["critic.model.0.weight"])
    return agent, snaps


def reference_policy(agent, params):
    """The policies.py module graph in float64 with the snapshotted parameters."""
    from xuanpolicy_b200.policies import make_policy
    H = agent.config.representation_hidden_size[-1]
    pol = make_policy(agent.observation_space, agent.action_space, hidden=(H,), device=agent.device).double()
    pol.load_state_dict({k: v.double() for k, v in params.items()})
    return pol.eval()


@torch.no_grad()
def reference_outputs(pol, x, discrete, chunk=1 << 18):
    """(value, logits | mu) of rows x [..., obs_dim] in float64."""
    flat = x.reshape(-1, x.shape[-1])
    vs, outs = [], []
    for i in range(0, flat.shape[0], chunk):
        # (the modules one by one: MLPRepresentation.forward would cast its input to float32)
        h = pol.representation.model(flat[i:i + chunk].double())
        dist = pol.actor(h)
        vs.append(pol.critic(h))
        outs.append(dist.logits if discrete else dist.mu)
    return torch.cat(vs).reshape(x.shape[:-1]), torch.cat(outs).reshape(*x.shape[:-1], -1)


class Normaliser:
    """RunningMeanStd of the device rollout: state (mean, var) float32, count float64; merges take fp64 batch moments and
    run the float32 Chan merge of normalize.cuh chan_merge (compiled without multiply-add contraction)."""

    def __init__(self, od):
        self.mean, self.var, self.count = np.zeros(od, np.float32), np.ones(od, np.float32), 1e-4

    def merge(self, x):
        xd = x.astype(np.float64)
        n = float(x.shape[0])
        bm = xd.sum(0) / n
        bv = np.maximum(np.square(xd).sum(0) / n - bm * bm, 0.0)
        bm, bv = bm.astype(np.float32), bv.astype(np.float32)
        fc, fb, ft = np.float32(self.count), np.float32(n), np.float32(self.count + n)
        delta = bm - self.mean
        m2 = self.var * fc + bv * fb + delta * delta * fc * fb / ft
        self.mean = self.mean + delta * fb / ft
        self.var = m2 / ft
        self.count = self.count + n

    def apply(self, x, clip):
        """norm_coeffs + norm_apply: (x - (float)mean) / (sqrtf((float)var) + 1e-8f), clipped."""
        den = np.sqrt(self.var) + np.float32(1e-8)
        return np.clip((x - self.mean) / den, np.float32(-clip), np.float32(clip)), den


def replay(agent, snaps, env_id):
    """Replays both rollouts' stored actions through the C oracle from the agent's seed.  Returns, per rollout, the
    policy inputs restated on the agent's schedule [T, N, od], the normalised terminal observations of every step with
    that step's normaliser state [T, N, od], the tolerance of the stored inputs [T, od] and the number of truncations."""
    from oracle import c_oracle
    N, od, norm = agent.n_envs, agent._obs_dim, agent.use_obsnorm
    ref = c_oracle.VecEnvC(env_id, N, seed=agent.seed, flavour="cr")
    rms = Normaliser(od)
    if norm:
        rms.merge(ref.obs[:, :od])               # the first observations, merged in the agent's constructor
    out = []
    for snap in snaps:
        act = snap["act"].cpu().numpy()
        T = act.shape[0]
        x_in, x_term = np.empty((T, N, od), np.float32), np.empty((T, N, od), np.float32)
        tol = np.zeros((T, od), np.float32)
        truncs = 0
        for t in range(T):
            raw = ref.obs[:, :od].copy()
            if norm:
                x_in[t], den = rms.apply(raw, agent.obsnorm_range)
                # (the float32 state can differ from the device's in its last bit where a sum is rounded differently; one
                #  ulp of the mean moves an input by ulp / den, the rest stays at float32 rounding)
                tol[t] = 2 * np.spacing(np.abs(rms.mean)) / den + 1e-6
            else:
                x_in[t] = raw
            a = act[t, :, 0] if not agent.discrete else act[t, :, 0].astype(np.int64)
            o = ref.step(a)
            x_term[t] = rms.apply(o["obs"][:, :od], agent.obsnorm_range)[0] if norm else o["obs"][:, :od]
            done = o["term"] | o["trunc"]
            truncs += int(o["trunc"].sum())
            ref.obs[done] = o["reset_obs"][done]
            if norm:                               # the step merges the observations the next step acts on
                rms.merge(ref.obs[:, :od])
        out.append((x_in, x_term, tol, truncs))
    return out


def rms_bar(agent):
    """RMS_BAR, doubled at H = 256: there every hidden unit and head output sums twice as many truncated fp32 products.
    Measured at C5 (262 144 envs): 3.8e-6 on the values and 5.5e-6 on the bootstrap values of rollout 1, whose inputs are
    mostly clipped to +-5 (a normaliser that has seen one step of identically seeded envs); H = 128: 1.7e-6 at most."""
    return RMS_BAR * (2 if agent.config.representation_hidden_size[-1] > 128 else 1)


def log_prob_errors(agent, pol, snap):
    """Values and log-probs of one rollout against the fp64 policy, on the stored observations.  Returns the measured
    errors and the standardised residuals of the draws [T, N] (z, or the residual of action 0), after asserting checks
    1 and 2 and the marginal part of 4."""
    od, T = agent._obs_dim, snap["obs"].shape[0]
    v64, out64 = reference_outputs(pol, snap["obs"][:, :, :od], agent.discrete)
    m = {"val": (rel_err(snap["val"], v64), rel_rms_err(snap["val"], v64))}
    assert m["val"][0] <= MAX_BAR and m["val"][1] <= rms_bar(agent), m
    if agent.discrete:
        A = out64.shape[-1]
        a = snap["act"][:, :, 0].long()
        lsm = torch.log_softmax(out64, -1)
        lp64 = lsm.gather(-1, a.unsqueeze(-1)).squeeze(-1)
        c = out64 - out64.mean(-1, keepdim=True)
        S = torch.maximum(c.abs().amax(-1), c.pow(2).mean().sqrt())
        bar = 2e-5 + 2 * MAX_BAR * S
        p = lsm.exp()
        for j in range(A):
            hit = (a == j).double()
            s = float((hit - p[..., j]).sum() / (p[..., j] * (1 - p[..., j])).sum().sqrt())
            assert abs(s) <= 5, ("action", j, s)
        p0 = p[..., 0].clamp(1e-6, 1 - 1e-6)
        resid = ((a == 0).double() - p0) / (p0 * (1 - p0)).sqrt()
    else:
        logstd = snap["params"]["actor.logstd"].double()
        sigma = logstd.exp()
        x = snap["act"].double()
        z = (x - out64) / sigma
        lp64 = (-0.5 * z * z - logstd - 0.5 * math.log(2 * math.pi)).sum(-1)
        S = torch.maximum(out64.abs(), out64.pow(2).mean().sqrt())
        bar = 2e-5 + (MAX_BAR * S * z.abs() / sigma).sum(-1)
        resid = z[..., 0]
        n = resid.numel()
        q = 0.04550026389635842                    # P(|z| > 2) of N(0, 1)
        stats = (float(resid.mean()) * math.sqrt(n), float(resid.pow(2).mean() - 1) / math.sqrt(2 / n),
                 (float((resid.abs() > 2).double().mean()) - q) / math.sqrt(q * (1 - q) / n))
        assert all(abs(s) <= 5 for s in stats), ("z mean / var / tail", stats)
    d = snap["logp"].double() - lp64
    m["logp"] = (float(d.abs().max()), float(d.pow(2).mean().sqrt()), float((d.abs() / bar).max()))
    assert bool((d.abs() <= bar).all()) and m["logp"][1] <= 1e-5, m
    assert resid.shape == (T, snap["obs"].shape[1])
    return m, resid


def corr_stat(x, y):
    """sum(x y) / sqrt(sum x^2 y^2): ~N(0, 1) when y has conditional mean 0 given x (martingale-difference residuals)."""
    x, y = x.double().reshape(-1), y.double().reshape(-1)
    return float((x * y).sum() / (x * x * y * y).sum().sqrt().clamp_min(1e-300))


@pytest.mark.parametrize("case", list(CASES))
def test_rollout_matches_fp64_policy(case):
    env_id, N, H, T, norm, nmb = CASES[case]
    agent, snaps = drive(env_id, N, H, T, norm, nmb)
    od = agent._obs_dim
    replays = replay(agent, snaps, env_id)
    resids, report = [], {}
    for r, (snap, (x_in, x_term, tol, truncs)) in enumerate(zip(snaps, replays)):
        # 0. the restated policy inputs are the stored observations
        stored = snap["obs"][:, :, :od].cpu().numpy()
        if norm:
            err = np.abs(stored - x_in) / tol[:, None, :]
            assert err.max() <= 1, (r, np.unravel_index(err.argmax(), err.shape), float(err.max()))
        else:
            assert np.array_equal(stored, x_in), r
        pol = reference_policy(agent, snap["params"])
        # 1, 2 and the marginals of 4
        m, resid = log_prob_errors(agent, pol, snap)
        resids.append(resid)
        # 3. bootstrap values: every stored one, truncated or not
        vb64, _ = reference_outputs(pol, torch.from_numpy(x_term).to(agent.device), agent.discrete)
        got = torch.cat([snap["boot"][:T - 1], snap["boot_last"][None]])
        m["boot"] = (rel_err(got, vb64), rel_rms_err(got, vb64))
        assert m["boot"][0] <= MAX_BAR and m["boot"][1] <= rms_bar(agent), (r, m)
        m["truncations"] = truncs
        report[r] = m
    if env_id in ("Pendulum-v1", "MountainCar-v0") and T >= 100:
        assert replays[1][3] > 0, "a Pendulum / MountainCar rollout pair must cross step 200"
    # 4. independence: step t vs t + 1, env e vs e + 1, rollout 1 vs rollout 2 at the same (t, e)
    ind = {}
    for r, x in enumerate(resids):
        if T > 1:
            ind["step%d" % r] = corr_stat(x[:-1], x[1:])
        ind["env%d" % r] = corr_stat(x[:, :-1], x[:, 1:])
    ind["rollouts"] = corr_stat(resids[0], resids[1])
    print("MEASURED %s %s independence %s" % (case, report, {k: round(v, 2) for k, v in ind.items()}))
    assert all(abs(v) <= 5 for v in ind.values()), ind


WORKER = r'''
import sys, torch
sys.path.insert(0, %r)
from xuanpolicy_b200 import dist as xd
from tests import test_gpu_rollout_fp64 as m
rank, local, world = xd.init_from_env("nccl")
agent, snaps = m.drive("CartPole-v1", 2048, 128, 16, True, 2)
assert agent.world_size == 2 and agent.learner._peer is not None and agent._shard_norm
resids = []
for snap in snaps:
    errs, resid = m.log_prob_errors(agent, m.reference_policy(agent, snap["params"]), snap)
    resids.append(resid)
    print("MEASURED rank %%d %%s" %% (rank, errs))
r = torch.stack(resids).contiguous()
rs = [torch.empty_like(r) for _ in range(world)]
torch.distributed.all_gather(rs, r)
obs = torch.stack([s["obs"] for s in snaps]).contiguous()
os_ = [torch.empty_like(obs) for _ in range(world)]
torch.distributed.all_gather(os_, obs)
if rank == 0:
    print("RESULT cross=%%.3f obs_differ=%%s" %% (m.corr_stat(rs[0], rs[1]), not torch.equal(os_[0], os_[1])))
torch.distributed.destroy_process_group()
''' % REPO


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_rollouts_match_fp64_policy_and_draw_independent_actions(tmp_path):
    """Env-sharded CartPole, 2048 envs per rank, the same config seed on both ranks (as bench runs C3), normalisers on and
    exchanged over peer memory.  Each rank checks its stored values and log-probs against the fp64 policy (the stored
    observations are the inputs); rank 0 gathers both ranks' standardised residuals: their correlation at the same
    (rollout, t, e) must be within +-5 sigma, and the ranks' observation buffers must differ — all trajectory diversity
    between the ranks comes from the rank folded into the sampling key."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, XB_PEER_COMM="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29563", str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    print("\n".join(l for l in out.stdout.splitlines() if l.startswith(("MEASURED", "RESULT"))))
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][-1]
    cross = float(line.split("cross=")[1].split()[0])
    assert abs(cross) <= 5 and "obs_differ=True" in line, line
