#!/usr/bin/env python
"""bench.py — PPO env-steps/s on B200 (BASELINE.json metric), with roofline, CPU baseline and clocks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload auto|c1|c2|c3|c5]
                    [--dump-outputs DIR]

A "step" is one PPO iteration of the hot path: a rollout of `horizon` vector steps over the env batch, the batched GAE,
and n_epoch x n_minibatch fused updates.  Observation / reward normalisation is ON (the reference yaml default,
xuance/configs/ppo/classic_control/*.yaml:34-35); the same measurement with it off rides along as `norm_off`.

Workloads (BASELINE.json configs; `--workload auto`, the default, picks by N):
  N = 1   headline = C2  "PPO-Clip Pendulum-v1 Gaussian policy, 4096 envs, horizon 128, on 1 B200";
          extra keys: `c3` (configs[2] on one GPU: the base of the strong-scaling series), `c1` (configs[0]: ours and the
          reference's CPU path on the full config), `e2e_compat`, `c4_gae`
  N > 1   headline = C3  "PPO-Clip CartPole-v1, 65536 envs, env-sharded across 2/4/8 B200" (STRONG scaling: 65536/N envs
          per rank); extra keys: `weak_c2` (C2 with 4096 envs on every rank), `c5` (configs[4], N = 8 only), `c4_gae`
          (configs[3] sharded over the ranks), `rank_parity` (replicas bit-identical; peer-memory gradient sum == NCCL sum)
For N > 1 launch with torchrun (RANK/LOCAL_RANK/WORLD_SIZE from the env).

Printed keys (one JSON line, rank 0):
  value  env-steps/s with everything device-resident (index permutations drawn on the GPU)
  e2e    the same loop through the public API `PPOCLIP_Agent.train` with HOST-drawn minibatch permutations copied
         H2D from pinned memory every epoch and the log scalars read back D2H every iteration
  e2e_compat    the three drop-ins in COMPAT mode (numpy in / numpy out, list-of-dict infos: what an unmodified reference
                agent calls) driven by the reference's agent loop as restated in oracle/ref_port.PPOAgentPort
  roofline      the kernel of ours with the largest share of the step, timed alone with CUDA events
  kernels       the same measurement for every hand-written kernel on the path + the GAE micro-benchmark shape
  cpu_baseline  the reference's CPU path on a FIXED sample of the workload (same policy as `--impl reference`)
`--impl reference` times the reference's own CPU implementation: the unmodified `PPOCLIP_Agent.train` of the copy
pip-installed into oracle/_ref (oracle/build_ref.py; kind "reference"), else its restatement oracle/ref_port.py (kind
"port"), on a fixed 1024-env sample of the same config with a fixed thread policy.
`--dump-outputs DIR` writes what the headline's last timed step computed (see dump_outputs); every input is seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
    # BASELINE.json configs[0..4]; hyper-parameters not named there default to the reference yaml
    "c1": dict(env_id="CartPole-v1", envs=16, horizon=256, hidden=64, gamma=0.99,
               name="PPO-Clip CartPole-v1, MLP 64x64, 16 envs, horizon 256"),
    "c2": dict(env_id="Pendulum-v1", envs=4096, horizon=128, hidden=128, gamma=0.98,
               name="PPO-Clip Pendulum-v1 Gaussian policy, 4096 envs, horizon 128"),
    "c3": dict(env_id="CartPole-v1", envs=65536, horizon=256, hidden=128, gamma=0.99, strong=True,
               name="PPO-Clip CartPole-v1, 65536 envs (total, env-sharded), horizon 256, gamma 0.99 lambda 0.95"),
    "c5": dict(env_id="Pendulum-v1", envs=262144, horizon=128, hidden=256, gamma=0.98, strong=True, minibatch=65536,
               name="PPO-Clip Pendulum-v1, MLP 256x256, 262144 envs (total), minibatch 65536"),
}
HBM_FALLBACK_GBS = 6650.0


def roofline_of(dom, kd, peak, peak_src, traffic):
    """The dominant kernel (largest CUDA-event time x launches per step) against the roof that bounds it: the tensor pipe when
    its TF32-pass fraction exceeds its HBM fraction (round 2: the dense kernels no longer move the hidden activations), else HBM."""
    hbm = {"achieved": kd["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": kd["frac"], "bytes_per_launch": kd["bytes_per_launch"]}
    note = ("kernel with the largest share of the step (CUDA-event time x launches per step); HBM: achieved = algorithmic bytes / "
            "time; tensor: achieved = fp32-equivalent GEMM flops x TF32 passes / time against 1/2 of the measured bf16 peak.  "
            "See c4_gae for the pure HBM-bound shape")
    if kd.get("tensor_frac_of_tf32_peak", 0.0) > kd["frac"]:
        return {"kernel": dom, "bound": "tensor", "achieved": kd["tensor_pipe_tflops_tf32"], "peak": round(measured_tf32_peak(), 1),
                "unit": "TFLOP/s", "frac": kd["tensor_frac_of_tf32_peak"], "traffic": traffic,
                "peak_source": "1/2 x measured cuBLAS bf16 (MEASURED_PEAKS.json)", "tf32_passes": kd.get("tf32_passes"),
                "gemm_tflops": kd.get("gemm_tflops"), "hbm": hbm, "note": note}
    return {"kernel": dom, "bound": "hbm", "achieved": kd["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": kd["frac"],
            "traffic": traffic, "peak_source": peak_src,
            "tensor": {k: kd[k] for k in ("gemm_tflops", "tensor_pipe_tflops_tf32", "tensor_frac_of_tf32_peak") if k in kd},
            "note": note}


def measured_tf32_peak():
    """Dense TF32 tensor-pipe ceiling in TFLOP/s: half the measured cuBLAS bf16 burst throughput (same pipe, K per
    instruction halves), else half the fallback."""
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["bf16_tflops"]) / 2
    return 1590.0 / 2


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nme, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------- our arm
def build_agent(wl, world, shuffle, sync_info, norm=True, pg=None):
    from xuanpolicy_b200.configs import build_ppo
    n_local = wl["envs"] // world if wl.get("strong") else wl["envs"]
    h = [wl["hidden"]]
    # every rank gets the SAME config seed: the agent folds the rank into its sampling / permutation keys itself
    return build_ppo(wl["env_id"], device="cuda", process_group=pg, parallels=n_local, n_steps=wl["horizon"],
                     gamma=wl["gamma"], gae_lambda=0.95, n_epoch=8, n_minibatch=n_minibatches(wl), representation_hidden_size=h,
                     actor_hidden_size=h, critic_hidden_size=h, shuffle=shuffle, sync_info=sync_info, seed=1, policy_seed=1,
                     use_obsnorm=norm, use_rewnorm=norm, running_steps=10 ** 9)


def n_minibatches(wl):
    if wl.get("minibatch"):
        return max(1, (wl["envs"] * wl["horizon"]) // wl["minibatch"])
    return 8


def mlp_params(wl):
    """Parameter count of the reference's actor-critic for this workload (Basic_MLP + ActorNet + CriticNet; + log-std)."""
    obs, act, gauss = {"CartPole-v1": (4, 2, False), "Pendulum-v1": (3, 1, True)}[wl["env_id"]]
    h = wl["hidden"]
    return (obs * h + h) + 2 * (h * h + h) + (h * act + act) + (h + 1) + (act if gauss else 0)


def config_of(wl, world):
    """The `config` object of the JSON line: a pure function of (workload, N) so that both arms print the same one."""
    n_local = wl["envs"] // world if wl.get("strong") else wl["envs"]
    mb = n_minibatches(wl)
    return {"workload": wl["name"], "envs_total": n_local * world, "envs_per_gpu": n_local, "horizon": wl["horizon"], "n_epoch": 8,
            "n_minibatch": mb, "minibatch_per_gpu": n_local * wl["horizon"] // mb, "mlp_hidden": wl["hidden"],
            "params": mlp_params(wl), "gamma": wl["gamma"], "gae_lambda": 0.95, "use_obsnorm": True, "use_rewnorm": True,
            "parallelism": "env-sharded dp%d" % world,
            "l2_flush": "256 MiB buffer written between timed steps (outside the event pairs)", "allow_tf32": False}


def time_agent(agent, steps, warmup, flush, world):
    """K timed PPO iterations, each bracketed by its own CUDA-event pair; an L2 flush (write of a buffer larger
    than L2) sits between iterations, outside the pairs.  Returns seconds (max over ranks)."""
    T = agent.n_steps
    for _ in range(warmup):
        agent.train(T)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    pairs = []
    for _ in range(steps):
        flush.add_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        agent.train(T)
        e.record()
        pairs.append((s, e))
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    total_ms = sum(s.elapsed_time(e) for s, e in pairs)
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item()) / 1e3


def time_phases(agent, flush):
    """CUDA-event time of one rollout graph replay and one epoch graph replay (single GPU, graphs captured)."""
    epoch_graph = agent._epoch_graph if agent._epoch_graph is not None else (agent._epoch_graphs or [None])[0]
    if agent._rollout_graph is None or epoch_graph is None:
        return None
    out = {}
    for name, g in (("rollout_graph_ms", agent._rollout_graph), ("epoch_graph_ms", epoch_graph)):
        ms = []
        for _ in range(5):
            flush.add_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            g.replay()
            e.record()
            torch.cuda.synchronize()
            ms.append(s.elapsed_time(e))
        out[name] = round(float(np.mean(ms)), 4)
    out["note"] = "one PPO iteration = 1 rollout graph + n_epoch epoch graphs (+ permutation draw/copy per epoch)"
    return out


def count_launches(agent):
    """Hand-written kernel launches inside one PPO iteration (counted from the calls the agent makes)."""
    T, E, M = agent.n_steps, agent.n_epoch, agent.n_updates_per_epoch
    if agent.learner._fused is not None:
        # rollout: weight split (1); per step the one-launch forward + the fused sample/env/store step; bootstrap forward (1);
        # GAE + record packing (2); counter (1)
        per_rollout = 1 + T * (2 if agent._fused_step else 4) + 1 + 2 + 1   # split; per step forward + fused step; bootstrap fwd
        # update: gather, weight split, trunk, hidden, loss, dgrad, wgrad, trunk wgrad, tail (all reduces), grad-norm, adam
        tail_norm = agent.world_size == 1 and os.environ.get("XB_TAIL_NORM", "1") != "0"   # norm taken by the tail launch
        adam_split = os.environ.get("XB_ADAM_SPLIT", "1") != "0"                          # weight split done by the Adam launch
        gather_trunk = os.environ.get("XB_GATHER_TRUNK", "1") != "0"                     # gather + first layer in one launch
        fused_loss = agent.learner._fused_loss_ok(agent.memory, agent.learner._fused)      # loss in the forward epilogue
        # gather(+trunk), [split], [trunk], hidden(+loss), [loss], dgrad, wgrad, trunk wgrad, tail(+norm), [norm], adam(+split)
        per_update = (1 + (0 if adam_split else 1) + (0 if gather_trunk else 1) + 1 + (0 if fused_loss else 1) + 1 + 1 + 1 + 1
                      + (1 if tail_norm else 2))
    else:
        per_rollout = T * (3 + 5) + 5 + 2 + 1  # per step: sample, env_step, store, 3 bias+act, 2 head; bootstrap fwd; GAE + pack; counter
        per_update = 1 + 1 + 2 + 5 + 3         # gather, loss, grad-norm + adam, fwd: 3 bias+act + 2 head, bwd: 2 head+act + 1 act+bias
    per_epoch = 2 if agent.shuffle != "host" else 0     # device permutation + its counter tick
    if agent._fused_norm:                               # statistics ride in the fused step, normalisation in the forward
        if agent.use_obsnorm and not (agent.learner._fused is not None and agent.learner._fused.fwd_from_obs_ok()
                                      and 2 * agent.n_envs >= agent.learner._fused.MIN_ROWS):
            per_rollout += T + 1                        # xb_rms_apply in front of a torch / multi-launch forward
    else:
        if agent.use_obsnorm:                           # per step: moments + normalise; + the bootstrap normalise; state copy
            per_rollout += 2 * T + 2
        if agent.use_rewnorm:                           # per step: return tracker + scalar merge
            per_rollout += 2 * T
    if agent._norm_peer is not None:                    # env-sharded: one statistics exchange per step (+ the merge launch)
        per_rollout += T * (2 if agent._fused_norm else 1)
    return per_rollout + E * (M * per_update + per_epoch)


def time_kernel(fn, flush, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        flush.add_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ms.append(s.elapsed_time(e))
    return float(np.mean(ms)), float(np.min(ms))


def kernel_rooflines(agent, flush, peak, launches_per_step, with_c4, world):
    """Times each hand-written kernel alone, with the arguments it gets inside the step, and derives achieved
    GB/s from the ALGORITHMIC bytes of DESIGN.md / SURVEY.md §8(d)."""
    from xuanpolicy_b200 import ops
    mem, env, lr = agent.memory, agent.envs, agent.learner
    N, T, B = agent.n_envs, agent.n_steps, agent.batch_size
    od, gauss = mem.obs_dim, not agent.discrete
    out = {}
    tf32_peak = measured_tf32_peak()

    def add(name, fn, bytes_per_launch, launches, flops=None, passes=3):
        mean_ms, min_ms = time_kernel(fn, flush)
        gbs = bytes_per_launch / (mean_ms * 1e-3) / 1e9
        out[name] = {"ms": round(mean_ms, 5), "min_ms": round(min_ms, 5), "launches_per_step": launches,
                     "bytes_per_launch": int(bytes_per_launch), "achieved_gbs": round(gbs, 2), "frac": round(gbs / peak, 5)}
        if flops:   # tensor-core kernels: fp32-equivalent GEMM flops (2MNK); the TF32 split issues `passes` x that on the tensor
            tf = flops / (mean_ms * 1e-3) / 1e12      # pipe (3: hi/lo of both operands; 2: binary-form wgrad, one operand exact)
            out[name].update({"gemm_tflops": round(tf, 2), "tf32_passes": passes, "tensor_pipe_tflops_tf32": round(passes * tf, 2),
                              "tensor_frac_of_tf32_peak": round(passes * tf / tf32_peak, 4)})

    with torch.no_grad():
        dist, v = agent._policy_forward(agent._x[agent._cur])
    x_cur, x_nxt = agent._x[agent._cur], agent._x[agent._cur ^ 1]
    snap = agent._snapshot()
    env_bytes = (78 if gauss else 118) * N
    sep = 0 if agent._fused_step else T      # the three per-step kernels are fused into one launch on the rollout path
    add("env_step", lambda: ops.env_step(env._kind, env._state, env._rng, env._elapsed, env._ep_score,
                                         agent._act.reshape(N), x_nxt[N:], x_nxt[:N], env._rew, env._term, env._trunc,
                                         env._reset_obs, env._ep_step_out, env._ep_score_out, env.max_episode_length,
                                         ep_stats=env.ep_stats), env_bytes, sep)
    agent._restore(snap)
    add("sample_logp", lambda: agent._sample(dist, 0), N * ((4 + 4 + 4) if gauss else (8 + 8 + 4)), sep)
    vN = v[:N].contiguous()
    add("store", lambda: mem.store_device(x_cur[:N], agent._act, env._rew, vN, env._term, env._trunc, agent._logp, 0),
        N * 2 * 36, sep)
    if agent._fused_step:
        snap = agent._snapshot()
        cur = agent._cur

        def one_step():
            agent._rollout_step(0)
        with torch.no_grad():
            dist0, v0 = dist, v
            prm = dist0.get_param()
            act_param = prm[:N] if not gauss else prm[0][:N]
            logstd = None if not gauss else agent.policy.actor.logstd.detach()
            add("rollout_step_fused", lambda: ops.rollout_step(
                env._kind, act_param, logstd, v0[:N], agent._sample_seed, agent._ctr, 0, env._state, env._rng, env._elapsed,
                env._ep_score, x_nxt[N:], x_nxt[:N], env._rew, env._term, env._trunc, env._reset_obs, env._ep_step_out,
                env._ep_score_out, env.ep_stats, env.max_episode_length, x_cur[:N], agent._act, agent._logp, mem._obs[0],
                mem._act[0], mem._rew[0], mem._val[0], mem._term[0], mem._trunc[0], mem._logp[0],
                boot_src=v0[N:], boot_row=mem._boot[0], trig_cache=agent._trig_cache),
                env_bytes + N * ((4 + 4 + 4) if gauss else (8 + 8 + 4)) + N * 36, T)
        agent._restore(snap)
        agent._cur = cur
    if agent.use_obsnorm and not agent._fused_norm:
        add("obs_moments", lambda: ops.moments4(x_cur[:N], agent._obs_sums, agent._obs_ws), N * 16, T)
        add("obs_normalize", lambda: ops.rms_normalize(x_cur, od, agent._obs_sums, agent._obs_rms[0], agent._obs_rms[1],
                                                       agent.obsnorm_range, agent._xn, 0), 2 * N * 32, T + 1)
    if agent.use_rewnorm and not agent._fused_norm:
        snap_r = agent._snapshot()
        add("returns_track", lambda: ops.returns_track(agent._returns, env._rew, env._term, env._trunc, agent.gamma,
                                                       agent._ret_sums, agent._ret_ws), N * (8 + 8 + 4 + 2), T)
        agent._restore(snap_r)
    add("gae_and_pack", lambda: mem.finish_rollout(agent._boot_last), (20 + 1 + (64 if mem._rec is not None else 0)) * N * T, 1)
    idx = agent._perm[:B]
    agent._device_permutation()
    fused = lr._fused if (lr._fused is not None and B >= lr._fused.MIN_ROWS) else None
    Hh = agent.config.representation_hidden_size[-1]
    mb = lr.stage_gather(mem, idx)
    if mb.get("trunk_done"):     # gather fused with the MLP's first layer: + the B x H activations it writes
        add("gather_trunk_fwd", lambda: lr.stage_gather(mem, idx), B * (8 + 32 + 4 * od + 16 + 4 * Hh), launches_per_step["updates"])
    else:
        add("gather_records" if mem.packed else "gather_obs_advstats", lambda: lr.stage_gather(mem, idx),
            B * ((8 + 32 + 4 * od + 16) if mem.packed else (8 + 16 + 4 * od + 4)), launches_per_step["updates"])
    with torch.no_grad():
        if fused is not None:
            act_out, v_pred = fused.forward(mb["obs"])
            a_dist = fused.dist_params(act_out)
        else:
            _, a_dist, v_pred = agent.policy(mb["obs"])
    vp = v_pred.contiguous()
    dv = torch.empty_like(vp)
    kw = dict(clip_range=lr.clip_range, vf_coef=lr.vf_coef, ent_coef=lr.ent_coef, inv_batch=1.0 / B, adv_stats=mb["stats"],
              adv_count=B)
    # with the loss riding in dense_fwd2's epilogue the stand-alone loss kernel is not launched in the step at all
    # (launches_per_step 0: listed for its own roofline only, never counted into the step)
    loss_launches = 0 if (fused is not None and lr._fused_loss_ok(mem, fused)) else launches_per_step["updates"]
    if mem.packed:
        kw.update(packed=mb["scal"])
        margs = (None, None, None, None)
    else:
        kw.update(idx=idx, T=T, N=N)
        margs = (mem._act, mem._ret, mem._adv, mem._logp)
    if gauss:
        mu, std = a_dist.get_param()
        mu = mu.contiguous()
        logstd = agent.policy.actor.logstd.detach() if std is None else std.log().contiguous()
        dmu = torch.empty_like(mu)
        dls = torch.empty(mu.shape[1], dtype=torch.float64, device="cuda")
        add("ppo_loss_fwd_bwd", lambda: ops.ppo_loss_gaussian(mu, logstd, vp, *margs, dmu, dls, dv, lr._scalars, **kw),
            B * (32 if mem.packed else 40), loss_launches)
    else:
        logits = a_dist.get_param().contiguous()
        dl = torch.empty_like(logits)
        add("ppo_loss_fwd_bwd", lambda: ops.ppo_loss_categorical(logits, vp, *margs, dl, dv, lr._scalars, **kw),
            B * (40 if mem.packed else 48), loss_launches)
    H = agent.config.representation_hidden_size[-1]
    upd = launches_per_step["updates"]
    A_out = 1 if gauss else 2
    if fused is not None:
        # the MLP on the tcgen05 dense kernels (csrc/dense_tc.cu) + the SIMT trunk layer (csrc/mlp_trunk.cu), update shape
        obs_u = mb["obs"]
        bu = fused._buffers(B)
        if bu["dz1"] is None:
            bu["dz1"] = torch.empty(B, H, dtype=torch.float32, device="cuda")
        dact = torch.randn((B, A_out), device="cuda") / B
        dv2 = torch.randn((B, 1), device="cuda") / B
        f4 = 4 * B * H
        adam_split = os.environ.get("XB_ADAM_SPLIT", "1") != "0"
        add("mlp_split_weights", lambda: fused.refresh_weights(), 2 * H * H * 4 * 5, 1 if adam_split else upd + 1)
        add("mlp_trunk_fwd", lambda: fused.stage_trunk(obs_u, bu), B * od * 4 + f4, 0 if mb.get("trunk_done") else upd)
        # round 2: with rank-1 head gradients (every BASELINE config) the hidden activations ya / yc are never stored — the
        # forward leaves one SIGN BIT per activation (B x 2H/32 words), dgrad and the binary-form wgrad read those
        pair = not gauss                               # categorical: the two logit gradients are a softmax pair
        if pair:
            dact[:, 1] = -dact[:, 0]
        skip_y = fused.can_skip_y(softmax_pair=pair)
        sgn = B * (2 * H // 32) * 4 if fused.sign_bits else 0
        heads = B * (A_out + 1) * 4
        add("dense_fwd2_tc", lambda: fused.stage_hidden(bu, keep_y=not skip_y), (1 if skip_y else 3) * f4 + sgn + heads, upd,
            flops=2 * 2.0 * B * H * H)
        add("dense_dgrad_tc", lambda: fused.stage_dgrad(bu, dact, dv2, softmax_pair=pair),
            (2 * f4 + sgn if fused.sign_dgrad else 4 * f4) + heads, upd, flops=2.0 * B * 2 * H * H)
        binw = fused.bin_wgrad and fused._rank1(pair)
        add("dense_wgrad_tc", lambda: fused.stage_wgrad(bu, dact, dv2, softmax_pair=pair), (f4 + sgn if binw else 3 * f4) + heads,
            upd, flops=2 * 2.0 * B * H * (H + 1), passes=2 if binw else 3)
        add("mlp_trunk_wgrad", lambda: fused.stage_trunk_wgrad(obs_u, bu), f4 + B * od * 4, upd)
        add("mlp_backward_tail", lambda: fused.stage_tail(), fused.ws_wgrad.numel() * 4 + fused.ws_trunk.numel() * 4, upd)
        # rollout shape: 2N rows (the obs to act on + the previous step's terminal obs)
        x_r = agent._x[agent._cur][:, :od]
        br = fused._buffers(2 * N)
        if od <= 4 and H <= 128:   # the whole forward in one launch: trunk generated in-kernel, heads only
            add("mlp_fwd_from_obs_rollout", lambda: fused.forward_inference(x_r), 2 * N * (od * 4 + (A_out + 1) * 4), T + 1,
                flops=2 * 2.0 * 2 * N * H * H)
        else:
            add("mlp_trunk_fwd_rollout", lambda: fused.stage_trunk(x_r, br), 2 * N * (od * 4 + H * 4), T + 1)
            add("dense_fwd2_tc_rollout", lambda: fused.stage_hidden(br), 3 * 4 * 2 * N * H, T + 1, flops=2 * 2.0 * 2 * N * H * H)
    else:
        # torch/cuBLAS GEMMs + the non-GEMM half of the MLP (csrc/mlp_epilogue.cu): per update, one forward and one
        # backward epilogue per Linear+LeakyReLU block (3 blocks: representation, actor hidden, critic hidden)
        yb = torch.randn((B, H), device="cuda")
        dyb = torch.randn((B, H), device="cuda")
        dzb, dbb = torch.empty_like(dyb), torch.empty(H, device="cuda")
        bias = torch.randn(H, device="cuda")
        ws32 = torch.zeros(4 + 592 * 1024, dtype=torch.float32, device="cuda")
        w2, b2 = torch.randn((A_out, H), device="cuda"), torch.randn(A_out, device="cuda")
        hout, dout = torch.empty((B, A_out), device="cuda"), torch.randn((B, A_out), device="cuda")
        dw2, db2 = torch.empty_like(w2), torch.empty_like(b2)
        add("mlp_bias_act_fwd", lambda: ops.bias_act_fwd(yb, bias, 0.01), B * H * 8, 3 * upd)
        add("mlp_head_fwd", lambda: ops.head_fwd(yb, w2, b2, hout), B * (H + A_out) * 4, 2 * upd)
        add("mlp_head_bwd_act", lambda: ops.head_bwd_act(dout, yb, w2, 0.01, dzb, dbb, dw2, db2, ws32), B * (2 * H + A_out) * 4, 2 * upd)
        add("mlp_act_bias_bwd", lambda: ops.act_bias_bwd(dyb, yb, 0.01, dzb, dbb, ws32), B * H * 12, 1 * upd)
    snap = agent._snapshot()
    def optimizer_stage():     # what the update graph runs after the backward tail: Adam (+ operand split); norm alone otherwise
        if fused is not None:
            fused.norm_done = agent.world_size == 1 and os.environ.get("XB_TAIL_NORM", "1") != "0"
        lr.stage_optimizer()
    add("adam_step", optimizer_stage, lr._flat.n * (16 + 12), launches_per_step["updates"])
    agent._restore(snap)
    if with_c4:
        out.update(large_shape_rooflines(flush, peak))
    return out


def c4_gae(flush, peak, world):
    """BASELINE.json configs[3]: GAE/return micro-benchmark, T = 2048 x N = 2^20 envs fp32 synthetic rewards / values /
    dones, the envs sharded over the ranks (no exchange: GAE is independent per env).  Both kernel variants; time = max
    over ranks of the mean CUDA-event time; GB/s = 20 B/element x ALL ranks' elements / that time."""
    from xuanpolicy_b200 import ops
    Tc, Nc = 2048, (1 << 20) // world
    rank = torch.distributed.get_rank() if world > 1 else 0
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    rew = torch.randn((Tc, Nc), device="cuda", generator=gen)
    val = torch.randn((Tc, Nc), device="cuda", generator=gen)
    term = (torch.rand((Tc, Nc), device="cuda", generator=gen) < 1 / 200).float()
    boot = torch.randn(Nc, device="cuda", generator=gen)
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    out = {"T": Tc, "N_total": Nc * world, "N_per_gpu": Nc, "bytes_per_element": 20}
    for variant in ("ldg", "tma"):
        if world > 1:
            torch.distributed.barrier()
        mean_ms, min_ms = time_kernel(lambda: ops.gae(rew, val, term, boot, adv, ret, 0.99, 0.95, variant=variant), flush, iters=10)
        t = torch.tensor([mean_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
        gbs = 20.0 * Tc * Nc * world / (ms * 1e-3) / 1e9
        out[variant] = {"ms": round(ms, 4), "min_ms_rank0": round(min_ms, 4), "achieved_gbs_all_gpus": round(gbs, 1),
                        "frac_of_hbm_peak_per_gpu": round(gbs / world / peak, 4),
                        "elements_per_s": round(Tc * Nc * world / (ms * 1e-3), 1)}
    del rew, val, term, adv, ret
    torch.cuda.empty_cache()
    return out


def large_shape_rooflines(flush, peak):
    """The env-step / store / gather / loss kernels at the C3 shape (CartPole, 65 536 envs x 256 steps, global
    minibatch 2 097 152): here the working set (738 MB) exceeds L2, so the HBM roofline is meaningful."""
    import xuanpolicy_b200 as xb
    from xuanpolicy_b200 import ops
    N, T, B = 65536, 256, 2097152
    out = {}

    def add(name, fn, nbytes):
        mean_ms, min_ms = time_kernel(fn, flush, iters=10)
        gbs = nbytes / (mean_ms * 1e-3) / 1e9
        out[name] = {"ms": round(mean_ms, 5), "min_ms": round(min_ms, 5), "launches_per_step": 0, "bytes_per_launch": int(nbytes),
                     "achieved_gbs": round(gbs, 2), "frac": round(gbs / peak, 5)}

    env = xb.DummyVecEnv_Gym(xb.make_env_fns("CartPole-v1", 1, N), device="cuda", native=True)
    env.reset()
    act = torch.randint(0, 2, (N,), device="cuda")
    add("env_step_c3_65536", lambda: env.step_device(act), 118 * N)
    obs_space, act_space = xb.make_spaces("CartPole-v1")
    mem = xb.DummyOnPolicyBuffer(obs_space, act_space, {"old_logp": ()}, N, T, device="cuda", native=True)
    gen = torch.Generator(device="cuda").manual_seed(7)
    for t in (mem._obs, mem._rew, mem._val, mem._logp, mem._adv, mem._ret):
        t.copy_(torch.randn(t.shape, device="cuda", generator=gen))
    mem._act.copy_(torch.randint(0, 2, mem._act.shape, device="cuda", generator=gen).float())
    val = torch.randn(N, device="cuda")
    add("store_c3_65536", lambda: mem.store_device(env._obs, act, env._rew, val, env._term, env._trunc, val, 3), 2 * 36 * N)
    idx = torch.randperm(N * T, device="cuda")[:B].contiguous()
    obs_out = torch.empty((B, 4), device="cuda")
    stats = torch.zeros(2, dtype=torch.float64, device="cuda")
    add("gather_obs_c3_2M", lambda: ops.gather_obs(idx, T, N, mem._obs, 4, obs_out, b_adv=mem._adv, stats=stats), B * (8 + 16 + 16 + 4))
    logits = torch.randn((B, 2), device="cuda")
    vp = torch.randn(B, device="cuda")
    dl, dv = torch.empty_like(logits), torch.empty_like(vp)
    scal64 = torch.zeros(8, dtype=torch.float64, device="cuda")
    add("ppo_loss_c3_2M", lambda: ops.ppo_loss_categorical(logits, vp, mem._act, mem._ret, mem._adv, mem._logp, dl, dv, scal64,
                                                           0.2, 0.25, 0.01, 1.0 / B, idx=idx, T=T, N=N, adv_stats=stats,
                                                           adv_count=B), B * 48)
    rec = torch.zeros((N * T, 8), device="cuda")
    add("pack_records_c3", lambda: ops.pack_records(mem._obs, mem._act, mem._logp, mem._adv, mem._ret, rec), N * T * 64)
    scal = torch.empty((B, 4), device="cuda")
    add("gather_records_c3_2M", lambda: ops.gather_records(idx, T, N, rec, 4, obs_out, scal, stats=stats), B * (8 + 32 + 16 + 16))
    add("ppo_loss_packed_c3_2M", lambda: ops.ppo_loss_categorical(logits, vp, None, None, None, None, dl, dv, scal64, 0.2, 0.25,
                                                                  0.01, 1.0 / B, adv_stats=stats, adv_count=B, packed=scal),
        B * (16 + 8 + 4 + 8 + 4))
    del mem, env, obs_out, logits, idx, rec, scal
    torch.cuda.empty_cache()
    return out


def measure(wl, world, steps, warmup, flush, shuffle, sync_info, norm=True):
    """Builds the agent for `wl`, times `steps` PPO iterations.  Returns (agent, env-steps/s over all ranks, ms per step)."""
    agent = build_agent(wl, world, shuffle, sync_info, norm=norm)
    secs = time_agent(agent, steps, warmup, flush, world)
    return agent, agent.n_envs * agent.n_steps * steps * world / secs, secs / steps * 1e3


DUMP_BYTES = 64 << 20          # --dump-outputs writes at most this much


def dump_outputs(agent, out_dir):
    """--dump-outputs: what the timed path's last PPO iteration computed, one DIR/<name>.npy each (float32 or float64): the
    log scalars train() returned, the policy parameters and running statistics it left, and the rollout it trained on
    (time-major [T, envs, ...]).  Rollouts larger than the budget keep a fixed, seeded sample of the envs.  With --gpus N > 1
    only rank 0 dumps, so the rollout is rank 0's env shard (envs_per_gpu of the config, not envs_total).  Run to run,
    everything is bit-identical except info_mean_episode_score (its fp64 episode totals are summed by atomics)."""
    mem = agent.memory
    out = {"info_" + k.replace("-", "_"): np.float64(v) for k, v in agent.last_info.items()}
    out.update({"param_" + k: v.detach().float().cpu().numpy() for k, v in agent.policy.state_dict().items()})
    out["obs_rms"] = agent._obs_rms[agent._rms_cur].cpu().numpy()        # fp64 mean[D], var[D], count
    out["ret_rms"] = agent._ret_rms.cpu().numpy()                       # fp64 mean, var, count
    rollout = {"obs": mem._obs[..., :mem.obs_dim], "act": mem._act, "rew": mem._rew, "val": mem._val, "term": mem._term,
               "logp": mem._logp, "adv": mem._adv, "ret": mem._ret}
    fixed = sum(a.nbytes for a in out.values())
    per_env = sum(t[:, 0].numel() * 4 for t in rollout.values())
    keep = min(mem.n_envs, (DUMP_BYTES - fixed) // per_env)
    envs = None
    if keep < mem.n_envs:
        envs = np.sort(np.random.default_rng(0).choice(mem.n_envs, keep, replace=False))
        envs = torch.as_tensor(envs, device=mem._rew.device)
    for k, t in rollout.items():
        out[k] = (t if envs is None else t.index_select(1, envs)).float().cpu().numpy()
    assert sum(a.nbytes for a in out.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return sorted(out)


def value_and_e2e(wl, world, steps, warmup, flush, norm=True, with_e2e=True):
    """{"value", "ms_per_step", "e2e": {...}} for a secondary workload (no kernel table)."""
    agent, value, ms = measure(wl, world, steps, warmup, flush, "device", False, norm)
    out = {"workload": wl["name"], "scaling": "strong" if wl.get("strong") else "weak", "value": round(value, 1),
           "unit": "env-steps/s", "ms_per_step": round(ms, 4), "steps": steps, "warmup": warmup,
           "envs_per_gpu": agent.n_envs, "minibatch_per_gpu": agent.batch_size, "use_obsnorm": norm, "use_rewnorm": norm,
           "gpu_launches_per_step": count_launches(agent)}
    del agent
    torch.cuda.empty_cache()
    if with_e2e:
        agent, e2e, ms = measure(wl, world, steps, warmup, flush, "host", True, norm)
        iters = steps + warmup
        out["e2e"] = {"value": round(e2e, 1), "unit": "env-steps/s", "ms_per_step": round(ms, 4),
                      "h2d_bytes_per_step": int(agent.h2d_bytes // iters), "d2h_bytes_per_step": int(agent.d2h_bytes // iters)}
        del agent
        torch.cuda.empty_cache()
    return out


def rank_parity(agent, world):
    """Self-check carried in the multi-GPU line: (1) the replicated parameters are bit-identical on every rank after the
    timed iterations; (2) the fused peer-memory gradient exchange (csrc/peer_comm.cu) gives every rank the same bits, equal
    to NCCL's all-reduce of the same data within fp32 summation-order rounding, and the norm of the sum."""
    d = torch.distributed
    fl, peer = agent.learner._flat, agent.learner._peer
    mine = fl.flat_param.clone()
    allp = [torch.empty_like(mine) for _ in range(world)]
    d.all_gather(allp, mine)
    out = {"params_bit_identical_across_ranks": bool(all(torch.equal(allp[0], x) for x in allp)),
           "exchange": "peer-memory kernels" if peer is not None else "nccl all-reduce"}
    # (3) env-sharded running statistics: every rank must hold the SAME global RunningMeanStd state after the timed rollouts
    #     (the per-step exchange + merge of xb_peer_allreduce_merge; the replicated parameters alone would not show a divergence)
    states = [getattr(agent, n, None) for n in ("_obs_rms", "_ret_rms", "_rew_std")]
    states = [t for s_ in states if s_ is not None for t in (s_ if isinstance(s_, (list, tuple)) else [s_]) if torch.is_tensor(t)]
    if states and (agent.use_obsnorm or agent.use_rewnorm):
        flat = torch.cat([t.detach().reshape(-1).double() for t in states])
        alls = [torch.empty_like(flat) for _ in range(world)]
        d.all_gather(alls, flat)
        out["normaliser_state_bit_identical_across_ranks"] = bool(all(torch.equal(alls[0], x) for x in alls))
    if peer is not None:
        snap = agent._snapshot()
        gen = torch.Generator(device="cuda").manual_seed(100 + d.get_rank())
        fl.flat_grad.copy_(torch.randn(fl.n, device="cuda", generator=gen))
        ref = fl.flat_grad.clone()
        d.all_reduce(ref)
        fl.apply_peer(peer, 0.5, 1.0)
        torch.cuda.synchronize()
        sums = [torch.empty_like(fl.grad_sum) for _ in range(world)]
        d.all_gather(sums, fl.grad_sum)
        n_ref = float(ref.double().norm().item())
        out.update({"peer_sum_bit_identical_across_ranks": bool(all(torch.equal(sums[0], x) for x in sums)),
                    "peer_sum_vs_nccl_max_abs_err": float((fl.grad_sum - ref).abs().max().item()),
                    "peer_sum_equals_nccl_sum": bool(torch.allclose(fl.grad_sum, ref, rtol=1e-6, atol=1e-6)),
                    "norm_of_sum_rel_err": abs(float(fl.gnorm.item()) - n_ref) / n_ref})
        agent._restore(snap)
    return out


def time_compat(wl, sample_envs, iters=2):
    """`e2e_compat`: the drop-ins in compat mode — numpy in / numpy out, list-of-dict infos, per-env finish_path calls,
    host-side normalisation — i.e. the calls an UNMODIFIED reference PPOCLIP_Agent makes (INTEGRATION.md §1), driven by
    that agent's loop as restated in oracle/ref_port.PPOAgentPort.  Host<->device copies on every call are inside the
    timed region.  The per-env Python loops of the reference's agent bound it, not the kernels."""
    import xuanpolicy_b200 as xb
    from oracle import ref_port
    n, T = sample_envs, wl["horizon"]
    torch.manual_seed(1)
    np.random.seed(1)
    envs = xb.DummyVecEnv_Gym(xb.make_env_fns(wl["env_id"], 1, n), device="cuda")
    envs.reset()
    policy = xb.make_policy(envs.observation_space, envs.action_space, hidden=(wl["hidden"],), device="cuda")
    opt = torch.optim.Adam(policy.parameters(), 4e-4, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=10 ** 9)
    memory = xb.DummyOnPolicyBuffer(envs.observation_space, envs.action_space, {"old_logp": ()}, n, T, True, True, wl["gamma"], 0.95)
    learner = xb.PPOCLIP_Learner(policy, opt, sched, "cuda", "/tmp", vf_coef=0.25, ent_coef=0.01, clip_range=0.2,
                                 clip_grad_norm=0.5, use_grad_clip=True)
    agent = ref_port.PPOAgentPort(envs, policy, opt, sched, T, 8, n_minibatches(wl), wl["gamma"], 0.95, use_obsnorm=True,
                                  use_rewnorm=True, memory=memory, update_fn=learner.update)
    agent.train(T)                                   # warm-up iteration
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    agent.train(T * iters)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": round(n * T * iters / dt, 1), "unit": "env-steps/s", "ms_per_step": round(dt / iters * 1e3, 2),
            "sample": "%d of %d envs x full horizon %d, %d timed PPO iterations after 1 warm-up (wall clock incl. every "
                      "H2D/D2H copy); compat drop-ins (DummyVecEnv_Gym.step / DummyOnPolicyBuffer.store, finish_path, "
                      "sample / PPOCLIP_Learner.update) under the reference agent's per-env Python loop" % (n, wl["envs"], T, iters)}


def c1_line(flush):
    """BASELINE.json configs[0] (CartPole-v1, MLP 64x64, 16 envs, horizon 256): ours (device-resident agent; the policy is
    below the tensor-core path's width and batch, so the MLP runs in torch) next to the reference's CPU path on the FULL
    config (the one config the reference runs as is)."""
    wl = WORKLOADS["c1"]
    agent, value, ms = measure(wl, 1, 5, 3, flush, "device", False, True)
    del agent
    torch.cuda.empty_cache()
    ref = time_reference_cpu(wl, wl["envs"], threads=1, warmup=1, steps=3)
    return {"workload": wl["name"], "ours": {"value": round(value, 1), "unit": "env-steps/s", "ms_per_step": round(ms, 3)},
            "reference_cpu": ref}


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    key = args.workload if args.workload != "auto" else ("c2" if world == 1 else "c3")
    wl = WORKLOADS[key]
    # strict fp32 GEMMs by default (the parity tolerances are stated for fp32); --tf32 lets cuBLAS use the TF32 tensor
    # cores where the torch MLP path runs (not the headline: the large-batch MLP runs on our 3xTF32 tcgen05 kernels)
    torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
    peak, peak_src = measured_peaks()
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device="cuda")   # 256 MiB > 126 MB L2
    sampler = ClockSampler(local) if rank == 0 else None
    extra = not args.headline_only

    # value: device-resident (permutations drawn on the GPU, one host sync at the end of train())
    agent, value, ms_step = measure(wl, world, args.steps, args.warmup, flush, "device", False, True)
    dumped = dump_outputs(agent, args.dump_outputs) if (args.dump_outputs and rank == 0) else None
    launches = count_launches(agent)
    phases = time_phases(agent, flush) if world == 1 else None
    launches_per_step = {"updates": agent.n_epoch * agent.n_updates_per_epoch}
    # (all ranks when env-sharded: the optimiser stage contains the cross-GPU exchange kernel, which waits for every peer)
    kernels = kernel_rooflines(agent, flush, peak, launches_per_step, with_c4=(extra and world == 1), world=world) if (rank == 0 or world > 1) else {}
    parity = rank_parity(agent, world) if world > 1 else None
    fused_on = agent.learner._fused is not None and agent.batch_size >= agent.learner._fused.MIN_ROWS
    del agent
    torch.cuda.empty_cache()

    # e2e: public API with host-drawn permutations (H2D from pinned memory each epoch) and D2H of the log each iteration
    agent, e2e, ms_e2e = measure(wl, world, args.steps, args.warmup, flush, "host", True, True)
    iters = args.steps + args.warmup
    h2d, d2h = agent.h2d_bytes // iters, agent.d2h_bytes // iters
    info = agent.last_info
    del agent
    torch.cuda.empty_cache()
    clocks = sampler.stop() if sampler else None

    side = {}
    if extra:
        short = dict(steps=min(args.steps, 5), warmup=3)
        side["norm_off"] = value_and_e2e(wl, world, flush=flush, norm=False, **short)
        side["norm_off"]["what"] = "the headline workload with use_obsnorm = use_rewnorm = False (round-1 setting)"
        if world == 1:
            if key != "c3":
                side["c3"] = value_and_e2e(WORKLOADS["c3"], 1, flush=flush, with_e2e=False, steps=3, warmup=3)
                side["c3"]["what"] = "BASELINE configs[2] on ONE GPU: the N = 1 point of the strong-scaling series bench.py --gpus 2/4/8 prints"
        else:
            if key != "c2":
                side["weak_c2"] = value_and_e2e(WORKLOADS["c2"], world, flush=flush, **short)
                side["weak_c2"]["what"] = "BASELINE configs[1] with 4096 envs on EVERY rank (weak scaling, round-1 headline)"
            if world == 8 and key != "c5":
                side["c5"] = value_and_e2e(WORKLOADS["c5"], world, flush=flush, with_e2e=False, steps=3, warmup=3)
                side["c5"]["what"] = "BASELINE configs[4]: Pendulum-v1, MLP 256x256, 262144 envs, minibatch 65536, at 8 B200"
        if not args.no_c4:
            side["c4_gae"] = c4_gae(flush, peak, world)
    if rank != 0:
        return
    if extra and world == 1:
        side["e2e_compat"] = time_compat(wl, sample_envs=min(1024, wl["envs"]))
        side["c1"] = c1_line(flush)
    step_share = {k: v["ms"] * v["launches_per_step"] for k, v in kernels.items() if v["launches_per_step"]}
    dom = max(step_share, key=step_share.get)
    kd = kernels[dom]
    traffic = None
    tpath = os.path.join(REPO, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and key == "c2":      # ncu DRAM bytes per launch of the same kernel at this shape
        traffic = json.load(open(tpath)).get(dom)
    cpu = None if args.no_cpu_baseline else cpu_baseline(wl)
    cfg = config_of(wl, world)
    line = {
        "metric": "PPO env-steps/s", "value": round(value, 1), "unit": "env-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 4),
        "higher_is_better": True, "scaling": "strong" if wl.get("strong") else "weak", "vs_baseline": None,
        "dtype": "tf32" if (args.tf32 and not fused_on) else "f32",
        "dtype_detail": ("f32-accurate MLP GEMMs (3xTF32 split on the tcgen05 tensor cores, fp32 accumulate)" if fused_on else
                         ("tf32 MLP GEMMs" if args.tf32 else "f32 MLP GEMMs (cuBLAS SIMT)")) + ", f32 loss/optimizer, f64 GAE carry, env physics and running statistics",
        "data": "synthetic",
        "config": cfg,
        "e2e": {"value": round(e2e, 1), "unit": "env-steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": round(ms_e2e, 4),
                "what": "PPOCLIP_Agent.train with host-drawn minibatch permutations (pinned H2D per epoch) and log scalars read back"},
        "gpu_launches": launches * args.steps,
        "roofline": roofline_of(dom, kd, peak, peak_src, traffic),
        "kernels": kernels,
        "phases": phases,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "last_info": {k: (float(v) if not isinstance(v, (int, float)) else v) for k, v in info.items()},
    }
    if parity is not None:
        line["rank_parity"] = parity
    if dumped is not None:
        line["dumped_outputs"] = dumped
    line.update(side)
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------- CPU arms
REF_SAMPLE_ENVS = 1024        # fixed sample of the env batch for the CPU arms (the reference's cost is linear in it)


def cpu_threads(sample_envs):
    """Fixed thread policy: tiny batches (C1) run fastest single-threaded (BASELINE.md §2: 2674 vs 970 env-steps/s at
    1 vs 8 threads), the 1024-env samples with every core (the minibatch GEMMs dominate)."""
    return 1 if sample_envs < 256 else min(os.cpu_count() or 1, 32)


def reference_kind():
    """"reference": the unmodified reference is importable (pip-installed copy in oracle/_ref, or the source tree in the
    build container); "port": only its restatement oracle/ref_port.py is."""
    from oracle import ref_loader
    return "reference" if ref_loader.available() else "port"


def _cpu_agent(wl, n_envs, threads):
    """(agent, kind): the LIVE reference PPOCLIP_Agent built by the reference's own get_runner on the restated libm physics
    (what gym executes on a host), or the port with the same hyper-parameters."""
    torch.set_num_threads(threads)
    h = [wl["hidden"]]
    if reference_kind() == "reference":
        from oracle import ref_agent
        runner = ref_agent.build_runner(wl["env_id"], trig="libm", parallels=n_envs, n_steps=wl["horizon"], seed=1, n_epoch=8,
                                        n_minibatch=n_minibatches(wl), gamma=wl["gamma"], gae_lambda=0.95, use_obsnorm=True,
                                        use_rewnorm=True, representation_hidden_size=h, actor_hidden_size=h, critic_hidden_size=h)
        import xuance.torch.agents.policy_gradient.ppoclip_agent as mod
        mod.tqdm = lambda x: x                         # no progress bar in the timed loop (module global, not a code edit)
        runner.agent.writer.add_scalar = lambda *a, **k: None      # tensorboard file I/O out of the timed loop
        runner.agent.writer.add_scalars = lambda *a, **k: None
        return runner.agent, "reference"
    from oracle import ref_port
    from xuanpolicy_b200 import policies
    torch.manual_seed(1)
    np.random.seed(1)
    envs = ref_port.VecEnvPort(wl["env_id"], n_envs, seed=1, trig="libm")
    envs.reset()
    pol = policies.make_policy(envs.observation_space, envs.action_space, hidden=(wl["hidden"],), device="cpu")
    opt = torch.optim.Adam(pol.parameters(), 4e-4, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=10 ** 9)
    return ref_port.PPOAgentPort(envs, pol, opt, sched, wl["horizon"], 8, n_minibatches(wl), wl["gamma"], 0.95,
                                 use_obsnorm=True, use_rewnorm=True), "port"


def time_reference_cpu(wl, sample_envs, threads, warmup, steps):
    agent, kind = _cpu_agent(wl, sample_envs, threads)
    T = wl["horizon"]
    if warmup:
        agent.train(T * warmup)
    per = []
    for _ in range(steps):
        t0 = time.perf_counter()
        agent.train(T)
        per.append(time.perf_counter() - t0)
    dt = float(sum(per))
    what = ("unmodified xuance PPOCLIP_Agent.train (oracle/_ref) over DummyVecEnv_Gym / DummyOnPolicyBuffer / PPOCLIP_Learner, "
            "torch CPU, restated gym 0.26.2 physics (libm)" if kind == "reference" else
            "oracle/ref_port.py = the reference's per-env Python loops + torch-CPU learner over libm physics")
    return {"value": round(sample_envs * T * steps / dt, 1), "unit": "env-steps/s", "cores": threads, "kind": kind,
            "host_cores_available": os.cpu_count() or 1,
            "ms_per_step_min_max": [round(min(per) * 1e3, 1), round(max(per) * 1e3, 1)],
            "sample": "%d of %d envs x full horizon %d per step, %d timed PPO iterations (8 epochs x %d minibatches) after %d "
                      "warm-up, use_obsnorm/use_rewnorm on; %s" % (sample_envs, wl["envs"], T, steps, n_minibatches(wl), warmup, what)}


def cpu_baseline(wl):
    n = min(REF_SAMPLE_ENVS, wl["envs"])
    return time_reference_cpu(wl, n, cpu_threads(n), warmup=1, steps=3)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = args.gpus
    key = args.workload if args.workload != "auto" else ("c2" if world == 1 else "c3")
    wl = WORKLOADS[key]
    n = min(REF_SAMPLE_ENVS, wl["envs"])
    threads = cpu_threads(n)
    steps = args.steps          # ~2-7 s per step on 16-32 host cores
    res = time_reference_cpu(wl, n, threads, warmup=max(1, min(args.warmup, 2)), steps=steps)
    print(json.dumps({
        "impl": "reference", "metric": "PPO env-steps/s", "value": res["value"], "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": max(1, min(args.warmup, 2)),
        "ms_per_step": round(n * wl["horizon"] / res["value"] * 1e3, 3),
        "higher_is_better": True, "scaling": "strong" if wl.get("strong") else "weak", "vs_baseline": None, "dtype": "f32",
        "dtype_detail": "f32 torch CPU learner, f64 physics", "data": "synthetic", "config": config_of(wl, world),
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto"] + sorted(WORKLOADS))
    ap.add_argument("--no-c4", action="store_true", help="skip the 40 GiB GAE micro-benchmark arrays")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="only the headline workload (no norm_off / c1 / c3 / weak_c2 / c5 / c4 keys)")
    ap.add_argument("--tf32", action="store_true", help="allow TF32 tensor-core GEMMs in the torch MLP (not the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the headline's last timed step computed to DIR/<name>.npy "
                    "(rank 0 only: with --gpus N > 1 the rollout is rank 0's env shard); bench_outputs/ is git-ignored")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the native arm (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
