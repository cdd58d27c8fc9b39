"""Env-sharded throughput of the configurations bench.py does not cover: PPG, PPO-KL, and PPO on the wide-row envs.

    torchrun --nproc-per-node N tools/bench_multi.py [--steps K] [--warmup W] [--only NAME ...]
    python tools/bench_multi.py ...                  (one GPU: the N = 1 point; no rank_parity)

Prints one JSON line per configuration (rank 0):
  * ppg_cartpole / ppg_pendulum — PPG_Agent at the ppg yaml defaults (n_steps 256, policy / value / aux epochs 4 / 8 / 8,
    use_obsnorm / use_rewnorm on) with 4096 envs on EVERY rank (weak scaling);
  * ppo_acrobot / ppo_mountaincar / ppo_mountaincar_continuous — PPOCLIP_Agent at bench.py's C3 shape (65536 envs in total,
    split over the ranks: strong scaling; horizon 256, 8 epochs x 8 minibatches, MLP 128) with both normalisers, on the 6-
    and 8-float observation rows (the last one with a Gaussian action);
  * ppokl_cartpole / ppo_cartpole — PPOKL_Agent and its PPO-Clip twin at the same C3 shape (no normalisers), target_kl 0.01;
  * ppokl_pendulum / ppo_pendulum — the same pair at bench.py's C2 shape (4096 envs per GPU x horizon 128, 8 x 8 minibatches,
    MLP 128, both normalisers on).
`--launches` adds `launches_per_minibatch`: the CUDA kernels, memsets and copies of one epoch issued eagerly under
torch.profiler (after the timed iterations), over the epoch's minibatches.
Each line carries `rank_parity` (parameters and normaliser states bit-identical across ranks after the timed iterations),
the card name and its power limit, read in the same run.  Writes nothing into the repository.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

CONFIGS = {
    "ppg_cartpole": dict(agent="ppg", env_id="CartPole-v1", envs=4096, strong=False),
    "ppg_pendulum": dict(agent="ppg", env_id="Pendulum-v1", envs=4096, strong=False),
    "ppo_acrobot": dict(agent="ppo", env_id="Acrobot-v1", envs=65536, strong=True),
    "ppo_mountaincar": dict(agent="ppo", env_id="MountainCar-v0", envs=65536, strong=True),
    "ppo_mountaincar_continuous": dict(agent="ppo", env_id="MountainCarContinuous-v0", envs=65536, strong=True),
    "ppokl_cartpole": dict(agent="ppokl", env_id="CartPole-v1", envs=65536, strong=True, T=256, norm=False),
    "ppo_cartpole": dict(agent="ppo", env_id="CartPole-v1", envs=65536, strong=True, T=256, norm=False),
    "ppokl_pendulum": dict(agent="ppokl", env_id="Pendulum-v1", envs=4096, strong=False, T=128, norm=True),
    "ppo_pendulum": dict(agent="ppo", env_id="Pendulum-v1", envs=4096, strong=False, T=128, norm=True),
}


def card(local):
    """(name, power limit) of this rank's GPU, as nvidia-smi reports them."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")[:2]]
        return {"name": name, "power_limit": limit}
    except Exception as e:                    # pragma: no cover - depends on the host's driver tools
        return {"name": torch.cuda.get_device_name(local), "power_limit": "unknown (%s)" % type(e).__name__}


def build(cfg, world):
    from xuanpolicy_b200.configs import build_ppg, build_ppo, build_ppokl
    n_local = cfg["envs"] // world if cfg["strong"] else cfg["envs"]
    if cfg["agent"] == "ppg":
        return build_ppg(cfg["env_id"], device="cuda", parallels=n_local, seed=1, running_steps=10 ** 9)
    h, norm = [128], cfg.get("norm", True)
    extra = dict(target_kl=0.01) if cfg["agent"] == "ppokl" else {}
    return (build_ppokl if cfg["agent"] == "ppokl" else build_ppo)(
        cfg["env_id"], device="cuda", parallels=n_local, n_steps=cfg.get("T", 256), gamma=0.99, gae_lambda=0.95, n_epoch=8,
        n_minibatch=8, representation_hidden_size=h, actor_hidden_size=h, critic_hidden_size=h, shuffle="device", seed=1,
        policy_seed=1, use_obsnorm=norm, use_rewnorm=norm, running_steps=10 ** 9, **extra)


def launches_per_minibatch(agent):
    """Device activities (kernels, memsets, copies) of one eagerly issued epoch, over its minibatches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        agent._epoch_peer() if agent.learner._peer is not None else agent._epoch_body()
        torch.cuda.synchronize()
    n = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    return round(n / agent.n_updates_per_epoch, 2)


def time_iterations(agent, steps, warmup, world):
    """Seconds of `steps` training iterations (one rollout + its update phase each) after `warmup`, max over ranks."""
    T = agent.n_steps
    for _ in range(warmup):
        agent.train(T)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        agent.train(T)
    e.record()
    torch.cuda.synchronize()
    t = torch.tensor([s.elapsed_time(e) / 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def rank_parity(agent, world):
    """Parameters and normaliser states bit-identical on every rank; the env states must differ (the ranks own different envs)."""
    d = torch.distributed

    def same(t):
        t = t.detach().reshape(-1).double().contiguous()
        all_ = [torch.empty_like(t) for _ in range(world)]
        d.all_gather(all_, t)
        return all(torch.equal(all_[0], x) for x in all_)
    params = torch.cat([p.detach().reshape(-1) for p in agent.policy.parameters()])
    norm = torch.cat([agent._obs_rms[agent._rms_cur], agent._ret_rms, agent._rew_std.double()])
    return {"params_bit_identical_across_ranks": same(params), "normaliser_state_bit_identical_across_ranks": same(norm),
            "env_states_differ_across_ranks": not same(agent.envs._state),
            "exchange": "peer-memory kernels" if agent.learner._peer is not None else "nccl all-reduce"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", nargs="*", default=None, choices=sorted(CONFIGS))
    ap.add_argument("--launches", action="store_true")
    args = ap.parse_args()
    from xuanpolicy_b200 import dist as xd
    rank, local, world = xd.init_from_env("nccl")
    torch.cuda.set_device(local)
    gpu = card(local)
    for name in args.only or list(CONFIGS):
        cfg = CONFIGS[name]
        agent = build(cfg, world)
        secs = time_iterations(agent, args.steps, args.warmup, world)
        parity = rank_parity(agent, world) if world > 1 else None
        line = {"config": name, "agent": type(agent).__name__, "env_id": cfg["env_id"], "n_gpus": world,
                "scaling": "strong" if cfg["strong"] else "weak", "envs_per_gpu": agent.n_envs, "envs_total": agent.n_envs * world,
                "horizon": agent.n_steps, "obs_row_floats": agent.memory.obs_row, "use_obsnorm": agent.use_obsnorm,
                "use_rewnorm": agent.use_rewnorm, "steps": args.steps, "warmup": args.warmup,
                "value": round(agent.n_envs * agent.n_steps * args.steps * world / secs, 1), "unit": "env-steps/s",
                "ms_per_iteration": round(secs / args.steps * 1e3, 3), "gpu": gpu["name"], "power_limit": gpu["power_limit"],
                "rank_parity": parity}
        if args.launches and cfg["agent"] != "ppg":
            line["launches_per_minibatch"] = launches_per_minibatch(agent)
        if rank == 0:
            print(json.dumps(line), flush=True)
        del agent
        torch.cuda.empty_cache()
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
