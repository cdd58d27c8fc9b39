"""Times `test()` (evaluation episodes): native device envs (the device evaluation loop) against compat numpy envs of the same
size (the host loop), for CartPole-v1 and Pendulum-v1 at N test envs with test_episode = N.

    python tools/bench_eval.py [--n 16 1024 8192 65536] [--envs CartPole-v1 Pendulum-v1] [--out FILE]
    python -m torch.distributed.run --nproc-per-node W tools/bench_eval.py [...]

Under torch.distributed.run each --n is the TOTAL env count, split evenly over the W ranks: the device path is the env-sharded
evaluation (one loop over all ranks' envs, exchanged over peer memory), the host path runs each rank's loop on its own envs to
test_episode = N, which is what an env-sharded run without the device path does.  Rank 0 prints the lines, with `world_size`.

Each path gets one warm-up call, then one timed call: a host clock around the call, which ends with the scores on the host
(the device path synchronises before it returns them).  A third call under torch.profiler counts what one call issues: device
-> host copies (each a host sync) and kernel launches, divided by the vector steps the call ran.  One JSON line per case, with
the card's name and power limit read in the same run.  Writes nothing into the repository unless --out points there."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def card(index=0):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout
        name, limit = [x.strip() for x in out.split(",")[:2]]
        return {"name": name, "power_limit": limit}
    except Exception as e:      # noqa: BLE001 - the card name from torch is still worth printing
        return {"name": torch.cuda.get_device_name(index), "power_limit": "unknown (%s)" % type(e).__name__}


class CountingEnvFn:
    """env_fn that also counts the vector steps taken on the envs it makes (the host loop's steps)."""

    def __init__(self, env_id, n, native, device="cuda"):
        self.env_id, self.n, self.native, self.device, self.steps = env_id, n, native, device, 0

    def __call__(self):
        import xuanpolicy_b200 as xb
        envs = xb.DummyVecEnv_Gym(xb.make_env_fns(self.env_id, 11, self.n), device=self.device, native=self.native)
        step = envs.step

        def counted(actions):
            self.steps += 1
            return step(actions)
        envs.step = counted
        return envs


def profile_call(agent, env_fn, test_episode):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        agent.test(env_fn, test_episode)
        torch.cuda.synchronize()
    d2h = launches = 0
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        if e.name.startswith("Memcpy DtoH"):
            d2h += 1
        elif not e.name.startswith(("Memcpy", "Memset")):
            launches += 1
    return d2h, launches


def run_path(agent, env_id, n, native, world=1):
    """n: the total env count, n // world on this rank."""
    fn = CountingEnvFn(env_id, n // world, native, agent.device)
    agent.test(fn, n)                                           # warm-up (the device path captures its chunk graph here)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    fn.steps = 0
    t0 = time.perf_counter()
    scores = agent.test(fn, n)
    wall = time.perf_counter() - t0
    steps = int(agent._evaluator.step.item()) if native else fn.steps
    d2h, launches = profile_call(agent, fn, n)
    return {"wall_s": round(wall, 6), "episodes": len(scores), "vector_steps": steps,
            "episodes_per_s": round(len(scores) / wall, 1), "env_steps_per_s": round(steps * n / wall, 1),
            "us_per_vector_step": round(wall / steps * 1e6, 2), "host_syncs_per_call": d2h,
            "launches_per_vector_step": round(launches / steps, 2)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--n", type=int, nargs="+", default=[16, 1024, 8192, 65536])
    ap.add_argument("--envs", nargs="+", default=["CartPole-v1", "Pendulum-v1"])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py measures on a CUDA device; none is available")
    from xuanpolicy_b200 import dist as xd
    from xuanpolicy_b200.configs import build_ppo
    from xuanpolicy_b200.fused_mlp import FusedActorCritic
    rank, local, world = xd.init_from_env("nccl")
    gpu = card(local)
    torch.cuda.set_device(local)
    for env_id in args.envs:
        for n in args.n:
            xd.shard_envs(n, world, rank)                       # refuses an N that does not split evenly
            agent = build_ppo(env_id, parallels=64, n_steps=16, n_epoch=1, n_minibatch=1, seed=1, device="cuda:%d" % local)
            with torch.no_grad():
                dev = run_path(agent, env_id, n, native=True, world=world)
                host = run_path(agent, env_id, n, native=False, world=world)
            line = {"bench": "eval", "env_id": env_id, "n_envs": n, "test_episode": n, "chunk": agent._eval_chunk,
                    "forward": "tcgen05" if n // world >= FusedActorCritic.MIN_ROWS and agent.learner._fused is not None else "torch",
                    "device": dev, "host": host, "speedup": round(host["wall_s"] / dev["wall_s"], 2),
                    "gpu": gpu["name"], "power_limit": gpu["power_limit"]}
            if world > 1:
                line["world_size"] = world
            if rank == 0:
                print(json.dumps(line), flush=True)
            if args.out and rank == 0:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
            del agent
            torch.cuda.empty_cache()
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
