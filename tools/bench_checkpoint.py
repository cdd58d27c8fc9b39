"""Wall time of agent.save_checkpoint / load_checkpoint at the C5 shape (BASELINE configs[4]: PPO-Clip Pendulum-v1,
MLP 256x256, 262144 envs, minibatch 65536), all envs on one GPU.

    python tools/bench_checkpoint.py [--envs N] [--dir DIR]

Prints one JSON line: save and load seconds and the file size, at a rollout boundary and half-way through a rollout (where
the buffer rows already written travel with the checkpoint), with the card name and its power limit read in the same run.
The checkpoint goes to a temporary directory (or --dir) and is removed afterwards.  Writes nothing into the repository.
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return round(time.perf_counter() - t0, 3)


def main():
    from bench_multi import card
    from xuanpolicy_b200.configs import build_ppo
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=262144)
    ap.add_argument("--dir", default=None, help="parent directory of the checkpoint (default: a temporary directory)")
    args = ap.parse_args()
    T, h = 128, [256]
    agent = build_ppo("Pendulum-v1", device="cuda", parallels=args.envs, n_steps=T, n_epoch=1, n_minibatch=args.envs * T // 65536,
                      representation_hidden_size=h, actor_hidden_size=h, critic_hidden_size=h, shuffle="device", seed=1,
                      use_obsnorm=True, use_rewnorm=True, running_steps=10 ** 9)
    root = tempfile.mkdtemp(prefix="xb200_ckpt_", dir=args.dir)
    out = {"what": "save_checkpoint / load_checkpoint, PPO-Clip Pendulum-v1, MLP 256, %d envs on one GPU, horizon %d" % (args.envs, T)}
    try:
        agent.train(T)
        for name, steps in (("boundary", 0), ("mid_rollout", T // 2)):
            agent.train(steps)
            path = os.path.join(root, name)
            out[name] = {"save_s": timed(lambda: agent.save_checkpoint(path)),
                         "load_s": timed(lambda: agent.load_checkpoint(path)),
                         "file_bytes": os.path.getsize(os.path.join(path, "rank0-of-1.pt")), "buffer_rows": agent._t}
    finally:
        shutil.rmtree(root, ignore_errors=True)
    gpu = card(0)
    out.update(gpu=gpu["name"], power_limit=gpu["power_limit"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
