"""On-disk training checkpoints of the device-resident agents (agent.save_checkpoint / load_checkpoint).

A checkpoint is a directory with one file per rank, `rank<r>-of-<W>.pt`, written by `torch.save` from CPU tensors:
{"meta": ..., "tensors": {name: tensor}, "host": {name: value}}.  `meta` identifies the run the file belongs to;
`check_compatible` decides whether another agent may resume from it.  This module holds the format and its rules only;
what goes into a file is enumerated by the agent (PPOCLIP_Agent._state_tensors and its checkpoint extras).
"""
import os

import torch

FORMAT_VERSION = 1

# config keys that only name places or logging: they may differ between the run that saved and the run that resumes
PLACE_KEYS = frozenset({"model_dir", "log_dir", "device", "feeder_threads", "sync_info"})

# identity fields of the metadata, checked in this order (world size before rank: a re-sharded run gets the clearer message)
_FIELDS = ("format_version", "agent_class", "env_id", "world_size", "rank", "n_envs", "n_steps", "obs_row")


def plain_config(config):
    """`vars(config)` with every value torch.load(weights_only=True) can read back: numbers, strings, None and lists of them
    stay; anything else is kept as its repr (still compared by check_compatible)."""
    def plain(v):
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        if isinstance(v, (list, tuple)):
            return [plain(x) for x in v]
        return repr(v)
    return {k: plain(v) for k, v in sorted(vars(config).items())}


def rank_file(path, rank, world_size):
    return os.path.join(path, "rank%d-of-%d.pt" % (rank, world_size))


def check_compatible(saved, current):
    """Raises ValueError naming the first field in which the checkpoint metadata `saved` differs from the resuming agent's
    `current`: the identity fields, the policy's parameter names and shapes, or any config key outside PLACE_KEYS.  The
    config seed gets its own message: the action-sampling and permutation keys derive from it (and the rank), so a run
    resumed under another seed would silently diverge."""
    for f in _FIELDS:
        if saved.get(f) != current.get(f):
            if f == "world_size":
                raise ValueError("checkpoint world_size is %r, this run has %r: resuming with a different number of ranks "
                                 "(re-sharding the envs) is not supported" % (saved.get(f), current.get(f)))
            raise ValueError("checkpoint %s is %r, this agent has %r" % (f, saved.get(f), current.get(f)))
    sp, cp = saved.get("params", []), current.get("params", [])
    if [n for n, _ in sp] != [n for n, _ in cp]:
        raise ValueError("checkpoint params (parameter names) %r differ from this policy's %r" % ([n for n, _ in sp], [n for n, _ in cp]))
    for (n, s), (_, c) in zip(sp, cp):
        if tuple(s) != tuple(c):
            raise ValueError("checkpoint params: parameter %r has shape %r, this policy's has %r" % (n, tuple(s), tuple(c)))
    scfg, ccfg = saved.get("config", {}), current.get("config", {})
    if scfg.get("seed") != ccfg.get("seed"):
        raise ValueError("checkpoint config seed is %r, this agent's is %r: the action-sampling and permutation keys derive "
                         "from the seed, so the run cannot resume under another one" % (scfg.get("seed"), ccfg.get("seed")))
    for k in sorted((set(scfg) | set(ccfg)) - PLACE_KEYS):
        if k not in scfg or k not in ccfg or scfg[k] != ccfg[k]:
            raise ValueError("checkpoint config key %r is %r, this agent's is %r"
                             % (k, scfg.get(k, "<absent>"), ccfg.get(k, "<absent>")))


def check_tensors(saved, live):
    """Raises ValueError naming the first tensor that is missing from either side or differs in shape or dtype."""
    for k in sorted(set(saved) | set(live)):
        if k not in saved or k not in live:
            raise ValueError("checkpoint tensor %r is %s" % (k, "missing from the file" if k not in saved else "not held by this agent"))
        s, c = saved[k], live[k]
        if tuple(s.shape) != tuple(c.shape) or s.dtype != c.dtype:
            raise ValueError("checkpoint tensor %r is %s %s, this agent's is %s %s" % (k, tuple(s.shape), s.dtype, tuple(c.shape), c.dtype))


def to_cpu(obj):
    """A copy of a nest of dicts / lists / tuples in which every tensor is a CPU tensor."""
    if torch.is_tensor(obj):
        return obj.detach().to("cpu", copy=True)
    if isinstance(obj, dict):
        return {k: to_cpu(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(to_cpu(v) for v in obj)
    return obj


# tensors every rank of an env-sharded run holds identically: parameters, optimiser state and the (global) normalisers
_REPLICATED = ("learner.flat_param", "learner.exp_avg", "learner.exp_avg_sq", "learner.step", "learner.lr", "learner.kl_coef",
               "policy.", "obs_rms", "ret_rms", "rew_std")


def replicated(payload):
    """(name, tensor) of the replicated part of one rank's payload, the torch optimiser's state included."""
    out = [(k, v) for k, v in sorted(payload["tensors"].items()) if k.startswith(_REPLICATED)]
    opt = payload["host"].get("learner", {}).get("optimizer")
    if opt is not None:
        for i, st in sorted(opt["state"].items()):
            out += [("optimizer.state.%s.%s" % (i, k), v) for k, v in sorted(st.items()) if torch.is_tensor(v)]
    return out


def differing_across_ranks(named, device, group=None):
    """Names of the tensors whose bytes are not the same on every rank (one all_gather of the concatenated bytes)."""
    import torch.distributed as dist
    parts = [t.detach().contiguous().reshape(-1).view(torch.uint8) for _, t in named]
    mine = torch.cat(parts).to(device) if parts else torch.zeros(0, dtype=torch.uint8, device=device)
    every = [torch.empty_like(mine) for _ in range(dist.get_world_size(group))]
    dist.all_gather(every, mine, group=group)
    bounds = [0]
    for p in parts:
        bounds.append(bounds[-1] + p.numel())
    return [n for i, (n, _) in enumerate(named)
            if any(not torch.equal(o[bounds[i]:bounds[i + 1]], every[0][bounds[i]:bounds[i + 1]]) for o in every[1:])]


def write_atomic(obj, path):
    """torch.save to a temporary name in the same directory, then os.replace: a save cut off part-way leaves the previous
    file (if any) under `path` and no partial file under that name."""
    tmp = "%s.tmp-%d" % (path, os.getpid())
    try:
        with open(tmp, "wb") as f:
            torch.save(obj, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise


def read(path, rank, world_size):
    """The payload of this rank's file.  A directory written by another number of ranks is refused by name."""
    f = rank_file(path, rank, world_size)
    if not os.path.exists(f):
        others = sorted(n for n in (os.listdir(path) if os.path.isdir(path) else []) if n.startswith("rank") and n.endswith(".pt"))
        if others:
            raise ValueError("checkpoint world_size: %s holds %s, not %s; resuming with a different number of ranks "
                             "(re-sharding the envs) is not supported" % (path, ", ".join(others), os.path.basename(f)))
        raise FileNotFoundError("no checkpoint file %s" % f)
    return torch.load(f, map_location="cpu", weights_only=True)
