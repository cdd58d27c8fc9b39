"""DummyOnPolicyBuffer drop-in: a device-resident, time-major rollout buffer.

Mirrors DummyOnPolicyBuffer (xuance/common/memory_tools.py:143-245): same constructor, `full`, `clear`, `store`,
`finish_path`, `sample`, and the attributes `observations, actions, rewards, returns, values, terminals,
advantages, auxiliary_infos, start_ids, ptr, size` (exposed env-major [n_envs, n_size, ...] like the reference).

Storage is time-major `[T, N]` on the GPU (see csrc/buffer.cu).  `finish_path(val, i)` keeps the reference's
per-env protocol but only RECORDS the segment end and its bootstrap value; the GAE for every env and segment is
computed by ONE reverse-scan kernel (csrc/gae.cu) the first time its results are needed (`sample`, `returns`,
`advantages`).  The native path skips the per-env calls altogether: `finish_rollout(boot_last)`.

Modes: compat (numpy in/out, the reference's types) and native (`native=True`, torch CUDA tensors in/out).
"""
import numpy as np
import torch

from . import ops
from .policies import OldDistBatch, old_dist_params
from .spaces import is_discrete


class DummyOnPolicyBuffer:
    def __init__(self, observation_space, action_space, auxiliary_shape, n_envs, n_size, use_gae=True,
                 use_advnorm=True, gamma=0.99, gae_lam=0.95, device=None, native=False, gae_variant="auto"):
        self.observation_space, self.action_space, self.auxiliary_shape = observation_space, action_space, auxiliary_shape
        self.n_envs, self.n_size = n_envs, n_size
        self.buffer_size = n_size * n_envs
        self.use_gae, self.use_advnorm = use_gae, use_advnorm
        self.gamma, self.gae_lam = gamma, gae_lam
        self.native, self.gae_variant = native, gae_variant
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("xuanpolicy_b200 buffers live on a CUDA device only (no CPU fallback)")
        obs_shape = tuple(observation_space.shape)
        if len(obs_shape) != 1 or not 1 <= obs_shape[0] <= 8:
            raise NotImplementedError("device buffer supports flat observations of 1..8 floats (classic control)")
        if auxiliary_shape and set(auxiliary_shape.keys()) not in ({"old_logp"}, {"old_dist"}):
            raise NotImplementedError("supported auxiliaries: {'old_logp': ()} (PPO-Clip), {'old_dist': None} "
                                      "(PPO-KL / PPG), or none (A2C / PG)")
        self._has_logp = bool(auxiliary_shape) and "old_logp" in auxiliary_shape
        # {"old_dist": None}: the reference keeps an [n_envs, n_size] numpy array of Python distribution objects
        # (memory_tools.py:28-30); here their parameters live in one device array [T, N, W] (W = A logits, or
        # A means + A stds), allocated at the first store
        self._has_dist = bool(auxiliary_shape) and "old_dist" in auxiliary_shape
        self._dist, self._dist_kind = None, None
        self.obs_dim = obs_shape[0]
        self.discrete = is_discrete(action_space)
        self.act_dim = 1 if self.discrete else int(np.prod(action_space.shape))
        self._act_shape = () if self.discrete else tuple(action_space.shape)
        self.start_ids = np.zeros(n_envs, np.int64)
        T, N, dev = n_size, n_envs, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs_row = 4 if self.obs_dim <= 4 else 8      # floats per stored observation row (one or two float4)
        self._obs = torch.zeros((T, N, self.obs_row), **f32)
        self._act = torch.zeros((T, N, self.act_dim), **f32)
        self._rew, self._val, self._term = torch.zeros((T, N), **f32), torch.zeros((T, N), **f32), torch.zeros((T, N), **f32)
        self._logp, self._adv, self._ret = torch.zeros((T, N), **f32), torch.zeros((T, N), **f32), torch.zeros((T, N), **f32)
        self._trunc = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self._boot = torch.zeros((T, N), **f32)
        self._boot_last = torch.zeros(N, **f32)
        # packed 32-byte records {obs[4], act, old_logp, adv, ret}: one DRAM sector per transition for the minibatch
        # gather (csrc/buffer.cu); built by finish_rollout, only for 1-dim actions
        self._rec = torch.zeros((T * N, 8), **f32) if (native and self.act_dim == 1 and self.obs_row == 4) else None
        self._rec_valid = False
        self._stats = torch.zeros(2, dtype=torch.float64, device=dev)        # whole-rollout (sum, sumsq) of adv
        self._mb_stats = torch.zeros(2, dtype=torch.float64, device=dev)     # per-minibatch (sum, sumsq)
        self._zero_u8 = torch.zeros(N, dtype=torch.uint8, device=dev)
        # host-side record of finish_path calls (compat protocol)
        self._h_segend = np.zeros((T, N), np.uint8)
        self._h_boot = np.zeros((T, N), np.float32)
        self._finished_upto = np.zeros(N, np.int64)
        self._gae_valid = False
        self.ptr, self.size = 0, 0

    # ---------------------------------------------------------------------------------------------- bookkeeping
    @property
    def full(self):
        return self.size >= self.n_size

    def clear(self):
        """Reference re-allocates zeroed arrays (memory_tools.py:185-194); here the same storage is zeroed."""
        self.ptr, self.size = 0, 0
        for t in (self._obs, self._act, self._rew, self._val, self._term, self._logp, self._adv, self._ret,
                  self._trunc, self._boot) + ((self._dist,) if self._dist is not None else ()):
            t.zero_()
        self._h_segend[...] = 0
        self._h_boot[...] = 0
        self._finished_upto[...] = 0
        self._gae_valid = False

    def clear_fast(self):
        """Native loop: every row is overwritten by the next rollout, so only the cursor is reset."""
        self.ptr, self.size = 0, 0
        self._gae_valid = False

    @property
    def packed(self):
        """True when the packed-record gather path is available for the current rollout."""
        return self._rec is not None and self._rec_valid

    # ---------------------------------------------------------------------------------------------- store
    def _dev(self, x, dtype):
        if torch.is_tensor(x):
            return x.to(device=self.device, dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(x)).to(device=self.device, dtype=dtype)

    def store(self, obs, acts, rews, value, terminals, aux_info=None, truncations=None):
        """memory[:, ptr] = data for every field (memory_tools.py:196-204).  `truncations` is an extension used by
        the native loop (segment ends that are not terminals); the reference signature works unchanged."""
        N, p = self.n_envs, self.ptr
        with torch.cuda.device(self.device):
            obs_t = self._dev(obs, torch.float32).reshape(N, self.obs_dim)
            if self.obs_dim != self.obs_row:
                padded = torch.zeros((N, self.obs_row), dtype=torch.float32, device=self.device)
                padded[:, :self.obs_dim] = obs_t
                obs_t = padded
            act_t = acts if (torch.is_tensor(acts) and acts.is_cuda) else torch.as_tensor(np.ascontiguousarray(acts)).to(self.device)
            if self.discrete:
                act_t = act_t.to(torch.int64).reshape(N).contiguous()
            else:
                act_t = act_t.to(torch.float32).reshape(N, self.act_dim).contiguous()
            logp = aux_info["old_logp"] if (aux_info and "old_logp" in aux_info) else torch.zeros(N)
            if self._has_dist:
                self._store_old_dist(aux_info["old_dist"], p)
            trunc = self._zero_u8 if truncations is None else self._dev(truncations, torch.uint8).reshape(N)
            self.store_device(obs_t, act_t, self._dev(rews, torch.float32).reshape(N),
                              self._dev(value, torch.float32).reshape(N), self._dev(terminals, torch.uint8).reshape(N),
                              trunc, self._dev(logp, torch.float32).reshape(N), p)
        self.ptr = (self.ptr + 1) % self.n_size
        self.size = min(self.size + 1, self.n_size)
        self._gae_valid = False

    def store_device(self, obs4, act, rew, val, term_u8, trunc_u8, logp, row, rew_std=None, rew_clip=0.0):
        """Raw device store of one step into row `row` (graph-capturable; all arguments are CUDA tensors;
        obs4 is [N, obs_row] float32)."""
        ops.store(obs4, act, rew, val, term_u8, trunc_u8, logp, self._obs[row], self._act[row], self._rew[row],
                  self._val[row], self._term[row], self._trunc[row], self._logp[row], rew_std, rew_clip)

    # ---------------------------------------------------------------------------------------------- old_dist
    def _dist_rows(self, dists, rows):
        """[rows, W] device rows (logits, or means | stds) of `rows` old distributions."""
        kind, p0, p1 = old_dist_params(dists, self.device)
        p0 = p0.reshape(rows, -1)
        w = p0 if kind == "categorical" else torch.cat([p0, p1.reshape(-1, p0.shape[1]).expand(rows, -1)], dim=1)
        if self._dist is None:
            self._dist_kind = kind
            self._dist = torch.zeros((self.n_size, self.n_envs, w.shape[1]), dtype=torch.float32, device=self.device)
        return w

    def _store_old_dist(self, dists, row):
        rows = self._dist_rows(dists, self.n_envs)      # allocates the device array at the first store
        self._dist[row].copy_(rows)

    def _old_dist_batch(self, w):
        if self._dist_kind == "categorical":
            return OldDistBatch("categorical", w)
        A = w.shape[-1] // 2
        return OldDistBatch("gaussian", w[..., :A].contiguous(), w[..., A:].contiguous())

    def set_old_dist(self, dists):
        """`memory.auxiliary_infos['old_dist'] = split_distributions(new_dist)` of PPG_Agent.train (ppg_agent.py:90-93):
        replaces the stored old distributions of the WHOLE buffer; `dists` is env-major [n_envs, n_size] like
        `memory.observations`."""
        rows = self._dist_rows(dists, self.n_envs * self.n_size).reshape(self.n_envs, self.n_size, -1)
        self._dist.copy_(rows.transpose(0, 1))

    # ---------------------------------------------------------------------------------------------- GAE
    def finish_path(self, val, i):
        """Reference protocol (memory_tools.py:206-229): closes env i's current path [start_ids[i], ptr or n_size)
        with bootstrap value `val`.  Only recorded here; the scan itself is batched (see `_run_gae`)."""
        end = self.n_size if self.full else self.ptr
        if end > self.start_ids[i]:
            self._h_segend[end - 1, i] = 1
            self._h_boot[end - 1, i] = val
            self._finished_upto[i] = end
        self.start_ids[i] = self.ptr
        self._gae_valid = False

    def finish_rollout(self, boot_last, variant=None, adv_from_ret=False):
        """Native path: one GAE scan for the whole rollout.  Segment ends come from the stored terminal /
        truncation flags, bootstrap values from `self._boot` (rows where trunc is set) and `boot_last` [N].
        `adv_from_ret`: the policy-gradient weights are the returns themselves (PG_Learner, pg_learner.py:24)."""
        ops.gae(self._rew, self._val, self._term, boot_last, self._adv, self._ret, self.gamma, self.gae_lam,
                trunc=self._trunc, boot=self._boot, stats=self._stats, use_gae=self.use_gae,
                variant=variant or self.gae_variant)
        if adv_from_ret:
            self._adv.copy_(self._ret)
        if self._rec is not None:
            ops.pack_records(self._obs, self._act, self._logp, self._adv, self._ret, self._rec)
            self._rec_valid = True
        self._gae_valid = True

    def _run_gae(self):
        if self._gae_valid:
            return
        T, N = self.n_size, self.n_envs
        with torch.cuda.device(self.device):
            self._trunc.copy_(torch.from_numpy(self._h_segend))
            self._boot.copy_(torch.from_numpy(self._h_boot))
            self._boot_last.copy_(torch.from_numpy(np.ascontiguousarray(self._h_boot[T - 1])))
            self.finish_rollout(self._boot_last)
            # transitions after an env's last finished path stay zero in the reference
            unfinished = self._finished_upto < self.size
            if unfinished.any():
                tt = torch.arange(T, device=self.device)[:, None]
                mask = tt >= torch.from_numpy(self._finished_upto).to(self.device)[None, :]
                self._adv.masked_fill_(mask, 0.0)
                self._ret.masked_fill_(mask, 0.0)
        self._gae_valid = True

    # ---------------------------------------------------------------------------------------------- sample
    def sample(self, indexes, adv_stats=None, adv_count=0):
        """memory_tools.py:231-245.  `adv_stats` (fp64 [2] CUDA, optional): the (sum adv, sum adv^2) over `adv_count` samples
        to normalise the advantages with instead of this minibatch's own — the global minibatch of an env-sharded agent."""
        assert self.full, "Not enough transitions for on-policy buffer to random sample"
        if not self.native:
            self._run_gae()
        with torch.cuda.device(self.device):
            idx = indexes if torch.is_tensor(indexes) else torch.from_numpy(np.ascontiguousarray(indexes, dtype=np.int64))
            idx = idx.to(device=self.device, dtype=torch.int64).contiguous()
            B = idx.numel()
            f32 = dict(dtype=torch.float32, device=self.device)
            obs = torch.empty((B, self.obs_dim), **f32)
            act = torch.empty((B, self.act_dim), **f32)
            ret, val, adv, logp = (torch.empty(B, **f32) for _ in range(4))
            local = self.use_advnorm and adv_stats is None
            ops.gather_batch(idx, self.n_size, self.n_envs, self._obs, self.obs_dim, self._act, self.act_dim, self._ret,
                             self._val, self._adv, self._logp, obs, act, ret, val, adv, logp,
                             stats=self._mb_stats if local else None)
            if local:
                ops.normalize_adv(adv, self._mb_stats, B)
            elif self.use_advnorm:
                ops.normalize_adv(adv, adv_stats, adv_count)
            act = act.reshape((B,) + self._act_shape)
            aux = {"old_logp": logp if self.native else logp.cpu().numpy()} if self._has_logp else {}
            if self._has_dist:       # stays on the device in both modes: the learner is its only consumer
                w = torch.empty((B, self._dist.shape[2]), **f32)
                ops.gather_rows(idx, self.n_size, self.n_envs, self._dist, w)
                aux["old_dist"] = self._old_dist_batch(w)
        if self.native:
            return obs, act, ret, val, adv, aux
        return obs.cpu().numpy(), act.cpu().numpy(), ret.cpu().numpy(), val.cpu().numpy(), adv.cpu().numpy(), aux

    # ---------------------------------------------------------------------------------------------- views
    def _env_major(self, t, trailing=None):
        v = t.transpose(0, 1)
        if trailing is not None:
            v = v[..., :trailing]
        return v if self.native else v.contiguous().cpu().numpy()

    @property
    def observations(self):
        return self._env_major(self._obs, self.obs_dim)

    @property
    def actions(self):
        a = self._env_major(self._act)
        return a.reshape((self.n_envs, self.n_size) + self._act_shape)

    @property
    def rewards(self):
        return self._env_major(self._rew)

    @property
    def values(self):
        return self._env_major(self._val)

    @property
    def terminals(self):
        return self._env_major(self._term)

    @property
    def returns(self):
        if not self.native:
            self._run_gae()
        return self._env_major(self._ret)

    @property
    def advantages(self):
        if not self.native:
            self._run_gae()
        return self._env_major(self._adv)

    @property
    def auxiliary_infos(self):
        if self._has_dist:
            return _AuxInfos(self)
        return {"old_logp": self._env_major(self._logp)} if self._has_logp else {}


class _AuxInfos(dict):
    """`memory.auxiliary_infos` for the "old_dist" auxiliary: reading gives the env-major [n_envs, n_size] batch,
    assigning replaces the stored distributions (the one write PPG_Agent.train performs, ppg_agent.py:93)."""

    def __init__(self, memory):
        super().__init__()
        self._memory = memory
        if memory._dist is not None:
            dict.__setitem__(self, "old_dist", memory._old_dist_batch(memory._dist.transpose(0, 1)))

    def __setitem__(self, key, value):
        if key != "old_dist":
            raise KeyError(key)
        self._memory.set_old_dist(value)
        dict.__setitem__(self, key, self._memory._old_dist_batch(self._memory._dist.transpose(0, 1)))
