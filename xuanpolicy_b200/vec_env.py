"""DummyVecEnv_Gym drop-in: all N classic-control environments live on the GPU and step in one kernel.

Mirrors (same names, arguments, attributes, exceptions)
    VecEnv, AlreadySteppingError, NotSteppingError   xuance/environment/vector_envs/vector_env.py:7-103
    DummyVecEnv_Gym                                  xuance/environment/gym/gym_vec_env.py:148-231
    Gym_Env bookkeeping (episode_step/episode_score)  xuance/environment/gym/gym_env.py:36-49

Two modes behind the same methods:
  * compat (default): numpy in / numpy out with list-of-dict `infos`, exactly the reference's types; every call
    does one H2D copy of the actions and D2H copies of the results.  Used for 1:1 parity tests and by an
    unmodified `PPOCLIP_Agent`.
  * native (`native=True`): torch CUDA tensors in / out, `infos` is a lazy array-backed view; nothing leaves
    the device.  Returned tensors alias the env's persistent output buffers (valid until the next step).
"""
from argparse import Namespace

import numpy as np
import torch

from . import ops
from .spaces import Box, Discrete

SPECS = {
    "CartPole-v1": dict(kind=0, state_dim=4, obs_dim=4, max_steps=500),
    "Pendulum-v1": dict(kind=1, state_dim=2, obs_dim=3, max_steps=200),
    # the reference's make_envs wraps MountainCar in a 4-frame stack (gym_env.py:50-83; environment/__init__.py:66-67):
    # that is what "MountainCar-v0" means under the drop-in; gym's bare 2-float env keeps the id "gym:MountainCar-v0"
    "MountainCar-v0": dict(kind=4, state_dim=8, obs_dim=8, max_steps=200),
    "gym:MountainCar-v0": dict(kind=2, state_dim=2, obs_dim=2, max_steps=200),
    "Acrobot-v1": dict(kind=3, state_dim=4, obs_dim=6, max_steps=500),
    # CartPole with gym's v0 registration: the same env, TimeLimit 200
    "CartPole-v0": dict(kind=0, state_dim=4, obs_dim=4, max_steps=200),
    # the 4-frame rule of make_envs holds for every id containing "MountainCar": the continuous env too
    "MountainCarContinuous-v0": dict(kind=6, state_dim=8, obs_dim=8, max_steps=999),
    "gym:MountainCarContinuous-v0": dict(kind=5, state_dim=2, obs_dim=2, max_steps=999),
}


class AlreadySteppingError(Exception):
    def __init__(self):
        Exception.__init__(self, "already running an async step")


class NotSteppingError(Exception):
    def __init__(self):
        Exception.__init__(self, "not running an async step")


def make_spaces(env_id):
    if env_id in ("CartPole-v1", "CartPole-v0"):
        high = np.array([4.8, np.finfo(np.float32).max, 24 * np.pi / 360 * 2, np.finfo(np.float32).max], np.float32)
        return Box(-high, high), Discrete(2)
    if env_id == "Pendulum-v1":
        high = np.array([1.0, 1.0, 8.0], np.float32)
        return Box(-high, high), Box(-2.0, 2.0, shape=(1,))
    if env_id == "MountainCar-v0":       # gym_env.py:55-57
        return Box(np.array([-1.2, -0.07] * 4, np.float32), np.array([0.6, 0.07] * 4, np.float32)), Discrete(3)
    if env_id == "gym:MountainCar-v0":
        return Box(np.array([-1.2, -0.07], np.float32), np.array([0.6, 0.07], np.float32)), Discrete(3)
    if env_id == "Acrobot-v1":
        high = np.array([1.0, 1.0, 1.0, 1.0, 4 * np.pi, 9 * np.pi], np.float32)
        return Box(-high, high), Discrete(3)
    if env_id == "MountainCarContinuous-v0":     # the 4-frame stack of gym_env.py:50-83 over gym's continuous env
        return (Box(np.array([-1.2, -0.07] * 4, np.float32), np.array([0.6, 0.07] * 4, np.float32)),
                Box(-1.0, 1.0, shape=(1,)))
    if env_id == "gym:MountainCarContinuous-v0":
        return Box(np.array([-1.2, -0.07], np.float32), np.array([0.6, 0.07], np.float32)), Box(-1.0, 1.0, shape=(1,))
    raise NotImplementedError("only CartPole-v1, CartPole-v0, Pendulum-v1, MountainCar-v0, MountainCarContinuous-v0 and "
                              "Acrobot-v1 have device kernels (got %r)" % (env_id,))


def continuous_actions(env_id):
    """True when the env's action is a Box (one float32 per env), False for Discrete; KeyError for an unknown id."""
    return ops.continuous_kind(SPECS[env_id]["kind"])


class EnvFn:
    """A thunk describing one env (what `make_envs`' `_thunk` closure carries: env_id and seed)."""

    def __init__(self, env_id, seed):
        self.env_id, self.seed = env_id, seed

    def __call__(self):
        raise RuntimeError("device envs are never instantiated one by one")


def make_env_fns(env_id, seed, parallels):
    return [EnvFn(env_id, seed) for _ in range(parallels)]


def _describe(fn):
    """(env_id, seed) of an env thunk: our EnvFn, or the reference's `_thunk` closure over `config`
    (xuance/environment/__init__.py:36-83)."""
    if hasattr(fn, "env_id") and hasattr(fn, "seed"):
        return fn.env_id, fn.seed
    for cell in getattr(fn, "__closure__", None) or ():
        cfg = cell.cell_contents
        if isinstance(cfg, Namespace) or (hasattr(cfg, "env_id") and hasattr(cfg, "seed")):
            return cfg.env_id, cfg.seed
    raise TypeError("cannot infer env_id/seed from env_fn %r; use xuanpolicy_b200.make_env_fns" % (fn,))


def pcg64_seed_state(seed):
    """numpy's PCG64(SeedSequence(seed)) initial (state_hi, state_lo, inc_hi, inc_lo) — gym.utils.seeding.np_random."""
    st = np.random.PCG64(np.random.SeedSequence(seed)).state["state"]
    m = (1 << 64) - 1
    return np.array([st["state"] >> 64, st["state"] & m, st["inc"] >> 64, st["inc"] & m], dtype=np.uint64)


class LazyInfos:
    """Array-backed stand-in for the reference's list of per-env info dicts (native mode)."""

    def __init__(self, env):
        self._env = env
        self.episode_step, self.episode_score = env._ep_step_out, env._ep_score_out
        self.reset_obs, self.next_obs = env._reset_obs[:, :env._obs_dim], env._next_obs[:, :env._obs_dim]
        self.done = None

    def __len__(self):
        return self._env.num_envs

    def __getitem__(self, i):
        d = {"episode_step": int(self.episode_step[i]), "episode_score": float(self.episode_score[i])}
        if bool(self._env._term[i]) or bool(self._env._trunc[i]):
            d["reset_obs"] = self.reset_obs[i].cpu().numpy()
        return d


class DummyVecEnv_Gym:
    def __init__(self, env_fns, device=None, native=False):
        self.waiting = False
        self.closed = False
        descr = [_describe(fn) for fn in env_fns]
        env_ids = {d[0] for d in descr}
        if len(env_ids) != 1:
            raise ValueError("all env_fns must describe the same env_id")
        self.env_id = descr[0][0]
        if self.env_id not in SPECS:
            raise NotImplementedError("no device kernel for %r" % (self.env_id,))
        spec = SPECS[self.env_id]
        self._kind, self._state_dim, self._obs_dim = spec["kind"], spec["state_dim"], spec["obs_dim"]
        self.num_envs = len(env_fns)
        self.observation_space, self.action_space = make_spaces(self.env_id)
        self.obs_shape = self.observation_space.shape
        self.max_episode_length = spec["max_steps"]
        self.native = native
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("xuanpolicy_b200 environments run on a CUDA device only (no CPU fallback)")
        N, dev = self.num_envs, self.device
        with torch.cuda.device(dev):
            # every env is seeded like the reference: Gym_Env.__init__ does env.reset(seed=seed) (gym_env.py:19)
            seeds = [d[1] for d in descr]
            uniq = {s: pcg64_seed_state(s) for s in set(seeds)}
            rng = np.stack([uniq[s] for s in seeds], axis=1)  # [4, N]
            self._rng = torch.from_numpy(rng.view(np.int64).copy()).to(dev)
            self._state = torch.zeros((self._state_dim, N), dtype=torch.float64, device=dev)
            self._elapsed = torch.zeros(N, dtype=torch.int32, device=dev)
            self._ep_score = torch.zeros(N, dtype=torch.float64, device=dev)
            # observation rows are whole float4s: 4 floats (obs_dim <= 4) or 8 (wide rows, Acrobot-v1's 6)
            self._obs_row = 4 if self._obs_dim <= 4 else 8
            self._obs = torch.zeros((N, self._obs_row), dtype=torch.float32, device=dev)
            self._next_obs = torch.zeros((N, self._obs_row), dtype=torch.float32, device=dev)
            self._reset_obs = torch.zeros((N, self._obs_row), dtype=torch.float32, device=dev)
            self._rew = torch.zeros(N, dtype=torch.float32, device=dev)
            self._term = torch.zeros(N, dtype=torch.uint8, device=dev)
            self._trunc = torch.zeros(N, dtype=torch.uint8, device=dev)
            self._ep_step_out = torch.zeros(N, dtype=torch.int32, device=dev)
            self._ep_score_out = torch.zeros(N, dtype=torch.float64, device=dev)
            self.ep_stats = torch.zeros(3, dtype=torch.float64, device=dev)  # finished episodes, sum score, sum length
            act_dtype = torch.float32 if ops.continuous_kind(self._kind) else torch.int64
            self._act = torch.zeros(N, dtype=act_dtype, device=dev)
            ops.env_reset(self._kind, self._state, self._rng, self._elapsed, self._ep_score, self._obs, 1)
        self.buf_obs = np.zeros((N,) + self.obs_shape, dtype=np.float32)
        self.buf_dones = np.zeros((N,), dtype=bool)
        self.buf_trunctions = np.zeros((N,), dtype=bool)
        self.buf_rews = np.zeros((N,), dtype=np.float32)
        self.buf_infos = [{} for _ in range(N)]
        self.actions = None

    # ---------------------------------------------------------------------------------------------- device API
    def reset_device(self):
        """env.reset() on every env; returns the [N, obs_dim] observation tensor (aliases the env buffer)."""
        with torch.cuda.device(self.device):
            ops.env_reset(self._kind, self._state, self._rng, self._elapsed, self._ep_score, self._obs, 1)
        self._next_obs.copy_(self._obs)
        return self._obs[:, :self._obs_dim]

    def step_device(self, actions):
        """One vector step on the current stream, entirely on device (graph-capturable).  `actions`: int64 [N], or float32
        [N] for a Box action."""
        ops.env_step(self._kind, self._state, self._rng, self._elapsed, self._ep_score, actions, self._obs,
                     self._next_obs, self._rew, self._term, self._trunc, self._reset_obs, self._ep_step_out,
                     self._ep_score_out, self.max_episode_length, ep_stats=self.ep_stats)

    # ---------------------------------------------------------------------------------------------- VecEnv API
    def reset(self):
        obs = self.reset_device()
        if self.native:
            return obs, LazyInfos(self)
        self.buf_obs[...] = obs.cpu().numpy()
        self.buf_infos = [{"episode_step": 0} for _ in range(self.num_envs)]
        return self.buf_obs.copy(), self.buf_infos.copy()

    def step_async(self, actions):
        if self.waiting:
            raise AlreadySteppingError
        listify = True
        try:
            if len(actions) == self.num_envs:
                listify = False
        except TypeError:
            pass
        if not listify:
            self.actions = actions
        else:
            assert self.num_envs == 1, "actions {} is either not a list or has a wrong size - cannot match to {} " \
                                       "environments".format(actions, self.num_envs)
            self.actions = [actions]
        self.waiting = True

    def step_wait(self):
        if not self.waiting:
            raise NotSteppingError
        with torch.cuda.device(self.device):
            a = self.actions
            if torch.is_tensor(a):
                a = a.to(device=self.device, dtype=self._act.dtype).reshape(self.num_envs)
                if not a.is_contiguous():
                    a = a.contiguous()
            else:
                self._act.copy_(torch.as_tensor(np.asarray(a).reshape(self.num_envs)).to(self._act.dtype))
                a = self._act
            self.step_device(a)
        self.waiting = False
        if self.native:
            return (self._obs[:, :self._obs_dim], self._rew, self._term.bool(), self._trunc.bool(), LazyInfos(self))
        self.buf_obs[...] = self._obs[:, :self._obs_dim].cpu().numpy()
        self.buf_rews[...] = self._rew.cpu().numpy()
        self.buf_dones[...] = self._term.cpu().numpy().astype(bool)
        self.buf_trunctions[...] = self._trunc.cpu().numpy().astype(bool)
        ep_step = self._ep_step_out.cpu().numpy()
        ep_score = self._ep_score_out.cpu().numpy()
        done = self.buf_dones | self.buf_trunctions
        reset_obs = self._reset_obs[:, :self._obs_dim].cpu().numpy() if done.any() else None
        infos = []
        for e in range(self.num_envs):
            info = {"episode_step": int(ep_step[e]), "episode_score": float(ep_score[e])}
            if done[e]:
                info["reset_obs"] = reset_obs[e].copy()
            infos.append(info)
        self.buf_infos = infos
        return (self.buf_obs.copy(), self.buf_rews.copy(), self.buf_dones.copy(), self.buf_trunctions.copy(),
                self.buf_infos.copy())

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close_extras(self):
        self.closed = True

    def close(self):
        if self.closed:
            return
        self.close_extras()
        self.closed = True

    def render(self, mode):
        raise NotImplementedError("device environments have no renderer")

    # ---------------------------------------------------------------------------------------------- test hooks
    def get_state(self):
        """fp64 env state as numpy [N, state_dim] (tests compare it bit-for-bit with the oracle)."""
        return self._state.t().contiguous().cpu().numpy()
