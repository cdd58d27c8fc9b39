"""Test oracles for MountainCarContinuous-v0 and CartPole-v0, the two ids of gym 0.26.2's classic-control set that the
restatements in oracle/ predate.  They extend those restatements from the outside:

    MountainCarContinuousRestated   Python restatement of Continuous_MountainCarEnv (both trig flavours of oracle/gym_restated)
    make / register                 gym_restated.make for the new ids; `register(monkeypatch)` lets oracle/ref_port.VecEnvPort
                                    build them for one test
    vec_env_c                       oracle/c_oracle.VecEnvC for every id: CartPole-v0 on the C oracle's CartPole with limit
                                    200, "gym:MountainCarContinuous-v0" on tests/classic_control_ext.c (compiled on first use
                                    into a temporary directory, never into the tree), "MountainCarContinuous-v0" as the
                                    reference's 4-frame stack over it (c_oracle.MountainCarStackC)
"""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import c_oracle, gym_restated
from oracle.gym_restated import CartPoleRestated, TimeLimitRestated, _Math, _Spaces, new_rng

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "classic_control_ext.c")
# the flags of oracle/Makefile: no FMA contraction, no fast-math, one rounding per operation
_CFLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-fexcess-precision=standard", "-fno-builtin-pow",
           "-fno-builtin-sin", "-fno-builtin-cos", "-Wall", "-Wextra"]


class MountainCarContinuousRestated:
    """gym 0.26.2 Continuous_MountainCarEnv (gym/envs/classic_control/continuous_mountain_car.py), goal_velocity = 0.

    Arithmetic of the pinned numpy 1.21.6, spelled out with explicit float(...) conversions (numpy 2's promotion, installed
    here, would compute `force * self.power` in float32).  The legacy rules are those of the "old result" column of NEP 50's
    table: a numpy scalar combined with a Python scalar promotes by type, not by value, so
      * `force * self.power`: force is action[0] (a float32 scalar) or a Python float (min / max return one operand) ->
        float32 scalar * Python float -> float64;
      * `3 * position`: after a step position is a float32 scalar -> float32 scalar * Python int -> float64 (exact);
      * `velocity += ...`: float32 scalar + float64 -> float64, and so on: every operation of step() is fp64;
      * `math.pow(action[0], 2)`: math converts the float32 to a double; the square of a float32 is exact in fp64;
      * `np.array([position, velocity], dtype=np.float32)`: the only rounding, at the end of the step.
    After reset() the state is the float64 array of the draw, so the first step of an episode runs on the unrounded position.
    """
    min_action = -1.0
    max_action = 1.0
    min_position = -1.2
    max_position = 0.6
    max_speed = 0.07
    goal_position = 0.45
    goal_velocity = 0
    power = 0.0015
    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 30}
    reward_range = (-float("inf"), float("inf"))

    def __init__(self, trig="libm", with_spaces=True):
        self.m = _Math(trig)
        self.np_random = None
        self.state = None
        if with_spaces:
            low = np.array([self.min_position, -self.max_speed], dtype=np.float32)
            high = np.array([self.max_position, self.max_speed], dtype=np.float32)
            self.observation_space = _Spaces.box(low, high)
            self.action_space = _Spaces.box(self.min_action, self.max_action, shape=(1,))

    def reset(self, seed=None):
        if seed is not None or self.np_random is None:
            self.np_random = new_rng(seed)
        self.state = (float(self.np_random.uniform(low=-0.6, high=-0.4)), 0.0)      # np.array([...]): float64
        return np.array(self.state, dtype=np.float32), {}

    def step(self, action):
        a = float(np.float32(np.asarray(action, dtype=np.float32).reshape(-1)[0]))     # action[0], a float32 scalar
        position, velocity = float(self.state[0]), float(self.state[1])
        force = min(max(a, self.min_action), self.max_action)
        velocity = velocity + (force * self.power - 0.0025 * self.m.cos(3.0 * position))
        if velocity > self.max_speed:
            velocity = self.max_speed
        if velocity < -self.max_speed:
            velocity = -self.max_speed
        position = position + velocity
        if position > self.max_position:
            position = self.max_position
        if position < self.min_position:
            position = self.min_position
        if position == self.min_position and velocity < 0:
            velocity = 0.0
        terminated = bool(position >= self.goal_position and velocity >= self.goal_velocity)
        reward = 100.0 if terminated else 0.0
        reward = reward - self.m.sq(a) * 0.1
        obs = np.array([position, velocity], dtype=np.float32)
        self.state = (float(obs[0]), float(obs[1]))
        return obs, reward, terminated, False, {}

    def close(self):
        pass

    def render(self):
        return None


SPECS = {"MountainCarContinuous-v0": (MountainCarContinuousRestated, 999), "CartPole-v0": (CartPoleRestated, 200)}


def make(env_id, trig=None):
    """gym.make(env_id) restated, for the new ids and every id of oracle/gym_restated."""
    cls, limit = SPECS[env_id] if env_id in SPECS else gym_restated.SPECS[env_id]
    return TimeLimitRestated(cls(trig=trig or gym_restated.DEFAULT_TRIG), limit)


def register(monkeypatch):
    """For the duration of one test, gym_restated.make (which oracle/ref_port.VecEnvPort calls) builds the new ids too."""
    for env_id, spec in SPECS.items():
        monkeypatch.setitem(gym_restated.SPECS, env_id, spec)


# ------------------------------------------------------------------------------------------------ C oracle
_lib = None


def lib():
    """tests/classic_control_ext.c as a shared library, built once per source version under the temporary directory."""
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), "xb200_oracle_ext_%d_%s" % (os.getuid(), hashlib.sha1(src).hexdigest()[:16]))
        so = os.path.join(d, "liboracle_ext.so")
        if not os.path.exists(so):
            os.makedirs(d, exist_ok=True)
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")     # oracle/Makefile's compiler
            tmp = "%s.%d" % (so, os.getpid())
            subprocess.check_call([cc] + _CFLAGS + ["-o", tmp, _SRC, "-lquadmath", "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


class VecEnvCExt(c_oracle.VecEnvC):
    """c_oracle.VecEnvC with CartPole-v0 and gym's bare MountainCarContinuous-v0 (float32 actions)."""
    NEW = {"CartPole-v0": dict(sdim=4, odim=4, max_steps=200, act=np.int64),
           "gym:MountainCarContinuous-v0": dict(sdim=2, odim=2, max_steps=999, act=np.float32)}
    SPEC = dict(c_oracle.VecEnvC.SPEC, **NEW)

    def reset_all(self, n_draws=1):
        if self.env_id not in self.NEW:
            return super().reset_all(n_draws)
        fn = c_oracle.lib().oc_cartpole_reset if self.env_id == "CartPole-v0" else lib().oc_mountaincar_continuous_reset
        p = c_oracle._p
        fn(p(self.state), p(self.rng), p(self.elapsed), p(self.ep_score), p(self.obs), C.c_int(n_draws), C.c_long(self.n))
        return self.obs.copy()

    def step(self, actions):
        if self.env_id not in self.NEW:
            return super().step(actions)
        n, p = self.n, c_oracle._p
        a = np.ascontiguousarray(np.asarray(actions).reshape(n), dtype=self.act_dtype)
        rew, term, trunc = np.empty(n, np.float32), np.empty(n, np.uint8), np.empty(n, np.uint8)
        reset_obs = np.zeros((n, self.odim), np.float32)
        ep_step, ep_score = np.empty(n, np.int32), np.empty(n, np.float64)
        fn = c_oracle.lib().oc_cartpole_step if self.env_id == "CartPole-v0" else lib().oc_mountaincar_continuous_step
        fn(p(self.state), p(self.rng), p(self.elapsed), p(self.ep_score), p(a), p(self.obs), p(rew), p(term), p(trunc),
           p(reset_obs), p(ep_step), p(ep_score), C.c_int(self.max_steps), C.c_long(n), C.c_int(self.flavour))
        return dict(obs=self.obs.copy(), rew=rew, term=term.astype(bool), trunc=trunc.astype(bool),
                    reset_obs=reset_obs, ep_step=ep_step, ep_score=ep_score, state=self.state.copy())


class MountainCarContinuousStackC(c_oracle.MountainCarStackC):
    """MountainCarContinuous-v0 as the reference's make_envs builds it: c_oracle.MountainCarStackC's 4-frame stack (state
    layout of the device kernel) over the bare continuous env."""

    def __init__(self, env_id, n, seed=1, flavour="cr", n_warm_resets=2, seeds=None):
        self.raw = VecEnvCExt("gym:MountainCarContinuous-v0", n, seed, flavour, n_warm_resets, seeds)
        self.env_id, self.n, self.sdim, self.odim, self.max_steps = env_id, n, 8, 8, self.raw.max_steps
        self.act_dtype = np.float32
        self._refill()


def vec_env_c(env_id, n, **kw):
    """The C oracle's vector env for any id the device runs."""
    if env_id == "MountainCarContinuous-v0":
        return MountainCarContinuousStackC(env_id, n, **kw)
    if env_id in VecEnvCExt.NEW:
        return VecEnvCExt(env_id, n, **kw)
    return c_oracle.VecEnvC(env_id, n, **kw)
