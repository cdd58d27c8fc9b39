"""Vectorised, device-resident PPOCLIP_Agent: the caller of the hot path.

Mirrors PPOCLIP_Agent (xuance/torch/agents/policy_gradient/ppoclip_agent.py:4-165): same constructor
`(config, envs, policy, optimizer, scheduler, device)`, same `train(train_steps)` semantics (train_steps vector
steps; one PPO update phase of n_epoch x n_minibatch SGD steps every n_steps), same hyper-parameter names.

What changes is the shape of the loop, not its arithmetic:
  * one rollout of n_steps vector steps is ONE CUDA graph: per step the whole actor-critic forward in one launch
    (csrc/dense_tc.cu xb_mlp_fwd_from_obs; the torch modules only below FusedActorCritic.MIN_ROWS rows or for
    unsupported policy shapes) and one fused sample + env step + store launch (csrc/env_classic.cu
    rollout_step_kernel), then the bootstrap forward and the batched GAE scan; the reference's O(N) Python loops
    (:71-75, :89-109), per-step D2H copies (:54-56) and list-of-dict infos are gone;
  * truncation bootstraps: the reference runs a full-batch forward per finished env (:99); here every step's
    forward also evaluates V(terminal obs of the previous step) on rows [N, 2N) of the same batch, so the
    values are there for whichever envs were truncated;
  * the update phase is n_epoch graph launches (n_minibatch fused updates each, every kernel hand-written); with
    env-sharded data parallelism the exchanges are kernels of ours over NVLink peer memory inside the same graph
    (csrc/peer_comm.cu); NCCL all-reduces between per-stage graphs are the fallback when CUDA IPC is unavailable.
Env-sharded runs: every rank may be given the SAME config seed — the action-sampling key and the permutation seeds
fold the rank in, so the ranks' rollouts are decorrelated (the envs themselves are all seeded alike, like the
reference's, gym_env.py:18-19, and diverge through their actions).
Index permutations follow the reference (`np.random.shuffle` of a persistent arange, :76-78) when
`config.shuffle == "host"` (copied H2D from pinned memory each epoch), or are drawn on device ("device").

`use_obsnorm` / `use_rewnorm` (SURVEY.md §8 f1) run on device too: RunningMeanStd moments + Chan merge + clip in
csrc/normalize.cu, two extra launches per step each; env-sharded, the per-step moments are exchanged over peer memory so
every rank holds the global statistics.
`train(train_steps)` accepts any step count (ppoclip_agent.py:59-61): whole rollouts replay the captured graph, a
partial rollout runs the same launches eagerly and the buffer position carries over to the next call.
"""
import os
import time

import numpy as np
import torch

from . import _lib, checkpoint, ops
from . import dist as xdist
from .buffer import DummyOnPolicyBuffer
from .learner import PPOCLIP_Learner
from .spaces import is_discrete
from .vec_env import DummyVecEnv_Gym


class HostPermutationFeeder:
    """Host side of the minibatch-index feed: the role of `np.random.shuffle(indexes)` (ppoclip_agent.py:76-78).
    Permutations for rollout k+1 are drawn by worker threads (native xb_host_permutation32, GIL released) into
    pinned int32 staging buffers while the GPU is busy with rollout k; two buffer sets alternate.  32-bit indices halve the
    pinned memory and the H2D bytes (the device widens them to the int64 the gather kernels take)."""

    def __init__(self, n, n_epoch, seed, workers=4):
        from concurrent.futures import ThreadPoolExecutor
        self.n, self.n_epoch, self.seed = n, n_epoch, seed
        self.sets = [[torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(n_epoch)] for _ in range(2)]
        self.pool = ThreadPoolExecutor(max_workers=max(1, workers))
        self.futures = {}
        self.consumed = [None, None]

    def _draw(self, buf, seed):
        _lib.call("xb_host_permutation32", buf.data_ptr(), self.n, seed)
        return buf

    def prefetch(self, iteration):
        if iteration in self.futures:
            return
        ev = self.consumed[iteration & 1]
        if ev is not None:
            ev.synchronize()                                        # the H2D copies that read this set have finished
        self.futures[iteration] = [self.pool.submit(self._draw, self.sets[iteration & 1][ep],
                                                    (self.seed * 1000003 + iteration) * 64 + ep)
                                   for ep in range(self.n_epoch)]

    def get(self, iteration, ep):
        self.prefetch(iteration)
        return self.futures[iteration][ep].result()

    def mark_consumed(self, iteration):
        ev = torch.cuda.Event()
        ev.record()
        self.consumed[iteration & 1] = ev
        self.futures.pop(iteration, None)

    def drain(self):
        """Waits for every outstanding draw and forgets it (before the iteration number changes under the feeder)."""
        for futures in self.futures.values():
            for f in futures:
                f.result()
        self.futures.clear()


def _mix64(x):
    """splitmix64's finaliser: a bijection of 64-bit integers that scatters nearby inputs."""
    m = (1 << 64) - 1
    x = (x + 0x9E3779B97F4A7C15) & m
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & m
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & m
    return x ^ (x >> 31)


def agree_eval_plan(plans):
    """The host check at the start of an env-sharded `test()`: `plans` holds one (device path, env count, env kind, test_episode)
    row per rank.  Returns True when every rank takes the device path with the same env count, env kind and episode target,
    False when no rank takes it (each rank then runs the host loop on its own envs), and raises ValueError otherwise, on every
    rank alike, before any rank reaches a cross-GPU barrier."""
    rows = [tuple(int(v) for v in p) for p in plans]
    device = [r for r, p in enumerate(rows) if p[0]]
    if not device:
        return False
    if len(device) < len(rows):
        raise ValueError("test(): ranks %s would run the device evaluation loop and ranks %s the host loop; every rank must "
                         "pass native device envs of the training env" % (device, [r for r in range(len(rows)) if r not in device]))
    for k, what in ((1, "test env counts"), (2, "env kinds"), (3, "test_episode values")):
        values = [p[k] for p in rows]
        if len(set(values)) > 1:
            raise ValueError("test(): the ranks' %s differ (%s); the env-sharded evaluation needs the same on every rank"
                             % (what, values))
    return True


def order_eval_scores(scores, steps):
    """The scores of an env-sharded evaluation in the order of the reference's loop over the global vector env, whose env
    r * n + e is env e of rank r: by step, then rank, then env.  scores[r] / steps[r]: rank r's episode queue and the step each
    score finished in (already in (step, env) order).  Returns a list of floats."""
    if len(scores) != len(steps) or any(len(a) != len(b) for a, b in zip(scores, steps)):
        raise ValueError("every rank needs one step tag per score")
    for t in steps:
        if np.any(np.diff(np.asarray(t, dtype=np.int64)) < 0):
            raise ValueError("a rank's episode queue is not in step order")
    flat = np.concatenate([np.asarray(s, dtype=np.float64) for s in scores]) if scores else np.zeros(0)
    step = np.concatenate([np.asarray(t, dtype=np.int64) for t in steps]) if steps else np.zeros(0, np.int64)
    rank = np.concatenate([np.full(len(s), r, np.int64) for r, s in enumerate(scores)]) if scores else np.zeros(0, np.int64)
    return flat[np.lexsort((rank, step))].tolist()         # a stable sort: each rank's env order is kept


class DeviceEvaluator:
    """The evaluation loop of `test()` (ppoclip_agent.py:113-165) on the device, for one test-env count N.  It owns the loop's
    state: env physics and RNG streams, the observation the policy acts on, the observation statistics being merged, and the
    episode queue (scores, count, step).  One captured graph runs `chunk` vector steps, each the agent's `_policy_forward` and
    one xb_eval_step launch.  The host replays it and reads the 8-byte queue count after every chunk: one sync per chunk.
    With a peer comm block (`peer`), the N envs are this rank's shard of a global vector env: each step is followed by the
    xb_peer_eval_merge exchange, `count` is the global episode count and the scores, tagged with their steps, go to a local
    queue of `local_count` entries."""

    def __init__(self, agent, envs, cap, chunk, tape_steps=0, peer=None):
        N, dev = envs.num_envs, agent.device
        f64, i64 = dict(dtype=torch.float64, device=dev), dict(dtype=torch.int64, device=dev)
        self.N, self.chunk, self.tape_steps, self.peer = N, chunk, tape_steps, peer
        self.kind, self.max_steps = envs._kind, envs.max_episode_length
        self.state, self.rng = torch.zeros_like(envs._state), torch.zeros_like(envs._rng)
        self.elapsed, self.ep_score = torch.zeros_like(envs._elapsed), torch.zeros_like(envs._ep_score)
        self.x = torch.zeros_like(envs._obs)                            # the observation the policy acts on [N, row]
        self.xn = torch.zeros_like(envs._obs)                           # its normalised form, where the forward needs one
        self.trig_cache = torch.full((3, N), float("nan"), **f64)
        D = envs._obs_row
        self.stats, self.stats_cand = torch.zeros(2 * D + 1, **f64), torch.zeros(2 * D + 1, **f64)
        self.scores = torch.zeros(cap, **f64)
        self.count, self.step, self.key, self.test_episode = (torch.zeros(1, **i64) for _ in range(4))
        ctas = -(-N // 32)                                              # CTAs of the widest launch (32 envs each)
        self.partials, self.workspace = torch.zeros(20 * ctas, **f64), torch.zeros(2 + ctas, **i64)
        self.tape = None
        if tape_steps:                  # test hook: the sampled actions, row = evaluation step
            act_dtype = torch.float32 if ops.continuous_kind(envs._kind) else torch.int64
            self.tape = torch.zeros((tape_steps, N), dtype=act_dtype, device=dev)
        self.local_count = self.score_step = self.record = None
        if peer is not None:
            self.local_count = torch.zeros(1, **i64)
            self.score_step = torch.zeros(cap, dtype=torch.int32, device=dev)
            self.record = torch.zeros(2 * D + 4, **f64)      # this rank's step record: sum x[D], sum x^2[D], N, 0, 0, finishers
            self.totals = torch.zeros(2 * D + 4, **f64)      # the global moments of the first / the latest observations
        self.graph = None

    def load(self, envs, key, test_episode):
        """The reset state of `envs` in, the queue emptied, this evaluation's Philox key and episode target set."""
        for dst, src in ((self.state, envs._state), (self.rng, envs._rng), (self.elapsed, envs._elapsed),
                         (self.ep_score, envs._ep_score), (self.x, envs._obs)):
            dst.copy_(src)
        self.count.zero_()
        self.step.zero_()
        if self.local_count is not None:
            self.local_count.zero_()
        self.key.fill_(key - (1 << 64) if key >= 1 << 63 else key)
        self.test_episode.fill_(test_episode)

    def steps(self, agent, k):
        N = self.N
        stats = self.stats if agent.use_obsnorm else None
        for _ in range(k):
            norm = (stats, stats, N, agent.obsnorm_range) if stats is not None else None
            dist, _ = agent._policy_forward(self.x, norm, xn=self.xn)
            act_param, logstd = agent._act_params(dist, N)
            ops.eval_step(self.kind, act_param, logstd, self.key, self.step, self.state, self.rng, self.elapsed, self.ep_score,
                          self.x, self.trig_cache, self.max_steps, self.scores, self.count, self.test_episode, self.partials,
                          self.workspace, obs_state=stats, obs_state_cand=self.stats_cand if stats is not None else None,
                          obs_dim=agent._obs_dim, act_tape=self.tape, local_count=self.local_count, score_step=self.score_step,
                          record=self.record)
            if self.peer is not None:
                ops.peer_eval_merge(self.peer, self.record, self.totals, self.count, self.test_episode, agent._NORM_INBOX, obs_state=stats,
                                    obs_state_cand=self.stats_cand if stats is not None else None, obs_dim=agent._obs_dim)

    def capture(self, agent):
        """Warm up one step on a side stream (lazy module state, library workspaces), then capture `chunk` steps."""
        s = torch.cuda.Stream(device=agent.device)
        s.wait_stream(torch.cuda.current_stream(agent.device))
        with torch.cuda.stream(s):
            self.steps(agent, 1)
        torch.cuda.current_stream(agent.device).wait_stream(s)
        torch.cuda.synchronize(agent.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.steps(agent, self.chunk)


class PPOCLIP_Agent:
    _mask_terminal_returns = True      # the reward normaliser's return tracker drops the running return on a terminal (:87)
    _bootstrap_truncations = True      # a truncated episode is closed with V(terminal obs) (:96-100); PG / PPG close it with 0
    _track_returns = True              # per-env return tracker + ret_rms.update (:87-92); PPG_Agent has neither
    _graph_updates = True              # the update phase is captured (epoch graphs); False: eager phases through a compat learner
    _aux_shape = {"old_logp": ()}

    def __init__(self, config, envs, policy, optimizer, scheduler=None, device=None, process_group=None):
        self.use_obsnorm = bool(getattr(config, "use_obsnorm", False))
        self.use_rewnorm = bool(getattr(config, "use_rewnorm", False))
        self.obsnorm_range = float(getattr(config, "obsnorm_range", 5))
        self.rewnorm_range = float(getattr(config, "rewnorm_range", 5))
        self.config, self.envs, self.policy = config, envs, policy
        self.device = torch.device(device if device is not None else "cuda")
        self.n_envs, self.n_steps = envs.num_envs, config.n_steps
        self.n_minibatch, self.n_epoch = config.n_minibatch, config.n_epoch
        self.gamma, self.gae_lam = config.gamma, config.gae_lambda
        self.observation_space, self.action_space = envs.observation_space, envs.action_space
        self.discrete = is_discrete(self.action_space)
        self.buffer_size = self.n_envs * self.n_steps
        self.batch_size = self.buffer_size // self.n_minibatch
        self.n_updates_per_epoch = -(-self.buffer_size // self.batch_size)      # incl. the short last minibatch, if any
        self.use_graphs = bool(getattr(config, "use_cuda_graphs", True))
        self.shuffle = getattr(config, "shuffle", "host")
        self.seed = int(getattr(config, "seed", 1))
        # Philox key of the action sampler: the rank is folded in so that ranks given the same config seed draw
        # different actions (otherwise W ranks would compute W bit-identical rollouts)
        self._sample_seed = self.seed + 1000003 * self._rank()
        self.memory = DummyOnPolicyBuffer(self.observation_space, self.action_space, dict(self._aux_shape), self.n_envs,
                                          self.n_steps, config.use_gae, config.use_advnorm, self.gamma, self.gae_lam,
                                          device=self.device, native=True,
                                          gae_variant=getattr(config, "gae_variant", "auto"))
        self.learner = self._make_learner(config, policy, optimizer, scheduler)
        if self._graph_updates:
            self.learner.enable_fused_optimizer(process_group)
        else:                 # eager update phases: the learner exchanges the gradients its torch optimiser steps on
            self.learner.enable_sharding(process_group)
        self.world_size = self.learner.world_size
        if self.world_size > 1:
            if self._graph_updates:       # replicated policy: every rank starts from rank 0's parameters
                xdist.broadcast_parameters(self.learner._flat.flat_param, 0, process_group)
            if self.buffer_size % self.batch_size:
                raise ValueError("env-sharded training needs n_envs * n_steps (%d) divisible by n_minibatch (%d): the ranks' "
                                 "minibatches must be equal for the global-minibatch statistics" % (self.buffer_size, self.n_minibatch))
        N, dev = self.n_envs, self.device
        obs_dim = self.memory.obs_dim
        self._obs_dim = obs_dim
        # ping-pong policy-input buffers: rows [0,N) = obs the policy acts on, rows [N,2N) = terminal obs of the last step
        self._x = [torch.zeros((2 * N, self.memory.obs_row), dtype=torch.float32, device=dev) for _ in range(2)]
        self._cur = 0
        self._act = torch.zeros(N if self.discrete else (N, self.memory.act_dim),
                                dtype=torch.int64 if self.discrete else torch.float32, device=dev)
        self._logp = torch.zeros(N, dtype=torch.float32, device=dev)
        self._boot_last = torch.zeros(N, dtype=torch.float32, device=dev)
        # (theta, sin, cos) of the last observation per env, keyed by theta (NaN = empty): see xb_rollout_step
        self._trig_cache = torch.full((3, N), float("nan"), dtype=torch.float64, device=dev)
        self._ctr = torch.zeros(1, dtype=torch.int64, device=dev)
        self._perm = torch.zeros(self.buffer_size, dtype=torch.int64, device=dev)
        self._perm_ctr = torch.zeros(1, dtype=torch.int64, device=dev)      # one tick per drawn device permutation
        self._mb_stats_all = torch.zeros(2 * max(1, self.buffer_size // self.batch_size), dtype=torch.float64, device=dev)
        self._perm_bufs = [self._perm, torch.zeros_like(self._perm)]        # host shuffle: double-buffered, widened on device
        self._perm32 = None
        self._perm_ready, self._perm_free, self._perm_staged = [None, None], [None, None], False
        self._copy_stream = torch.cuda.Stream(device=dev)
        self._epoch_graphs = None
        self._perm_seed = self.seed * 2654435761 + 7919 * self._rank() + 1
        self._feeder = None
        if self.shuffle == "host":
            import os as _os0
            local_world = int(_os0.environ.get("LOCAL_WORLD_SIZE", "1"))
            auto = max(1, min(self.n_epoch, (_os0.cpu_count() or 4) // max(1, local_world)))   # one epoch's draw per thread
            self._feeder = HostPermutationFeeder(self.buffer_size, self.n_epoch, self.seed + 7919 * self._rank(),
                                                 workers=int(getattr(config, "feeder_threads", auto)))
            self._perm32 = [torch.zeros(self.buffer_size, dtype=torch.int32, device=dev) for _ in range(2)]
            self._feeder.prefetch(0)
        self._iteration = 0
        self._t = 0                        # vector steps already taken in the current (unfinished) rollout
        self.sync_info = bool(getattr(config, "sync_info", True))
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        # device-side RunningMeanStd (statistic_tools.py:35-48: mean 0, var 1, count 1e-4), obs state ping-pongs
        # state layout fp64 [2D + 1] = mean[D], var[D], count with D = floats per observation row (4, or 8 for wide rows)
        f64 = dict(dtype=torch.float64, device=dev)
        D = self.memory.obs_row
        init = torch.tensor([0.0] * D + [1.0] * D + [1e-4], **f64)
        self._obs_rms = [init.clone(), init.clone()]
        self._rms_cur = 0
        self._norm_n = 2 * D + 4          # one step's sums: sum x[D], sum x^2[D], N, sum R, sum R^2, n finished
        self._obs_sums = torch.zeros(9, **f64)
        self._obs_ws = torch.zeros(8 + 8 * 1184, **f64)
        self._xn = torch.zeros((2 * N, D), dtype=torch.float32, device=dev)      # normalised policy input
        self._ret_rms = torch.tensor([0.0, 1.0, 1e-4], **f64)
        self._ret_sums = torch.zeros(3, **f64)
        self._ret_ws = torch.zeros(8 + 8 * 1184, **f64)
        self._returns = torch.zeros(N, dtype=torch.float64, device=dev)
        self._rew_std = torch.ones(1, dtype=torch.float32, device=dev)
        # env-sharded normalisers: the per-step observation moments [2D + 1] and finished-episode return sums [3] are exchanged
        # over peer memory (the analogue of mpi_moments, statistic_tools.py:6-32) so every rank keeps the GLOBAL statistics;
        # they live at the end of the comm block's statistics region (its start carries the per-epoch advantage sums)
        self._norm_peer = self.learner._peer if (self.use_obsnorm or self.use_rewnorm) else None
        if (self.use_obsnorm or self.use_rewnorm) and self.learner.world_size > 1 and self._norm_peer is None:
            raise NotImplementedError("use_obsnorm / use_rewnorm with env sharding need the peer-memory exchange "
                                      "(XB_PEER_COMM=1 and CUDA IPC available)")
        if self._norm_peer is not None:
            self._norm_off = self._norm_peer.stats.numel() - self._norm_n
            self._norm_local = self._norm_peer.stats[self._norm_off:]
            self._norm_local.zero_()
            self._norm_global = torch.zeros(self._norm_n, **f64)
        # one launch per vector step (sample + env step + store) for the two classic-control action shapes
        import os as _os
        self._fused_step = (_os.environ.get("XB_FUSED_STEP", "1") != "0" and
                            ((self.discrete and int(self.action_space.n) == {0: 2, 2: 3, 3: 3, 4: 3}.get(envs._kind, -1)) or
                             (not self.discrete and self.memory.act_dim == 1)))
        # running statistics carried by the fused rollout step (csrc/normalize.cuh StepStats): no moments / normalise /
        # return-tracker launches per step; the rollout forward normalises the raw observations itself.  Env-sharded, the
        # step writes this rank's sums and ONE launch with one cross-GPU barrier exchanges them over peer memory and merges the
        # normalisers (xb_peer_allreduce_merge; every rank keeps the GLOBAL statistics, bit-identical).
        self._fused_norm = (self._fused_step and (self.use_obsnorm or self.use_rewnorm)
                            and _os.environ.get("XB_FUSED_NORM", "1") != "0"
                            and (self.world_size == 1 or self._norm_peer is not None))
        self._shard_norm = self._fused_norm and self.world_size > 1
        self._norm_push = _os.environ.get("XB_NORM_PUSH", "1") != "0"      # one-barrier push exchange + merge in one launch
        if self.use_obsnorm and not self._fused_norm and self.memory.obs_row != 4:
            raise NotImplementedError("observations wider than 4 floats are normalised on the fused rollout path only "
                                      "(XB_FUSED_STEP / XB_FUSED_NORM on)")
        self._stat_partials = torch.zeros(20 * max(148, N // 32 + 2), **f64)
        self._stat_ticket = torch.zeros(1, dtype=torch.int32, device=dev)
        self._zero_v = {}                  # rows -> the zero value vector of an actor-only policy
        self._chain = False
        self._rollout_graph = None
        self._epoch_graph = None
        self._stage_graphs = None
        self.current_step = 0
        self.current_episode = 0
        self.last_info = {}
        # test() on native device envs: DeviceEvaluator of the latest test-env count, vector steps per captured chunk, the
        # number of device evaluations so far (it keys their action sampler) and, for tests, the steps of actions to record
        self._evaluator = None
        self._eval_chunk = 32
        self._eval_index = 0
        self._eval_tape_steps = 0
        # the comm block of the env-sharded device evaluation (None: one rank, the plain device loop)
        self._eval_peer = self.learner._peer if self.world_size > 1 else None
        # first observation: whatever the envs currently hold (Runner_Base calls envs.reset() before the agent, runner_basic.py:12)
        self._x[0][:N].copy_(envs._obs)
        self._x[0][N:].copy_(envs._obs)
        if self._fused_norm and self.use_obsnorm:
            # `obs_rms.update(obs)` for the very first observations (ppoclip_agent.py:62); from here on every fused rollout
            # step merges the moments of the observations it produces
            if self._shard_norm:
                ops.moments4(self._x[0][:N], self._norm_local[:2 * D + 1], self._obs_ws)
                ops.peer_allreduce_f64(self._norm_peer, self._norm_n, self._norm_global, offset=self._norm_off)
                ops.rms_merge_sums(self._norm_global, self._obs_rms[0], self._obs_rms[1], obs_dim, None, None)
                self._norm_local.zero_()
            else:
                ops.rms_update_rows(self._x[0][:N], obs_dim, self._obs_rms[0], self._obs_rms[1], self._stat_partials,
                                    self._stat_ticket)
            self._obs_rms[0].copy_(self._obs_rms[1])

    def _make_learner(self, config, policy, optimizer, scheduler):
        return PPOCLIP_Learner(policy, optimizer, scheduler, self.device, getattr(config, "model_dir", "./"),
                               vf_coef=config.vf_coef, ent_coef=config.ent_coef, clip_range=config.clip_range,
                               clip_grad_norm=config.clip_grad_norm, use_grad_clip=config.use_grad_clip,
                               value_clip=getattr(config, "value_clip", None))

    def _store_extra(self, t, dist):
        """Per-step auxiliaries beyond old_logp (PPG: the old action distribution's parameters)."""

    def _dist_out(self, t):
        """Row t of the old-distribution array when the fused rollout step writes it (PPO-KL), else None."""
        return None

    @staticmethod
    def _rank():
        d = torch.distributed
        return d.get_rank() if (d.is_available() and d.is_initialized()) else 0

    # ---------------------------------------------------------------------------------------------- rollout
    def _policy_forward(self, x, norm=None, xn=None):
        """norm = (state_new, state_old, n_new_rows, clip): `x` holds raw observations (fused-statistics path); the
        one-launch rollout forward normalises them itself, otherwise xb_rms_apply does in front of the MLP, into `xn`
        (default: the rollout's buffer of 2 * n_envs rows)."""
        fused = self.learner._fused
        if fused is not None and x.shape[0] >= fused.MIN_ROWS:     # weights were split at the start of the rollout
            if norm is not None and not fused.fwd_from_obs_ok():
                x, norm = self._apply_norm(x, norm, xn), None
            # (`_chain`: the launch before this forward is a rollout step of this loop, which writes no weights — the
            #  forward's set-up and weight loads may then overlap it: programmatic dependent launch, csrc/common.cuh)
            act_out, v = fused.forward_inference(x[:, :self._obs_dim], norm=norm, weights_stable=self._chain)
            return fused.dist_params(act_out), v
        if norm is not None:
            x = self._apply_norm(x, norm, xn)
        out = self.policy(x[:, :self._obs_dim])       # (outputs, dist, v) | actor-only (outputs, dist) | PPG (outputs, dist, v, aux_v)
        if len(out) < 3:
            # one vector per row count: a captured graph keeps reading the one it was captured with
            zero = self._zero_v.get(x.shape[0])
            if zero is None:
                zero = self._zero_v[x.shape[0]] = torch.zeros(x.shape[0], dtype=torch.float32, device=self.device)
            return out[1], zero
        return out[1], out[2]

    def _apply_norm(self, x, norm, xn=None):
        xn = self._xn if xn is None else xn
        ops.rms_apply(x, self._obs_dim, norm[0], norm[1], norm[2], norm[3], xn)
        return xn

    def _obs_norm_args(self):
        if not self.use_obsnorm:
            return None
        c = self._rms_cur     # rows [0, N): statistics incl. these observations; rows [N, 2N): the step before (agent.py:104-116)
        return (self._obs_rms[c], self._obs_rms[c ^ 1], self.n_envs, self.obsnorm_range)

    def _sample(self, dist, offset):
        N = self.n_envs
        if self.discrete:
            logits = dist.get_param()
            ops.sample_categorical(logits[:N].contiguous(), self._sample_seed, self._ctr, offset, self._act, self._logp)
        else:
            mu, std = dist.get_param()
            logstd = getattr(getattr(self.policy, "actor", None), "logstd", None)   # gaussian.py:25
            logstd = logstd.detach() if logstd is not None else std.log().contiguous()
            ops.sample_gaussian(mu[:N].contiguous(), logstd, self._sample_seed, self._ctr, offset, self._act, self._logp)

    def _act_params(self, dist, N):
        """(action parameters of rows [0, N), log-std) as the fused step kernels take them: logits, or mu and the log-std."""
        prm = dist.get_param()
        if self.discrete:
            return prm[:N], None
        logstd = getattr(getattr(self.policy, "actor", None), "logstd", None)
        return prm[0][:N], (logstd.detach() if logstd is not None else prm[1].log().contiguous())

    _NORM_INBOX = 1024      # doubles [1024, 1280) of the comm block's statistics area (the epoch's advantage sums use [0, 2 M))

    def _rollout_step(self, t):
        """One vector step into buffer row t (reference loop body, ppoclip_agent.py:62-68,88,101)."""
        N, env, mem = self.n_envs, self.envs, self.memory
        x_cur, x_nxt = self._x[self._cur], self._x[self._cur ^ 1]
        if self._fused_norm:
            # (the step kernel folds the moments of the observations it produces into the normaliser: csrc/normalize.cuh.
            # Leaving only per-CTA partial sums and merging them in the forward's prologue was tried and measured slower, 3.11 vs
            # 2.96 ms per C2 rollout: the reduction then sits in front of the forward's first operand tile)
            dist, v = self._policy_forward(x_cur, self._obs_norm_args())
            act_param, logstd = self._act_params(dist, N)
            stats = dict(partials=self._stat_partials, ticket=self._stat_ticket, gamma=self.gamma,
                         mask_terminal=self._mask_terminal_returns)
            if self.use_obsnorm:
                c = self._rms_cur
                stats.update(obs_in=self._obs_rms[c], obs_out=self._obs_rms[c ^ 1], obs_dim=self._obs_dim,
                             obs_clip=self.obsnorm_range)
            if self.use_rewnorm and self._track_returns:
                stats.update(ret_state=self._ret_rms, returns=self._returns)
            if self._shard_norm:
                stats.update(sums_out=self._norm_local)
            if "obs_in" not in stats and "returns" not in stats:
                stats = None
            self._store_extra(t, dist)
            boot = t > 0 and self._bootstrap_truncations
            ops.rollout_step(env._kind, act_param, logstd, v[:N], self._sample_seed, self._ctr, t, env._state, env._rng,
                             env._elapsed, env._ep_score, x_nxt[N:], x_nxt[:N], env._rew, env._term, env._trunc,
                             env._reset_obs, env._ep_step_out, env._ep_score_out, env.ep_stats, env.max_episode_length,
                             x_cur[:N], self._act, self._logp, mem._obs[t], mem._act[t], mem._rew[t], mem._val[t],
                             mem._term[t], mem._trunc[t], mem._logp[t],
                             rew_std=self._rew_std if self.use_rewnorm else None, rew_clip=self.rewnorm_range,
                             boot_src=v[N:] if boot else None, boot_row=mem._boot[t - 1] if boot else None,
                             trig_cache=self._trig_cache, stats=stats, dist_row=self._dist_out(t))
            if self._shard_norm:      # the ranks' sums of this step -> global sums -> merged normalisers (for the next step)
                c = self._rms_cur
                if self._norm_push:
                    # one kernel, one cross-GPU barrier (push into a parity double-buffered inbox), merge included
                    ops.peer_allreduce_merge(self._norm_peer, self._norm_local, self._norm_n, self._norm_global, self._NORM_INBOX,
                                             self._obs_rms[c] if self.use_obsnorm else None,
                                             self._obs_rms[c ^ 1] if self.use_obsnorm else None, self._obs_dim,
                                             self._ret_rms if self.use_rewnorm else None,
                                             self._rew_std if self.use_rewnorm else None)
                else:                 # pull form: two barriers + a separate merge launch
                    ops.peer_allreduce_f64(self._norm_peer, self._norm_n, self._norm_global, offset=self._norm_off)
                    ops.rms_merge_sums(self._norm_global, self._obs_rms[c] if self.use_obsnorm else None,
                                       self._obs_rms[c ^ 1] if self.use_obsnorm else None, self._obs_dim,
                                       self._ret_rms if self.use_rewnorm else None, self._rew_std if self.use_rewnorm else None)
            if self.use_obsnorm:
                self._rms_cur ^= 1
            self._cur ^= 1
            self._chain = True
            return
        if self._norm_peer is not None:
            # sharded: this step's observation moments + the previous step's return sums in ONE exchange, then the global
            # return normaliser is merged before this step's rewards are scaled (same order as the reference, :87-92)
            r = self._norm_n - 3              # the return sums follow the 2D + 1 observation moments
            if self.use_obsnorm:
                ops.moments4(x_cur[:N], self._norm_local[:r], self._obs_ws)
            ops.peer_allreduce_f64(self._norm_peer, self._norm_n, self._norm_global, offset=self._norm_off)
            if self.use_rewnorm:
                ops.rms_merge_scalar(self._norm_global[r:], self._ret_rms, self._rew_std)
        x_in = self._normalize_obs(x_cur, update=True)            # obs_rms.update(obs); _process_observation (:63-64)
        dist, v = self._policy_forward(x_in)                      # V on [obs_t ; terminal obs of step t-1]
        boot = t > 0 and self._bootstrap_truncations
        if boot and not self._fused_step:
            mem._boot[t - 1].copy_(v[N:])                         # bootstrap for envs truncated at step t-1 (:99)
        self._store_extra(t, dist)
        if self._fused_step:
            # sample + env step + store in one launch (csrc/env_classic.cu: rollout_step_kernel)
            act_param, logstd = self._act_params(dist, N)
            ops.rollout_step(env._kind, act_param, logstd, v[:N], self._sample_seed, self._ctr, t, env._state, env._rng,
                             env._elapsed, env._ep_score, x_nxt[N:], x_nxt[:N], env._rew, env._term, env._trunc,
                             env._reset_obs, env._ep_step_out, env._ep_score_out, env.ep_stats, env.max_episode_length,
                             x_in[:N], self._act, self._logp, mem._obs[t], mem._act[t], mem._rew[t], mem._val[t],
                             mem._term[t], mem._trunc[t], mem._logp[t],
                             rew_std=self._rew_std if self.use_rewnorm else None, rew_clip=self.rewnorm_range,
                             boot_src=v[N:] if boot else None, boot_row=mem._boot[t - 1] if boot else None,
                             trig_cache=self._trig_cache, dist_row=self._dist_out(t))
        else:
            self._sample(dist, t)
            ops.env_step(env._kind, env._state, env._rng, env._elapsed, env._ep_score, self._act.reshape(N),
                         x_nxt[N:], x_nxt[:N], env._rew, env._term, env._trunc, env._reset_obs, env._ep_step_out,
                         env._ep_score_out, env.max_episode_length, ep_stats=env.ep_stats)
            mem.store_device(x_in[:N], self._act, env._rew, v[:N].contiguous(), env._term, env._trunc, self._logp, t,
                             rew_std=self._rew_std if self.use_rewnorm else None, rew_clip=self.rewnorm_range)
        if self.use_rewnorm and self._track_returns:              # returns tracker + ret_rms.update (:87,:91-92)
            if self._norm_peer is not None:      # merged globally at the start of the next step (see above)
                ops.returns_track(self._returns, env._rew, env._term, env._trunc, self.gamma, self._norm_local[self._norm_n - 3:], self._ret_ws,
                                  mask_terminal=self._mask_terminal_returns)
            else:
                ops.returns_track(self._returns, env._rew, env._term, env._trunc, self.gamma, self._ret_sums, self._ret_ws,
                                  mask_terminal=self._mask_terminal_returns)
                ops.rms_merge_scalar(self._ret_sums, self._ret_rms, self._rew_std)
        self._cur ^= 1
        self._chain = True            # (nothing in this loop writes weights)

    def _normalize_obs(self, x, update):
        """rows [0,N): the observations the agent acts on — merged into obs_rms first when `update`; rows [N,2N): the
        previous step's terminal observations, normalised with the statistics of that step (agent.py:104-116)."""
        if not self.use_obsnorm:
            return x
        N = self.n_envs
        s_in, s_out = self._obs_rms[self._rms_cur], self._obs_rms[self._rms_cur ^ 1]
        sums = self._obs_sums
        if update and self._norm_peer is not None:
            sums = self._norm_global[:self._norm_n - 3]     # global moments, exchanged by _rollout_step
        elif update:
            ops.moments4(x[:N], self._obs_sums, self._obs_ws)
        ops.rms_normalize(x, self._obs_dim, sums, s_in, s_out, self.obsnorm_range, self._xn, N if update else 0)
        self._rms_cur ^= 1
        return self._xn

    def _rollout_begin(self):
        self._chain = False
        if self.learner._fused is not None:
            self.learner._fused.refresh_weights()

    def _rollout_end(self):
        """The bootstrap forward (:70), the batched GAE for every env and segment (:71-75), counter / ping-pong upkeep."""
        self._close_paths()
        self._rollout_upkeep()

    def _close_paths(self):
        N = self.n_envs
        if self._fused_norm:      # terminal observations of the last step, normalised with that step's statistics
            _, v = self._policy_forward(self._x[self._cur], self._obs_norm_args())
        else:
            _, v = self._policy_forward(self._normalize_obs(self._x[self._cur], update=False))
        self._boot_last.copy_(v[N:])
        self.memory.finish_rollout(self._boot_last)

    def _rollout_upkeep(self):
        self._chain = False
        ops.counter_add(self._ctr, self.n_steps)
        if self.n_steps % 2:   # keep the ping-pong phase identical for every replay of the captured graph
            self._x[self._cur ^ 1].copy_(self._x[self._cur])
            self._cur ^= 1
        if self._rms_cur:      # same for the normaliser state (n_steps + 1 publications per rollout)
            self._obs_rms[0].copy_(self._obs_rms[1])
            self._rms_cur = 0

    def _rollout(self):
        """n_steps vector steps, the bootstrap forward and the GAE scan: the body of the captured rollout graph."""
        with torch.no_grad():
            self._rollout_begin()
            for t in range(self.n_steps):
                self._rollout_step(t)
            self._rollout_end()

    # ---------------------------------------------------------------------------------------------- update phase
    def _device_permutation(self):
        """np.random.shuffle(indexes) (ppoclip_agent.py:76-78) as one launch: a keyed bijection of [0, buffer_size)
        (csrc/sample.cu: random_permutation_kernel); the device counter makes every graph replay draw a new one."""
        ops.random_permutation(self._perm, self._perm_seed, self._perm_ctr, 0)
        ops.counter_add(self._perm_ctr, 1)

    def _epoch_start(self):
        """Called at the top of every (captured) epoch / first-minibatch stage.  The tf32 hi/lo operand copies of the
        hidden-layer weights are only known to be current if the optimiser launch re-splits them (adam_apply_split);
        on every other path the first minibatch of the epoch re-splits unconditionally — the `splits_fresh` flag is
        Python state evaluated at capture time and must not leak from the capture of the rollout graph."""
        fused = self.learner._fused
        if fused is not None and not self.learner.adam_resplits():
            fused.splits_fresh = False

    def _epoch_body(self, perm=None):
        B = self.batch_size
        self._epoch_start()
        if self.shuffle != "host":
            self._device_permutation()
        perm = self._perm if perm is None else perm
        # like the reference (`range(0, buffer_size, batch_size)`, ppoclip_agent.py:79-83): when buffer_size is not a
        # multiple of n_minibatch the last, short minibatch is trained on too
        for start in range(0, self.buffer_size, B):
            idx = perm[start:start + B]
            mb = self.learner.stage_gather(self.memory, idx)
            self.learner.stage_forward_backward(self.memory, idx, mb)
            self.learner.stage_optimizer()

    def _epoch_peer(self, perm=None):
        """Env-sharded epoch over NVLink peer memory — no NCCL call, so the whole epoch is ONE captured graph:
        the (sum adv, sum adv^2) of all minibatches of the epoch are computed in one pass and exchanged once
        (global-minibatch advantage normalisation, memory_tools.py:241-242), and every update's gradient exchange is
        fused into the first optimiser kernel (csrc/peer_comm.cu)."""
        B, lr, mem, peer = self.batch_size, self.learner, self.memory, self.learner._peer
        M = self.buffer_size // B
        self._epoch_start()
        if self.shuffle != "host":
            self._device_permutation()
        perm = self._perm if perm is None else perm
        if mem.use_advnorm:
            if mem.packed and lr.value_clip <= 0:
                adv, stride = mem._rec.view(-1)[6:], 8          # adv lane of the packed 32-byte records
            else:
                adv, stride = mem._adv, 1
            ops.adv_stats_minibatches(perm, M, B, mem.n_size, mem.n_envs, adv, stride, peer.stats)
            ops.peer_allreduce_f64(peer, 2 * M, self._mb_stats_all)
        for k, start in enumerate(range(0, self.buffer_size - B + 1, B)):
            idx = perm[start:start + B]
            mb = lr.stage_gather(mem, idx, compute_stats=False)
            lr.stage_forward_backward(mem, idx, mb, stats=self._mb_stats_all[2 * k:2 * k + 2])
            lr.stage_optimizer()

    def _epoch_distributed(self):
        """Env-sharded data parallel epoch: every rank updates on its local minibatch; the only exchanges are the
        two-scalar advantage statistics and the flat gradient (SURVEY.md §8(e)), between (graph) stages."""
        if self.learner._peer is not None:
            return self._epoch_peer()
        B, lr, mem = self.batch_size, self.learner, self.memory
        if self._stage_graphs is None:
            self._epoch_start()
        for k, start in enumerate(range(0, self.buffer_size - B + 1, B)):
            idx = self._perm[start:start + B]
            g = self._stage_graphs[k] if self._stage_graphs is not None else None
            if g is not None:
                g[0].replay()
                mb = lr._mb[(B, mem.obs_dim)]
            else:
                mb = lr.stage_gather(mem, idx)
            if mem.use_advnorm:
                xdist.allreduce_adv_stats(mb["stats"], lr.process_group)
            if g is not None:
                g[1].replay()
            else:
                lr.stage_forward_backward(mem, idx, mb)
            lr.allreduce_grads()
            if g is not None:
                g[2].replay()
            else:
                lr.stage_optimizer()

    def _stage_host_perm(self, ep):
        """H2D copy of epoch `ep`'s host-drawn permutation into device buffer ep & 1 on the copy stream, so it overlaps
        the previous epoch's graph (which reads the other buffer)."""
        k = ep & 1
        src = self._feeder.get(self._iteration, ep)
        cs = self._copy_stream
        if self._perm_free[k] is not None:
            cs.wait_event(self._perm_free[k])                      # the epoch that last read this buffer has finished
        with torch.cuda.stream(cs):
            self._perm32[k].copy_(src, non_blocking=True)          # int32 from pinned memory
            self._perm_bufs[k].copy_(self._perm32[k])              # widened on the device (copy stream)
            ev = torch.cuda.Event()
            ev.record(cs)
        self._perm_ready[k] = ev
        self.h2d_bytes += src.numel() * 4

    def _update_phase_overlapped(self):
        """Host-shuffle update phase with double-buffered permutations: two captured epoch graphs, one per buffer."""
        main = torch.cuda.current_stream(self.device)
        if not self._perm_staged:
            self._stage_host_perm(0)
        self._perm_staged = False
        self._feeder.prefetch(self._iteration + 1)
        for ep in range(self.n_epoch):
            if ep + 1 < self.n_epoch:
                self._stage_host_perm(ep + 1)
            k = ep & 1
            main.wait_event(self._perm_ready[k])
            self._epoch_graphs[k].replay()
            ev = torch.cuda.Event()
            ev.record(main)
            self._perm_free[k] = ev
        self._feeder.mark_consumed(self._iteration)
        self.learner.iterations += self.n_epoch * self.n_updates_per_epoch
        self._iteration += 1

    def _update_phase(self):
        if self._epoch_graphs is not None:
            return self._update_phase_overlapped()
        n_updates = self.n_epoch * self.n_updates_per_epoch
        if self.shuffle == "host":
            self._feeder.prefetch(self._iteration + 1)             # next rollout's permutations, drawn while the GPU works
        for ep in range(self.n_epoch):
            if self.shuffle == "host":
                src = self._feeder.get(self._iteration, ep)
                self._perm32[0].copy_(src, non_blocking=True)      # H2D from pinned memory (int32), widened on the device
                self._perm.copy_(self._perm32[0])
                self.h2d_bytes += src.numel() * 4
            elif self.world_size > 1 and self.learner._peer is None:   # otherwise drawn inside the epoch graph
                self._device_permutation()
            if self._epoch_graph is not None:
                self._epoch_graph.replay()
            elif self.world_size > 1:
                self._epoch_distributed()
            else:
                self._epoch_body()
        if self.shuffle == "host":
            self._feeder.mark_consumed(self._iteration)
        self.learner.iterations += n_updates
        self._iteration += 1

    # ---------------------------------------------------------------------------------------------- graphs
    def _capture(self):
        """Warm up eagerly on a side stream (cuBLAS workspaces, autograd, lazy module state), then capture."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        snap = self._snapshot()
        with torch.cuda.stream(s):
            self._rollout()
            if not self._graph_updates:
                pass
            elif self.shuffle == "host" or (self.world_size > 1 and self.learner._peer is None):
                self._device_permutation()                 # a valid permutation for the warm-up epoch
            if not self._graph_updates:
                pass
            elif self.world_size > 1:
                self._epoch_distributed()
            else:
                self._epoch_body()
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        self._restore(snap)
        self._rollout_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._rollout_graph):
            self._rollout()
        if not self._graph_updates:        # the update phases run eagerly through the learner's own methods
            torch.cuda.synchronize(self.device)
            self._restore(snap)
            return
        peer = self.learner._peer is not None
        epoch = self._epoch_peer if peer else self._epoch_body
        if (self.world_size == 1 or peer) and self.shuffle == "host":
            # one epoch graph per permutation buffer: the H2D copy of the next permutation overlaps the running epoch
            self._epoch_graphs = []
            for k in range(2):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    epoch(self._perm_bufs[k])
                self._epoch_graphs.append(g)
        elif self.world_size == 1:
            self._epoch_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._epoch_graph):
                self._epoch_body()
        elif self.learner._peer is not None:
            self._epoch_graph = torch.cuda.CUDAGraph()      # peer-memory exchange: plain kernels, one graph per epoch
            with torch.cuda.graph(self._epoch_graph):
                self._epoch_peer()
        elif self._capture_distributed_epoch():
            pass          # one graph per epoch with the NCCL all-reduces inside it
        else:
            B, lr, mem = self.batch_size, self.learner, self.memory
            graphs = []
            for start in range(0, self.buffer_size - B + 1, B):
                idx = self._perm[start:start + B]
                if start == 0:
                    self._epoch_start()
                ga, gb, gc = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with torch.cuda.graph(ga):
                    mb = lr.stage_gather(mem, idx)
                with torch.cuda.graph(gb):
                    lr.stage_forward_backward(mem, idx, mb)
                with torch.cuda.graph(gc):
                    lr.stage_optimizer()
                graphs.append((ga, gb, gc))
            self._stage_graphs = graphs
        torch.cuda.synchronize(self.device)
        self._restore(snap)   # capture does not execute, but keep the state exactly as before either way

    def _capture_distributed_epoch(self):
        """Env-sharded epoch as ONE CUDA graph: NCCL collectives are graph-capturable, so the two all-reduces of every
        update are recorded between the kernels instead of being launched from the host (5 host launches per update
        otherwise).  Returns False (and leaves the per-stage graphs to be captured) if the capture is refused."""
        import os
        # opt-in: +3 % at 2 GPUs (65.2 M vs 63.1 M env-steps/s at C2), but the small-batch 2-rank test hung once with the
        # collectives inside the graph, so the per-stage graphs with host-launched all-reduces stay the default
        if os.environ.get("XB_DIST_EPOCH_GRAPH", "0") != "1":
            return False
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._epoch_distributed_eager()
            self._epoch_graph = g
            return True
        except Exception as e:        # pragma: no cover - depends on the NCCL / driver combination
            import warnings
            warnings.warn("distributed epoch graph capture failed (%s); using per-stage graphs" % (e,))
            self._epoch_graph = None
            torch.cuda.synchronize(self.device)
            return False

    def _epoch_distributed_eager(self):
        B, lr, mem = self.batch_size, self.learner, self.memory
        self._epoch_start()
        for start in range(0, self.buffer_size - B + 1, B):
            idx = self._perm[start:start + B]
            mb = lr.stage_gather(mem, idx)
            if mem.use_advnorm:
                xdist.allreduce_adv_stats(mb["stats"], lr.process_group)
            lr.stage_forward_backward(mem, idx, mb)
            lr.allreduce_grads()
            lr.stage_optimizer()

    def _state_tensors(self):
        """The device tensors of the training state, by name: everything a rollout or an update phase carries forward.
        Graph capture snapshots and restores them around its warm-up (_snapshot); checkpoints save them with the buffer
        rows and host counters on top (_checkpoint_tensors, _host_state).  Left out because nothing reads them before
        rewriting them: scratch (statistics partials, tickets, workspaces, minibatch buffers), the trig cache (results do
        not depend on it), the tf32 operand copies and the folded head (derived from the weights), peer comm blocks."""
        env = self.envs
        named = {"env.state": env._state, "env.rng": env._rng, "env.elapsed": env._elapsed, "env.ep_score": env._ep_score,
                 "env.ep_stats": env.ep_stats, "ctr": self._ctr, "perm_ctr": self._perm_ctr, "x0": self._x[0], "x1": self._x[1],
                 "obs_rms0": self._obs_rms[0], "obs_rms1": self._obs_rms[1], "ret_rms": self._ret_rms,
                 "returns": self._returns, "rew_std": self._rew_std}
        if self._norm_peer is not None:
            named["norm_local"] = self._norm_local      # pending return sums of the last step (merged at the next step)
        named.update(self.learner.state_tensors())
        return named

    def _snapshot(self):
        """Everything a warm-up rollout/update mutates, so that capturing leaves training state untouched."""
        return [(t, t.clone()) for t in self._state_tensors().values()] + [("cur", self._cur)]

    def _restore(self, snap):
        for t, c in snap:
            if isinstance(t, str):
                self._cur = c
            else:
                t.copy_(c)

    # ---------------------------------------------------------------------------------------------- checkpoints
    def _checkpoint_tensors(self, t):
        """_state_tensors plus rows [0, t) of every per-step array the rollout writes: the part of an unfinished rollout
        that is already in the buffer (at a rollout boundary, t = 0, the next rollout overwrites every row)."""
        named = self._state_tensors()
        if t > 0:
            mem = self.memory
            for n in ("_obs", "_act", "_rew", "_val", "_term", "_trunc", "_logp", "_boot", "_dist"):
                if getattr(mem, n) is not None:
                    named["buffer." + n[1:]] = getattr(mem, n)[:t]
        return named

    def _host_state(self):
        mem = self.memory
        return {"t": self._t, "cur": self._cur, "rms_cur": self._rms_cur, "iteration": self._iteration,
                "current_step": self.current_step, "current_episode": self.current_episode, "memory_ptr": mem.ptr,
                "memory_size": mem.size, "last_info": self.last_info, "learner": self.learner.host_state(),
                "eval_index": self._eval_index}

    def _load_host_state(self, st):
        self._t, self._cur, self._rms_cur, self._iteration = st["t"], st["cur"], st["rms_cur"], st["iteration"]
        self.current_step, self.current_episode = st["current_step"], st["current_episode"]
        self.memory.ptr, self.memory.size = st["memory_ptr"], st["memory_size"]
        self.last_info = st["last_info"]
        self.learner.load_host_state(st["learner"])
        self._eval_index = st.get("eval_index", 0)        # absent from checkpoints written before device evaluation

    def _checkpoint_meta(self):
        return {"format_version": checkpoint.FORMAT_VERSION, "agent_class": type(self).__name__, "env_id": self.envs.env_id,
                "n_envs": self.n_envs, "n_steps": self.n_steps, "obs_row": self.memory.obs_row, "world_size": self.world_size,
                "rank": self._rank(), "params": [(n, list(p.shape)) for n, p in self.policy.named_parameters()],
                "config": checkpoint.plain_config(self.config)}

    def _rebuild_derived(self):
        """The tf32 hi/lo operand copies and the folded Discrete(3) head follow the weights; a rollout resumed part-way runs
        its forwards without the refresh at the rollout's start, so they are rebuilt from the loaded weights here."""
        if self.learner._fused is not None:
            self.learner._fused.refresh_weights()

    def save_checkpoint(self, path):
        """Writes the full training state into the directory `path`, one file per rank (`rank<r>-of-<W>.pt`): env physics
        and RNG streams, sampling and permutation counters, observation ping-pong, normalisers, optimiser state, the
        buffer rows of an unfinished rollout and the host counters.  A fresh agent built with the same config continues
        from it with `load_checkpoint` as if the run had never stopped.  Call it between `train()` calls (mid-rollout
        included).  Each file is written under a temporary name and moved into place, so a save that is cut off leaves
        the previous checkpoint.  Env-sharded, every rank calls it; they pass one barrier after writing."""
        with torch.cuda.device(self.device):
            tensors = {k: v.detach().to("cpu", copy=True) for k, v in self._checkpoint_tensors(self._t).items()}
        payload = {"meta": self._checkpoint_meta(), "tensors": tensors, "host": checkpoint.to_cpu(self._host_state())}
        os.makedirs(path, exist_ok=True)
        checkpoint.write_atomic(payload, checkpoint.rank_file(path, self._rank(), self.world_size))
        if self.world_size > 1:
            torch.distributed.barrier(group=self.learner.process_group)

    def load_checkpoint(self, path):
        """Restores what `save_checkpoint` wrote.  Refuses with a ValueError naming the field, before anything is copied,
        when the checkpoint belongs to another agent class, env, env count, horizon, world size or rank, another policy
        shape, or another config (keys that only name places or logging, checkpoint.PLACE_KEYS, may differ).  Every tensor
        is copied in place, so CUDA graphs the agent has already captured stay valid.  Env-sharded, every rank calls it;
        the replicated tensors (parameters, optimiser state, normalisers) must be bit-identical across the ranks' files."""
        rank, world = self._rank(), self.world_size
        err = None
        try:
            payload = checkpoint.read(path, rank, world)
            checkpoint.check_compatible(payload["meta"], self._checkpoint_meta())
            t = payload["host"]["t"]
            if not 0 <= t < self.n_steps:
                raise ValueError("checkpoint t (steps into the rollout) is %r, outside [0, %d)" % (t, self.n_steps))
            live = self._checkpoint_tensors(t)
            checkpoint.check_tensors(payload["tensors"], live)
        except (ValueError, FileNotFoundError) as e:
            err = e
        if world > 1:          # every rank refuses together, or none does
            group = self.learner.process_group
            bad = torch.tensor([int(err is not None)], dtype=torch.int32, device=self.device)
            torch.distributed.all_reduce(bad, group=group)
            if err is None and int(bad.item()):
                err = ValueError("checkpoint refused on another rank")
            if err is None:
                differ = checkpoint.differing_across_ranks(checkpoint.replicated(payload), self.device, group)
                if differ:
                    err = ValueError("checkpoint replicated tensors differ across the ranks' files: %s" % ", ".join(differ))
        if err is not None:
            raise err
        with torch.cuda.device(self.device), torch.no_grad():
            if self._feeder is not None:     # outstanding draws write pinned sets that the new iteration may reuse
                self._feeder.drain()
            for k, v in live.items():
                v.copy_(payload["tensors"][k])
            self._trig_cache.fill_(float("nan"))
            self._load_host_state(payload["host"])
            self._perm_staged = False
            self._rebuild_derived()
            torch.cuda.synchronize(self.device)
            if self._feeder is not None:
                self._feeder.prefetch(self._iteration)

    def save_model(self, model_name):
        """The reference's Agent.save_model: the policy's state_dict (learner.save_model) into
        `<config.model_dir>/seed_<seed>_<time>/<model_name>` (one directory per agent, the layout learner.load_model
        searches), and with `use_obsnorm` the observation statistics as `obs_rms.npy` beside it.  Weights only: a run is
        resumed from save_checkpoint.  Env-sharded, rank 0 writes (policy and statistics are replicated)."""
        if self._rank() != 0:
            return
        if getattr(self, "_model_dir_save", None) is None:
            stamp = time.asctime().replace(" ", "").replace(":", "_")
            self._model_dir_save = os.path.join(getattr(self.config, "model_dir", "./"), "seed_%d_%s" % (self.seed, stamp))
        os.makedirs(self._model_dir_save, exist_ok=True)
        self.learner.save_model(os.path.join(self._model_dir_save, model_name))
        if self.use_obsnorm:
            st, D, od = self._obs_rms[self._rms_cur].cpu().numpy(), self.memory.obs_row, self._obs_dim
            np.save(os.path.join(self._model_dir_save, "obs_rms.npy"),
                    {"count": float(st[2 * D]), "mean": st[:od].copy(), "var": st[D:D + od].copy()})

    def load_model(self, path, seed=1):
        """The reference's Agent.load_model: the newest policy file of the `seed_<seed>` directory under `path`, and with
        `use_obsnorm` its `obs_rms.npy` into both observation-statistics slots.  Returns the directory it read."""
        path = self.learner.load_model(path, seed)
        with torch.cuda.device(self.device):
            self._rebuild_derived()
            if self.use_obsnorm:
                f = os.path.join(path, "obs_rms.npy")
                if not os.path.exists(f):
                    raise RuntimeError("Failed to load observation status file 'obs_rms.npy' from %s!" % f)
                stat = np.load(f, allow_pickle=True).item()
                D, od = self.memory.obs_row, self._obs_dim
                for st in self._obs_rms:
                    st[:od].copy_(torch.from_numpy(np.asarray(stat["mean"], np.float64).reshape(od)))
                    st[D:D + od].copy_(torch.from_numpy(np.asarray(stat["var"], np.float64).reshape(od)))
                    st[2 * D].fill_(float(stat["count"]))
        return path

    # ---------------------------------------------------------------------------------------------- public API
    def train(self, train_steps):
        """train_steps vector steps (reference: `for _ in tqdm(range(train_steps))`, ppoclip_agent.py:59-61); a PPO update
        phase every time the buffer fills (every n_steps of them, counted across calls like the reference's `memory.ptr`).
        Whole rollouts replay the captured graph; a partial rollout (train_steps not a multiple of n_steps, or a call that
        starts mid-rollout) issues the same launches eagerly.  Returns the log dict of the last update phase (also kept in
        `self.last_info`)."""
        remaining = int(train_steps)
        with torch.cuda.device(self.device):
            while remaining > 0:
                if self._t == 0 and remaining >= self.n_steps:
                    if self.use_graphs and self._rollout_graph is None:
                        self._capture()            # only ever at a rollout boundary: the warm-up rollout overwrites the buffer
                    if self._epoch_graphs is not None and not self._perm_staged:
                        self._stage_host_perm(0)                   # first permutation travels while the rollout runs
                        self._perm_staged = True
                    if self._rollout_graph is not None:
                        self._rollout_graph.replay()
                    else:
                        self._rollout()
                    remaining -= self.n_steps
                else:                                              # partial rollout: the same launches, eagerly
                    k = min(remaining, self.n_steps - self._t)
                    with torch.no_grad():
                        self._chain = False
                        if self._t == 0:
                            self._rollout_begin()
                        for t in range(self._t, self._t + k):
                            self._rollout_step(t)
                        self._t += k
                        remaining -= k
                        self.memory.ptr = self.memory.size = self._t
                        if self._t < self.n_steps:
                            break
                        self._rollout_end()
                self._t = 0
                self.memory.ptr, self.memory.size = 0, self.n_steps
                self._update_phase()
                self.memory.clear_fast()
                self.current_step += self.n_envs * self.n_steps
                if self.sync_info:
                    self.last_info = self._collect_info()
            if not self.sync_info:
                self.last_info = self._collect_info()
        return self.last_info

    def _collect_info(self):
        """One host sync per rollout: learner scalars + episode totals (reference logs at :84,:102-109)."""
        last_mb = self.buffer_size - (self.n_updates_per_epoch - 1) * self.batch_size   # size of the last minibatch trained on
        info = self.learner.info(last_mb)
        if self.learner._peer is not None:
            self.learner._peer.check()
        st = self.envs.ep_stats.cpu().numpy()
        self.d2h_bytes += 8 * 8 + 3 * 8 + 4 + 8
        n_ep = int(st[0]) - self.current_episode
        info["episodes"] = int(st[0])
        self.current_episode = int(st[0])
        info["new_episodes"] = n_ep
        info["mean_episode_score"] = float(st[1] / st[0]) if st[0] > 0 else float("nan")
        info["mean_episode_steps"] = float(st[2] / st[0]) if st[0] > 0 else float("nan")
        return info

    def _test_observation(self, obs):
        """`self.obs_rms.update(obs); obs = self._process_observation(obs)` of the reference's test loop
        (ppoclip_agent.py:126-127): evaluation observations are merged into the running statistics too."""
        if not self.use_obsnorm:
            return obs
        od, st = self._obs_dim, self._obs_rms[self._rms_cur]
        half = (st.numel() - 1) // 2
        x = obs[:, :od].double()
        n = x.shape[0]
        mean, var, cnt = st[:od], st[half:half + od], st[2 * half]
        delta, tot = x.mean(0) - mean, cnt + n
        m2 = var * cnt + x.var(0, unbiased=False) * n + delta * delta * cnt * n / tot
        mean.add_(delta * n / tot)
        var.copy_(m2 / tot)
        st[2 * half] = tot
        return torch.clamp((x - mean) / (var.sqrt() + 1e-8), -self.obsnorm_range, self.obsnorm_range).float()

    def test(self, env_fn, test_episode):
        """Evaluation episodes on fresh envs (reference :113-165): stochastic actions, scores of finished episodes, in (step,
        env index) order; the loop stops at the first step after which there are at least `test_episode` of them.  With
        `use_obsnorm`, every observation the policy acts on is merged into the observation statistics first.
        Native device envs of the training env on this device run the loop on the device (_test_device).  Env-sharded, every
        rank calls test() together and `env_fn()` returns the rank's shard of the test envs: the W ranks' envs form one vector
        env (env r * n + e = env e of rank r), the stop rule counts the episodes of all ranks, the statistics merge the
        observations of all ranks, and every rank returns the same scores in (step, rank, env) order; this needs the peer
        memory exchange (`_eval_peer`).  Any other envs (compat numpy envs, other vec envs, no peer memory) run the loop on the
        host, each rank on its own envs."""
        envs = env_fn()
        obs, _ = envs.reset()
        index = lambda d: d.index if d.index is not None else torch.cuda.current_device()
        device = (isinstance(envs, DummyVecEnv_Gym) and envs.native and index(envs.device) == index(self.device)
                  and envs._kind == self.envs._kind and (self.world_size == 1 or self._eval_peer is not None))
        if self.world_size > 1:
            plan = torch.tensor([int(device), envs.num_envs if device else 0, envs._kind if device else -1, int(test_episode)],
                                dtype=torch.int64, device=self.device)
            plans = torch.empty((self.world_size, 4), dtype=torch.int64, device=self.device)
            torch.distributed.all_gather_into_tensor(plans, plan, group=self.learner.process_group)
            try:
                device = agree_eval_plan(plans.cpu().tolist())
            except ValueError:
                envs.close()
                raise
        if device:
            return self._test_device(envs, int(test_episode))
        scores = []
        with torch.no_grad(), torch.cuda.device(self.device):
            while len(scores) < test_episode:
                obs = obs if torch.is_tensor(obs) else torch.as_tensor(obs, device=self.device)
                dist = self.policy(self._test_observation(obs))[1]
                acts = dist.stochastic_sample()
                obs, _, term, trunc, infos = envs.step(acts if envs.native else acts.cpu().numpy())
                done = (term | trunc)
                done = done.cpu().numpy() if torch.is_tensor(done) else done
                for i in np.nonzero(done)[0]:
                    scores.append(infos[int(i)]["episode_score"])
                if envs.native:
                    obs = infos.next_obs
                else:
                    for i in np.nonzero(done)[0]:
                        obs[i] = infos[int(i)]["reset_obs"]
        envs.close()
        return scores

    def _test_device(self, envs, test_episode):
        """test() on the device: the reset state of `envs` is copied into the DeviceEvaluator of this env count, the first
        observations are merged into the statistics, and chunks of captured steps run until the episode queue holds
        `test_episode` scores.  The Philox key of the sampler derives from (seed, evaluation index), not from the training
        sampler's key or counter; the only training state that changes is the current observation statistics."""
        if test_episode <= 0:
            envs.close()
            return []
        N, peer = envs.num_envs, self._eval_peer
        with torch.no_grad(), torch.cuda.device(self.device):
            ev = self._evaluator
            if (ev is None or ev.N != N or ev.scores.numel() < test_episode + N - 1 or ev.chunk != self._eval_chunk
                    or ev.tape_steps != self._eval_tape_steps or ev.peer is not peer):
                self._evaluator = None           # (its graph and buffers go before the new ones are made)
                ev = self._evaluator = DeviceEvaluator(self, envs, test_episode + N - 1, self._eval_chunk, self._eval_tape_steps,
                                                       peer)
            key = _mix64((self._sample_seed & ((1 << 64) - 1)) ^ _mix64(0xE7A1 + self._eval_index))
            self._chain = False
            if self.learner._fused is not None:
                self.learner._fused.refresh_weights()        # tf32 operand copies of the current weights
            if self.use_graphs and ev.graph is None:
                ev.load(envs, key, test_episode)
                ev.capture(self)
            ev.load(envs, key, test_episode)
            envs.close()
            if self.use_obsnorm and peer is None:           # `obs_rms.update(obs)` of the first loop iteration
                ops.rms_update_rows(ev.x, self._obs_dim, self._obs_rms[self._rms_cur], ev.stats, self._stat_partials,
                                    self._stat_ticket)
            elif self.use_obsnorm:         # ... over the observations of every rank (the exchange of __init__)
                m = 2 * self.memory.obs_row + 1
                off = peer.stats.numel() - ev.record.numel()
                ops.moments4(ev.x, peer.stats[off:off + m], self._obs_ws)
                ops.peer_allreduce_f64(peer, m, ev.totals[:m], offset=off)
                ops.rms_merge_sums(ev.totals, self._obs_rms[self._rms_cur], ev.stats, self._obs_dim, None, None)
            while True:
                if ev.graph is not None:
                    ev.graph.replay()
                else:
                    ev.steps(self, ev.chunk)
                count = int(ev.count.item())
                if peer is not None:
                    peer.check()
                if count >= test_episode:
                    break
            scores = ev.scores[:count].tolist() if peer is None else self._gather_eval_scores(ev, test_episode + N - 1, count)
            if self.use_obsnorm:
                self._obs_rms[self._rms_cur].copy_(ev.stats)
        self._eval_index += 1
        return scores

    def _gather_eval_scores(self, ev, cap, count):
        """Every rank's queue (local count, scores, step tags) in one all_gather and one device -> host copy, in (step, rank,
        env) order."""
        mine = torch.cat([ev.local_count.double(), ev.scores[:cap], ev.score_step[:cap].double()])
        if self.world_size > 1:
            rows = torch.empty((self.world_size, mine.numel()), dtype=torch.float64, device=self.device)
            torch.distributed.all_gather_into_tensor(rows, mine, group=self.learner.process_group)
        else:
            rows = mine[None]
        rows = rows.cpu().numpy()
        k = rows[:, 0].astype(np.int64)
        if int(k.sum()) != count:
            raise RuntimeError("env-sharded test(): the ranks' queues hold %d scores, the global count is %d" % (k.sum(), count))
        return order_eval_scores([r[1:1 + n] for r, n in zip(rows, k)], [r[1 + cap:1 + cap + n] for r, n in zip(rows, k)])


class A2C_Agent(PPOCLIP_Agent):
    """A2C_Agent drop-in (xuance/torch/agents/policy_gradient/a2c_agent.py:6-100), vectorised like PPOCLIP_Agent: the same
    device-resident rollout / GAE / minibatch loop — the reference's two `train` bodies differ only in the learner
    (A2C surrogate -(adv * log_prob).mean(), a2c_learner.py:24-35, always gradient-clipped with `config.clip_grad`, :36),
    the absent old_logp auxiliary, and the reward normaliser's return tracker, which does not mask terminals (:85).
    The fused kernels select the A2C surrogate with clip_range = 0."""

    _mask_terminal_returns = False

    def __init__(self, config, envs, policy, optimizer, scheduler=None, device=None, process_group=None):
        from argparse import Namespace
        cfg = Namespace(**vars(config))
        cfg.clip_range = 0.0                                   # A2C surrogate in the loss kernels
        cfg.clip_grad_norm = getattr(config, "clip_grad", getattr(config, "clip_grad_norm", 0.5))
        cfg.use_grad_clip = True
        super().__init__(cfg, envs, policy, optimizer, scheduler, device, process_group)

    def _collect_info(self):
        info = super()._collect_info()
        info.pop("clip_ratio", None)                           # a2c_learner.py:42-48 logs no clip ratio
        return info


class PG_Agent(PPOCLIP_Agent):
    """PG_Agent drop-in (xuance/torch/agents/policy_gradient/pg_agent.py:4-96): the device-resident loop above with the
    reference's PG protocol — an actor-only policy (`policy(obs) -> (outputs, dist)`), value 0 stored (:59), every path
    still open when the buffer fills closed with that step's processed reward as bootstrap (:60-62), paths that end inside
    the rollout closed with 0 (:81, truncations included), minibatches of `buffer_size // n_epoch` samples (:28), the return
    tracker of the reward normaliser not masked by terminals (:74), and PG_Learner's loss (pg_learner.py:17-31:
    -(returns * log_prob).mean() - ent_coef * entropy, gradient norm clipped to `clip_grad`) — the fused loss kernels'
    A2C surrogate with the returns as weights and no value term, so the whole update phase is the captured one."""
    _mask_terminal_returns = False
    _bootstrap_truncations = False
    _aux_shape = {}

    def __init__(self, config, envs, policy, optimizer, scheduler=None, device=None, process_group=None):
        from argparse import Namespace
        cfg = Namespace(**vars(config))
        cfg.n_minibatch = config.n_epoch                       # batch_size = buffer_size // n_epoch (:28)
        cfg.use_advnorm = False                                # `sample` normalises advantages nobody reads (:70)
        cfg.clip_range, cfg.vf_coef = 0.0, 0.0
        cfg.clip_grad_norm = getattr(config, "clip_grad", None)
        cfg.use_grad_clip = cfg.clip_grad_norm is not None
        super().__init__(cfg, envs, policy, optimizer, scheduler, device, process_group)
        self._term_save = torch.zeros(self.n_envs, dtype=torch.float32, device=self.device)

    def _close_paths(self):
        mem, last = self.memory, self.n_steps - 1
        self._boot_last.copy_(mem._rew[last])                  # finish_path(self._process_reward(rewards)[i], i)
        if not mem.use_gae:
            # discount_cumsum appends the bootstrap to the rewards whether or not the last step was terminal
            # (memory_tools.py:224-225); the batched scan masks a terminal's bootstrap, so the flag is lifted for it
            self._term_save.copy_(mem._term[last])
            mem._term[last].zero_()
        mem.finish_rollout(self._boot_last, adv_from_ret=True)
        if not mem.use_gae:
            mem._term[last].copy_(self._term_save)

    def _collect_info(self):
        info = super()._collect_info()
        for k in ("critic-loss", "predict_value", "clip_ratio"):    # pg_learner.py:38-42 logs three scalars
            info.pop(k, None)
        return info


class PPOKL_Agent(PPOCLIP_Agent):
    """PPOKL_Agent (xuance/torch/agents/policy_gradient/ppokl_agent.py) on the device loop above: PPOCLIP_Agent's training
    loop with the old action distribution stored per transition (`{"old_dist": dists}`, device rows [T, N, W]: the logits,
    or mu and std) and PPOKL_Learner's update: a_loss = -(ratio * adv).mean() + kl_coef * KL(new || old).mean(), no gradient
    clipping, the coefficient adapted on the device after every minibatch from that minibatch's KL (x2 above 1.5 target_kl,
    /2 below 0.5 target_kl, clipped to [0.1, 20]; the update that measured the KL used the old value).  The update phase is
    the captured epoch graphs: the coefficient changes between replays on the device.  The fused rollout step writes the old
    distribution in the same launch; the unfused step stores it from the forward's parameters.
    The reference's own train loop cannot run (ppokl_agent.py:22, 26 and 80-82, see DESIGN.md §8 f3); this is the loop
    those lines evidently intend: PPOCLIP_Agent's, with the auxiliary and the five-argument `PPOKL_Learner.update`."""
    _aux_shape = {"old_dist": None}

    def __init__(self, config, envs, policy, optimizer, scheduler=None, device=None, process_group=None):
        super().__init__(config, envs, policy, optimizer, scheduler, device, process_group)
        M = self.buffer_size // self.batch_size
        if self.learner._peer is not None and 2 * M > self._NORM_INBOX:
            # the epoch's advantage sums take doubles [0, 2M) of the comm block's statistics area: they must stay clear of
            # the normaliser inbox [1024, 1344) and of the KL slot (PPOKL_Learner._KL_SLOT)
            raise ValueError("env-sharded PPO-KL over peer memory supports n_minibatch <= %d (got %d minibatches per epoch)"
                             % (self._NORM_INBOX // 2, M))
        mem, A = self.memory, (int(self.action_space.n) if self.discrete else self.memory.act_dim)
        mem._dist_kind = "categorical" if self.discrete else "gaussian"
        mem._dist = torch.zeros((self.n_steps, self.n_envs, A if self.discrete else 2 * A), dtype=torch.float32,
                                device=self.device)
        self._n_act = A

    def _make_learner(self, config, policy, optimizer, scheduler):
        from .learner import PPOKL_Learner
        return PPOKL_Learner(policy, optimizer, scheduler, self.device, getattr(config, "model_dir", "./"),
                             vf_coef=config.vf_coef, ent_coef=config.ent_coef, target_kl=config.target_kl)

    def _dist_out(self, t):
        return self.memory._dist[t] if self._fused_step else None

    def _store_extra(self, t, dist):
        if self._fused_step:
            return
        out, prm, N, A = self.memory._dist[t], dist.get_param(), self.n_envs, self._n_act
        if self.discrete:
            out.copy_(prm[:N])
            return
        out[:, :A].copy_(prm[0][:N])
        std = prm[1]
        if std is None:                 # the tensor-core forward returns mu only; the log-std is the policy's parameter
            std = self.policy.actor.logstd.detach().exp()
        out[:, A:].copy_(std.reshape(-1, A).expand(N, A) if std.numel() == A else std[:N])

    def _collect_info(self):
        info = super()._collect_info()
        info.pop("clip_ratio", None)
        return info


class PPG_Agent(PPOCLIP_Agent):
    """PPG_Agent drop-in (xuance/torch/agents/policy_gradient/ppg_agent.py:4-109).  The rollout is the captured device loop
    above with PPG's protocol: `policy(obs) -> (outputs, dist, v, aux_v)`, the old action distribution's parameters stored
    per transition (:63; device rows [T, N, W] instead of Python objects), paths that end inside the rollout closed with 0
    (:103), no return tracker (`ret_rms` is never updated: `_process_reward` only clips), minibatches of
    `buffer_size // n_epoch` samples (:29).  The update (:69-98) — policy phase, critic phase, refresh of every stored old
    distribution from the current policy, auxiliary phase — runs on device minibatches (`memory.sample`, nothing crosses
    PCIe) through PPG_Learner's three fused loss launches and the torch optimiser the caller built.
    Env-sharded (a process group of W > 1 ranks): every rank trains on minibatches of its own envs, normalises their advantages
    with the GLOBAL minibatch statistics, and steps its optimiser on the rank-mean gradient (PPG_Learner.enable_sharding), so
    the replicas stay bit-identical; the refresh of the stored old distributions stays local to each rank's shard."""
    _bootstrap_truncations = False
    _track_returns = False
    _graph_updates = False
    _aux_shape = {"old_dist": None}

    def __init__(self, config, envs, policy, optimizer, scheduler=None, device=None, process_group=None):
        from argparse import Namespace
        cfg = Namespace(**vars(config))
        cfg.n_minibatch = config.n_epoch                       # batch_size = buffer_size // n_epoch (:29)
        cfg.shuffle = "device"                                 # np.random.shuffle -> one keyed-bijection launch per epoch
        self.policy_nepoch, self.value_nepoch, self.aux_nepoch = config.policy_nepoch, config.value_nepoch, config.aux_nepoch
        super().__init__(cfg, envs, policy, optimizer, scheduler, device, process_group)
        mem, A = self.memory, (int(self.action_space.n) if self.discrete else self.memory.act_dim)
        mem._dist_kind = "categorical" if self.discrete else "gaussian"
        mem._dist = torch.zeros((self.n_steps, self.n_envs, A if self.discrete else 2 * A), dtype=torch.float32,
                                device=self.device)
        self._n_act = A

    def _make_learner(self, config, policy, optimizer, scheduler):
        from .learner import PPG_Learner
        return PPG_Learner(policy, optimizer, scheduler, self.device, getattr(config, "model_dir", "./"),
                           ent_coef=config.ent_coef, clip_range=config.clip_range, kl_beta=config.kl_beta)

    def _dist_rows(self, dist, rows, out):
        prm = dist.get_param()
        if self.discrete:
            out.copy_(prm[:rows])
        else:
            A = self._n_act
            out[:, :A].copy_(prm[0][:rows])
            out[:, A:].copy_(prm[1].reshape(-1, A).expand(rows, A) if prm[1].numel() == A else prm[1][:rows])

    def _store_extra(self, t, dist):
        self._dist_rows(dist, self.n_envs, self.memory._dist[t])          # {"old_dist": dists} (:63)

    def _draw_permutation(self):
        self._device_permutation()
        return self._perm

    def _global_adv_stats(self, perm):
        """(sum adv, sum adv^2) of every minibatch of the epoch, summed over the ranks (memory_tools.py:241-242 on the global
        minibatch): one pass over the permutation and one exchange, as PPOCLIP_Agent._epoch_peer does."""
        mem, B, lr = self.memory, self.batch_size, self.learner
        M = self.buffer_size // B
        if lr._peer is not None:
            ops.adv_stats_minibatches(perm, M, B, mem.n_size, mem.n_envs, mem._adv, 1, lr._peer.stats)
            ops.peer_allreduce_f64(lr._peer, 2 * M, self._mb_stats_all)
        else:
            ops.adv_stats_minibatches(perm, M, B, mem.n_size, mem.n_envs, mem._adv, 1, self._mb_stats_all)
            xdist.allreduce_adv_stats(self._mb_stats_all[:2 * M], lr.process_group)
        return self._mb_stats_all

    def _phase(self, n_epoch, update):
        mem, B, info = self.memory, self.batch_size, {}
        for ep in range(n_epoch):
            perm = self._draw_permutation()
            stats = self._global_adv_stats(perm) if (self.world_size > 1 and mem.use_advnorm) else None
            for k, start in enumerate(range(0, self.buffer_size, B)):
                kw = {} if stats is None else dict(adv_stats=stats[2 * k:2 * k + 2], adv_count=B * self.world_size)
                obs, act, ret, _, adv, aux = mem.sample(perm[start:start + B], **kw)
                # log scalars are read back for the last update of a phase only (one sync per phase, not per update)
                self.learner.read_back = ep == n_epoch - 1 and start + B >= self.buffer_size
                info = update(obs, act, ret, adv, aux["old_dist"])
        self.learner.read_back = True
        return info

    def _update_phase(self):
        mem, L, info = self.memory, self.learner, {}
        info.update(self._phase(self.policy_nepoch, L.update_policy))
        info.update(self._phase(self.value_nepoch, L.update_critic))
        with torch.no_grad():            # old_dist <- the current policy on every stored observation (:90-93)
            rows = mem._obs.reshape(self.buffer_size, mem.obs_row)[:, :self._obs_dim]
            _, new_dist, _, _ = self.policy(rows)
            self._dist_rows(new_dist, self.buffer_size, mem._dist.reshape(self.buffer_size, -1))
        info.update(self._phase(self.aux_nepoch, L.update_auxiliary))
        self._phase_info = info
        self._iteration += 1

    def _host_state(self):
        return dict(super()._host_state(), phase_info=getattr(self, "_phase_info", {}))

    def _load_host_state(self, st):
        super()._load_host_state(st)
        self._phase_info = st["phase_info"]

    def _collect_info(self):
        info = dict(getattr(self, "_phase_info", {}))
        if self.learner._peer is not None:
            self.learner._peer.check()
        st = self.envs.ep_stats.cpu().numpy()
        info["new_episodes"] = int(st[0]) - self.current_episode
        info["episodes"] = self.current_episode = int(st[0])
        info["mean_episode_score"] = float(st[1] / st[0]) if st[0] > 0 else float("nan")
        info["mean_episode_steps"] = float(st[2] / st[0]) if st[0] > 0 else float("nan")
        return info
