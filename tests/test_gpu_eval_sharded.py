"""GPU, one process: the env-sharded evaluation loop of `test()` (sharded xb_eval_step + xb_peer_eval_merge).

On a comm block mapped by this process alone (W = 1) the sharded path must give today's one-rank device loop bit for bit.  The
exchange kernel is also driven at W = 2 in one process: rank 1's record and barrier flag are written into the block rank 0 reads
before the launch, so rank 0's launch never waits."""
import ctypes as C

import numpy as np
import pytest
import torch

import xuanpolicy_b200 as xb
from xuanpolicy_b200.configs import build_ppg, build_ppo

pytestmark = pytest.mark.gpu
ENVS = ["CartPole-v1", "Pendulum-v1", "Acrobot-v1", "MountainCar-v0", "gym:MountainCar-v0"]
EVAL_SEED = 11
PUSH_SLOT, ERR_SLOT, INBOX, ROW = 61, 62, 1024, 20      # peer_comm.cu: kPeerPushSlot, kPeerErrSlot, the agent's inbox, kPeerPushMax


def _view(ptr, count, typestr):
    from xuanpolicy_b200.dist import _DeviceMemory
    return torch.as_tensor(_DeviceMemory(ptr, count, typestr), device="cuda")


class _OneRankComm:
    """The attributes ops.* and the agent read from a dist.PeerComm, for one rank without a process group."""

    def __init__(self, n=64):
        from xuanpolicy_b200 import _lib
        lib = _lib.load()
        self.rank, self.world, self.n = 0, 1, (n + 3) // 4 * 4
        ptr = C.c_void_p()
        _lib.call("xb_peer_alloc", C.byref(ptr), lib.xb_peer_block_bytes(self.n))
        self._own = ptr.value
        self.bases = (C.c_void_p * 1)(self._own)
        self.tickets = torch.zeros(64, dtype=torch.int32, device="cuda")
        self.stats = _view(self._own + lib.xb_peer_stats_offset(), lib.xb_peer_stats_max(), "<f8")
        self.flags = _view(self._own, 64 * 8, "<i4")

    def check(self):
        assert int(self.tickets[ERR_SLOT].item()) == 0

    def close(self):
        from xuanpolicy_b200 import _lib
        torch.cuda.synchronize()
        _lib.call("xb_peer_free", C.c_void_p(self._own))


@pytest.fixture
def comm():
    c = _OneRankComm()
    yield c
    c.close()


def _env_fn(env_id, n):
    return lambda: xb.DummyVecEnv_Gym(xb.make_env_fns(env_id, EVAL_SEED, n), device="cuda", native=True)


def _after(agent):
    ev = agent._evaluator
    torch.cuda.synchronize()
    count = int(ev.count.item())
    return [t.clone() for t in (ev.state, ev.rng, ev.elapsed, ev.ep_score, ev.x, ev.step, ev.count, ev.stats,
                                agent._obs_rms[0], agent._obs_rms[1])], count


@pytest.mark.parametrize("n", [16, 4096])
@pytest.mark.parametrize("use_obsnorm", [False, True])
@pytest.mark.parametrize("env_id", ENVS)
def test_one_rank_sharded_path_equals_the_device_loop(comm, env_id, use_obsnorm, n):
    kw = dict(parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=use_obsnorm, seed=3)
    plain, sharded = build_ppo(env_id, **kw), build_ppo(env_id, **kw)
    assert plain._eval_peer is None
    sharded._eval_peer = comm
    want = plain.test(_env_fn(env_id, n), n)
    got = sharded.test(_env_fn(env_id, n), n)
    assert sharded._evaluator.peer is comm and plain._evaluator.peer is None
    assert got == want and len(got) >= n
    (a, count_a), (b, count_b) = _after(plain), _after(sharded)
    assert count_a == count_b == int(sharded._evaluator.local_count.item())
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert sharded._evaluator.score_step[:count_b].cpu().tolist() == sorted(sharded._evaluator.score_step[:count_b].cpu().tolist())
    comm.check()


@pytest.mark.parametrize("build,env_id", [(build_ppg, "Pendulum-v1"), (build_ppo, "Acrobot-v1")])
def test_one_rank_sharded_path_equals_the_device_loop_ppg_and_repeat(comm, build, env_id):
    """PPG's four-output policy; a second evaluation on the same evaluator (the next evaluation index)."""
    plain, sharded = build(env_id, parallels=16, n_steps=8, seed=4), build(env_id, parallels=16, n_steps=8, seed=4)
    sharded._eval_peer = comm
    for _ in range(2):
        assert sharded.test(_env_fn(env_id, 64), 40) == plain.test(_env_fn(env_id, 64), 40)
    assert sharded._eval_index == plain._eval_index == 2


@pytest.mark.parametrize("env_id", ["CartPole-v1", "Pendulum-v1"])
def test_chunk_sizes_and_stop_rule(comm, env_id):
    """K = 1, 5 and 32 steps per chunk agree; a chunk replayed after the stop changes nothing, the barrier tickets included."""
    runs = []
    for k in (1, 5, 32):
        agent = build_ppo(env_id, parallels=16, n_steps=8, n_epoch=1, n_minibatch=1, use_obsnorm=True, seed=6)
        agent._eval_peer = comm
        agent._eval_chunk = k
        scores = agent.test(_env_fn(env_id, 300), 100)
        before, _ = _after(agent)
        ev = agent._evaluator
        tickets, local, queue = comm.tickets.clone(), ev.local_count.clone(), ev.score_step.clone()
        with torch.no_grad():
            ev.graph.replay()                               # a whole chunk after the stop
        after, _ = _after(agent)
        for x, y in zip(before, after):
            assert torch.equal(x, y)
        assert torch.equal(tickets, comm.tickets) and torch.equal(local, ev.local_count) and torch.equal(queue, ev.score_step)
        runs.append((scores, before))
    for scores, st in runs[1:]:
        assert scores == runs[0][0]
        for x, y in zip(st, runs[0][1]):
            assert torch.equal(x, y)
    comm.check()


# ------------------------------------------------------------------------------------------------ the exchange kernel at W = 2
def _merge_numpy(state, totals, D, dim):
    """The observation merge of xb_peer_eval_merge in float32 / float64 with every operation rounded on its own (numpy never
    contracts a multiply-add): the bits the kernel must produce."""
    out = state.copy()
    n, count = totals[2 * D], state[2 * D]
    for d in range(dim):
        bm = totals[d] / n
        bv = max(totals[D + d] / n - bm * bm, 0.0)
        nm, nv = np.float32(state[d]), np.float32(state[D + d])
        fc, fb, ft = np.float32(count), np.float32(n), np.float32(count + n)
        delta = np.float32(bm) - nm
        m2 = nv * fc + np.float32(bv) * fb + delta * delta * fc * fb / ft
        out[d], out[D + d] = nm + delta * fb / ft, m2 / ft
    out[2 * D] = count + n
    return out


class _TwoBlocks:
    """Two comm blocks in this process: rank 0 launches, rank 1's side is written by hand."""

    def __init__(self):
        self.blocks = [_OneRankComm(), _OneRankComm()]
        self.bases = (C.c_void_p * 2)(self.blocks[0]._own, self.blocks[1]._own)
        self.rank, self.world, self.tickets = 0, 2, self.blocks[0].tickets

    def stage_rank1(self, record, ticket):
        """Rank 1's record in rank 0's inbox row [parity][1], and rank 1's barrier flag for this ticket in rank 0's flags."""
        b0, parity = self.blocks[0], ticket & 1
        row = INBOX + (parity * 8 + 1) * ROW
        b0.stats[row:row + record.numel()] = record
        b0.flags[PUSH_SLOT * 8 + 1] = ticket
        torch.cuda.synchronize()
        assert int(b0.flags[PUSH_SLOT * 8 + 1].item()) == ticket

    def close(self):
        for b in self.blocks:
            b.close()


def _record(D, N, fin, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((N, D)) * rng.uniform(0.5, 2, D) + rng.uniform(-1, 1, D)).astype(np.float32).astype(np.float64)
    return np.concatenate([x.sum(0), (x * x).sum(0), [N, 0.0, 0.0, fin]])


@pytest.mark.parametrize("D,dim", [(4, 4), (8, 6)])
def test_exchange_at_two_ranks(D, dim):
    from xuanpolicy_b200 import ops
    f64, i64 = dict(dtype=torch.float64, device="cuda"), dict(dtype=torch.int64, device="cuda")
    pair = _TwoBlocks()
    try:
        r0, r1 = _record(D, 300, 7, 1), _record(D, 300, 5, 2)
        state_h = np.concatenate([np.float32(np.linspace(-1, 1, D)), np.float32(np.linspace(0.5, 2, D)), [1234.0]])
        state, cand = torch.tensor(state_h, **f64), torch.zeros(2 * D + 1, **f64)
        record, totals = torch.tensor(r0, **f64), torch.zeros(2 * D + 4, **f64)
        count, target = torch.tensor([10], **i64), torch.tensor([100], **i64)
        b1 = pair.blocks[1]
        # (1) a step that goes round again: totals in rank order, count + both ranks' finishers, merge
        pair.stage_rank1(torch.tensor(r1, **f64), 1)
        ops.peer_eval_merge(pair, record, totals, count, target, INBOX, state, cand, dim)
        torch.cuda.synchronize()
        want = (0.0 + r0) + r1
        assert np.array_equal(totals.cpu().numpy(), want)
        assert int(count.item()) == 10 + 12
        assert np.array_equal(state.cpu().numpy(), _merge_numpy(state_h, want, D, dim))
        row = INBOX + (1 * 8 + 0) * ROW                                   # rank 0's push reached rank 1's inbox, flag set
        assert np.array_equal(b1.stats[row:row + 2 * D + 4].cpu().numpy(), r0)
        assert int(b1.flags[PUSH_SLOT * 8 + 0].item()) == 1 and int(pair.tickets[PUSH_SLOT].item()) == 1
        # (2) the step that reaches the target: the count advances, no merge
        count.fill_(90)
        state1 = state.clone()
        pair.stage_rank1(torch.tensor(r1, **f64), 2)
        ops.peer_eval_merge(pair, record, totals, count, target, INBOX, state, cand, dim)
        torch.cuda.synchronize()
        assert int(count.item()) == 102 and torch.equal(state, state1) and int(pair.tickets[PUSH_SLOT].item()) == 2
        # (3) the target already met: no push, no barrier, nothing written
        inbox1, flags1, totals1 = b1.stats.clone(), b1.flags.clone(), totals.clone()
        ops.peer_eval_merge(pair, record, totals, count, target, INBOX, state, cand, dim)
        torch.cuda.synchronize()
        assert int(count.item()) == 102 and torch.equal(state, state1) and torch.equal(totals, totals1)
        assert torch.equal(b1.stats, inbox1) and torch.equal(b1.flags, flags1) and int(pair.tickets[PUSH_SLOT].item()) == 2
        assert int(pair.tickets[ERR_SLOT].item()) == 0
    finally:
        pair.close()


def test_bad_arguments_raise(comm):
    from xuanpolicy_b200 import _lib, ops
    f64, i64 = dict(dtype=torch.float64, device="cuda"), dict(dtype=torch.int64, device="cuda")
    rec, tot, st, cand = torch.zeros(12, **f64), torch.zeros(12, **f64), torch.zeros(9, **f64), torch.zeros(9, **f64)
    cnt, tgt = torch.zeros(1, **i64), torch.ones(1, **i64)
    p = lambda t: t.data_ptr() if t is not None else None

    def merge(bases=comm.bases, rank=0, W=1, record=rec, n=12, inbox=INBOX, totals=tot, count=cnt, obs=None, c=None, dim=0):
        _lib.call("xb_peer_eval_merge", bases, rank, W, p(record), n, inbox, p(totals), p(count), p(tgt), p(obs), p(c), dim,
                  comm.tickets.data_ptr(), None)

    N = 64
    state, rng = torch.zeros((4, N), **f64), torch.zeros((2, N), **i64)
    el, eps, x = torch.zeros(N, dtype=torch.int32, device="cuda"), torch.zeros(N, **f64), torch.zeros((N, 4), device="cuda")
    logits, key, step = torch.zeros((N, 2), device="cuda"), torch.zeros(1, **i64), torch.zeros(1, **i64)
    scores, part, ws = torch.zeros(N, **f64), torch.zeros(20 * 2, **f64), torch.zeros(4, **i64)
    local, tags = torch.zeros(1, **i64), torch.zeros(N, dtype=torch.int32, device="cuda")

    def step_(**kw):
        a = dict(local_count=local, score_step=tags, record=rec)
        a.update(kw)
        ops.eval_step(0, logits, None, key, step, state, rng, el, eps, x, None, 500, scores, cnt, tgt, part, ws, **a)

    bad = [
        lambda: merge(n=13),                                   # not 2D + 4 for D = 4 or 8
        lambda: merge(n=20, record=torch.zeros(20, **f64), totals=None),
        lambda: merge(record=None),
        lambda: merge(count=None),
        lambda: merge(inbox=2048 - 320 + 1),                   # the inbox leaves the statistics area
        lambda: merge(inbox=-1),
        lambda: merge(obs=st, c=None, dim=4),                  # the merge needs its scratch
        lambda: merge(obs=st, c=st, dim=4),
        lambda: merge(obs=st, c=cand, dim=5),                  # dim > D
        lambda: merge(W=0),
        lambda: merge(rank=1),
        lambda: ops.peer_eval_merge(comm, rec, torch.zeros(11, **f64), cnt, tgt, INBOX),     # totals shorter than the record
        lambda: step_(record=None),                            # the sharded form needs all three
        lambda: step_(local_count=None),
        lambda: step_(score_step=None, record=None),
        lambda: step_(score_step=tags[:N - 1]),                # a step tag per queue slot
        lambda: step_(obs_state=st, obs_dim=9),
        lambda: step_(local_count=None, score_step=None, record=None, obs_state=st, obs_dim=4),   # one-rank form: scratch needed
    ]
    for i, f in enumerate(bad):
        with pytest.raises(_lib.XB200Error):
            f()
            pytest.fail("case %d did not raise" % i)
    torch.cuda.synchronize()
    assert int(step.item()) == 0 and int(comm.tickets[PUSH_SLOT].item()) == 0
