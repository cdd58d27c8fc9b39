"""GPU, one rank: the exchange kernels behind env-sharded PPG and the env-sharded running statistics of 8-float observation
rows (csrc/peer_comm.cu, csrc/normalize.cu), on a comm block mapped by this process alone (W = 1)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


class _OneRankComm:
    """The attributes ops.* read from a dist.PeerComm, for one rank without a process group."""

    def __init__(self, n):
        from xuanpolicy_b200 import _lib
        lib = _lib.load()
        self.rank, self.world, self.n = 0, 1, (n + 3) // 4 * 4
        ptr = C.c_void_p()
        _lib.call("xb_peer_alloc", C.byref(ptr), lib.xb_peer_block_bytes(self.n))
        self._own = ptr.value
        self.bases = (C.c_void_p * 1)(self._own)
        self.tickets = torch.zeros(64, dtype=torch.int32, device="cuda")

    def close(self):
        from xuanpolicy_b200 import _lib
        torch.cuda.synchronize()
        _lib.call("xb_peer_free", C.c_void_p(self._own))


@pytest.fixture
def comm():
    c = _OneRankComm(50_000)
    yield c
    c.close()


def test_grad_mean_returns_its_input_bit_for_bit(comm):
    from xuanpolicy_b200 import ops
    g = torch.randn(comm.n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) * 1e-3
    g[::7] = torch.tensor(float("-0.0"))
    for _ in range(3):                          # both halves of the parity double-buffered inbox, and back
        out = torch.full_like(g, float("nan"))
        ops.peer_allreduce_mean(comm, g, out)
        torch.cuda.synchronize()
        assert torch.equal(out.view(torch.int32), g.view(torch.int32))
    assert int(comm.tickets[62].item()) == 0


def _wide_batch(dim, N, seed):
    rng = np.random.default_rng(seed)
    x = np.zeros((N, 8), np.float32)
    x[:, :dim] = (rng.standard_normal((N, dim)) * rng.uniform(0.5, 4, dim) + rng.uniform(-3, 3, dim)).astype(np.float32)
    return x


def test_moments_of_8_float_rows_equal_fp64_column_sums():
    from xuanpolicy_b200 import ops
    f64 = dict(dtype=torch.float64, device="cuda")
    ws = torch.zeros(8 + 8 * 1184, **f64)
    for N in (37, 4096, 300_000):
        x = _wide_batch(8, N, N)
        sums = torch.full((17,), float("nan"), **f64)
        ops.moments4(torch.from_numpy(x).cuda(), sums, ws)
        x64 = x.astype(np.float64)
        want = np.concatenate([x64.sum(0), (x64 * x64).sum(0), [N]])
        np.testing.assert_allclose(sums.cpu().numpy(), want, rtol=1e-12, atol=1e-9)


def _chan_f32(state, sums, D, dim):
    """RunningMeanStd.update_from_moments (statistic_tools.py:101-112) on float32 arrays, the batch moments from the sums."""
    mean, var, count = state[:D].astype(np.float32), state[D:2 * D].astype(np.float32), state[2 * D]
    n = sums[2 * D]
    bm = sums[:D] / n
    bv = np.maximum(sums[D:2 * D] / n - bm * bm, 0.0)
    tot = count + n
    fc, fb, ft = np.float32(count), np.float32(n), np.float32(tot)
    delta = bm.astype(np.float32) - mean
    new_mean = mean + delta * fb / ft
    new_var = (var * fc + bv.astype(np.float32) * fb + delta * delta * fc * fb / ft) / ft
    keep = np.arange(D) < dim
    return np.where(keep, new_mean, mean), np.where(keep, new_var, var), tot


@pytest.mark.parametrize("dim", [6, 8])
def test_wide_statistics_exchange_matches_pull_form_and_numpy(comm, dim):
    from xuanpolicy_b200 import ops
    D, n = 8, 20
    f64 = dict(dtype=torch.float64, device="cuda")
    x = _wide_batch(dim, 5000, dim).astype(np.float64)
    R = np.random.default_rng(dim).standard_normal(300) * 4 + 1
    src_h = np.concatenate([x.sum(0), (x * x).sum(0), [x.shape[0]], [R.sum(), (R * R).sum(), R.size]])
    state_h = np.concatenate([np.float32(np.linspace(-1, 1, D)), np.float32(np.linspace(0.5, 2, D)), [1234.0]]).astype(np.float64)
    ret_h = np.array([0.3, 2.5, 77.0])
    src = torch.tensor(src_h, **f64)
    push = dict(obs_out=torch.zeros(2 * D + 1, **f64), ret=torch.tensor(ret_h, **f64), std=torch.zeros(1, device="cuda"))
    pull = dict(obs_out=torch.zeros(2 * D + 1, **f64), ret=torch.tensor(ret_h, **f64), std=torch.zeros(1, device="cuda"))
    state = torch.tensor(state_h, **f64)
    out = torch.zeros(n, **f64)
    ops.peer_allreduce_merge(comm, src, n, out, 1024, state, push["obs_out"], dim, push["ret"], push["std"])
    ops.rms_merge_sums(src, state, pull["obs_out"], dim, pull["ret"], pull["std"])
    torch.cuda.synchronize()
    assert torch.equal(out, src)                                   # one rank: the totals are its own sums
    for k in ("obs_out", "ret", "std"):
        assert torch.equal(push[k], pull[k]), k
    mean, var, tot = _chan_f32(state_h, src_h, D, dim)
    got = push["obs_out"].cpu().numpy()
    np.testing.assert_allclose(got[:D], mean, rtol=2e-6, atol=1e-6)
    np.testing.assert_allclose(got[D:2 * D], var, rtol=2e-6, atol=1e-6)
    assert got[2 * D] == tot
    assert np.all(got[:2 * D] == got[:2 * D].astype(np.float32))   # mean / var hold float32 values, like the reference's arrays
    bm, bv, c = R.mean(), R.var(), ret_h[2]                        # return normaliser: Chan in fp64
    d_, t_ = bm - ret_h[0], c + R.size
    want_ret = [ret_h[0] + d_ * R.size / t_, (ret_h[1] * c + bv * R.size + d_ * d_ * c * R.size / t_) / t_, t_]
    np.testing.assert_allclose(push["ret"].cpu().numpy(), want_ret, rtol=1e-12)
    assert abs(float(push["std"].item()) - np.clip(np.sqrt(want_ret[1]), 0.1, 100)) <= 1e-6 * np.sqrt(want_ret[1])


def test_bad_arguments_raise(comm):
    from xuanpolicy_b200 import _lib, ops
    f64 = dict(dtype=torch.float64, device="cuda")
    s20, s12, st17, st9 = (torch.zeros(k, **f64) for k in (20, 12, 17, 9))
    o17, o9, ret, std = torch.zeros(17, **f64), torch.zeros(9, **f64), torch.zeros(3, **f64), torch.zeros(1, device="cuda")
    g = torch.zeros(comm.n, device="cuda")
    bad = [
        lambda: ops.peer_allreduce_merge(comm, s20, 21, torch.zeros(21, **f64), 1024),          # n > 20
        lambda: ops.peer_allreduce_merge(comm, s20, 16, s20, 1024, st17, o17, 8),                 # merge needs n = 12 or 20
        lambda: ops.peer_allreduce_merge(comm, s20, 20, s20, 1024, st17, o17, 9),                 # dim > 8
        lambda: ops.peer_allreduce_merge(comm, s12, 12, s12, 1024, st9, o9, 5),                   # dim > 4 with 4-float sums
        lambda: ops.peer_allreduce_merge(comm, s20, 20, s20, 2048 - 320 + 1),                     # inbox leaves the area
        lambda: ops.rms_merge_sums(torch.zeros(13, **f64), st9, o9, 4, None, None),               # n not 2D + 4
        lambda: ops.rms_merge_sums(s20, st17, o17, 9, None, None),                                # dim > 8
        lambda: ops.rms_merge_sums(s20, None, None, 0, ret, None),                                # ret_state without rew_std
        lambda: _lib.call("xb_moments4", g.data_ptr(), 6, s20.data_ptr(), st17.data_ptr(), 4, None),   # row width 6
        lambda: _lib.call("xb_moments4", None, 8, s20.data_ptr(), st17.data_ptr(), 4, None),
        lambda: _lib.call("xb_peer_allreduce_mean", comm.bases, 0, 1, comm.n - 2, g.data_ptr(), g.data_ptr(),
                          comm.tickets.data_ptr(), None),                                          # n not a multiple of 4
        lambda: _lib.call("xb_peer_allreduce_mean", comm.bases, 0, 1, comm.n, None, g.data_ptr(), comm.tickets.data_ptr(), None),
        lambda: _lib.call("xb_peer_allreduce_mean", comm.bases, 0, 1, comm.n, g.data_ptr(), g.data_ptr(), None, None),
        lambda: _lib.call("xb_peer_allreduce_mean", comm.bases, 0, 0, comm.n, g.data_ptr(), g.data_ptr(),
                          comm.tickets.data_ptr(), None),                                          # W = 0
        lambda: _lib.call("xb_peer_allreduce_mean", comm.bases, 1, 1, comm.n, g.data_ptr(), g.data_ptr(),
                          comm.tickets.data_ptr(), None),                                          # rank >= W
    ]
    for i, f in enumerate(bad):
        with pytest.raises(_lib.XB200Error):
            f()
            pytest.fail("case %d did not raise" % i)
    torch.cuda.synchronize()
