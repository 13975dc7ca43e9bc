"""Lazy m2v planes of the Potts grid. A sweep stores the m2v messages of its first and last rows only; the first read of an
m2v plane after a sweep (cxb_grid_get_messages 0..3) rebuilds the other rows from the m2f planes that sweep read
(k_potts_m2v). CXB_GRID_EAGER_M2V=1 stores every m2v every sweep. Every message plane and the marginals of the two modes
must agree bit for bit, on one shard and on row shards, before, between and after sweeps, across a reset and after a
pipelined host job."""
import hashlib
import os

import numpy as np
import pytest

from tests._pkg import pkg as C
from tests.test_device_parity import _d2d

cap = C.capi
pytestmark = pytest.mark.gpu

F32, F64 = cap.F32, cap.F64
# every lanes-per-pixel instantiation (K / 4 for fp32, K / 2 for fp64: 1 .. 32) and the degenerate one-row / one-column grids
CASES = [(F32, s) for s in ((1, 1, 4), (1, 7, 4), (6, 1, 4), (5, 7, 8), (9, 33, 16), (64, 64, 32), (7, 9, 64), (8, 8, 128))] + \
        [(F64, s) for s in ((5, 6, 2), (1, 7, 4), (6, 1, 4), (5, 7, 8), (9, 33, 16), (64, 64, 32), (8, 8, 64))]


def _npdt(dtype):
    return np.float32 if dtype == F32 else np.float64


def _unary(H, W, K, dtype, seed):
    return np.random.Generator(np.random.PCG64(seed)).dirichlet(np.ones(K), size=(H, W)).astype(_npdt(dtype))


def _grid(monkeypatch, eager, H, W, K, beta, dtype=F32, **kw):
    """the mode is read when the grid is created"""
    monkeypatch.setenv("CXB_GRID_EAGER_M2V", "1" if eager else "0")
    return C.PottsGrid(H, W, K, beta, dtype=dtype, **kw)


def _planes(g):
    """m2v from / m2f towards the (up, left, right, down) factor, then the marginals"""
    return [g.get_messages(w) for w in range(8)] + [g.get_marginals()]


def _assert_equal(got, want, what):
    for w, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), f"{what}: plane {w} differs"


def _launches():
    return C.default_api().kernel_launches()


@pytest.mark.parametrize("dtype,shape", CASES, ids=[f"{'f32' if d == F32 else 'f64'}-{h}x{w}xK{k}" for d, (h, w, k) in CASES])
def test_lazy_m2v_planes_equal_the_stored_ones(monkeypatch, dtype, shape):
    H, W, K = shape
    unary = _unary(H, W, K, dtype, 1234)
    eager, lazy = (_grid(monkeypatch, e, H, W, K, 0.7, dtype) for e in (True, False))
    for g in (eager, lazy):
        g.set_unary(unary)
        g.reset_messages()
    # before any sweep the m2v planes read as zeros
    for w in range(4):
        assert not np.any(lazy.get_messages(w)) and not np.any(eager.get_messages(w))
    for s in range(3):
        assert eager.sweep() == lazy.sweep()
        _assert_equal(_planes(lazy), _planes(eager), f"after sweep {s}")
    # one rebuild per sweep, none in eager mode or on a second read
    eager.sweep()
    lazy.sweep()
    l0 = _launches()
    first = lazy.get_messages(2)
    assert _launches() - l0 == (1 if H > 2 else 0)
    l0 = _launches()
    assert np.array_equal(lazy.get_messages(2), first) and np.array_equal(lazy.get_messages(0), lazy.get_messages(0))
    assert np.array_equal(eager.get_messages(1), lazy.get_messages(1))
    assert _launches() == l0
    assert np.array_equal(first, eager.get_messages(2))
    # a reset keeps the m2v planes of the last sweep; the next sweep starts from uniform messages again
    eager.sweep()
    lazy.sweep()
    for g in (eager, lazy):
        g.reset_messages()
    _assert_equal(_planes(lazy), _planes(eager), "after reset_messages")
    for g in (eager, lazy):
        g.sweep()
    _assert_equal(_planes(lazy), _planes(eager), "first sweep after reset_messages")


@pytest.mark.parametrize("eager", [True, False])
def test_sweep_is_one_launch_in_both_modes(monkeypatch, eager):
    g = _grid(monkeypatch, eager, 9, 33, 16, 0.7)
    g.set_unary(_unary(9, 33, 16, F32, 5))
    g.reset_messages()
    for _ in range(3):
        l0 = _launches()
        g.sweep()
        assert _launches() - l0 == 1


def test_lazy_m2v_after_a_pipelined_host_job(monkeypatch):
    import torch

    H, W, K, sweeps = 37, 29, 16, 3
    rng = np.random.Generator(np.random.PCG64(21))
    unaries = [rng.dirichlet(np.ones(K), size=(H, W)).astype(np.float32) for _ in range(2)]
    host_in = [torch.from_numpy(u).pin_memory() for u in unaries]
    host_out = torch.empty((H, W, K), dtype=torch.float32).pin_memory()
    got = {}
    for eager in (True, False):
        g = _grid(monkeypatch, eager, H, W, K, 0.7)
        g.reset_messages()
        for u in host_in:
            g.infer_host(u.data_ptr(), host_out.data_ptr(), sweeps)
        g.sync()
        got[eager] = _planes(g)
    _assert_equal(got[False], got[True], "after infer_host")


def test_two_shards_with_caller_exchange(monkeypatch):
    """The halo exchange of tests/test_device_parity.py::test_potts_grid_row_sharding_is_bit_identical, in both modes, against
    one unsharded grid."""
    H, W, K, beta, sweeps = 10, 12, 16, 0.7, 4
    unary = _unary(H, W, K, F32, 3)
    full = _grid(monkeypatch, False, H, W, K, beta)
    full.set_unary(unary)
    full.reset_messages()
    for s in range(sweeps):
        full.sweep()
    want = _planes(full)
    for eager in (True, False):
        top = _grid(monkeypatch, eager, 4, W, K, beta, has_lower=True)
        bot = _grid(monkeypatch, eager, 6, W, K, beta, has_upper=True)
        top.set_unary(unary[:4])
        bot.set_unary(unary[4:])
        top.reset_messages()
        bot.reset_messages()
        nbytes = top.halo_elems * 4
        for s in range(sweeps):
            top.sweep()
            bot.sweep()
            top.sync()
            bot.sync()
            _d2d(bot.halo_recv_ptr(0), top.halo_send_ptr(1), nbytes)
            _d2d(top.halo_recv_ptr(1), bot.halo_send_ptr(0), nbytes)
        got = [np.concatenate([a, b], axis=0) for a, b in zip(_planes(top), _planes(bot))]
        _assert_equal(got, want, f"eager={eager}")


@pytest.mark.parametrize("dtype", [F32, F64])
def test_three_fused_shards(monkeypatch, dtype):
    """Three row shards connected through cxb_grid_p2p_connect_local (the sweep kernel stores the cut-edge messages into the
    neighbours' halo buffers), read between sweeps, in both modes, against one unsharded grid. The boundary rows' m2v come
    from halo buffers that the neighbours overwrite with their next sweep, so those rows must be the stored ones."""
    H, W, K, beta, sweeps = 13, 9, 8, 0.45, 5
    unary = _unary(H, W, K, dtype, 8)
    cuts = [0, 4, 9, H]
    full = _grid(monkeypatch, True, H, W, K, beta, dtype)
    full.set_unary(unary)
    full.reset_messages()
    want = []
    for s in range(sweeps):
        full.sweep()
        want.append(_planes(full))
    for eager in (True, False):
        shards = [_grid(monkeypatch, eager, cuts[i + 1] - cuts[i], W, K, beta, dtype, has_upper=i > 0, has_lower=i < 2) for i in range(3)]
        for i, sh in enumerate(shards):
            sh.set_unary(unary[cuts[i]:cuts[i + 1]])
            sh.reset_messages()
        for i, sh in enumerate(shards):
            if i > 0:
                sh.p2p_connect_local(0, shards[i - 1])
            if i < 2:
                sh.p2p_connect_local(1, shards[i + 1])
        for s in range(sweeps):
            for sh in shards:  # every shard enqueues sweep s before any shard enqueues sweep s + 1
                sh.sweep()
            # read only the m2v planes of the middle shard now; the others after their neighbours' next sweep
            mid = [shards[1].get_messages(w) for w in range(4)]
            for w in range(4):
                assert np.array_equal(mid[w], want[s][w][cuts[1]:cuts[2]]), f"eager={eager}, sweep {s}, middle shard, m2v plane {w}"
        for sh in shards:
            sh.sync()
        got = [np.concatenate(p, axis=0) for p in zip(*(_planes(sh) for sh in shards))]
        _assert_equal(got, want[-1], f"eager={eager}")


@pytest.mark.skipif(os.environ.get("CXB_SKIP_FULLSIZE") == "1", reason="CXB_SKIP_FULLSIZE=1")
def test_full_size_8192_squared(monkeypatch):
    """The benchmarked grid (8192^2, K = 16, fp32), two sweeps: SHA-256 of every m2v plane and of the marginals, one mode after
    the other (each grid holds 60 GB of device memory)."""
    N, K, beta, sweeps = 8192, 16, 0.7, 2
    rng = np.random.Generator(np.random.PCG64(1234))
    unary = np.empty((N, N, K), dtype=np.float32)
    for i in range(0, N, 256):
        e = rng.standard_exponential((256, N, K), dtype=np.float32)
        unary[i:i + 256] = e / e.sum(axis=-1, keepdims=True)
    digests = {}
    for eager in (True, False):
        g = _grid(monkeypatch, eager, N, N, K, beta)
        g.set_unary(unary)
        g.reset_messages()
        for _ in range(sweeps):
            g.sweep()
        digests[eager] = [hashlib.sha256(g.get_messages(w).data).hexdigest() for w in range(4)]
        digests[eager].append(hashlib.sha256(g.get_marginals().data).hexdigest())
        del g
    assert digests[False] == digests[True]
