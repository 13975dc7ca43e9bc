"""Lazy marginals of the Potts grid. A sweep stores the marginals of its first and last rows only (every row when
CXB_GRID_EAGER_M2V=1, and in the last sweep of an infer_host job); the first cxb_grid_get_marginals after a sweep rebuilds
the others from the m2f planes and the evidence that sweep read (k_potts_m2v). Every hazard to those inputs is exercised
here against eager mode, bit for bit: new evidence set before the read, infer_host jobs uploading into the evidence buffer
of a pending sweep, reads at irregular points, and fused row shards whose halo buffers the neighbours overwrite before the
read."""
import numpy as np
import pytest

from tests._pkg import pkg as C
from tests.test_potts_lazy_m2v import CASES, _assert_equal, _grid, _launches, _npdt, _planes, _unary

pytestmark = pytest.mark.gpu

F32, F64 = C.capi.F32, C.capi.F64
# the lanes-per-pixel instantiations of test_potts_lazy_m2v plus H = 2 and 3 (no interior row / one interior row)
ALL = CASES + [(F32, (2, 5, 8)), (F32, (3, 6, 16)), (F64, (2, 5, 4)), (F64, (3, 6, 16))]
IDS = [f"{'f32' if d == F32 else 'f64'}-{h}x{w}xK{k}" for d, (h, w, k) in ALL]


def _pair(monkeypatch, H, W, K, dtype, beta=0.7, **kw):
    return {e: _grid(monkeypatch, e, H, W, K, beta, dtype, **kw) for e in (True, False)}


@pytest.mark.parametrize("dtype,shape", ALL, ids=IDS)
def test_new_evidence_before_the_read(monkeypatch, dtype, shape):
    """set_unary between a sweep and get_marginals: the marginals are those of the evidence the sweep read."""
    H, W, K = shape
    u0, u1 = (_unary(H, W, K, dtype, s) for s in (11, 12))
    g = _pair(monkeypatch, H, W, K, dtype)
    for e in g.values():
        e.set_unary(u0)
        e.reset_messages()
        assert not np.any(e.get_marginals())  # before any sweep: the zeros of init
    for s in range(3):
        for e in g.values():
            e.sweep()
        for e in g.values():
            e.set_unary(u1 if s % 2 == 0 else u0)
        _assert_equal([g[False].get_marginals()], [g[True].get_marginals()], f"after sweep {s} and set_unary")
    # a sweep is one launch; the first read after it rebuilds once when there are interior rows, a second read launches nothing
    l0 = _launches()
    g[False].sweep()
    assert _launches() - l0 == 1
    l0 = _launches()
    first = g[False].get_marginals()
    assert _launches() - l0 == (1 if H > 2 else 0)
    l0 = _launches()
    assert np.array_equal(g[False].get_marginals(), first)
    assert _launches() == l0
    g[True].sweep()
    assert np.array_equal(first, g[True].get_marginals())


@pytest.mark.parametrize("dtype,shape", ALL, ids=IDS)
def test_reads_at_irregular_points(monkeypatch, dtype, shape):
    """Marginals read after every other sweep, twice in a row; m2f reads flush nothing, m2v reads flush only the m2v."""
    H, W, K = shape
    unary = _unary(H, W, K, dtype, 31)
    g = _pair(monkeypatch, H, W, K, dtype, beta=0.45)
    for e in g.values():
        e.set_unary(unary)
        e.reset_messages()
    for s in range(6):
        for e in g.values():
            e.sweep()
        if s % 2:
            want = g[True].get_marginals()
            for _ in range(2):
                assert np.array_equal(g[False].get_marginals(), want), f"sweep {s}"
        elif s == 2:
            l0 = _launches()
            m2f = [g[False].get_messages(w) for w in range(4, 8)]
            assert _launches() == l0
            g[False].get_messages(0)
            assert _launches() - l0 == (1 if H > 2 else 0)  # the m2v only: the marginals are still pending
            l0 = _launches()
            _assert_equal(m2f + [g[False].get_marginals()], [g[True].get_messages(w) for w in range(4, 8)] + [g[True].get_marginals()],
                          f"sweep {s}")
            assert _launches() - l0 == (1 if H > 2 else 0)
    # a reset keeps the last sweep's marginals
    for e in g.values():
        e.sweep()
        e.reset_messages()
    _assert_equal(_planes(g[False]), _planes(g[True]), "after reset_messages")


@pytest.mark.parametrize("dtype,shape", [(F32, (37, 29, 16)), (F64, (3, 6, 16)), (F32, (2, 5, 8)), (F64, (9, 33, 16))],
                         ids=["f32-37x29xK16", "f64-3x6xK16", "f32-2x5xK8", "f64-9x33xK16"])
def test_plain_sweeps_then_host_jobs(monkeypatch, dtype, shape):
    """Plain sweeps leave marginals pending; infer_host jobs follow with no read in between (the first job uploads into
    the evidence buffer those sweeps read). Every job's host output and the final marginals equal eager mode; a job
    launches only its sweeps once nothing is pending."""
    import torch

    H, W, K = shape
    sweeps, jobs = 3, 4
    tdt = torch.float32 if dtype == F32 else torch.float64
    rng = np.random.Generator(np.random.PCG64(77))
    plain = _unary(H, W, K, dtype, 78)
    host_in = [torch.from_numpy(rng.dirichlet(np.ones(K), size=(H, W)).astype(_npdt(dtype))).pin_memory() for _ in range(2 * jobs)]
    got = {}
    for eager in (True, False):
        g = _grid(monkeypatch, eager, H, W, K, 0.7, dtype)
        g.set_unary(plain)
        g.reset_messages()
        outs = [torch.empty((H, W, K), dtype=tdt).pin_memory() for _ in range(2 * jobs)]
        for rnd in range(2):  # plain sweeps, then jobs; twice, so the second round starts from the jobs' evidence buffers
            # a job's output is complete after sync(); a plain sweep before it would write the buffer still being downloaded
            g.sync()
            for _ in range(2):
                g.sweep()
            for k in range(jobs):
                j = rnd * jobs + k
                l0 = _launches()
                g.infer_host(host_in[j].data_ptr(), outs[j].data_ptr(), sweeps)
                n = _launches() - l0
                rebuild = 1 if (not eager and k == 0 and H > 2) else 0  # only the marginals the plain sweeps left pending
                assert n == sweeps + rebuild, f"eager={eager}, job {j}: {n} launches"
        g.sync()
        l0 = _launches()
        got[eager] = [o.numpy().copy() for o in outs] + [g.get_marginals()]
        assert _launches() == l0  # the last job stored every marginal
        del g
    _assert_equal(got[False], got[True], "host jobs")


@pytest.mark.parametrize("dtype", [F32, F64])
def test_fused_shards_read_after_the_neighbours_ran_ahead(monkeypatch, dtype):
    """Three fused row shards. The outer shards run sweep s + 1 before the middle shard's marginals of sweep s are read:
    by then they have overwritten the halo buffer the middle shard read, so its boundary rows must be the stored values.
    Against one unsharded grid, in both modes."""
    H, W, K, beta, sweeps = 14, 9, 8, 0.45, 5
    unary = _unary(H, W, K, dtype, 8)
    cuts = [0, 4, 10, H]
    full = _grid(monkeypatch, True, H, W, K, beta, dtype)
    full.set_unary(unary)
    full.reset_messages()
    want = []
    for s in range(sweeps):
        full.sweep()
        want.append(full.get_marginals())
    for eager in (True, False):
        sh = [_grid(monkeypatch, eager, cuts[i + 1] - cuts[i], W, K, beta, dtype, has_upper=i > 0, has_lower=i < 2) for i in range(3)]
        for i, x in enumerate(sh):
            x.set_unary(unary[cuts[i]:cuts[i + 1]])
            x.reset_messages()
        for i, x in enumerate(sh):
            if i > 0:
                x.p2p_connect_local(0, sh[i - 1])
            if i < 2:
                x.p2p_connect_local(1, sh[i + 1])
        for x in sh:
            x.sweep()
        for s in range(sweeps - 1):
            sh[0].sweep()
            sh[2].sweep()
            sh[0].sync()
            sh[2].sync()  # sweep s + 1 of the outer shards has stored into the middle shard's halo buffer of sweep s
            mid = sh[1].get_marginals()
            assert np.array_equal(mid, want[s][cuts[1]:cuts[2]]), f"eager={eager}, sweep {s}, middle shard"
            for i in (0, 2):
                assert np.array_equal(sh[i].get_marginals(), want[s + 1][cuts[i]:cuts[i + 1]]), f"eager={eager}, sweep {s + 1}, shard {i}"
            sh[1].sweep()
        for x in sh:
            x.sync()
        got = np.concatenate([x.get_marginals() for x in sh], axis=0)
        assert np.array_equal(got, want[-1]), f"eager={eager}, last sweep"
