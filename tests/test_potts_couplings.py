"""Per-edge coupling strengths of the Potts grid (cxb_grid_set_couplings / PottsGrid.set_couplings): factor e carries
psi_e[a][b] = exp(beta_e [a==b]). Checked against the oracle's explicit graph (one POTTS form per distinct beta), against an
independent fp64 numpy flooding BP, against the uniform grid when every coupling equals the create-time beta, lazy against
eager rebuilds, row shards against one shard, pipelined host jobs against plain calls, and refused input. The slicing of
global couplings into row shards (sharding.shard_couplings) is checked without a GPU."""
import numpy as np
import pytest

from tests import models
from tests._pkg import pkg as C
from tests.test_device_parity import _d2d
from tests.test_potts_lazy_m2v import _assert_equal, _grid, _launches, _npdt, _planes, _unary

cap = C.capi
F32, F64 = cap.F32, cap.F64
PALETTE = np.array([0.0, -0.6, 0.25, 0.7, 1.3, 2.1])


def _palette_couplings(H, W, seed):
    """global horizontal [H][W-1] and vertical [H-1][W] couplings drawn from PALETTE"""
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.choice(PALETTE, size=(H, W - 1)), rng.choice(PALETTE, size=(max(H - 1, 0), W))


def _smooth_couplings(H, W, seed, lam=1.5, sigma=0.1):
    """contrast-sensitive couplings lam * exp(-|I_i - I_j|^2 / 2 sigma^2) of a random image (continuous values)"""
    img = np.random.Generator(np.random.PCG64(seed)).random((H, W))
    hz = lam * np.exp(-(img[:, 1:] - img[:, :-1]) ** 2 / (2 * sigma ** 2))
    vt = lam * np.exp(-(img[1:, :] - img[:-1, :]) ** 2 / (2 * sigma ** 2))
    return hz, vt


def _per_edge_grid_model(H, W, K, hz, vt, api):
    """The explicit graph of tests/models.py::make_grid_model (pixels row-major, one unary leaf factor per pixel, pairwise
    factors created per pixel as (right, down), protocol-B links) with the factor between (i, j) and (i, j + 1) given
    beta hz[i, j] and the one between (i, j) and (i + 1, j) beta vt[i, j]: one POTTS form per distinct value."""
    g = C.BipartiteFactorGraph()
    pix = [[g.add_variable(C.Variable(name="s", index=(i, j))) for j in range(W)] for i in range(H)]
    un = [[g.add_factor(C.Factor(functional_form="unary")) for j in range(W)] for i in range(H)]
    for i in range(H):
        for j in range(W):
            g.add_edge(pix[i][j], un[i][j], C.Connection(label="out"))
    forms = {}  # beta -> functional form
    pair = []
    for i in range(H):
        for j in range(W):
            for di, dj, b in ((0, 1, hz[i, j] if j + 1 < W else None), (1, 0, vt[i, j] if i + 1 < H else None)):
                if b is None:
                    continue
                f = g.add_factor(C.Factor(functional_form=forms.setdefault(float(b), f"pair{len(forms)}")))
                g.add_edge(pix[i][j], f, C.Connection(label="a"))
                g.add_edge(pix[i + di][j + dj], f, C.Connection(label="b"))
                pair.append((f, pix[i][j], pix[i + di][j + dj]))
    rules = {name: (cap.RULE_POTTS, [b]) for b, name in forms.items()} or {"pair": (cap.RULE_POTTS, [0.0])}
    proc = C.RuleProcessor(rules, family=cap.FAMILY_CATEGORICAL, value_dim=K)
    engine = C.InferenceEngine(model_engine=g, dependency_resolver=C.DefaultDependencyResolver(),
                               inference_request_processor=proc, dtype=cap.F64, api=api)
    models.protocol_b_link(engine, [v for row in pix for v in row])
    return engine, pix, un, pair


def _set(g, hz, vt, row0=0):
    g.set_couplings(*C.shard_couplings(hz, vt, row0, g.H))


# ---- CPU: slicing of global couplings into row shards ----------------------------------------------------------------------
def test_shard_couplings_slices_and_cut_edges_agree():
    H, W = 11, 6
    hz, vt = _smooth_couplings(H, W, 3)
    cuts = [0, 3, 4, 8, H]
    prev = None
    for s in range(len(cuts) - 1):
        row0, rows = cuts[s], cuts[s + 1] - cuts[s]
        h, v = C.shard_couplings(hz, vt, row0, rows)
        assert h.shape == (rows, W - 1) and v.shape == (rows + 1, W) and h.dtype == v.dtype == np.float64
        assert np.array_equal(h, hz[row0:row0 + rows])
        for r in range(rows + 1):  # local row r: the factor between global rows row0 + r - 1 and row0 + r
            gr = row0 + r - 1
            want = vt[gr] if 0 <= gr < H - 1 else np.zeros(W)
            assert np.array_equal(v[r], want), (s, r)
        if prev is not None:
            assert np.array_equal(prev[-1], v[0])  # the shared cut edge: same values on both sides
        prev = v
    # one shard covering the grid: no cut edges
    h, v = C.shard_couplings(hz, vt, 0, H)
    assert not v[0].any() and not v[H].any() and np.array_equal(v[1:H], vt)
    # degenerate grids and bad arguments
    h, v = C.shard_couplings(np.zeros((1, 4)), np.zeros((0, 5)), 0, 1)
    assert h.shape == (1, 4) and v.shape == (2, 5) and not v.any()
    h, v = C.shard_couplings(np.zeros((4, 0)), np.ones((3, 1)), 1, 2)
    assert h.shape == (2, 0) and np.array_equal(v, np.ones((3, 1)))
    with pytest.raises(ValueError):
        C.shard_couplings(hz, vt[:-1], 0, 2)
    with pytest.raises(ValueError):
        C.shard_couplings(hz, vt, 9, 3)


# ---- against the oracle's explicit graph --------------------------------------------------------------------------------------
# every lanes-per-pixel instantiation (K / 4 for fp32, K / 2 for fp64: 1 .. 32) and the one-pixel / one-row / one-column grids
ORACLE_CASES = [(F32, s) for s in ((1, 1, 4), (1, 7, 4), (6, 1, 4), (5, 6, 4), (5, 7, 8), (6, 5, 16), (4, 6, 32), (4, 5, 64),
                                   (3, 4, 128))] + \
               [(F64, s) for s in ((1, 1, 2), (1, 7, 4), (6, 1, 4), (5, 6, 2), (5, 7, 4), (6, 5, 8), (4, 6, 16), (4, 5, 32),
                                   (3, 4, 64))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,shape", ORACLE_CASES, ids=[f"{'f32' if d == F32 else 'f64'}-{h}x{w}xK{k}" for d, (h, w, k) in ORACLE_CASES])
def test_per_edge_grid_vs_oracle(oracle_api, dtype, shape):
    """Three protocol-B sweeps; the marginals and all 8 message planes against the explicit graph with one factor type per
    distinct beta (palette with 0 and a negative value)."""
    H, W, K = shape
    beta, sweeps = 0.7, 3
    hz, vt = _palette_couplings(H, W, 5 + H * W + K)
    unary = np.random.Generator(np.random.PCG64(1234)).dirichlet(np.ones(K), size=(H, W))
    gr = C.PottsGrid(H, W, K, beta, dtype=dtype)
    gr.set_unary(unary)
    _set(gr, hz, vt)
    gr.reset_messages()
    e, pix, un, pair = _per_edge_grid_model(H, W, K, hz, vt, oracle_api)
    vids = [v for row in pix for v in row]
    models.protocol_b_init(e, vids, K)
    usig = [C.get_connection_message_to_variable(e, pix[i][j], un[i][j]) for i in range(H) for j in range(W)]
    unary_used = unary.astype(gr.np_dtype).astype(np.float64)
    for s in range(sweeps):
        st = models.protocol_b_sweep(e, vids, usig, unary_used.reshape(-1, K))
        assert gr.sweep() == st.updates  # n_updates does not depend on the couplings
    want = C.get_values([C.get_variable_marginal(C.get_variable(e, v)) for v in vids]).reshape(H, W, K)
    models.assert_values_close(gr.get_marginals(), want, dtype)
    nb = {0: (-1, 0), 1: (0, -1), 2: (0, 1), 3: (1, 0)}
    fac = {}
    for f, a, b in pair:
        fac[(a, b)] = f
        fac[(b, a)] = f
    for d, (di, dj) in nb.items():
        got_v, got_f = gr.get_messages(d), gr.get_messages(4 + d)
        for i in range(H):
            for j in range(W):
                if 0 <= i + di < H and 0 <= j + dj < W:
                    f = fac[(pix[i][j], pix[i + di][j + dj])]
                    models.assert_values_close(got_v[i, j], C.get_value(C.get_connection_message_to_variable(e, pix[i][j], f)), dtype)
                    models.assert_values_close(got_f[i, j], C.get_value(C.get_connection_message_to_factor(e, pix[i][j], f)), dtype)


# ---- against an independent fp64 numpy flooding BP ----------------------------------------------------------------------------
def _flooding_reference(H, W, K, unary, hz, vt, sweeps):
    """dense numpy flooding BP on the grid with psi_e = exp(beta_e [a==b]) (tests/test_schedules.py::_sync_bp_reference with
    a table per edge; psi_e is symmetric)"""
    nbrs = lambda i, j: [(a, b) for a, b in ((i - 1, j), (i + 1, j), (i, j - 1), (i, j + 1)) if 0 <= a < H and 0 <= b < W]  # noqa: E731

    def psi(p, q):
        (a, b), (c, d) = sorted((p, q))
        return models.potts_table(K, hz[a, b] if a == c else vt[a, b])

    v2f = {((i, j), n): np.full(K, 1.0 / K) for i in range(H) for j in range(W) for n in nbrs(i, j)}
    marg = np.zeros((H, W, K))
    for _ in range(sweeps):
        f2v = {}
        for (src, dst), m in v2f.items():
            out = psi(src, dst) @ m
            f2v[(src, dst)] = out / out.sum()
        new = {}
        for i in range(H):
            for j in range(W):
                inc = {n: f2v[(n, (i, j))] for n in nbrs(i, j)}
                b = unary[i, j].copy()
                for n in sorted(inc):
                    b = b * inc[n]
                marg[i, j] = b / b.sum()
                for n in inc:
                    o = unary[i, j].copy()
                    for n2 in sorted(inc):
                        if n2 != n:
                            o = o * inc[n2]
                    new[((i, j), n)] = o / o.sum()
        v2f = new
    return marg


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,K", [(F32, 4), (F32, 16), (F64, 2), (F64, 8)])
def test_per_edge_grid_vs_numpy_flooding(dtype, K):
    H, W, sweeps = 7, 9, 6
    hz, vt = _smooth_couplings(H, W, 17)
    hz[0, :3] = [-0.4, 0.0, 2.5]  # a repulsive, a vanishing and a strong coupling among the continuous values
    unary = np.random.Generator(np.random.PCG64(99)).dirichlet(np.ones(K), size=(H, W))
    gr = C.PottsGrid(H, W, K, 0.7, dtype=dtype)
    gr.set_unary(unary)
    _set(gr, hz, vt)
    gr.reset_messages()
    for _ in range(sweeps):
        gr.sweep()
    want = _flooding_reference(H, W, K, unary.astype(_npdt(dtype)).astype(np.float64), hz, vt, sweeps)
    models.assert_values_close(gr.get_marginals(), want, dtype)


# ---- equal couplings are the uniform grid -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eager", [False, True], ids=["lazy", "eager"])
@pytest.mark.parametrize("dtype,shape", [(F32, (9, 33, 16)), (F32, (5, 7, 128)), (F64, (9, 33, 16)), (F64, (6, 1, 2))],
                         ids=["f32-9x33xK16", "f32-5x7xK128", "f64-9x33xK16", "f64-6x1xK2"])
def test_equal_couplings_are_the_uniform_grid(monkeypatch, eager, dtype, shape):
    """Every coupling = the create-time beta gives the uniform grid bit for bit (every plane and the marginals); after
    set_couplings(None, None) the grid equals one that never had couplings."""
    H, W, K = shape
    beta = 0.45
    unary = _unary(H, W, K, dtype, 41)
    ref, per = (_grid(monkeypatch, eager, H, W, K, beta, dtype) for _ in range(2))
    per.set_couplings(np.full((H, W - 1), beta), np.full((H + 1, W), beta))
    for g in (ref, per):
        g.set_unary(unary)
        g.reset_messages()
    for s in range(3):
        assert ref.sweep() == per.sweep()
        _assert_equal(_planes(per), _planes(ref), f"sweep {s}")
    # different couplings, then back to the uniform beta: a reset grid then runs exactly like the never-coupled one
    hz, vt = _palette_couplings(H, W, 2)
    _set(per, hz, vt)
    per.sweep()
    per.set_couplings(None, None)
    for g in (ref, per):
        g.reset_messages()
        g.sweep()
        g.sweep()
    _assert_equal(_planes(per), _planes(ref), "after set_couplings(None, None)")


# ---- lazy rebuilds against eager stores ---------------------------------------------------------------------------------------
LAZY_CASES = [(F32, (1, 7, 4)), (F32, (2, 5, 8)), (F32, (3, 6, 16)), (F32, (9, 33, 16)), (F32, (7, 9, 64)), (F32, (6, 5, 128)),
              (F64, (6, 1, 4)), (F64, (3, 6, 2)), (F64, (9, 33, 16)), (F64, (8, 8, 64))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,shape", LAZY_CASES, ids=[f"{'f32' if d == F32 else 'f64'}-{h}x{w}xK{k}" for d, (h, w, k) in LAZY_CASES])
def test_lazy_equals_eager_with_couplings(monkeypatch, dtype, shape):
    """With per-edge couplings the lazily rebuilt m2v planes and marginals equal eager mode's stored ones bit for bit. A
    set_couplings between a sweep and the read leaves the read with the couplings that sweep used: the pending rows are
    rebuilt (one launch) before the new couplings land, and the read launches nothing."""
    H, W, K = shape
    unary = _unary(H, W, K, dtype, 7)
    couplings = [_palette_couplings(H, W, 10 + s) for s in range(4)]
    g = {e: _grid(monkeypatch, e, H, W, K, 0.7, dtype) for e in (True, False)}
    for e in g.values():
        e.set_unary(unary)
        _set(e, *couplings[0])
        e.reset_messages()
    for s in range(3):
        for e in g.values():
            e.sweep()
        _assert_equal(_planes(g[False]), _planes(g[True]), f"sweep {s}")
    for s in range(1, 4):
        for e in g.values():
            e.sweep()
        l0 = _launches()
        _set(g[False], *couplings[s])
        assert _launches() - l0 == (1 if H > 2 else 0), f"set_couplings after sweep: {s}"
        l0 = _launches()
        _set(g[True], *couplings[s])
        assert _launches() == l0  # eager mode has nothing pending
        l0 = _launches()
        lazy = _planes(g[False])
        assert _launches() == l0  # nothing left to rebuild
        _assert_equal(lazy, _planes(g[True]), f"couplings changed after sweep {s}")
    # the new couplings are in effect from the next sweep, and the sweep stays one launch
    l0 = _launches()
    for e in g.values():
        e.sweep()
    assert _launches() - l0 == 2
    _assert_equal(_planes(g[False]), _planes(g[True]), "first sweep with the last couplings")


@pytest.mark.gpu
def test_set_couplings_reads_back_the_sweep_that_used_the_old_ones(monkeypatch):
    """The values read after set_couplings are those of a grid that never saw the new couplings."""
    H, W, K, dtype = 9, 13, 16, F32
    unary = _unary(H, W, K, dtype, 4)
    old, new = _palette_couplings(H, W, 1), _palette_couplings(H, W, 2)
    a, b = (_grid(monkeypatch, False, H, W, K, 0.7, dtype) for _ in range(2))
    for g in (a, b):
        g.set_unary(unary)
        _set(g, *old)
        g.reset_messages()
        g.sweep()
        g.sweep()
    _set(a, *new)
    _assert_equal(_planes(a), _planes(b), "read after set_couplings")
    a.sweep()
    _set(b, *new)
    b.sweep()
    _assert_equal(_planes(a), _planes(b), "sweep after set_couplings")


# ---- row shards ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eager", [False, True], ids=["lazy", "eager"])
def test_two_shards_with_caller_exchange(monkeypatch, eager):
    H, W, K, beta, sweeps = 10, 12, 16, 0.7, 4
    unary = _unary(H, W, K, F32, 3)
    hz, vt = _smooth_couplings(H, W, 5)
    vt[3] = np.linspace(-0.5, 2.0, W)  # the cut edge between the two shards: non-uniform, one repulsive coupling
    full = _grid(monkeypatch, eager, H, W, K, beta)
    full.set_unary(unary)
    _set(full, hz, vt)
    full.reset_messages()
    for _ in range(sweeps):
        full.sweep()
    want = _planes(full)
    top = _grid(monkeypatch, eager, 4, W, K, beta, has_lower=True)
    bot = _grid(monkeypatch, eager, 6, W, K, beta, has_upper=True)
    for sh, row0 in ((top, 0), (bot, 4)):
        sh.set_unary(unary[row0:row0 + sh.H])
        _set(sh, hz, vt, row0)
        sh.reset_messages()
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


@pytest.mark.gpu
@pytest.mark.parametrize("eager", [False, True], ids=["lazy", "eager"])
@pytest.mark.parametrize("dtype", [F32, F64])
def test_three_fused_shards(monkeypatch, dtype, eager):
    """Three row shards connected through cxb_grid_p2p_connect_local, couplings cut by shard_couplings (non-uniform cut
    edges), read between sweeps; the couplings change halfway. Against one unsharded grid."""
    H, W, K, beta, sweeps = 13, 9, 8, 0.45, 6
    unary = _unary(H, W, K, dtype, 8)
    cuts = [0, 4, 9, H]
    cpl = [_palette_couplings(H, W, 21), _smooth_couplings(H, W, 22)]
    full = _grid(monkeypatch, True, H, W, K, beta, dtype)
    full.set_unary(unary)
    full.reset_messages()
    want = []
    for s in range(sweeps):
        if s % 3 == 0:
            _set(full, *cpl[s // 3])
        full.sweep()
        want.append(_planes(full))
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
        if s % 3 == 0:
            for i, sh in enumerate(shards):
                _set(sh, *cpl[s // 3], row0=cuts[i])
        for sh in shards:  # every shard enqueues sweep s before any shard enqueues sweep s + 1
            sh.sweep()
        mid = [shards[1].get_messages(w) for w in range(4)]
        for w in range(4):
            assert np.array_equal(mid[w], want[s][w][cuts[1]:cuts[2]]), f"sweep {s}, middle shard, m2v plane {w}"
    for sh in shards:
        sh.sync()
    got = [np.concatenate(p, axis=0) for p in zip(*(_planes(sh) for sh in shards))]
    _assert_equal(got, want[-1], "last sweep")


# ---- pipelined host jobs ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("eager", [False, True], ids=["lazy", "eager"])
def test_host_jobs_with_couplings_equal_the_plain_calls(monkeypatch, eager):
    """infer_host jobs with couplings set equal set_unary / sweep / get_marginals; a set_couplings between two jobs takes
    effect from the next job."""
    import torch

    H, W, K, sweeps, jobs = 37, 29, 16, 3, 5
    rng = np.random.Generator(np.random.PCG64(21))
    unaries = [rng.dirichlet(np.ones(K), size=(H, W)).astype(np.float32) for _ in range(jobs)]
    cpl = [_smooth_couplings(H, W, 31), _palette_couplings(H, W, 32)]
    switch = 2  # the couplings change before this job
    plain = _grid(monkeypatch, eager, H, W, K, 0.7)
    plain.reset_messages()
    want = []
    for j, u in enumerate(unaries):
        if j in (0, switch):
            _set(plain, *cpl[j > 0])
        plain.set_unary(u)
        for _ in range(sweeps):
            plain.sweep()
        want.append(plain.get_marginals())
    want_planes = _planes(plain)
    piped = _grid(monkeypatch, eager, H, W, K, 0.7)
    piped.reset_messages()
    host_in = [torch.from_numpy(u).pin_memory() for u in unaries]
    host_out = [torch.empty((H, W, K), dtype=torch.float32).pin_memory() for _ in range(jobs)]
    for j in range(jobs):
        if j in (0, switch):
            _set(piped, *cpl[j > 0])
        piped.infer_host(host_in[j].data_ptr(), host_out[j].data_ptr(), sweeps)
    piped.sync()
    for j in range(jobs):
        assert np.array_equal(host_out[j].numpy(), want[j]), f"job {j}"
    _assert_equal(_planes(piped), want_planes, "after the jobs")


# ---- refused input ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F32, F64])
def test_bad_couplings_are_refused_and_change_nothing(monkeypatch, dtype):
    H, W, K, beta = 6, 7, 8, 0.7
    unary = _unary(H, W, K, dtype, 12)
    api = C.default_api()
    bad = [np.nan, np.inf, -np.inf] + ([89.0] if dtype == F32 else [710.0])  # exp(beta) - 1 overflows the engine dtype
    good = _palette_couplings(H, W, 6)
    for start in (None, good):  # a uniform grid, and one with couplings set
        ref, g = (_grid(monkeypatch, False, H, W, K, beta, dtype) for _ in range(2))
        for x in (ref, g):
            x.set_unary(unary)
            if start is not None:
                _set(x, *start)
            x.reset_messages()
            x.sweep()
        for b in bad:
            for where in ("h", "v"):
                hz, vt = (np.full((H, W - 1), 0.3), np.full((H + 1, W), 0.3))
                (hz if where == "h" else vt)[2, 3] = b
                assert api.grid_set_couplings(g.h, hz.ctypes.data_as(cap.f64p), vt.ctypes.data_as(cap.f64p)) == cap.ERR_BAD_ARG
                with pytest.raises(ValueError):
                    g.set_couplings(hz, vt)
        hz = np.zeros((H, W - 1))
        assert api.grid_set_couplings(g.h, hz.ctypes.data_as(cap.f64p), None) == cap.ERR_BAD_ARG  # one array without the other
        with pytest.raises(ValueError):
            g.set_couplings(np.zeros((H, W)), np.zeros((H + 1, W)))  # wrong shape
        _assert_equal(_planes(g), _planes(ref), "after the refused calls")
        for x in (ref, g):
            x.sweep()
        _assert_equal(_planes(g), _planes(ref), "next sweep")
    # fp64 holds what fp32 cannot
    if dtype == F64:
        g = _grid(monkeypatch, False, H, W, K, beta, dtype)
        g.set_couplings(np.full((H, W - 1), 89.0), np.full((H + 1, W), 89.0))


@pytest.mark.gpu
def test_cut_edge_rows_without_a_neighbour_are_not_read(monkeypatch):
    """Rows 0 and H of the vertical couplings are the cut edges: without a neighbour they are neither read nor checked."""
    H, W, K = 5, 6, 8
    unary = _unary(H, W, K, F32, 13)
    hz, vt = _palette_couplings(H, W, 14)
    a, b = (_grid(monkeypatch, False, H, W, K, 0.7) for _ in range(2))
    _set(a, hz, vt)
    h, v = C.shard_couplings(hz, vt, 0, H)
    v[0], v[H] = np.nan, 3.0
    b.set_couplings(h, v)
    for g in (a, b):
        g.set_unary(unary)
        g.reset_messages()
        g.sweep()
        g.sweep()
    _assert_equal(_planes(b), _planes(a), "cut-edge rows ignored")
