"""The generic engine's categorical rules (products, POTTS, CAT_TABLE, HMM_EMIT) at every value width K, on every device path
that serves K, against an independent fp64 numpy reference and against the oracle's sequential schedule.

Which device code evaluates a categorical rule depends on K, the graph size and the schedule:
- K <= 64 on graphs of at most 65,536 signals: one warp per signal (rule_cat_warp) inside the resident level loop, the
  resident memo replay and the sequential executor;
- the per-level schedule (larger graphs, K > 64, tracing on, CXB_ENGINE_RESIDENT=0) and its memo replay: k_rule_cat<T, G,
  MAXC>, G = the next power of two >= K capped at 32 lanes per signal, MAXC = ceil(K / G) components per lane.
The widths below reach every (G, MAXC) instantiation, both sides of every power of two, the resident / per-level boundary at
64 and the two width limits of k_rule_cat (shared memory of CAT_TABLE, MAXC <= 16)."""
from types import SimpleNamespace

import numpy as np
import pytest

from tests import models
from tests._pkg import pkg as C

cap = C.capi
NP = {cap.F32: np.float32, cap.F64: np.float64}
WIDTHS = [2, 3, 5, 8, 12, 16, 17, 31, 32, 33, 48, 63, 64, 65, 96, 100, 128, 200, 256, 500, 512]
# CAT_TABLE stages both orientations of the K x K table plus eight K-wide inputs in at most 200 KiB of shared memory:
# 8K^2 + 32K bytes in fp32, 16K^2 + 64K in fp64
TABLE_MAX = {cap.F32: 158, cap.F64: 111}
POTTS_MAX = 512  # 32 lanes x 16 components
MODELS = ["grid_potts", "grid_table", "row_potts", "hmm", "powerlaw"]
TABLE_MODELS = {"grid_table", "hmm", "powerlaw"}
SWEEPS = 4
BETA = 0.7
HMM_T, HMM_M = 6, 7  # M is not a power of two; the last observation is symbol M - 1


# ---- fp64 reference (numpy, independent of the oracle) -------------------------------------------------------------------
def _normalise(x):
    return x / x.sum(axis=-1, keepdims=True)


def potts_rule(inc, beta):
    """m2v = exp(beta * I) @ in, normalised: sum_b in[b] + (e^beta - 1) in[a]."""
    return _normalise(inc.sum(axis=-1, keepdims=True) + np.expm1(beta) * inc)


def table_rule(inc, table, u_is_low):
    """CAT_TABLE: table[x_lo, x_hi] is indexed by (lower variable id, higher variable id). A message from the lower variable u
    to the higher v is out[a] = sum_b table[b, a] in[b]; from the higher to the lower, out[a] = sum_b table[a, b] in[b]."""
    return _normalise(inc @ table if u_is_low else inc @ table.T)


def hmm_emit_rule(E, o):
    """HMM_EMIT with emission table E[K, M] and observed symbol o: E[:, o], normalised."""
    return _normalise(E[:, int(o)])


class Reference:
    """Belief propagation on an explicit edge list, fp64. Variables 0..n-1 (ids ascend with the index); pairs[p] = (u, v, rule)
    with u < v and rule ("potts", beta) or ("table", T[x_u, x_v]); leaf messages (unary evidence, prior, emission) enter as
    one product per variable. Directed slot 2p is factor p -> v (its input is the m2f of u), slot 2p + 1 is p -> u."""

    def __init__(self, K, n, pairs):
        self.K, self.n, self.pairs = K, n, pairs
        self.tgt = np.array([x for (u, v, _) in pairs for x in (v, u)], dtype=np.int64)
        self.incoming = [np.flatnonzero(self.tgt == i) for i in range(n)]
        self.m2f = np.full((2 * len(pairs), K), 1.0 / K)  # m2f[s]: variable tgt[s] -> the factor of slot s
        self.m2v = np.zeros((2 * len(pairs), K))
        self.marginal = np.zeros((n, K))

    def sweep(self, leaf):
        """Protocol B (SURVEY Appendix B) sweep: every m2v from the m2f held before the sweep, then the marginals and the
        linked m2f from the new m2v. leaf[i]: product of the leaf messages of variable i."""
        new = np.empty_like(self.m2v)
        for p, (u, v, rule) in enumerate(self.pairs):
            for s, low in ((2 * p, True), (2 * p + 1, False)):
                inc = self.m2f[s ^ 1]
                new[s] = potts_rule(inc, rule[1]) if rule[0] == "potts" else table_rule(inc, rule[1], low)
        self.m2v = new
        for i in range(self.n):
            sl = self.incoming[i]
            msgs = self.m2v[sl]
            self.marginal[i] = _normalise(leaf[i] * np.prod(msgs, axis=0))
            for j, s in enumerate(sl):
                self.m2f[s] = _normalise(leaf[i] * np.prod(np.delete(msgs, j, axis=0), axis=0))


def exact_row_marginals(leaf, pairs, K):
    """Brute-force marginals of a chain of len(leaf) variables (K^W states)."""
    W = len(leaf)
    joint = np.ones((K,) * W)
    for i in range(W):
        joint = joint * leaf[i].reshape([K if d == i else 1 for d in range(W)])
    for (u, v, rule) in pairs:
        psi = np.exp(rule[1] * np.eye(K)) if rule[0] == "potts" else rule[1]
        joint = joint * psi.reshape([K if d in (u, v) else 1 for d in range(W)])
    return np.stack([_normalise(joint.sum(axis=tuple(d for d in range(W) if d != i))) for i in range(W)])


def forward_backward(prior, A, E, obs):
    """Exact smoothed marginals of an HMM: p(z_0) = prior, p(z_t+1 | z_t) ∝ A[z_t, z_t+1], p(y_t | z_t) ∝ E[z_t, y_t]."""
    T = len(obs)
    alpha, beta = np.zeros((T, len(prior))), np.ones((T, len(prior)))
    alpha[0] = _normalise(prior * E[:, obs[0]])
    for t in range(1, T):
        alpha[t] = _normalise((alpha[t - 1] @ A) * E[:, obs[t]])
    for t in range(T - 2, -1, -1):
        beta[t] = _normalise(A @ (E[:, obs[t + 1]] * beta[t + 1]))
    return _normalise(alpha * beta)


# ---- models: one seeded instance per (model, K, dtype), inputs rounded to the engine dtype --------------------------------
def _round(x, dtype):
    return np.asarray(x, dtype=np.float64).astype(NP[dtype]).astype(np.float64)


def _grid_pairs(H, W):
    """4-neighbourhood, horizontal then vertical edge of each pixel in row-major order (tests/models.py::make_grid_model)."""
    out = []
    for i in range(H):
        for j in range(W):
            if j + 1 < W:
                out.append((i * W + j, i * W + j + 1))
            if i + 1 < H:
                out.append((i * W + j, (i + 1) * W + j))
    return out


class Model:
    """Seeded model description shared by the reference, the oracle and the device engines."""

    def __init__(self, kind, K, dtype, seed=0):
        self.kind, self.K, self.dtype = kind, K, dtype
        rng = np.random.Generator(np.random.PCG64([K, sum(map(ord, kind)), seed]))
        if kind == "hmm":
            self.n = HMM_T
            self.A = _round(rng.dirichlet(np.ones(K), size=K) * K, dtype)
            self.E = _round(rng.dirichlet(np.ones(K), size=HMM_M).T * K, dtype)
            self.pairs = [(t, t + 1, ("table", self.A)) for t in range(HMM_T - 1)]
            obs = rng.integers(0, HMM_M, size=HMM_T)
            obs[-1] = HMM_M - 1
            self.obs = obs
            return
        if kind in ("grid_potts", "grid_table", "potts80"):
            H, W = (80, 80) if kind == "potts80" else (3, 4)
            edges = _grid_pairs(H, W)
            self.n = H * W
        elif kind == "row_potts":
            W = 4 if K <= 8 else 3 if K <= 40 else 2  # K^W states enumerated
            edges = [(i, i + 1) for i in range(W - 1)]
            self.n = W
        else:  # powerlaw: Chung-Lu graph with a hub (the resolver gives it segment-tree product nodes)
            self.n = 40
            edges = models.chung_lu_edges(self.n, 80, seed=7)
        if kind == "grid_table" or kind == "powerlaw":
            n_tables = 1 if kind == "grid_table" else 3
            self.tables = [_round(np.exp(0.5 * rng.standard_normal((K, K))), dtype) for _ in range(n_tables)]  # asymmetric
            self.pairs = [(u, v, ("table", self.tables[p % n_tables])) for p, (u, v) in enumerate(edges)]
        else:
            self.pairs = [(u, v, ("potts", BETA)) for (u, v) in edges]

    def unary(self, sweep):
        """Evidence of a sweep: fresh on loopy graphs, constant on trees (so that BP converges to the exact marginals)."""
        tree = self.kind == "row_potts"
        rng = np.random.Generator(np.random.PCG64(99 if tree else 100 + sweep))
        return _round(rng.dirichlet(np.ones(self.K), size=self.n), self.dtype)

    def leaf(self, sweep):
        if self.kind != "hmm":
            return self.unary(sweep)
        leaf = np.stack([hmm_emit_rule(self.E, o) for o in self.obs])
        leaf[0] = leaf[0] * (1.0 / self.K)
        return leaf

    # -- engines --
    def build(self, api, dtype):
        """An engine of the model and the signal ids the checks read, as one handle."""
        K, h = self.K, SimpleNamespace()
        if self.kind == "hmm":
            e, z, y, prior, em, tr = models.make_hmm_model(HMM_T, K, HMM_M, self.A, self.E, api, dtype=dtype)
            h.vs, h.fac, h.hmm = z, tr, (z, y, prior, em)
            h.emit_sigs = [C.get_connection_message_to_variable(e, z[t], em[t]).sid for t in range(HMM_T)]
            h.data_sigs = [C.get_connection_message_to_factor(e, y[t], em[t]).sid for t in range(HMM_T)]
            h.data_sigs.append(C.get_connection_message_to_variable(e, z[0], prior).sid)
        else:
            g = C.BipartiteFactorGraph()
            vs = [g.add_variable(C.Variable(name="v", index=(i,))) for i in range(self.n)]
            un = [g.add_factor(C.Factor(functional_form="unary")) for _ in range(self.n)]
            for i in range(self.n):
                g.add_edge(vs[i], un[i], C.Connection(label="out"))
            fac, rules = [], {}
            for p, (u, v, rule) in enumerate(self.pairs):
                form = rule[0] if rule[0] == "potts" else f"table{next(i for i, t in enumerate(self.tables) if t is rule[1])}"
                rules[form] = (cap.RULE_POTTS, [rule[1]]) if rule[0] == "potts" else (cap.RULE_CAT_TABLE, rule[1].ravel())
                f = g.add_factor(C.Factor(functional_form=form))
                g.add_edge(vs[u], f, C.Connection(label="a"))
                g.add_edge(vs[v], f, C.Connection(label="b"))
                fac.append(f)
            proc = C.RuleProcessor(rules, family=cap.FAMILY_CATEGORICAL, value_dim=K)
            e = C.InferenceEngine(model_engine=g, dependency_resolver=C.DefaultDependencyResolver(),
                                  inference_request_processor=proc, dtype=dtype, api=api)
            models.protocol_b_link(e, vs)
            models.protocol_b_init(e, vs, K)
            h.unary_sigs = [C.get_connection_message_to_variable(e, vs[i], un[i]) for i in range(self.n)]
            h.vs, h.fac, h.emit_sigs, h.data_sigs = vs, fac, [], [s.sid for s in h.unary_sigs]
        m2v, m2f = [], []
        for p, (u, v, _) in enumerate(self.pairs):
            for t in (v, u):
                m2v.append(C.get_connection_message_to_variable(e, h.vs[t], h.fac[p]).sid)
                m2f.append(C.get_connection_message_to_factor(e, h.vs[t], h.fac[p]).sid)
        h.e, h.m2v_sigs, h.m2f_sigs = e, np.array(m2v), np.array(m2f)
        h.marg_sigs = np.array([C.get_variable(e, v).marginal.sid for v in h.vs])
        return h

    def set_data(self, h, sweep, obs=None):
        """The evidence of a sweep: observations and prior (HMM), unary messages (protocol B)."""
        if self.kind == "hmm":
            z, y, prior, em = h.hmm
            models.hmm_set_data(h.e, z, y, prior, em, self.obs if obs is None else obs, self.K)
        else:
            C.set_values(h.unary_sigs, self.unary(sweep))

    def run_sweep(self, h, sweep, schedule, obs=None):
        self.set_data(h, sweep, obs)
        return C.update_marginals(h.e, h.vs, schedule=schedule)


def reference_sweeps(model, n_sweeps):
    """[(m2v, m2f, marginal)] after every sweep. The HMM is one request on a tree: the engine computes the converged messages,
    which flooding sweeps reach after as many sweeps as the chain is long."""
    ref = Reference(model.K, model.n, model.pairs)
    out = []
    for s in range(n_sweeps):
        for _ in range(HMM_T if model.kind == "hmm" else 1):
            ref.sweep(model.leaf(s))
        out.append((ref.m2v.copy(), ref.m2f.copy(), ref.marginal.copy()))
    return out


def exact_marginals(model):
    if model.kind == "hmm":
        return forward_backward(np.full(model.K, 1.0 / model.K), model.A, model.E, model.obs)
    return exact_row_marginals(model.leaf(0), model.pairs, model.K)


def widths_of(kind, dtype):
    """CAT_TABLE models stop at the table limit; test_width_limits checks the limit itself."""
    return [K for K in WIDTHS if kind not in TABLE_MODELS or K <= TABLE_MAX[dtype]]


def _values(h):
    st = h.e.store
    return C.get_values([C.Signal(st, s) for s in range(st.n_signals())])


def check_against_reference(model, h, vals, ref, tol_dtype, what):
    m2v, m2f, marg = ref
    models.assert_values_close(vals[h.m2v_sigs], m2v, tol_dtype, err_msg=f"{what}: m2v")
    models.assert_values_close(vals[h.m2f_sigs], m2f, tol_dtype, err_msg=f"{what}: m2f")
    models.assert_values_close(vals[h.marg_sigs], marg, tol_dtype, err_msg=f"{what}: marginals")
    if h.emit_sigs:
        want = np.stack([hmm_emit_rule(model.E, o) for o in model.obs])
        models.assert_values_close(vals[h.emit_sigs], want, tol_dtype, err_msg=f"{what}: HMM_EMIT m2v")


def check_sums(h, state, vals, dtype, what):
    """Every message a rule computed sums to 1 (the data signals are set by the caller)."""
    computed = np.array([c for (c, _p, _n) in state], dtype=bool)
    computed[h.data_sigs] = False
    sums = vals[computed].sum(axis=1)
    bad = np.abs(sums - 1.0) > models.TOL[dtype]
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} messages do not sum to 1 (worst {sums[bad][np.argmax(np.abs(sums[bad] - 1))]!r})"


def _set_env(mp, env):
    for k in ("CXB_MEMO", "CXB_ENGINE_RESIDENT", "CXB_CERTIFY", "CXB_PLAN"):
        mp.delenv(k, raising=False)
    for k, v in env.items():
        mp.setenv(k, v)


# ---- (b) the reference itself against the oracle, on the CPU ----------------------------------------------------------------
@pytest.mark.parametrize("kind,K", [(kind, K) for kind in MODELS for K in widths_of(kind, cap.F32)])
def test_reference_equals_oracle_sequential(oracle_api, kind, K):
    model = Model(kind, K, cap.F64)
    h = model.build(oracle_api, cap.F64)
    ref = reference_sweeps(model, SWEEPS)
    for s in range(SWEEPS):
        model.run_sweep(h, s, "seq")
        check_against_reference(model, h, _values(h), ref[s], cap.F64, f"sweep {s}")
    check_sums(h, models.engine_state(h.e)[0], _values(h), cap.F64, "oracle")
    if kind in ("hmm", "row_potts"):
        models.assert_values_close(_values(h)[h.marg_sigs], exact_marginals(model), cap.F64, err_msg="exact marginals")
    if kind == "powerlaw":
        assert max(len(C.get_connected_factor_ids(h.e, v)) for v in h.vs) > 6  # a hub: the resolver builds product nodes


# ---- (c)-(f) every device path at every width ------------------------------------------------------------------------------
# path: (environment, schedule, tracing)
PATHS = {
    "resident": ({"CXB_MEMO": "0"}, "lvl", False),
    "level": ({"CXB_MEMO": "0", "CXB_ENGINE_RESIDENT": "0"}, "lvl", False),
    "traced": ({"CXB_MEMO": "0"}, "lvl", True),
    "seq": ({"CXB_MEMO": "0"}, "seq", False),
    "replay_resident": ({}, "auto", False),
    "replay_level": ({"CXB_ENGINE_RESIDENT": "0"}, "auto", False),
}


def paths_of(K):
    return list(PATHS) if K <= 64 else ["level", "traced", "replay_level"]


def _build_on_path(model, device_api, path, mp):
    env, schedule, traced = PATHS[path]
    _set_env(mp, env)
    h = model.build(device_api, model.dtype)
    if traced:
        h.e.store.check(h.e.api.trace_enable(h.e.store.h, 1))
    return h, schedule


def _run_path(model, device_api, path, oracle_states, ref, monkeypatch):
    dtype = model.dtype
    with monkeypatch.context() as mp:
        h, schedule = _build_on_path(model, device_api, path, mp)
        ran, launches = [], []
        for s in range(SWEEPS):
            st = model.run_sweep(h, s, schedule)
            ran.append(C.last_schedule(h.e))
            launches.append(st.kernel_launches)
            what = f"{path}, sweep {s}"
            if path.startswith("replay"):
                vals = _values(h)  # engine_state would evaluate is_pending and change the flag state the memo is keyed on
            else:
                state, vals = models.engine_state(h.e)
                assert state == oracle_states[s][0], f"{what}: computed / pending flags or nibbles differ from the oracle"
                check_sums(h, state, vals, dtype, what)
            models.assert_values_close(vals, oracle_states[s][1], dtype, err_msg=f"{what}: values vs oracle")
            check_against_reference(model, h, vals, ref[s], dtype, what)
        state, vals = models.engine_state(h.e)
        assert state == oracle_states[-1][0], f"{path}: flags or nibbles differ from the oracle"
        check_sums(h, state, vals, dtype, path)
    if path in ("resident", "level", "traced"):
        assert ran == [cap.SCHEDULE_LEVEL] * SWEEPS, (path, ran)
    if path == "resident":
        assert max(launches) <= 3, (path, launches)  # request + request check + one resident level loop
    if path in ("level", "traced"):
        assert min(launches) > 3, (path, launches)  # frontier discovery and rule kernels, level by level
    if path == "seq":
        assert ran == [cap.SCHEDULE_SEQUENTIAL] * SWEEPS, ran
    if path.startswith("replay"):
        assert ran[-1] == cap.RAN_REPLAY, (path, ran)
    return h, state, vals, launches


@pytest.mark.gpu
@pytest.mark.parametrize("kind,K,dtype", [(kind, K, dtype) for kind in MODELS for dtype in (cap.F64, cap.F32) for K in widths_of(kind, dtype)])
def test_every_path_at_every_width(oracle_api, device_api, monkeypatch, kind, K, dtype):
    model = Model(kind, K, dtype)
    ho = model.build(oracle_api, cap.F64)
    oracle_states = []
    for s in range(SWEEPS):
        model.run_sweep(ho, s, "seq")
        oracle_states.append(models.engine_state(ho.e))
    ref = reference_sweeps(model, SWEEPS)
    finals = {path: _run_path(model, device_api, path, oracle_states, ref, monkeypatch) for path in paths_of(K)}
    if kind in ("hmm", "row_potts"):  # trees: converged BP is exact
        for path, (h, _st, vals, _l) in finals.items():
            models.assert_values_close(vals[h.marg_sigs], exact_marginals(model), dtype, err_msg=f"{path}: exact marginals")
    # rule_cat_warp reduces over 32 lanes, k_rule_cat over G: with the padding at zero, the extra lanes add exact zeros
    # first, and every path leaves the same bits
    first = next(iter(finals))
    for path, (_h, st, vals, _l) in finals.items():
        assert st == finals[first][1], (first, path)
        np.testing.assert_array_equal(vals, finals[first][2], err_msg=f"{path} vs {first}")
    if "replay_resident" in finals:  # one replay launch vs the recorded levels' rule kernels
        assert finals["replay_resident"][3][-1] < finals["replay_level"][3][-1]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
def test_potts_80x80_default_routing_reaches_the_per_level_kernel(oracle_api, device_api, monkeypatch, dtype):
    """69,760 signals: above the resident limit of 65,536, so the default schedule runs k_rule_cat at K = 5 (G = 8, one
    component per lane, three padding lanes)."""
    _set_env(monkeypatch, {})
    model = Model("potts80", 5, dtype)
    ho = model.build(oracle_api, cap.F64)
    hd = model.build(device_api, dtype)
    assert hd.e.store.n_signals() == 69760
    ref = Reference(model.K, model.n, model.pairs)
    for s in range(3):
        model.run_sweep(ho, s, "seq")
        st = model.run_sweep(hd, s, "auto")
        assert C.last_schedule(hd.e) in (cap.SCHEDULE_LEVEL, cap.RAN_REPLAY) and st.kernel_launches > 3, (C.last_schedule(hd.e), st.kernel_launches)
        ref.sweep(model.leaf(s))
        so, vo = models.engine_state(ho.e)
        sd, vd = models.engine_state(hd.e)
        assert so == sd
        models.assert_values_close(vd, vo, dtype, err_msg=f"sweep {s}: values vs oracle")
        check_against_reference(model, hd, vd, (ref.m2v, ref.m2f, ref.marginal), dtype, f"sweep {s}")
        check_sums(hd, sd, vd, dtype, f"sweep {s}")


# ---- (g) width limits ----------------------------------------------------------------------------------------------------
def _limit_model(kind, K, dtype):
    """pair: one factor between two variables (the refused rule is the first level of the request); hmm: the CAT_TABLE
    levels come after the HMM_EMIT level and a level of m2f products; grid_potts: the 3 x 4 grid."""
    model = Model("grid_table" if kind == "pair_table" else "grid_potts" if kind == "pair_potts" else kind, K, dtype, seed=5)
    if kind.startswith("pair"):
        model.n, model.pairs = 2, [(0, 1, model.pairs[0][2])]
    return model


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
@pytest.mark.parametrize("kind", ["pair_table", "hmm", "pair_potts", "grid_potts"])
def test_width_limits(oracle_api, device_api, dtype, kind):
    """The widest K each rule serves runs and matches the oracle; one more is refused with ValueError before the request
    changes anything, also where the refused rule is not in the first level."""
    K_max = POTTS_MAX if kind.endswith("potts") else TABLE_MAX[dtype]
    for K in (K_max, K_max + 1):
        model = _limit_model(kind, K, dtype)
        hd = model.build(device_api, dtype)
        if K == K_max:
            ho = model.build(oracle_api, cap.F64)
            model.run_sweep(ho, 0, "seq")
            model.run_sweep(hd, 0, "auto")
            so, vo = models.engine_state(ho.e)
            sd, vd = models.engine_state(hd.e)
            assert so == sd
            models.assert_values_close(vd, vo, dtype)
            check_sums(hd, sd, vd, dtype, f"K = {K}")
            continue
        model.set_data(hd, 0)
        before = models.engine_state(hd.e)
        with pytest.raises(ValueError, match="value_dim too large"):
            C.update_marginals(hd.e, hd.vs)
        after = models.engine_state(hd.e)
        assert before[0] == after[0], "computed / pending flags or nibbles changed by a refused request"
        np.testing.assert_array_equal(after[1], before[1], err_msg="values changed by a refused request")


# ---- (h) rule-argument errors --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("K", [5, 100])
def test_hmm_symbol_out_of_range_raises_the_same_error_everywhere(oracle_api, device_api, monkeypatch, K):
    """A symbol equal to M is a bad argument: ValueError from the oracle and from every device path."""
    model = Model("hmm", K, cap.F64)
    bad = model.obs.copy()
    bad[2] = HMM_M
    ho = model.build(oracle_api, cap.F64)
    with pytest.raises(ValueError, match="symbol out of range"):
        model.run_sweep(ho, 0, "seq", obs=bad)
    for path in paths_of(K):
        with monkeypatch.context() as mp:
            h, schedule = _build_on_path(model, device_api, path, mp)
            if path.startswith("replay"):
                ran = []
                for s in range(3):
                    model.run_sweep(h, s, schedule)
                    ran.append(C.last_schedule(h.e))
                assert ran[-1] == cap.RAN_REPLAY, (path, ran)
            with pytest.raises(ValueError, match="symbol out of range"):
                model.run_sweep(h, 0, schedule, obs=bad)
            if path.startswith("replay"):  # the bad request itself was replayed (the rule kernels of the replay refused it)
                assert C.last_schedule(h.e) == cap.RAN_REPLAY, path
            elif path != "seq":
                assert C.last_schedule(h.e) == cap.SCHEDULE_LEVEL, path
