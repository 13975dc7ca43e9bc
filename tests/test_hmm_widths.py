"""The structured HMM engine (cxb_hmm_*) on every kernel path, at state counts, symbol counts, lengths and batch sizes on
both sides of every boundary of its dispatch rule, in fp32 and fp64, against an independent fp64 forward-backward.

Which kernel runs (Hmm::launch_t in hmm.cu; `hmm_path` below is a copy of the rule):
- fp32, K = 64: k_hmm64_pass, the emission table in shared memory for M <= 128, else read from global memory;
- fp32, K a multiple of 64 in [128, 1024], M <= 64: the tcgen05 path, k_hmm_tc_step_pair<NT>, NT = 32 while
  (chain tiles of 128) x (K / 32) x 2 CTAs fit one per SM (148 on a B200), else 64;
- K = 32: k_hmm_pass with the table in registers;
- everything else: k_hmm_pass with the K x K table in shared memory, whole when it fits next to the staging, else streamed
  in row tiles; the emission table in shared memory when it and one table row fit in 200 KiB, else in global memory.
Vectors are compared at the north-star tolerance (tests/models.py::assert_values_close) for every chain and time step."""
import itertools

import numpy as np
import pytest

from tests import models
from tests._pkg import pkg as C
from tests.test_device_parity import HMM_TC_SHAPES

cap = C.capi
gpu = pytest.mark.gpu
NP = {cap.F32: np.float32, cap.F64: np.float64}
DTYPES = [cap.F32, cap.F64]
N_SM = 148  # B200
SMEM_BUDGET = 200 * 1024  # bytes of shared memory k_hmm_pass plans with
HMM_WARPS = 8  # chains per CTA of k_hmm_pass


def _id(d):
    return "f32" if d == cap.F32 else "f64"


# ---- the dispatch rule of hmm.cu -----------------------------------------------------------------------------------------
def simt_plan(dtype, K, M):
    """(emission table in shared memory, table rows per tile) of the streamed k_hmm_pass."""
    esz = 4 if dtype == cap.F32 else 8
    stage, em, row = HMM_WARPS * K * esz, M * K * esz, K * esz
    em_smem = stage + em + row <= SMEM_BUDGET
    return em_smem, min(K, (SMEM_BUDGET - stage - (em if em_smem else 0)) // row)


def hmm_path(dtype, K, M, B, no_tc=False):
    if dtype == cap.F32 and K == 64:
        return "k64/smem" if M <= 128 else "k64/global"
    if dtype == cap.F32 and not no_tc and K % 64 == 0 and 128 <= K <= 1024 and M <= 64:
        return "tc32" if -(-B // 128) * (K // 32) * 2 <= N_SM else "tc64"
    if K == 32:
        return "register"
    em_smem, rows = simt_plan(dtype, K, M)
    return ("whole" if rows >= K else "tiled") + ("/smem" if em_smem else "/global")


SIMT_LABELS = ["register", "whole/smem", "tiled/smem", "whole/global", "tiled/global"]
LABELS = {cap.F64: SIMT_LABELS, cap.F32: SIMT_LABELS + ["k64/smem", "k64/global", "tc32", "tc64"]}


# ---- the GPU matrix ------------------------------------------------------------------------------------------------------
KS = [2, 3, 5, 17, 31, 32, 33, 63, 64, 65, 96, 100, 127, 128, 129, 160, 192, 210, 255, 256, 320, 500, 512, 700, 1000, 1024]
MS = [1, 7, 64, 65, 128, 129, 256]  # both sides of M <= 64 (tcgen05) and M <= 128 (k_hmm64_pass), and the largest M
B_MATRIX, T_MATRIX = 9, 40  # a CTA of k_hmm_pass with one live warp; T crosses one 32-step observation block
# (K, M, B, T) beyond the cross product: fp32 whole / global at (200, 256), tiled / global at (255, 200) and (1000, 44);
# tcgen05 with NT = 64 (5 x 16 x 2 and 3 x 32 x 2 CTAs)
EXTRA = {cap.F32: [(200, 256, B_MATRIX, T_MATRIX), (255, 200, B_MATRIX, T_MATRIX), (1000, 44, B_MATRIX, T_MATRIX),
                   (512, 16, 513, 6), (1024, 8, 300, 5)],
         cap.F64: []}


def matrix(dtype):
    return [(K, M, B_MATRIX, T_MATRIX) for K, M in itertools.product(KS, MS)] + EXTRA[dtype]


# one shape (K, M, B) of each path, for the length, batch, state and error tests
REPRESENTATIVE = {
    cap.F32: {"register": (32, 7, 9), "whole/smem": (33, 7, 9), "tiled/smem": (192, 128, 9), "whole/global": (210, 256, 9),
              "tiled/global": (255, 200, 9), "k64/smem": (64, 7, 9), "k64/global": (64, 200, 9), "tc32": (128, 7, 9),
              "tc64": (512, 16, 513)},
    cap.F64: {"register": (32, 7, 9), "whole/smem": (100, 7, 9), "tiled/smem": (1000, 7, 9), "whole/global": (100, 256, 9),
              "tiled/global": (192, 128, 9)},
}


def rep_cases(skip=()):
    return [pytest.param(d, lbl, id=f"{_id(d)}-{lbl}") for d in DTYPES for lbl in LABELS[d] if lbl not in skip]


# ---- fp64 reference ------------------------------------------------------------------------------------------------------
def reference(A, E, obs):
    """Scaled forward-backward, fp64, vectorised over chains. A[K][K] as the engine stores it, E[K][M] raw, obs[T][B].
    Returns (forward messages m2f(z_t, tr_t), marginals), each [T][B][K] and normalised."""
    A = np.asarray(A, dtype=np.float64)
    En = E / E.sum(axis=0, keepdims=True)  # m2v(z_t, em_t) = normalise(E[:, o_t]) (HMM_EMIT)
    em = En.T[np.asarray(obs, dtype=np.int64)]  # [T][B][K]
    T = em.shape[0]
    fwd, marg = np.empty_like(em), np.empty_like(em)
    v = em[0] / em[0].sum(axis=-1, keepdims=True)
    fwd[0] = v
    for t in range(1, T):
        v = em[t] * (v @ A)
        v /= v.sum(axis=-1, keepdims=True)
        fwd[t] = v
    marg[T - 1] = fwd[T - 1]
    w = em[T - 1] / em[T - 1].sum(axis=-1, keepdims=True)
    for t in range(T - 2, -1, -1):
        back = w @ A.T
        g = fwd[t] * back
        marg[t] = g / g.sum(axis=-1, keepdims=True)
        w = em[t] * back
        w /= w.sum(axis=-1, keepdims=True)
    return fwd, marg


def brute_force_marginals(A, E, o):
    """p(z_t | y_1..T) of one chain (uniform prior on z_1) by enumerating every state path."""
    K, T = A.shape[0], len(o)
    marg = np.zeros((T, K))
    for path in itertools.product(range(K), repeat=T):
        p = E[path[0], o[0]]
        for t in range(1, T):
            p *= A[path[t - 1], path[t]] * E[path[t], o[t]]
        marg[np.arange(T), path] += p
    return marg / marg.sum(axis=-1, keepdims=True)


def make_inputs(K, M, B, T, seed, obs=None):
    rng = np.random.Generator(np.random.PCG64(seed))
    A = rng.dirichlet(np.full(K, 0.5), size=K)
    E = rng.gamma(0.7, size=(K, M)) + 1e-3  # columns do not sum to 1: the host normalisation matters
    if obs is None:
        obs = rng.integers(0, M, size=(T, B), dtype=np.uint8)
        obs[-1, -1] = M - 1  # the largest symbol occurs
    return A, E, obs


def run(dtype, A, E, obs, M, check_launches=None):
    T, B = obs.shape
    K = A.shape[0]
    hm = C.HmmBatch(B, T, K, M, dtype=dtype)
    hm.set_tables(A, E)
    hm.set_observations(obs)
    api = C.default_api()
    l0 = api.kernel_launches()
    assert hm.update_marginals() == B * (6 * T - 4)
    launches = api.kernel_launches() - l0
    if check_launches is not None:
        assert launches == (T + 4 if check_launches.startswith("tc") else 2), (check_launches, launches)
    return hm, hm.get_forward(), hm.get_marginals()


def check(dtype, got_f, got_m, A, E, obs, what=""):
    want_f, want_m = reference(A.astype(NP[dtype]).astype(np.float64), E, obs)
    models.assert_values_close(got_f, want_f, dtype, err_msg=f"{what}: forward messages")
    models.assert_values_close(got_m, want_m, dtype, err_msg=f"{what}: marginals")
    for name, x in (("forward", got_f), ("marginal", got_m)):
        s = x.astype(np.float64).sum(axis=-1)
        bad = np.abs(s - 1.0) > models.TOL[dtype]
        assert not bad.any(), f"{what}: {int(bad.sum())} {name} vectors do not sum to 1 (worst {s.flat[np.argmax(np.abs(s - 1))]!r})"


def run_and_check(dtype, K, M, B, T, seed, label=None, obs=None):
    A, E, obs = make_inputs(K, M, B, T, seed, obs)
    hm, got_f, got_m = run(dtype, A, E, obs, M, check_launches=label)
    check(dtype, got_f, got_m, A, E, obs, what=f"{_id(dtype)} K={K} M={M} B={B} T={T} {label}")
    return hm


# ---- CPU: the reference and the rule -------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,M,T", [(2, 2, 1), (2, 3, 5), (3, 2, 4), (4, 3, 5), (3, 1, 3)])
def test_reference_equals_brute_force(K, M, T):
    B = 3
    A, E, obs = make_inputs(K, M, B, T, seed=10 * K + T)
    fwd, marg = reference(A, E, obs)
    for b in range(B):
        np.testing.assert_allclose(marg[:, b], brute_force_marginals(A, E, obs[:, b]), rtol=1e-12, atol=0)
        for t in range(T):  # the forward message m2f(z_t, tr_t) is the filtering distribution: the last marginal of y_1..t
            np.testing.assert_allclose(fwd[t, b], brute_force_marginals(A, E, obs[: t + 1, b])[t], rtol=1e-12, atol=0)


@pytest.mark.parametrize("K,M", [(2, 1), (3, 5), (33, 7)])
def test_reference_equals_oracle_explicit_graph(oracle_api, K, M):
    B, T = 3, 12
    A, E, obs = make_inputs(K, M, B, T, seed=K + M)
    fwd, marg = reference(A, E, obs)
    for b in range(B):
        e, z, y, prior, em, tr = models.make_hmm_model(T, K, M, A, E, oracle_api)
        models.hmm_set_data(e, z, y, prior, em, obs[:, b], K)
        C.update_marginals(e, z, schedule="seq")
        want_m = C.get_values([C.get_variable_marginal(C.get_variable(e, v)) for v in z])
        want_f = C.get_values([C.get_connection_message_to_factor(e, z[t], tr[t]) for t in range(T - 1)])
        np.testing.assert_allclose(marg[:, b], want_m, rtol=1e-12, atol=1e-300)
        np.testing.assert_allclose(fwd[:-1, b], want_f, rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("dtype", DTYPES, ids=_id)
def test_matrix_reaches_every_path(dtype):
    """Every path of the rule is run at least twice by the GPU matrix, and the shapes named in hmm.cu's history land where
    the arithmetic of launch_t puts them."""
    seen = {}
    for K, M, B, T in matrix(dtype):
        seen.setdefault(hmm_path(dtype, K, M, B), []).append((K, M))
    for label in LABELS[dtype]:
        assert len(seen.get(label, [])) >= 2, (label, seen.get(label))
    assert set(seen) == set(LABELS[dtype])
    for label, (K, M, B) in REPRESENTATIVE[dtype].items():
        assert hmm_path(dtype, K, M, B) == label, (label, K, M, B)
    named = {cap.F32: {(210, 256): "whole/global", (255, 200): "tiled/global", (512, 128): "tiled/global",
                       (1000, 44): "tiled/global", (1024, 256): "tiled/global", (192, 128): "tiled/smem",
                       (320, 129): "tiled/smem", (500, 64): "tiled/smem"},
             cap.F64: {(100, 256): "whole/global", (192, 128): "tiled/global", (512, 64): "tiled/global",
                       (1024, 256): "tiled/global", (96, 256): "tiled/smem", (1000, 7): "tiled/smem"}}[dtype]
    for (K, M), label in named.items():
        assert hmm_path(dtype, K, M, B_MATRIX) == label, (K, M)
    if dtype == cap.F64:
        assert simt_plan(dtype, 96, 256) == (True, 2)


def test_every_accepted_shape_fits_shared_memory():
    """Every (K, M) that cxb_hmm_create accepts gets at least one table row and at most 200 KiB of shared memory."""
    K = np.arange(2, 1025)[:, None]
    M = np.arange(1, 257)[None, :]
    for esz in (4, 8):
        stage, em, row = HMM_WARPS * K * esz, M * K * esz, K * esz
        em_smem = stage + em + row <= SMEM_BUDGET
        rows = np.minimum(K, (SMEM_BUDGET - stage - np.where(em_smem, em, 0)) // row)
        smem = stage + np.where(em_smem, em, 0) + rows * row
        assert rows.min() >= 1 and smem.max() <= SMEM_BUDGET


# ---- GPU: the matrix -----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype,K,M,B,T", [(d,) + s for d in DTYPES for s in matrix(d)],
                         ids=[f"{_id(d)}-K{s[0]}-M{s[1]}-B{s[2]}-T{s[3]}" for d in DTYPES for s in matrix(d)])
def test_matrix_vs_reference(device_api, dtype, K, M, B, T):
    run_and_check(dtype, K, M, B, T, seed=1000 * K + M, label=hmm_path(dtype, K, M, B))


@gpu
@pytest.mark.parametrize("T", [1, 2, 31, 32, 33, 64, 65])
@pytest.mark.parametrize("dtype,label", rep_cases())
def test_lengths_vs_reference(device_api, dtype, label, T):
    """T on both sides of the 32-step observation blocks, the 4-step pipeline of k_hmm64_pass and the hand-over of the
    tcgen05 path."""
    K, M, B = REPRESENTATIVE[dtype][label]
    run_and_check(dtype, K, M, B, T, seed=7 * T + K, label=label)


@gpu
@pytest.mark.parametrize("B", [1, 7, 8, 9, 17])
@pytest.mark.parametrize("dtype,label", rep_cases(skip=("tc64",)))  # NT = 64 needs hundreds of chains
def test_batch_vs_reference(device_api, dtype, label, B):
    """Batches that leave dead warps in the last CTA of k_hmm_pass (8 chains per CTA) and ragged chain tiles."""
    K, M, _ = REPRESENTATIVE[dtype][label]
    assert hmm_path(dtype, K, M, B) == label
    run_and_check(dtype, K, M, B, 37, seed=11 * B + K, label=label)


@gpu
@pytest.mark.parametrize("dtype,K,M,B", [(cap.F64, 192, 128, 3), (cap.F32, 33, 7, 3)], ids=["f64-tiled-global", "f32-K33"])
def test_long_chain_vs_reference(device_api, dtype, K, M, B):
    run_and_check(dtype, K, M, B, 3000, seed=3000 + K, label=hmm_path(dtype, K, M, B))


@gpu
@pytest.mark.parametrize("K,B,T,M", HMM_TC_SHAPES)
def test_simt_path_on_tensor_core_shapes(device_api, monkeypatch, K, B, T, M):
    """CXB_HMM_NO_TC=1 on every tcgen05 shape: the SIMT kernel against the reference, and against the tcgen05 path."""
    A, E, obs = make_inputs(K, M, B, T, seed=2024 + K)
    res = {}
    for no_tc in ("0", "1"):
        monkeypatch.setenv("CXB_HMM_NO_TC", no_tc)
        label = hmm_path(cap.F32, K, M, B, no_tc=no_tc == "1")
        _, res[no_tc + "f"], res[no_tc + "m"] = run(cap.F32, A, E, obs, M, check_launches=label)
    check(cap.F32, res["1f"], res["1m"], A, E, obs, what=f"SIMT K={K} B={B} T={T} M={M}")
    models.assert_values_close(res["1f"], res["0f"], cap.F32, err_msg="forward messages: SIMT vs tcgen05")
    models.assert_values_close(res["1m"], res["0m"], cap.F32, err_msg="marginals: SIMT vs tcgen05")


@gpu
@pytest.mark.parametrize("dtype,K,M,span", [(cap.F32, 33, 6, 18), (cap.F64, 100, 6, 18), (cap.F32, 255, 200, 10)],
                         ids=["f32-K33", "f64-K100", "f32-K255-tiled"])
def test_sparse_transitions_and_tiny_emissions(device_api, dtype, K, M, span):
    """Banded transitions (all but three entries per row exactly zero) and emissions spanning 10^-span .. 1 on the SIMT
    paths. At K = 255 the banded chain moves mass further than fp32 can follow with emissions below 1e-10: the largest
    entry of forward x backward message then falls below the smallest fp32 subnormal (7e-46 at 1e-18), so no fp32
    recursion that normalises every step can get those marginals right, the numpy one included."""
    B, T = 6, 300
    rng = np.random.Generator(np.random.PCG64(404 + K))
    A = np.zeros((K, K))
    for i in range(K):
        for dlt, w in ((0, 0.6), (1, 0.3), (2, 0.1)):
            A[i, (i + dlt) % K] += w
    E = 10.0 ** rng.uniform(-span, 0.0, size=(K, M))
    obs = rng.integers(0, M, size=(T, B), dtype=np.uint8)
    _, got_f, got_m = run(dtype, A, E, obs, M, check_launches=hmm_path(dtype, K, M, B))
    assert np.all(np.isfinite(got_f)) and np.all(np.isfinite(got_m))
    check(dtype, got_f, got_m, A, E, obs, what=f"banded K={K}")


@gpu
@pytest.mark.parametrize("dtype,label", rep_cases())
def test_handle_reuse_equals_fresh_handle(device_api, dtype, label):
    """set_tables, set_observations and update_marginals twice on one handle give bit for bit what a fresh handle gives for
    the final inputs (the tcgen05 ping-pong buffers persist between calls); time slices equal slices of the full read."""
    K, M, B = REPRESENTATIVE[dtype][label]
    T = 23
    A1, E1, o1 = make_inputs(K, M, B, T, seed=1)
    A2, E2, o2 = make_inputs(K, M, B, T, seed=2)
    hm = C.HmmBatch(B, T, K, M, dtype=dtype)
    hm.set_tables(A1, E1)
    hm.set_observations(o1)
    hm.update_marginals()
    hm.set_tables(A2, E2)
    hm.set_observations(o2)
    hm.update_marginals()
    _, fresh_f, fresh_m = run(dtype, A2, E2, o2, M)
    got_f, got_m = hm.get_forward(), hm.get_marginals()
    np.testing.assert_array_equal(got_f, fresh_f)
    np.testing.assert_array_equal(got_m, fresh_m)
    for t0, t1 in ((0, 1), (5, 6), (3, 17), (T - 1, T), (0, T)):
        np.testing.assert_array_equal(hm.get_marginals(t0, t1), got_m[t0:t1])
        np.testing.assert_array_equal(hm.get_forward(t0, t1), got_f[t0:t1])
    check(dtype, got_f, got_m, A2, E2, o2, what=label)


@gpu
@pytest.mark.parametrize("M", [1, 7, 200])
@pytest.mark.parametrize("dtype,label", rep_cases())
def test_out_of_range_symbol_is_refused(device_api, dtype, label, M):
    """A byte >= M makes set_observations raise ValueError and leaves the handle without observations; valid ones work
    again afterwards."""
    K, _, B = REPRESENTATIVE[dtype][label]
    T = 37  # T * B is not a multiple of 16: the last bytes are checked one by one
    A, E, obs = make_inputs(K, M, B, T, seed=M)
    hm = C.HmmBatch(B, T, K, M, dtype=dtype)
    hm.set_tables(A, E)
    for pos, val in (((0, 0), M), ((T - 1, B - 1), M), ((T // 2, B // 2), 255), ((T - 1, 0), M + 1)):
        bad = obs.copy()
        bad[pos] = val
        with pytest.raises(ValueError, match="symbol out of range"):
            hm.set_observations(bad)
        with pytest.raises(C.CortexError):
            hm.update_marginals()
    hm.set_observations(obs)
    hm.update_marginals()
    check(dtype, hm.get_forward(), hm.get_marginals(), A, E, obs, what=f"{label} M={M} after a refused call")


@gpu
@pytest.mark.parametrize("dtype,label", rep_cases(skip=("tc32", "tc64")))
def test_256_symbols_accept_every_byte(device_api, dtype, label):
    K, _, B = REPRESENTATIVE[dtype][label]
    M, T = 256, 40
    obs = (np.arange(T * B) % 256).astype(np.uint8).reshape(T, B)
    run_and_check(dtype, K, M, B, T, seed=256 + K, label=hmm_path(dtype, K, M, B), obs=obs)


@gpu
def test_out_of_range_symbol_in_a_large_batch(device_api):
    """A bad byte anywhere in 4.5 MB of observations (a grid-stride loop over many CTAs) is found."""
    B, T, K, M = 4096, 1101, 2, 9
    rng = np.random.Generator(np.random.PCG64(9))
    obs = rng.integers(0, M, size=(T, B), dtype=np.uint8)
    hm = C.HmmBatch(B, T, K, M, dtype=cap.F32)
    hm.set_tables(np.full((K, K), 0.5), np.ones((K, M)))
    hm.set_observations(obs)
    for pos in ((0, 0), (T - 1, B - 1), (T - 1, B - 16), (T // 3, 1234), (T - 2, 4095)):
        bad = obs.copy()
        bad[pos] = M
        with pytest.raises(ValueError, match="symbol out of range"):
            hm.set_observations(bad)
    hm.set_observations(obs)
    assert hm.update_marginals() == B * (6 * T - 4)
