"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs. Bar (BASELINE.json north_star): bit-exact frontier / wiring / pending state; values within
rel 1e-12 (fp64) and 1e-5 (fp32) of the oracle."""
import numpy as np
import pytest

from tests._pkg import pkg
from tests import models

C = pkg
cap = pkg.capi
pytestmark = pytest.mark.gpu
TOL = models.TOL


def assert_close(got, want, dtype, err_msg="", kind="prob"):
    """Element-wise, at the north-star tolerance (rel 1e-5 fp32 / 1e-12 fp64): tests/models.py::assert_values_close."""
    models.assert_values_close(got, want, dtype, kind=kind, err_msg=err_msg)


def _wiring(engine):
    st = engine.store
    out = []
    for s in range(st.n_signals()):
        sig = C.Signal(st, s)
        out.append((C.get_variant(sig), [d.sid for d in C.get_dependencies(sig)], C.get_dependency_props(sig),
                    [l.sid for l in C.get_listeners(sig)], C.get_listenmask(sig)))
    return out


def _compare(e_dev, e_ora, dtype):
    so, vo = models.engine_state(e_ora)
    sd, vd = models.engine_state(e_dev)
    assert so == sd  # is_computed / is_pending / nibbles of every signal: bit-exact
    family = e_ora.store.family
    kind = "prob" if family == cap.FAMILY_CATEGORICAL else "canon" if family == cap.FAMILY_GAUSS_CANON and vo.shape[-1] == 2 else "plain"
    assert_close(vd, vo, dtype, kind=kind)


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
def test_chain_engine_parity(oracle_api, device_api, dtype):
    T = 64
    data = np.cumsum(np.random.Generator(np.random.PCG64(1234)).standard_normal(T))
    eng = {}
    for name, api in (("o", oracle_api), ("d", device_api)):
        e, x, y, lik, tr = models.make_ssm_model(T, api, form="canon", q=0.7, r=1.3, dtype=dtype, trace=True)
        models.ssm_set_data(e, y, lik, data)
        eng[name] = (e, x)
    assert _wiring(eng["o"][0]) == _wiring(eng["d"][0])  # dependency resolution: bit-exact
    # frontier of the fresh request (scan_inference_request)
    so = C.scan_inference_request(C.request_inference_for(eng["o"][0], eng["o"][1]))
    sd = C.scan_inference_request(C.request_inference_for(eng["d"][0], eng["d"][1]))
    assert [s.sid for s in so] == [s.sid for s in sd] and len(so) == T
    sto = C.update_marginals(eng["o"][0], eng["o"][1], schedule="lvl")
    std = C.update_marginals(eng["d"][0], eng["d"][1], schedule="lvl")
    assert (sto.updates, sto.levels, list(sto.updates_by_kind)) == (std.updates, std.levels, list(std.updates_by_kind))
    assert std.updates == 6 * T - 4 and std.levels == 2 * T - 1 and std.kernel_launches > 0
    assert models.level_trace(eng["o"][0]) == models.level_trace(eng["d"][0])  # per-level frontier lists: bit-exact
    _compare(eng["d"][0], eng["o"][0], dtype)
    assert C.update_marginals(eng["d"][0], eng["d"][1]).updates == 0


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
@pytest.mark.parametrize("rule", ["potts", "table"])
def test_grid_protocol_b_engine_parity(oracle_api, device_api, dtype, rule):
    H, W, K, beta, sweeps = 5, 6, 4, 0.7, 4
    unary = np.random.Generator(np.random.PCG64(1234)).dirichlet(np.ones(K), size=(H, W))
    eng = {}
    for name, api in (("o", oracle_api), ("d", device_api)):
        e, pix, un, pair = models.make_grid_model(H, W, K, beta, api, dtype=dtype, rule=rule)
        e.store.check(e.api.trace_enable(e.store.h, 1))
        vids = [v for row in pix for v in row]
        models.protocol_b_init(e, vids, K)
        usig = [C.get_connection_message_to_variable(e, pix[i][j], un[i][j]) for i in range(H) for j in range(W)]
        eng[name] = (e, vids, usig)
    assert _wiring(eng["o"][0]) == _wiring(eng["d"][0])
    for s in range(sweeps):
        st = {}
        for name in ("o", "d"):
            e, vids, usig = eng[name]
            st[name] = models.protocol_b_sweep(e, vids, usig, unary.reshape(-1, K))
        assert st["o"].updates == st["d"].updates and st["o"].levels == st["d"].levels == 1
        assert (st["o"].final_marginals, st["o"].final_linked) == (st["d"].final_marginals, st["d"].final_linked)
        assert models.level_trace(eng["o"][0]) == models.level_trace(eng["d"][0])
    _compare(eng["d"][0], eng["o"][0], dtype)


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
def test_powerlaw_segment_tree_engine_parity(oracle_api, device_api, dtype):
    n, m, K, sweeps = 80, 220, 8, 3
    eng = {}
    for name, api in (("o", oracle_api), ("d", device_api)):
        e, vs, un, pair, unary, tables, ttype = models.make_powerlaw_model(n, m, K, api, dtype=dtype)
        e.store.check(e.api.trace_enable(e.store.h, 1))
        models.protocol_b_init(e, vs, K)
        usig = [C.get_connection_message_to_variable(e, vs[i], un[i]) for i in range(n)]
        eng[name] = (e, vs, usig, unary)
    assert _wiring(eng["o"][0]) == _wiring(eng["d"][0])
    assert max(len(C.get_connected_factor_ids(eng["d"][0], v)) for v in eng["d"][1]) > 5
    for s in range(sweeps):
        st = {}
        for name in ("o", "d"):
            e, vs, usig, unary = eng[name]
            st[name] = models.protocol_b_sweep(e, vs, usig, unary)
        assert st["o"].updates == st["d"].updates and st["o"].levels == st["d"].levels > 1
        assert list(st["o"].updates_by_kind) == list(st["d"].updates_by_kind)
        assert models.level_trace(eng["o"][0]) == models.level_trace(eng["d"][0])
    _compare(eng["d"][0], eng["o"][0], dtype)


def test_out_of_contract_is_refused_not_silently_different(oracle_api, device_api):
    """Appendix B's naive loopy protocol, call 2, is Gauss-Seidel in the reference: the level schedule refuses it and leaves
    the engine untouched; the default schedule answers it exactly as the reference does (sequential executor)."""
    H, W, K = 3, 3, 4
    unary = np.random.Generator(np.random.PCG64(5)).dirichlet(np.ones(K), size=(H, W))
    eng = {}
    for name, api in (("o", oracle_api), ("d", device_api)):
        e, pix, un, pair = models.make_grid_model(H, W, K, 0.5, api, link=False)
        vids = [v for row in pix for v in row]
        models.protocol_b_init(e, vids, K)
        usig = [C.get_connection_message_to_variable(e, pix[i][j], un[i][j]) for i in range(H) for j in range(W)]
        C.set_values(usig, unary.reshape(-1, K))
        C.update_marginals(e, vids, schedule="lvl" if name == "d" else "seq")
        eng[name] = (e, vids)
    e, vids = eng["d"]
    before = models.engine_state(e)
    with pytest.raises(C.OutOfContractError):
        C.update_marginals(e, vids, schedule="lvl")
    after = models.engine_state(e)
    assert before[0] == after[0] and np.array_equal(before[1], after[1], equal_nan=True)
    st_d = C.update_marginals(e, vids)
    assert C.last_schedule(e) == cap.SCHEDULE_SEQUENTIAL
    st_o = C.update_marginals(eng["o"][0], eng["o"][1], schedule="seq")
    assert st_d.updates == st_o.updates > 0 and list(st_d.updates_by_kind) == list(st_o.updates_by_kind)
    _compare(e, eng["o"][0], cap.F64)


@pytest.mark.parametrize("model", ["ssm", "beta", "hmm", "potts"])
def test_resident_level_loop_equals_per_level_kernels(device_api, model, monkeypatch):
    """update_marginals! of a small graph in ONE launch (k_update_resident) leaves exactly the state, values and
    statistics of the per-level kernels (frontier discovery -> host -> rule kernels -> apply, one round trip per level)."""
    out = []
    monkeypatch.setenv("CXB_MEMO", "0")  # the level loop itself: no memo look-up, recording or certification around it
    for resident in ("1", "0"):
        monkeypatch.setenv("CXB_ENGINE_RESIDENT", resident)
        if model == "ssm":
            T = 60
            e, x, y, lik, tr = models.make_ssm_model(T, device_api, form="canon", q=0.7, r=1.3)
            data = np.cumsum(np.random.Generator(np.random.PCG64(5)).standard_normal(T))
            st = []
            for rep in range(2):  # a second request with fresh data exercises the epochs
                models.ssm_set_data(e, y, lik, data + rep)
                st.append(C.update_marginals(e, x))
            assert st[0].updates == 6 * T - 4 and st[1].updates == 6 * T - 4
        elif model == "hmm":  # categorical family: CAT_TABLE, HMM_EMIT and family-reduce rules, one warp per signal
            T, K, M = 9, 8, 5
            rng = np.random.Generator(np.random.PCG64(12))
            A = rng.dirichlet(np.ones(K), size=K)
            E = rng.dirichlet(np.ones(K), size=M).T * K
            e, z, yv, prior, em, tr = models.make_hmm_model(T, K, M, A, E, device_api)
            models.hmm_set_data(e, z, yv, prior, em, rng.integers(0, M, size=T), K)
            st = [C.update_marginals(e, z)]
            assert st[0].updates == 6 * T - 4
        elif model == "potts":  # loopy grid, protocol B: Potts rule + linked m2f signals in the final phase
            H, W, K = 3, 4, 16
            e, pix, un, pair = models.make_grid_model(H, W, K, 0.7, device_api)
            flat = [v for row in pix for v in row]
            usig = [C.get_connection_message_to_variable(e, pix[i][j], un[i][j]) for i in range(H) for j in range(W)]
            unary = np.random.Generator(np.random.PCG64(13)).dirichlet(np.ones(K), size=len(flat))
            models.protocol_b_init(e, flat, K)
            st = [models.protocol_b_sweep(e, flat, usig, unary, schedule="lvl") for _ in range(2)]
        else:
            n = 40
            e, p, o, f = models.make_beta_bernoulli_model(n, device_api)
            obs = np.random.Generator(np.random.PCG64(6)).integers(0, 2, size=n).astype(np.float64)
            C.set_values([C.get_connection_message_to_factor(e, o[i], f[i]) for i in range(n)], obs.reshape(-1, 1))
            st = [C.update_marginals(e, p)]
            assert st[0].updates == 2 * n - 1  # n m2v + (n - 2) products + 1 marginal
        out.append((models.engine_state(e), [(s.levels, s.updates, s.final_marginals, s.final_linked, tuple(s.updates_by_kind)) for s in st],
                    [s.kernel_launches for s in st]))
    (state_r, stats_r, launches_r), (state_h, stats_h, launches_h) = out
    assert stats_r == stats_h
    assert max(launches_r) <= 3 < min(launches_h)  # request + request check + ONE resident loop vs a dozen launches per level
    assert state_r[0] == state_h[0]  # computed / pending flags and dependency nibbles of every signal
    np.testing.assert_array_equal(state_r[1], state_h[1])  # values, bit for bit


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
def test_hmm_engine_parity(oracle_api, device_api, dtype):
    T, K, M = 12, 8, 5
    rng = np.random.Generator(np.random.PCG64(1234))
    A = rng.dirichlet(np.ones(K), size=K)
    E = rng.dirichlet(np.ones(K), size=M).T * K
    obs = rng.integers(0, M, size=T)
    eng = {}
    for name, api in (("o", oracle_api), ("d", device_api)):
        e, z, y, prior, em, tr = models.make_hmm_model(T, K, M, A, E, api, dtype=dtype)
        models.hmm_set_data(e, z, y, prior, em, obs, K)
        st = C.update_marginals(e, z)
        assert st.updates == 6 * T - 4
        eng[name] = e
    _compare(eng["d"], eng["o"], dtype)


# ---- structured engines against the oracle -------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
@pytest.mark.parametrize("shape", [(1, 1), (3, 2), (70, 37), (300, 129)])
def test_chain_batch_kernel_vs_oracle(oracle_api, dtype, shape):
    B, T = shape
    rng = np.random.Generator(np.random.PCG64(1234))
    q, r = rng.uniform(0.5, 2.0, B), rng.uniform(0.5, 2.0, B)
    x = np.cumsum(rng.standard_normal((T, B)) * np.sqrt(q), axis=0)
    y = x + rng.standard_normal((T, B)) * np.sqrt(r)
    ch = C.GaussianChainBatch(B, T, dtype=dtype)
    ch.set_noise(q, r)
    ch.set_observations(y)
    assert ch.update_marginals() == B * (6 * T - 4)
    y_used = y.astype(ch.np_dtype).astype(np.float64)  # the oracle sees the same (rounded) observations
    ref = np.zeros((6, T, B, 2))
    oracle_api.chains_reference(B, T, q.ctypes.data_as(cap.f64p), r.ctypes.data_as(cap.f64p),
                                np.ascontiguousarray(y_used).ctypes.data_as(cap.f64p), ref.ctypes.data_as(cap.f64p))
    for m in range(6):
        assert_close(ch.get_messages(m).astype(np.float64), ref[m], dtype, err_msg=C.GaussianChainBatch.MESSAGE_CLASSES[m], kind="canon")
    assert ch.last_kernel_ms() > 0


def test_chain_batch_kernel_vs_explicit_graph_engine(oracle_api):
    """The structured plan is the same graph/wiring/schedule as the explicit BipartiteFactorGraph + DEFAULT_BP."""
    B, T = 3, 17
    rng = np.random.Generator(np.random.PCG64(99))
    q, r = rng.uniform(0.5, 2.0, B), rng.uniform(0.5, 2.0, B)
    y = rng.standard_normal((T, B)) * 3
    ch = C.GaussianChainBatch(B, T, dtype=cap.F64)
    ch.set_noise(q, r)
    ch.set_observations(y)
    ch.update_marginals()
    for b in range(B):
        e, x, yv, lik, tr = models.make_ssm_model(T, oracle_api, form="canon", q=q[b], r=r[b])
        models.ssm_set_data(e, yv, lik, y[:, b])
        C.update_marginals(e, x, schedule="seq")
        want = {0: [C.get_connection_message_to_variable(e, x[t], lik[t]) for t in range(T)],
                1: [None] + [C.get_connection_message_to_variable(e, x[t], tr[t - 1]) for t in range(1, T)],
                2: [C.get_connection_message_to_factor(e, x[t], tr[t]) for t in range(T - 1)] + [None],
                3: [C.get_connection_message_to_variable(e, x[t], tr[t]) for t in range(T - 1)] + [None],
                4: [None] + [C.get_connection_message_to_factor(e, x[t], tr[t - 1]) for t in range(1, T)],
                5: [C.get_variable_marginal(C.get_variable(e, x[t])) for t in range(T)]}
        for m, sigs in want.items():
            got = ch.get_messages(m)[:, b, :]
            for t, s in enumerate(sigs):
                if s is not None:
                    np.testing.assert_allclose(got[t], C.get_value(s), rtol=1e-12)


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
@pytest.mark.parametrize("shape", [(1, 1, 4), (1, 7, 4), (6, 1, 4), (5, 7, 8), (9, 33, 16)])
def test_potts_grid_kernel_vs_oracle(oracle_api, dtype, shape):
    H, W, K = shape
    beta, sweeps = 0.7, 3
    unary = np.random.Generator(np.random.PCG64(1234)).dirichlet(np.ones(K), size=(H, W))
    gr = C.PottsGrid(H, W, K, beta, dtype=dtype)
    gr.set_unary(unary)
    gr.reset_messages()
    e, pix, un, pair = models.make_grid_model(H, W, K, beta, oracle_api)
    vids = [v for row in pix for v in row]
    models.protocol_b_init(e, vids, K)
    usig = [C.get_connection_message_to_variable(e, pix[i][j], un[i][j]) for i in range(H) for j in range(W)]
    unary_used = unary.astype(gr.np_dtype).astype(np.float64)
    for s in range(sweeps):
        st = models.protocol_b_sweep(e, vids, usig, unary_used.reshape(-1, K))
        assert gr.sweep() == st.updates
    want = C.get_values([C.get_variable_marginal(C.get_variable(e, v)) for v in vids]).reshape(H, W, K)
    assert_close(gr.get_marginals(), want, dtype)
    # every message plane: m2v from / m2f towards the (up, left, right, down) factor
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
                    assert_close(got_v[i, j], C.get_value(C.get_connection_message_to_variable(e, pix[i][j], f)), dtype)
                    assert_close(got_f[i, j], C.get_value(C.get_connection_message_to_factor(e, pix[i][j], f)), dtype)


def test_potts_grid_row_sharding_is_bit_identical():
    """Two shards exchanging halo rows give exactly the single-shard result (SURVEY §8e)."""
    H, W, K, beta, sweeps = 10, 12, 16, 0.7, 4
    unary = np.random.Generator(np.random.PCG64(3)).dirichlet(np.ones(K), size=(H, W)).astype(np.float32)
    full = C.PottsGrid(H, W, K, beta)
    full.set_unary(unary)
    full.reset_messages()
    top = C.PottsGrid(4, W, K, beta, has_lower=True)
    bot = C.PottsGrid(6, W, K, beta, has_upper=True)
    top.set_unary(unary[:4])
    bot.set_unary(unary[4:])
    top.reset_messages()
    bot.reset_messages()
    nbytes = top.halo_elems * 4
    for s in range(sweeps):
        full.sweep()
        top.sweep()
        bot.sweep()
        top.sync()
        bot.sync()
        # top sends its `down` row to bot's upper halo; bot sends its `up` row to top's lower halo
        _d2d(bot.halo_recv_ptr(0), top.halo_send_ptr(1), nbytes)
        _d2d(top.halo_recv_ptr(1), bot.halo_send_ptr(0), nbytes)
    got = np.concatenate([top.get_marginals(), bot.get_marginals()], axis=0)
    assert np.array_equal(got, full.get_marginals())
    assert top.sweep() + bot.sweep() == full.sweep()  # same number of message updates


@pytest.mark.parametrize("dtype", [cap.F32, cap.F64])
def test_potts_grid_fused_peer_halo_is_bit_identical(dtype):
    """Three row shards connected through cxb_grid_p2p_connect_local: the sweep kernel itself stores the cut-edge messages
    into the neighbours' halo buffers and the sweep counters order the sweeps; no exchange call, result == one shard."""
    H, W, K, beta, sweeps = 13, 9, 8, 0.45, 5
    npdt = np.float32 if dtype == cap.F32 else np.float64
    unary = np.random.Generator(np.random.PCG64(8)).dirichlet(np.ones(K), size=(H, W)).astype(npdt)
    full = C.PottsGrid(H, W, K, beta, dtype=dtype)
    full.set_unary(unary)
    full.reset_messages()
    cuts = [0, 4, 9, H]
    shards = [C.PottsGrid(cuts[i + 1] - cuts[i], W, K, beta, dtype=dtype, has_upper=i > 0, has_lower=i < 2) for i in range(3)]
    for i, sh in enumerate(shards):
        sh.set_unary(unary[cuts[i]:cuts[i + 1]])
        sh.reset_messages()
    for i, sh in enumerate(shards):
        if i > 0:
            sh.p2p_connect_local(0, shards[i - 1])
        if i < 2:
            sh.p2p_connect_local(1, shards[i + 1])
    n_upd = 0
    for s in range(sweeps):
        full.sweep()
        n_upd = sum(sh.sweep() for sh in shards)  # every shard enqueues sweep s before any shard enqueues sweep s + 1
    got = np.concatenate([sh.get_marginals() for sh in shards], axis=0)
    assert np.array_equal(got, full.get_marginals())
    assert n_upd == full.sweep()
    # a reset (all shards idle) restarts the counters: the same answer again
    for sh in shards:
        sh.sync()
    for sh in shards:
        sh.reset_messages()
    for sh in shards:
        sh.sync()
    full.reset_messages()
    for s in range(2):
        full.sweep()
        for sh in shards:
            sh.sweep()
    assert np.array_equal(np.concatenate([sh.get_marginals() for sh in shards], axis=0), full.get_marginals())


def _d2d(dst, src, nbytes):
    """raw device-to-device copy (plumbing only)"""
    import ctypes

    rt = ctypes.CDLL("libcudart.so.12")
    rt.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    assert rt.cudaMemcpy(dst, src, nbytes, 3) == 0  # 3 = cudaMemcpyDeviceToDevice


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
@pytest.mark.parametrize("B,T,chunks", [(1, 3, 8), (70, 9, 8), (1000, 33, 8), (1000, 33, 1), (4099, 17, 32)])
def test_chain_batch_host_entry_point_is_bit_identical(dtype, B, T, chunks, monkeypatch):
    """cxb_chains_infer_host (chunk-pipelined host->device / compute / device->host) == set_observations +
    update_marginals + get_marginals, bit for bit, for ragged chunkings; repeated calls reuse the buffers safely."""
    import torch

    monkeypatch.setenv("CXB_CHAINS_HOST_CHUNKS", str(chunks))
    rng = np.random.Generator(np.random.PCG64(99))
    ch = C.GaussianChainBatch(B, T, dtype=dtype)
    ch.set_noise(rng.uniform(0.5, 2.0, B), rng.uniform(0.5, 2.0, B))
    tdt = torch.float32 if dtype == cap.F32 else torch.float64
    for rep in range(2):
        y = rng.standard_normal((T, B)).astype(ch.np_dtype)
        ch.set_observations(y)
        ch.update_marginals()
        want = ch.get_messages(5).copy()
        ch.set_observations(np.zeros_like(y))  # make sure the host path really uploads
        y_host = torch.from_numpy(y.copy()).pin_memory()
        out_host = torch.zeros((T, B, 2), dtype=tdt).pin_memory()
        assert ch.infer_host(y_host.data_ptr(), out_host.data_ptr()) == B * (6 * T - 4)
        np.testing.assert_array_equal(out_host.numpy(), want.reshape(T, B, 2))


@pytest.mark.parametrize("dtype,K", [(cap.F32, 64), (cap.F64, 64), (cap.F32, 32), (cap.F32, 8), (cap.F32, 96)])
def test_hmm_kernel_vs_oracle(oracle_api, dtype, K):
    B, T, M = 11, 40, 7
    rng = np.random.Generator(np.random.PCG64(1234))
    A = rng.dirichlet(np.ones(K), size=K)
    E = rng.dirichlet(np.ones(K), size=M).T * K
    obs = rng.integers(0, M, size=(T, B)).astype(np.uint8)
    hm = C.HmmBatch(B, T, K, M, dtype=dtype)
    hm.set_tables(A, E)
    hm.set_observations(obs)
    assert hm.update_marginals() == B * (6 * T - 4)
    got_m, got_f = hm.get_marginals(), hm.get_forward()
    A_used = A.astype(hm.np_dtype).astype(np.float64)
    for b in (0, B - 1):
        e, z, y, prior, em, tr = models.make_hmm_model(T, K, M, A_used, E, oracle_api)
        models.hmm_set_data(e, z, y, prior, em, obs[:, b], K)
        C.update_marginals(e, z, schedule="seq")
        want_m = C.get_values([C.get_variable_marginal(C.get_variable(e, v)) for v in z])
        assert_close(got_m[:, b, :], want_m, dtype)
        want_f = C.get_values([C.get_connection_message_to_factor(e, z[t], tr[t]) for t in range(T - 1)])
        assert_close(got_f[:-1, b, :], want_f, dtype)


def _hmm_numpy(A, E, obs):
    """Independent dense fp64 scaled forward-backward: forward messages m2f(z_t, tr_t) and marginals, all normalised."""
    T = len(obs)
    K = A.shape[0]
    En = E / E.sum(axis=0, keepdims=True)
    fwd = np.zeros((T, K))
    v = En[:, obs[0]].copy()
    fwd[0] = v / v.sum()
    for t in range(1, T):
        v = En[:, obs[t]] * (fwd[t - 1] @ A)
        fwd[t] = v / v.sum()
    marg = np.zeros((T, K))
    marg[T - 1] = fwd[T - 1]
    w = En[:, obs[T - 1]].copy()
    w /= w.sum()
    for t in range(T - 2, -1, -1):
        back = A @ w
        g = fwd[t] * back
        marg[t] = g / g.sum()
        w = En[:, obs[t]] * back
        w /= w.sum()
    return fwd, marg


@pytest.mark.parametrize("B,T,M", [(5, 1, 3), (5, 2, 3), (5, 3, 3), (5, 4, 5), (5, 5, 5), (5, 9, 32), (5, 70, 100), (5, 3000, 32),
                                   (1, 1, 3), (4, 301, 200)])
def test_hmm64_kernel_lengths_and_long_chain_vs_numpy(B, T, M):
    """K = 64 fp32 register kernel: the late write-out (T around the pipeline depth), a single chain, emission tables in
    shared memory (M <= 128) and in global memory (M = 200), and the drift-free power-of-two scaling over a long chain."""
    K = 64
    rng = np.random.Generator(np.random.PCG64(77))
    A = rng.dirichlet(np.ones(K) * 0.3, size=K)
    E = rng.dirichlet(np.ones(K) * 0.5, size=M).T * K
    obs = rng.integers(0, M, size=(T, B)).astype(np.uint8)
    hm = C.HmmBatch(B, T, K, M, dtype=cap.F32)
    hm.set_tables(A, E)
    hm.set_observations(obs)
    assert hm.update_marginals() == B * (6 * T - 4)
    got_m, got_f = hm.get_marginals(), hm.get_forward()
    A_used = A.astype(np.float32).astype(np.float64)
    for b in (0, B - 1):
        want_f, want_m = _hmm_numpy(A_used, E, obs[:, b])
        assert_close(got_f[:, b, :], want_f, cap.F32)
        assert_close(got_m[:, b, :], want_m, cap.F32)
        np.testing.assert_allclose(got_f[:, b, :].sum(axis=-1), 1.0, rtol=0, atol=2e-6)
        np.testing.assert_allclose(got_m[:, b, :].sum(axis=-1), 1.0, rtol=0, atol=2e-6)


# The slice width follows the grid: 32 output states per CTA while (chain tiles) x (K / 32) x 2 CTAs fit one per SM,
# else 64. On a 148-SM B200 the last five shapes are the ones that get NT = 64 (5 x 16 x 2 = 160, 3 x 32 x 2 = 192,
# 14 x 6 x 2 = 168 and 9 x 10 x 2 = 180 CTAs): T = 1 and 2 for the hand-over, and K / 64 odd.
HMM_TC_SHAPES = [(128, 5, 1, 4), (128, 5, 2, 4), (128, 130, 3, 7), (256, 7, 6, 32), (512, 131, 5, 32), (512, 3, 40, 64),
                 (320, 9, 12, 5), (512, 2, 1200, 16), (192, 3, 700, 9), (512, 600, 5, 16), (1024, 300, 3, 8),
                 (512, 600, 2, 16), (192, 1700, 1, 4), (320, 1100, 2, 5)]


@pytest.mark.parametrize("K,B,T,M", HMM_TC_SHAPES)
def test_hmm_tensor_core_kernel_vs_numpy(K, B, T, M):
    """K >= 128 fp32: tcgen05 path (bf16 split operands, fp32 TMEM accumulators, one launch per time step running both
    passes), ragged chain tiles (B not a multiple of 128), every pipeline depth, both slice widths, against the dense fp64
    forward-backward. T = 1, 2, 3 exercise the hand-over between stored predictions and direct marginals."""
    rng = np.random.Generator(np.random.PCG64(2024 + K))
    A = rng.dirichlet(np.ones(K) * 0.5, size=K)
    E = rng.dirichlet(np.ones(K) * 0.5, size=M).T * K
    obs = rng.integers(0, M, size=(T, B)).astype(np.uint8)
    hm = C.HmmBatch(B, T, K, M, dtype=cap.F32)
    hm.set_tables(A, E)
    hm.set_observations(obs)
    assert hm.update_marginals() == B * (6 * T - 4)
    got_m, got_f = hm.get_marginals(), hm.get_forward()
    A_used = A.astype(np.float32).astype(np.float64)
    for b in sorted({0, B // 2, B - 1}):
        want_f, want_m = _hmm_numpy(A_used, E, obs[:, b])
        assert_close(got_f[:, b, :], want_f, cap.F32)
        assert_close(got_m[:, b, :], want_m, cap.F32)
        np.testing.assert_allclose(got_m[:, b, :].sum(axis=-1), 1.0, rtol=0, atol=4e-6)


def test_hmm_tensor_core_kernel_matches_simt_kernel(monkeypatch):
    """The tcgen05 path against the library's own fp32 SIMT path on the same inputs (K = 128)."""
    K, B, T, M = 128, 40, 9, 6
    rng = np.random.Generator(np.random.PCG64(5))
    A = rng.dirichlet(np.ones(K), size=K)
    E = rng.dirichlet(np.ones(K), size=M).T * K
    obs = rng.integers(0, M, size=(T, B)).astype(np.uint8)
    res = []
    for no_tc in ("0", "1"):
        monkeypatch.setenv("CXB_HMM_NO_TC", no_tc)
        hm = C.HmmBatch(B, T, K, M, dtype=cap.F32)
        hm.set_tables(A, E)
        hm.set_observations(obs)
        hm.update_marginals()
        res.append((hm.get_forward(), hm.get_marginals()))
    assert_close(res[0][0], res[1][0], cap.F32)
    assert_close(res[0][1], res[1][1], cap.F32)


def _pairwise_vs_oracle(oracle_api, dtype, n, edges, K, sweeps, seed=7):
    rng = np.random.Generator(np.random.PCG64(seed))
    n_tables = 5
    tables = np.exp(rng.standard_normal((n_tables, K, K)))
    ttype = rng.integers(0, n_tables, size=len(edges))
    unary = rng.dirichlet(np.ones(K), size=n)
    pw = C.PairwiseGraph(n, [e[0] for e in edges], [e[1] for e in edges], ttype, tables, dtype=dtype)
    pw.set_unary(unary)
    pw.reset_messages()
    # the same model as an explicit graph on the oracle (tests/models.py conventions: unary factors first)
    g = C.BipartiteFactorGraph()
    vs = [g.add_variable(C.Variable(name="v", index=(i,))) for i in range(n)]
    un = [g.add_factor(C.Factor(functional_form="unary")) for _ in range(n)]
    for i in range(n):
        g.add_edge(vs[i], un[i], C.Connection(label="out"))
    fac = []
    for (u, v), t in zip(edges, ttype):
        f = g.add_factor(C.Factor(functional_form=f"pair{int(t)}"))
        g.add_edge(vs[u], f, C.Connection(label="a"))
        g.add_edge(vs[v], f, C.Connection(label="b"))
        fac.append(f)
    tables_used = tables.astype(pw.np_dtype).astype(np.float64)
    proc = C.RuleProcessor({f"pair{t}": (cap.RULE_CAT_TABLE, tables_used[t].ravel()) for t in range(n_tables)},
                           family=cap.FAMILY_CATEGORICAL, value_dim=K)
    e = C.InferenceEngine(model_engine=g, dependency_resolver=C.DefaultDependencyResolver(), inference_request_processor=proc,
                          api=oracle_api)
    models.protocol_b_link(e, vs)
    models.protocol_b_init(e, vs, K)
    usig = [C.get_connection_message_to_variable(e, vs[i], un[i]) for i in range(n)]
    unary_used = unary.astype(pw.np_dtype).astype(np.float64)
    for _ in range(sweeps):
        st = models.protocol_b_sweep(e, vs, usig, unary_used, schedule="lvl")
        assert pw.sweep() == st.updates  # same number of reference signal updates (incl. ProductOfMessages nodes)
    want = C.get_values([C.get_variable_marginal(C.get_variable(e, v)) for v in vs])
    assert_close(pw.get_marginals(), want, dtype)
    got_v, got_f = pw.get_messages(0), pw.get_messages(1)
    want_v = np.zeros((len(edges), 2, K))
    want_f = np.zeros((len(edges), 2, K))
    for k, ((u, v), f) in enumerate(zip(edges, fac)):
        for side, x in enumerate((u, v)):
            want_v[k, side] = C.get_value(C.get_connection_message_to_variable(e, vs[x], f))
            want_f[k, side] = C.get_value(C.get_connection_message_to_factor(e, vs[x], f))
    assert_close(got_v, want_v, dtype)
    assert_close(got_f, want_f, dtype)


@pytest.mark.parametrize("dtype", [cap.F64, cap.F32])
@pytest.mark.parametrize("K", [8, 4])
def test_pairwise_kernel_powerlaw_vs_oracle(oracle_api, dtype, K):
    n, m = 120, 330
    edges = models.chung_lu_edges(n, m, seed=11)
    deg = np.bincount(np.asarray(edges).ravel(), minlength=n)
    assert deg.max() > 4 and deg.min() == 0 or deg.max() > 4  # small path + hub path both exercised
    _pairwise_vs_oracle(oracle_api, dtype, n, edges, K, sweeps=3)


@pytest.mark.parametrize("K,dtype", [(8, cap.F32), (16, cap.F32), (32, cap.F32), (2, cap.F32), (4, cap.F64), (16, cap.F64)])
def test_pairwise_kernel_every_degree_bin(oracle_api, K, dtype):
    """Hubs whose degrees sit on both sides of every bin boundary of pairwise.cu (exact <= 4, teams of 1..16 groups of 8
    slots, chunked hubs), all sharing one pool of leaves so that leaves have mixed small degrees."""
    hub_degrees = [1, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 200, 257, 300]
    n_hubs, n_leaves = len(hub_degrees), 300
    rng = np.random.Generator(np.random.PCG64(5))
    edges = []
    for h, d in enumerate(hub_degrees):
        for leaf in sorted(rng.choice(n_leaves, size=d, replace=False)):
            edges.append((h, n_hubs + int(leaf)))
    edges += [(0, 1), (1, 2), (5, 9)]  # hub-hub factors
    edges = sorted(set(edges))
    _pairwise_vs_oracle(oracle_api, dtype, n_hubs + n_leaves + 2, edges, K, sweeps=2)


def test_pairwise_kernel_big_hub_and_isolated_variables(oracle_api):
    """A star with 1,100 leaves (block-per-hub path), a medium hub, a chain and two isolated variables."""
    n = 1150
    edges = [(0, i) for i in range(1, 1101)]                 # big hub: degree 1100 >= 1024
    edges += [(1101, i) for i in range(1102, 1122)]          # medium hub: degree 20
    edges += [(i, i + 1) for i in range(1122, 1147)]         # chain
    edges = sorted(edges)
    _pairwise_vs_oracle(oracle_api, cap.F32, n, edges, 8, sweeps=2)


# ---- degenerate shapes: nothing may crash, results stay normalised / equal to the closed form ----------------------------
def test_degenerate_shapes_of_the_structured_engines():
    # pairwise graph without factors: marginal = normalised unary, no message updates beyond the marginals
    n, K = 5, 8
    unary = np.random.Generator(np.random.PCG64(1)).dirichlet(np.ones(K), size=n)
    pw = C.PairwiseGraph(n, [], [], np.zeros(0, dtype=np.int32), np.ones((1, K, K)), dtype=cap.F64)
    pw.set_unary(unary)
    pw.reset_messages()
    assert pw.sweep() == n
    np.testing.assert_allclose(pw.get_marginals(), unary, rtol=1e-12)
    # 1 x 1 and 1 x 7 grids: a lone pixel's marginal is its unary evidence
    for H, W in ((1, 1), (1, 7), (6, 1)):
        un = np.random.Generator(np.random.PCG64(2)).dirichlet(np.ones(16), size=(H, W)).astype(np.float32)
        gr = C.PottsGrid(H, W, 16, 0.7)
        gr.set_unary(un)
        gr.reset_messages()
        gr.sweep()
        gr.sweep()
        m = gr.get_marginals()
        np.testing.assert_allclose(m.sum(axis=-1), 1.0, atol=1e-6)
        if H * W == 1:
            np.testing.assert_allclose(m, un, rtol=1e-6)
    # one chain, one step
    ch = C.GaussianChainBatch(1, 1, dtype=cap.F64)
    ch.set_noise([1.0], [2.0])
    ch.set_observations(np.array([[3.0]]))
    assert ch.update_marginals() == 2
    np.testing.assert_allclose(ch.get_marginals()[0, 0], [0.5, 1.5], rtol=1e-14)  # (1 / r, y / r)
    # tensor-core HMM with a single chain (127 padding rows in the tile)
    K, T, M = 128, 4, 3
    rng = np.random.Generator(np.random.PCG64(3))
    A = rng.dirichlet(np.ones(K), size=K)
    E = rng.dirichlet(np.ones(K), size=M).T * K
    obs = rng.integers(0, M, size=(T, 1)).astype(np.uint8)
    hm = C.HmmBatch(1, T, K, M, dtype=cap.F32)
    hm.set_tables(A, E)
    hm.set_observations(obs)
    hm.update_marginals()
    want_f, want_m = _hmm_numpy(A.astype(np.float32).astype(np.float64), E, obs[:, 0])
    assert_close(hm.get_marginals()[:, 0, :], want_m, cap.F32)


# ---- numerically awkward inputs ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [64, 128])
def test_hmm_sparse_transitions_and_peaked_emissions(K):
    """Banded transition matrix (most entries exactly zero) and emissions spanning 8 orders of magnitude: the
    power-of-two scaling of the K = 64 and tensor-core kernels must neither overflow nor lose the small states."""
    B, T, M = 6, 400, 6
    rng = np.random.Generator(np.random.PCG64(404 + K))
    A = np.zeros((K, K))
    for i in range(K):
        for dlt, w in ((0, 0.6), (1, 0.3), (2, 0.1)):
            A[i, (i + dlt) % K] += w
    E = np.exp(rng.uniform(-18.0, 0.0, size=(K, M)))
    obs = rng.integers(0, M, size=(T, B)).astype(np.uint8)
    hm = C.HmmBatch(B, T, K, M, dtype=cap.F32)
    hm.set_tables(A, E)
    hm.set_observations(obs)
    hm.update_marginals()
    got_m, got_f = hm.get_marginals(), hm.get_forward()
    assert np.all(np.isfinite(got_m)) and np.all(np.isfinite(got_f))
    A_used = A.astype(np.float32).astype(np.float64)
    for b in (0, B - 1):
        want_f, want_m = _hmm_numpy(A_used, E, obs[:, b])
        # entries far below the fp32 resolution of a normalised vector carry no information: compare above 1e-7 of the max
        for got, want in ((got_f[:, b, :], want_f), (got_m[:, b, :], want_m)):
            np.testing.assert_allclose(got, want, rtol=2e-5, atol=2e-5 * 1e-2)
            np.testing.assert_allclose(got.sum(axis=-1), 1.0, atol=4e-6)


def test_chain_batch_extreme_noise(oracle_api):
    """q = 0 (the state is a constant), very small and very large observation noise, fp64 against the oracle."""
    T = 30
    rng = np.random.Generator(np.random.PCG64(9))
    q = np.array([0.0, 1e-8, 1e6, 1.0])
    r = np.array([1.0, 1e-6, 1e-6, 1e8])
    B = len(q)
    y = rng.standard_normal((T, B)) * 3.0
    ch = C.GaussianChainBatch(B, T, dtype=cap.F64)
    ch.set_noise(q, r)
    ch.set_observations(y)
    ch.update_marginals()
    got = ch.get_marginals()
    for b in range(B):
        e, x, yv, lik, tr = models.make_ssm_model(T, oracle_api, form="canon", q=float(q[b]), r=float(r[b]))
        models.ssm_set_data(e, yv, lik, y[:, b])
        C.update_marginals(e, x, schedule="seq")
        want = C.get_values([C.get_variable_marginal(C.get_variable(e, v)) for v in x])
        np.testing.assert_allclose(got[:, b, :], want, rtol=1e-12, atol=0)


def test_potts_grid_halo_wait_is_bounded(monkeypatch):
    """A row neighbour that never enqueues its sweep must not hang the stream: the wait gives up after the time-out and the
    next synchronising call reports it (VERDICT r1: k_halo_wait spun for ever)."""
    monkeypatch.setenv("CXB_GRID_HALO_TIMEOUT_MS", "50")
    H, W, K = 6, 5, 8
    unary = np.random.Generator(np.random.PCG64(8)).dirichlet(np.ones(K), size=(H, W)).astype(np.float32)
    top = C.PottsGrid(3, W, K, 0.4, dtype=cap.F32, has_lower=True)
    bottom = C.PottsGrid(3, W, K, 0.4, dtype=cap.F32, has_upper=True)
    for g, rows in ((top, unary[:3]), (bottom, unary[3:])):
        g.set_unary(rows)
        g.reset_messages()
    top.p2p_connect_local(1, bottom)
    bottom.p2p_connect_local(0, top)
    top.sweep()
    top.sweep()  # waits for the sweep counter of `bottom`, which never sweeps
    with pytest.raises(C.CortexError, match="did not deliver"):
        top.sync()


def test_potts_grid_pipelined_host_jobs_equal_the_plain_calls():
    """cxb_grid_infer_host: evidence in, sweeps, marginals out, pipelined over three streams across jobs - bit-identical to
    set_unary / sweep / get_marginals one after the other (the messages carry over from job to job in both)."""
    import torch

    H, W, K, sweeps, jobs = 37, 29, 16, 3, 5
    rng = np.random.Generator(np.random.PCG64(21))
    unaries = [rng.dirichlet(np.ones(K), size=(H, W)).astype(np.float32) for _ in range(jobs)]
    plain = C.PottsGrid(H, W, K, 0.7, dtype=cap.F32)
    plain.reset_messages()
    want = []
    for u in unaries:
        plain.set_unary(u)
        for _ in range(sweeps):
            plain.sweep()
        want.append(plain.get_marginals())
    piped = C.PottsGrid(H, W, K, 0.7, dtype=cap.F32)
    piped.reset_messages()
    host_in = [torch.from_numpy(u).pin_memory() for u in unaries]
    host_out = [torch.empty((H, W, K), dtype=torch.float32).pin_memory() for _ in range(jobs)]
    for j in range(jobs):  # nothing waits between the calls
        assert piped.infer_host(host_in[j].data_ptr(), host_out[j].data_ptr(), sweeps) > 0
    piped.sync()
    for j in range(jobs):
        assert np.array_equal(host_out[j].numpy(), want[j]), f"job {j}"
    assert np.array_equal(piped.get_marginals(), want[-1])
