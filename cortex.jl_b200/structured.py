"""Structured model engines: closed-form plans of the fixed-stencil graph families (SURVEY §8a).

Each class is the host-side face of one `cxb_<family>_*` group of the C ABI.  They stand for the SAME graph,
wiring and schedule as an explicit `InferenceEngine` on the equivalent `BipartiteFactorGraph` (that is what the
parity tests compare them with); `update_marginals()` is `update_marginals!(engine, all state variables)`.
Host arrays are numpy; nothing here computes — all arithmetic happens in the CUDA library.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi as capi
from .inference_signal import CortexError, raise_for_status


def _np_dtype(dtype):
    return np.float32 if dtype == capi.F32 else np.float64


class _Handle:
    _prefix = ""

    def _fn(self, name):
        return getattr(self.api, f"{self._prefix}_{name}")

    def check(self, status):
        if status != capi.OK:
            msg = self._fn("last_error")(self.h)
            raise_for_status(status, msg.decode() if msg else f"status {status}")

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self._fn("destroy")(self.h)
                self.h = None
        except Exception:
            pass

    def sync(self):
        self.check(self._fn("sync")(self.h))

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        self.check(self._fn("last_kernel_ms")(self.h, C.byref(ms)))
        return float(ms.value)

    @property
    def stream(self) -> int:
        return int(self._fn("stream")(self.h) or 0)


class GaussianChainBatch(_Handle):
    """B independent random-walk chains of length T (graph of test/inference_engine_tests.jl:436-462)."""
    _prefix = "chains"
    MESSAGE_CLASSES = ("m2v(x_t,lik_t)", "m2v(x_t,tr_{t-1})", "m2f(x_t,tr_t)", "m2v(x_t,tr_t)", "m2f(x_t,tr_{t-1})", "marginal(x_t)")

    def __init__(self, n_chains, n_steps, dtype=capi.F32, device=0, api=None):
        self.api = api or capi.default_api()
        self.B, self.T, self.dtype, self.device = int(n_chains), int(n_steps), dtype, device
        self.np_dtype = _np_dtype(dtype)
        h = C.c_void_p()
        st = self.api.chains_create(device, dtype, self.B, self.T, C.byref(h))
        if st != capi.OK or not h:
            raise CortexError(st, "cxb_chains_create failed (CUDA device required; there is no CPU fallback)")
        self.h = h

    @property
    def n_updates(self):
        return self.B * (6 * self.T - 4)

    def set_noise(self, q, r):
        q = np.ascontiguousarray(np.broadcast_to(np.asarray(q, dtype=np.float64), (self.B,)))
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(r, dtype=np.float64), (self.B,)))
        self.check(self.api.chains_set_noise(self.h, q.ctypes.data_as(capi.f64p), r.ctypes.data_as(capi.f64p)))

    def set_observations(self, y):
        y = np.ascontiguousarray(y, dtype=self.np_dtype)
        assert y.shape == (self.T, self.B), "observations are time-major [T][B]"
        self.check(self.api.chains_set_observations(self.h, y.ctypes.data))

    def set_observations_device(self, ptr: int):
        self.check(self.api.chains_set_observations_device(self.h, ptr))

    def update_marginals(self) -> int:
        n = C.c_int64()
        self.check(self.api.chains_update_marginals(self.h, C.byref(n)))
        return int(n.value)

    def get_messages(self, message_class: int) -> np.ndarray:
        out = np.empty((self.T, self.B, 2), dtype=self.np_dtype)
        self.check(self.api.chains_get_messages(self.h, message_class, out.ctypes.data))
        return out

    def get_marginals(self) -> np.ndarray:
        return self.get_messages(5)

    def device_ptr(self, which: int) -> int:
        return int(self.api.chains_device_ptr(self.h, which) or 0)

    def infer_host(self, y_ptr: int, out_ptr: int) -> int:
        """H2D observations + update + D2H marginals on raw (pinned) host pointers — the end-to-end path."""
        n = C.c_int64()
        self.check(self.api.chains_infer_host(self.h, y_ptr, out_ptr, C.byref(n)))
        return int(n.value)


class PottsGrid(_Handle):
    """rows x cols shard of a Potts grid (K labels), synchronous sweeps = protocol B (SURVEY Appendix B)."""
    _prefix = "grid"
    M2V_PLANES = ("up", "left", "right", "down")

    def __init__(self, rows, cols, n_labels, beta, dtype=capi.F32, device=0, has_upper=False, has_lower=False, api=None):
        self.api = api or capi.default_api()
        self.H, self.W, self.K, self.beta, self.dtype, self.device = int(rows), int(cols), int(n_labels), float(beta), dtype, device
        self.has_upper, self.has_lower = bool(has_upper), bool(has_lower)
        self.np_dtype = _np_dtype(dtype)
        h = C.c_void_p()
        st = self.api.grid_create(device, dtype, self.H, self.W, self.K, self.beta, int(has_upper), int(has_lower), C.byref(h))
        if st != capi.OK or not h:
            raise CortexError(st, "cxb_grid_create failed (CUDA device required; there is no CPU fallback)")
        self.h = h

    def set_unary(self, unary):
        u = np.ascontiguousarray(unary, dtype=self.np_dtype)
        assert u.shape == (self.H, self.W, self.K)
        self.check(self.api.grid_set_unary(self.h, u.ctypes.data))

    def set_couplings(self, horizontal, vertical):
        """Per-edge coupling strengths, psi_e[a][b] = exp(beta_e [a==b]) (``cxb_grid_set_couplings``): ``horizontal[rows][cols-1]``
        between (i, j) and (i, j+1); ``vertical[rows+1][cols]`` between local rows i-1 and i, row 0 and row ``rows`` being the cut
        edges to the shards above and below (``sharding.shard_couplings`` cuts them from global arrays). ``None, None``
        returns to the create-time beta. Sweeps already enqueued keep the couplings they were enqueued with."""
        if horizontal is None and vertical is None:
            self.check(self.api.grid_set_couplings(self.h, None, None))
            return
        hz = np.ascontiguousarray(horizontal, dtype=np.float64)
        vt = np.ascontiguousarray(vertical, dtype=np.float64)
        if hz.shape != (self.H, self.W - 1) or vt.shape != (self.H + 1, self.W):
            raise ValueError(f"couplings of a {self.H} x {self.W} shard are horizontal [{self.H}][{self.W - 1}] and vertical "
                             f"[{self.H + 1}][{self.W}], got {hz.shape} and {vt.shape}")
        hz = hz if hz.size else np.zeros(1)  # a one-column shard has no horizontal factor; the library still wants a pointer
        self.check(self.api.grid_set_couplings(self.h, hz.ctypes.data_as(capi.f64p), vt.ctypes.data_as(capi.f64p)))

    def reset_messages(self):
        self.check(self.api.grid_reset_messages(self.h))

    def sweep(self) -> int:
        n = C.c_int64()
        self.check(self.api.grid_sweep(self.h, C.byref(n)))
        return int(n.value)

    def get_marginals(self):
        out = np.empty((self.H, self.W, self.K), dtype=self.np_dtype)
        self.check(self.api.grid_get_marginals(self.h, out.ctypes.data))
        return out

    def infer_host(self, unary_ptr: int, marginals_out_ptr: int, n_sweeps: int) -> int:
        """One job through (pinned) host buffers, asynchronous and pipelined across calls (``cxb_grid_infer_host``): the
        results are complete after ``sync()``."""
        n = C.c_int64()
        self.check(self.api.grid_infer_host(self.h, C.c_void_p(int(unary_ptr)), C.c_void_p(int(marginals_out_ptr)), int(n_sweeps), C.byref(n)))
        return int(n.value)

    def get_messages(self, which: int):
        out = np.empty((self.H, self.W, self.K), dtype=self.np_dtype)
        self.check(self.api.grid_get_messages(self.h, which, out.ctypes.data))
        return out

    def halo_send_ptr(self, direction: int) -> int:
        return int(self.api.grid_halo_send_ptr(self.h, direction) or 0)

    def halo_recv_ptr(self, direction: int) -> int:
        return int(self.api.grid_halo_recv_ptr(self.h, direction) or 0)

    @property
    def halo_elems(self) -> int:
        return int(self.api.grid_halo_elems(self.h))

    # ---- fused halo exchange over peer memory (cxb_grid_p2p_*): after connecting, sweep() delivers the cut-edge messages
    def p2p_export(self) -> bytes:
        buf = C.create_string_buffer(128)
        self.check(self.api.grid_p2p_export(self.h, buf))
        return buf.raw

    def p2p_connect_ipc(self, direction: int, handles: bytes) -> None:
        buf = C.create_string_buffer(bytes(handles), 128)
        self.check(self.api.grid_p2p_connect_ipc(self.h, direction, buf))

    def p2p_connect_local(self, direction: int, neighbour: "PottsGrid") -> None:
        self.check(self.api.grid_p2p_connect_local(self.h, direction, neighbour.h))


class HmmBatch(_Handle):
    """B discrete HMMs (K states, M symbols, T steps): scaled forward-backward (SURVEY Appendix C)."""
    _prefix = "hmm"

    def __init__(self, n_chains, n_steps, n_states, n_symbols, dtype=capi.F32, device=0, api=None):
        self.api = api or capi.default_api()
        self.B, self.T, self.K, self.M, self.dtype = int(n_chains), int(n_steps), int(n_states), int(n_symbols), dtype
        self.np_dtype = _np_dtype(dtype)
        h = C.c_void_p()
        st = self.api.hmm_create(device, dtype, self.B, self.T, self.K, self.M, C.byref(h))
        if st != capi.OK or not h:
            raise CortexError(st, "cxb_hmm_create failed (CUDA device required; there is no CPU fallback)")
        self.h = h

    @property
    def n_updates(self):
        return self.B * (6 * self.T - 4)

    def set_tables(self, transition, emission):
        a = np.ascontiguousarray(transition, dtype=np.float64)
        e = np.ascontiguousarray(emission, dtype=np.float64)
        assert a.shape == (self.K, self.K) and e.shape == (self.K, self.M)
        self.check(self.api.hmm_set_tables(self.h, a.ctypes.data_as(capi.f64p), e.ctypes.data_as(capi.f64p)))

    def set_observations(self, obs):
        o = np.ascontiguousarray(obs, dtype=np.uint8)
        assert o.shape == (self.T, self.B)
        self.check(self.api.hmm_set_observations(self.h, o.ctypes.data_as(capi.u8p)))

    def update_marginals(self) -> int:
        n = C.c_int64()
        self.check(self.api.hmm_update_marginals(self.h, C.byref(n)))
        return int(n.value)

    def get_marginals(self, t0=0, t1=None):
        t1 = self.T if t1 is None else t1
        out = np.empty((t1 - t0, self.B, self.K), dtype=self.np_dtype)
        self.check(self.api.hmm_get_marginals(self.h, t0, t1, out.ctypes.data))
        return out

    def get_forward(self, t0=0, t1=None):
        t1 = self.T if t1 is None else t1
        out = np.empty((t1 - t0, self.B, self.K), dtype=self.np_dtype)
        self.check(self.api.hmm_get_forward(self.h, t0, t1, out.ctypes.data))
        return out


class PairwiseGraph(_Handle):
    """Arbitrary pairwise categorical graph (one unary leaf factor per variable + pairwise table factors), synchronous
    sweeps = protocol B. `factors` = (u, v, table) with u < v in ascending factor id."""
    _prefix = "pairwise"

    def __init__(self, n_variables, fac_u, fac_v, fac_table, tables, dtype=capi.F32, device=0, api=None):
        self.api = api or capi.default_api()
        tables = np.ascontiguousarray(tables, dtype=np.float64)
        self.n, self.m, self.K, self.n_tables, self.dtype = int(n_variables), len(fac_u), tables.shape[-1], tables.shape[0], dtype
        self.np_dtype = _np_dtype(dtype)
        h = C.c_void_p()
        st = self.api.pairwise_create(device, dtype, self.n, self.m, self.K, self.n_tables, C.byref(h))
        if st != capi.OK or not h:
            raise CortexError(st, "cxb_pairwise_create failed (CUDA device required; there is no CPU fallback)")
        self.h = h
        fu = np.ascontiguousarray(fac_u, dtype=np.int64)
        fv = np.ascontiguousarray(fac_v, dtype=np.int64)
        ft = np.ascontiguousarray(fac_table, dtype=np.int32)
        self.check(self.api.pairwise_set_graph(self.h, fu.ctypes.data_as(capi.i64p), fv.ctypes.data_as(capi.i64p),
                                               ft.ctypes.data_as(capi.i32p)))
        self.check(self.api.pairwise_set_tables(self.h, tables.ctypes.data_as(capi.f64p)))

    def set_unary(self, unary):
        u = np.ascontiguousarray(unary, dtype=self.np_dtype)
        assert u.shape == (self.n, self.K)
        self.check(self.api.pairwise_set_unary(self.h, u.ctypes.data))

    def reset_messages(self):
        self.check(self.api.pairwise_reset_messages(self.h))

    def sweep(self) -> int:
        n = C.c_int64()
        self.check(self.api.pairwise_sweep(self.h, C.byref(n)))
        return int(n.value)

    def get_marginals(self):
        out = np.empty((self.n, self.K), dtype=self.np_dtype)
        self.check(self.api.pairwise_get_marginals(self.h, out.ctypes.data))
        return out

    def get_messages(self, which: int):
        out = np.empty((self.m, 2, self.K), dtype=self.np_dtype)
        self.check(self.api.pairwise_get_messages(self.h, which, out.ctypes.data))
        return out

    @property
    def algorithmic_bytes(self) -> int:
        return int(self.api.pairwise_algorithmic_bytes(self.h))
