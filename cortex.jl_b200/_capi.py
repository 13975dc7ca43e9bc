"""ctypes binding of the C ABI declared in ``include/cortex_b200.h``.

The package only ever binds ``csrc/libcortex_b200.so`` (prefix ``cxb_``).  The binder is
prefix-parametrised so that the test-suite can bind the CPU oracle (``oracle/liboracle.so``,
prefix ``cxo_``) to the *same* host-side frontend and diff the two; the package itself never
loads anything under ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

HERE = Path(__file__).resolve().parent
DEFAULT_LIB = HERE / "csrc" / "libcortex_b200.so"

# enums of include/cortex_b200.h
OK, ERR_NOT_PENDING, ERR_NO_RULE, ERR_OUT_OF_CONTRACT, ERR_BAD_ARG, ERR_UNSUPPORTED_ENGINE, ERR_CUDA, ERR_STATE, ERR_INTERNAL = range(9)
F32, F64 = 0, 1
KIND_UNSPECIFIED, KIND_M2F, KIND_M2V, KIND_PRODUCT, KIND_MARGINAL, KIND_JOINT = range(6)
DEP_INTERMEDIATE, DEP_WEAK, DEP_NO_LISTEN, DEP_NO_CHECK_COMPUTED = 1, 2, 16, 32
NIB_INTERMEDIATE, NIB_WEAK, NIB_COMPUTED, NIB_FRESH = 1, 2, 4, 8
(FAMILY_GAUSS_CANON, FAMILY_CATEGORICAL, FAMILY_GAUSS_MV, FAMILY_BETA, FAMILY_SUM, FAMILY_GAUSS_MP, FAMILY_GAMMA,
 FAMILY_POINT) = range(8)
(RULE_NONE, RULE_GAUSS_OBS, RULE_GAUSS_RW, RULE_CAT_TABLE, RULE_POTTS, RULE_HMM_EMIT, RULE_GAUSS_MV_OBS,
 RULE_GAUSS_MV_RW, RULE_BETA_BERNOULLI, RULE_SCALE2, RULE_NORMAL_MEAN_FIELD, RULE_NORMAL_STRUCTURED, RULE_PROGRAM) = range(13)
(OP_DEP, OP_CONST, OP_PARAM, OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_NEG, OP_EXP, OP_LOG, OP_SQRT, OP_STORE, OP_TSET, OP_TGET,
 OP_NDEPS) = range(1, 16)
RESOLVER_NONE, RESOLVER_DEFAULT_BP, RESOLVER_MEAN_FIELD = range(3)
SCHEDULE_AUTO, SCHEDULE_LEVEL, SCHEDULE_SEQUENTIAL, RAN_REPLAY, RAN_PLAN = range(5)

i32, i64, u8p, i32p, i64p, f64p, vp = (C.c_int32, C.c_int64, C.POINTER(C.c_uint8), C.POINTER(C.c_int32),
                                       C.POINTER(C.c_int64), C.POINTER(C.c_double), C.c_void_p)


class UpdateStats(C.Structure):
    _fields_ = [("levels", i64), ("updates", i64), ("updates_by_kind", i64 * 6), ("final_marginals", i64),
                ("final_linked", i64), ("kernel_launches", i64)]


RULE_CB = C.CFUNCTYPE(i32, vp, i64, i32, i64, i64, i64, i64p, f64p, f64p)
VISIT_CB = C.CFUNCTYPE(i32, vp, i64)

# name -> (restype, argtypes): the generic-engine part of the ABI, shared by cxb_ and cxo_
_COMMON = {
    "create": (i32, [i32, i32, i32, i32, C.POINTER(vp)]),
    "destroy": (None, [vp]),
    "last_error": (C.c_char_p, [vp]),
    "graph_build": (i32, [vp, i64, u8p, i32p, i64, i64p, i64p]),
    "register_rule": (i32, [vp, i32, i32, f64p, i64]),
    "set_factor_params": (i32, [vp, i64, i64p, f64p]),
    "set_variable_families": (i32, [vp, i64, i64p, i32p]),
    "create_signal": (i64, [vp]),
    "add_dependency": (i32, [vp, i64, i64, i32]),
    "resolve_dependencies": (i32, [vp, i32]),
    "resolve_factor_dependencies": (i32, [vp, i32, i64]),
    "resolve_variable_dependencies": (i32, [vp, i32, i64]),
    "set_signal_variant": (i32, [vp, i64, i32, i64, i64]),
    "link_signal": (i32, [vp, i64, i64]),
    "link_signals": (i32, [vp, i64, i64p, i64p]),
    "n_signals": (i64, [vp]),
    "signal_id": (i64, [vp, i32, i64, i64]),
    "signal_info": (i32, [vp, i64, i64p]),
    "get_dependencies": (i64, [vp, i64, i64p, u8p, i64]),
    "get_listeners": (i64, [vp, i64, i64p, u8p, i64]),
    "get_warnings": (i64, [vp, i64p, i64]),
    "set_values": (i32, [vp, i64, i64p, f64p, i64]),
    "get_values": (i32, [vp, i64, i64p, f64p, i64]),
    "is_pending": (i32, [vp, i64]),
    "is_computed": (i32, [vp, i64]),
    "compute": (i32, [vp, i64, i32, i32]),
    "request_inference": (i32, [vp, i64, i64p]),
    "scan": (i64, [vp, i64p, i64]),
    "update_marginals": (i32, [vp, i64, i64p, C.POINTER(UpdateStats)]),
    "prepare_signals": (i64, [vp, i64, i64p]),
    "set_values_prepared": (i32, [vp, i64, vp, i32]),
    "get_values_prepared": (i32, [vp, i64, vp, i32]),
    "prepare_request": (i64, [vp, i64, i64p]),
    "update_marginals_prepared": (i32, [vp, i64, C.POINTER(UpdateStats)]),
    "set_schedule": (i32, [vp, i32]),
    "last_schedule": (i32, [vp]),
    "scan_dfs": (i64, [vp, i64p, i64]),
    "process_dependencies_table": (i64, [vp, i64, i32, u8p, i64p, i64, i32p]),
    "trace_get_variables": (i64, [vp, i64p, i64]),
    "trace_enable": (i32, [vp, i32]),
    "trace_get": (i64, [vp, i64p, i64p, i64]),
    "trace_get_times": (i64, [vp, i64p, i64]),
}

# structured engines, cxb_ only
_STRUCTURED = {
    "stream": (vp, [vp]),
    "version": (C.c_char_p, []),
    "kernel_launches": (C.c_uint64, []),
    "chains_create": (i32, [i32, i32, i64, i64, C.POINTER(vp)]),
    "chains_destroy": (None, [vp]),
    "chains_last_error": (C.c_char_p, [vp]),
    "chains_set_noise": (i32, [vp, f64p, f64p]),
    "chains_set_observations": (i32, [vp, vp]),
    "chains_set_observations_device": (i32, [vp, vp]),
    "chains_update_marginals": (i32, [vp, i64p]),
    "chains_get_marginals": (i32, [vp, vp]),
    "chains_get_messages": (i32, [vp, i32, vp]),
    "chains_device_ptr": (vp, [vp, i32]),
    "chains_infer_host": (i32, [vp, vp, vp, i64p]),
    "chains_stream": (vp, [vp]),
    "chains_last_kernel_ms": (i32, [vp, C.POINTER(C.c_float)]),
    "chains_sync": (i32, [vp]),
    "grid_create": (i32, [i32, i32, i64, i64, i32, C.c_double, i32, i32, C.POINTER(vp)]),
    "grid_destroy": (None, [vp]),
    "grid_last_error": (C.c_char_p, [vp]),
    "grid_set_unary": (i32, [vp, vp]),
    "grid_set_couplings": (i32, [vp, f64p, f64p]),
    "grid_reset_messages": (i32, [vp]),
    "grid_sweep": (i32, [vp, i64p]),
    "grid_halo_send_ptr": (vp, [vp, i32]),
    "grid_halo_recv_ptr": (vp, [vp, i32]),
    "grid_halo_elems": (i64, [vp]),
    "grid_p2p_export": (i32, [vp, vp]),
    "grid_p2p_connect_ipc": (i32, [vp, i32, vp]),
    "grid_p2p_connect_local": (i32, [vp, i32, vp]),
    "grid_get_marginals": (i32, [vp, vp]),
    "grid_infer_host": (i32, [vp, vp, vp, i32, i64p]),
    "grid_get_messages": (i32, [vp, i32, vp]),
    "grid_stream": (vp, [vp]),
    "grid_last_kernel_ms": (i32, [vp, C.POINTER(C.c_float)]),
    "grid_sync": (i32, [vp]),
    "hmm_create": (i32, [i32, i32, i64, i64, i32, i32, C.POINTER(vp)]),
    "hmm_destroy": (None, [vp]),
    "hmm_last_error": (C.c_char_p, [vp]),
    "hmm_set_tables": (i32, [vp, f64p, f64p]),
    "hmm_set_observations": (i32, [vp, u8p]),
    "hmm_update_marginals": (i32, [vp, i64p]),
    "hmm_get_marginals": (i32, [vp, i64, i64, vp]),
    "hmm_get_forward": (i32, [vp, i64, i64, vp]),
    "hmm_stream": (vp, [vp]),
    "hmm_last_kernel_ms": (i32, [vp, C.POINTER(C.c_float)]),
    "hmm_sync": (i32, [vp]),
    "pairwise_create": (i32, [i32, i32, i64, i64, i32, i32, C.POINTER(vp)]),
    "pairwise_destroy": (None, [vp]),
    "pairwise_last_error": (C.c_char_p, [vp]),
    "pairwise_set_graph": (i32, [vp, i64p, i64p, i32p]),
    "pairwise_set_tables": (i32, [vp, f64p]),
    "pairwise_set_unary": (i32, [vp, vp]),
    "pairwise_reset_messages": (i32, [vp]),
    "pairwise_sweep": (i32, [vp, i64p]),
    "pairwise_get_marginals": (i32, [vp, vp]),
    "pairwise_get_messages": (i32, [vp, i32, vp]),
    "pairwise_algorithmic_bytes": (i64, [vp]),
    "pairwise_stream": (vp, [vp]),
    "pairwise_last_kernel_ms": (i32, [vp, C.POINTER(C.c_float)]),
    "pairwise_sync": (i32, [vp]),
}

# oracle-only extras (bound when present)
_ORACLE_EXTRA = {
    "set_rule_callback": (i32, [vp, RULE_CB, vp]),
    "raw_props": (i32, [vp, i64]),
    "update_marginals_seq": (i32, [vp, i64, i64p, C.POINTER(UpdateStats)]),
    "count_is_pending_calls": (i64, [vp]),
    "process_dependencies": (i32, [vp, i64, i32, VISIT_CB, vp]),
    "chains_reference": (i32, [i64, i64, f64p, f64p, f64p, f64p]),
}


def exported_symbols(prefix: str = "cxb_"):
    """Every symbol include/cortex_b200.h declares (used by the CPU-side ABI test)."""
    return [prefix + n for n in list(_COMMON) + list(_STRUCTURED)]


class CApi:
    """Binds one shared library exposing the ABI under ``prefix``."""

    def __init__(self, path=None, prefix: str = "cxb_"):
        path = Path(path) if path is not None else DEFAULT_LIB
        if not path.exists():
            raise ImportError(
                f"{path} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                "There is no CPU fallback."
            )
        self.path = str(path)
        self.prefix = prefix
        self.lib = C.CDLL(self.path, mode=os.RTLD_GLOBAL if hasattr(os, "RTLD_GLOBAL") else 0)
        tables = [_COMMON]
        if prefix == "cxb_":
            tables.append(_STRUCTURED)
        for table in tables:
            for name, (res, args) in table.items():
                fn = getattr(self.lib, prefix + name)
                fn.restype, fn.argtypes = res, args
                setattr(self, name, fn)
        for name, (res, args) in _ORACLE_EXTRA.items():
            fn = getattr(self.lib, prefix + name, None)
            if fn is not None:
                fn.restype, fn.argtypes = res, args
                setattr(self, name, fn)

    @property
    def is_device(self) -> bool:
        return self.prefix == "cxb_"


_default_api = None


def default_api() -> CApi:
    """The product library (hand-written sm_100a kernels). Fails loudly when it is not built."""
    global _default_api
    if _default_api is None:
        _default_api = CApi(DEFAULT_LIB, "cxb_")
    return _default_api
