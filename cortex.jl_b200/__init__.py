"""cortex.jl_b200 — B200-native batched belief-propagation engine behind Cortex.jl's API.

Only what the `update_marginals!` hot path needs lives here:
  csrc/               hand-written sm_100a CUDA kernels + the C ABI (include/cortex_b200.h)
  _capi.py            ctypes binding of that ABI
  inference_signal.py / model_engine.py / inference_engine.py
                      host-side mirror of the reference interface (same names and semantics)
  structured.py       structured model engines (closed-form plans of the fixed-stencil graphs)
  julia/CortexB200.jl the `ccall` glue a Cortex.jl maintainer adds (cannot run in this image)

The directory name contains a dot, so import it through `__graft_entry__.load_package()`
(registers the package as module `cortex_jl_b200`).
"""
from . import _capi as capi  # noqa: F401
from ._capi import CApi, default_api, exported_symbols  # noqa: F401
from .inference_signal import *  # noqa: F401,F403
from .inference_signal import (CortexError, NoRuleError, NotPendingError, OutOfContractError, Signal,  # noqa: F401
                               SignalStore)
from .model_engine import *  # noqa: F401,F403
from .inference_engine import *  # noqa: F401,F403
from .inference_engine import _as_ids  # noqa: F401
from .structured import GaussianChainBatch, HmmBatch, PairwiseGraph, PottsGrid  # noqa: F401
from .debug import signal_to_dot  # noqa: F401
from .sharding import HaloExchanger, batch_shard, connect_row_neighbours, device_tensor, row_shard, shard_couplings  # noqa: F401

__version__ = "0.1.0"
