"""Multi-GPU plumbing (one process per GPU, torch.distributed): how the hot path shards (SURVEY §8e).

* batches of independent chains (configs 2, 3): `batch_shard` — no data-path collective;
* row-sharded grid (config 4): `row_shard` + `HaloExchanger` — per sweep every rank sends the m2f messages of its
  first/last row to the row-neighbour ranks and receives theirs (8192*K*4 B = 512 KiB per direction at config 4).
The exchange is expressed on torch tensors, so the same code runs over NCCL (tensors wrapping the library's device
halo buffers) and over gloo on CPU (tests/test_sharding_gloo.py).
"""
from __future__ import annotations

from typing import Optional, Tuple


def batch_shard(n_items: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous split of `n_items` independent units: (first, count) of this rank (remainder to the low ranks)."""
    base, rem = divmod(n_items, world)
    first = rank * base + min(rank, rem)
    return first, base + (1 if rank < rem else 0)


def row_shard(n_rows: int, world: int, rank: int) -> Tuple[int, int, bool, bool]:
    """(row0, rows, has_upper_neighbour, has_lower_neighbour) of this rank's row block."""
    row0, rows = batch_shard(n_rows, world, rank)
    if rows == 0:
        raise ValueError("more ranks than grid rows")
    return row0, rows, rank > 0, rank < world - 1


def shard_couplings(horizontal, vertical, row0: int, rows: int):
    """This row block's arguments of `PottsGrid.set_couplings`, from the global per-edge couplings of an H x W grid:
    `horizontal[H][W-1]` (between (i, j) and (i, j+1)) and `vertical[H-1][W]` (between rows i and i+1). Returns
    (horizontal[rows][W-1], vertical[rows+1][W]): local row r of the vertical array is the factor between global rows
    row0 + r - 1 and row0 + r, so rows 0 and `rows` are the cut edges, zeros where there is no neighbour. Two neighbours
    cut their shared edge from the same global row, so they agree on it."""
    import numpy as np

    hz = np.asarray(horizontal, dtype=np.float64)
    vt = np.asarray(vertical, dtype=np.float64)
    H = hz.shape[0]
    W = vt.shape[1] if vt.ndim == 2 else hz.shape[1] + 1
    if hz.shape != (H, W - 1) or vt.shape != (H - 1, W):
        raise ValueError(f"global couplings must be horizontal [H][W-1] and vertical [H-1][W], got {hz.shape} and {vt.shape}")
    if not (0 <= row0 and rows > 0 and row0 + rows <= H):
        raise ValueError(f"rows [{row0}, {row0 + rows}) are not inside a grid of {H} rows")
    v = np.zeros((rows + 1, W))
    lo, hi = max(row0, 1), min(row0 + rows, H - 1)  # local row r <-> global edge row row0 + r - 1, which exists for 1..H-1
    v[lo - row0:hi - row0 + 1] = vt[lo - 1:hi]
    return np.ascontiguousarray(hz[row0:row0 + rows]), v


class HaloExchanger:
    """Per-sweep halo exchange between row-neighbour ranks. `dist` is torch.distributed (any backend)."""

    def __init__(self, dist, rank: int, world: int):
        self.dist, self.rank, self.world = dist, rank, world

    def exchange(self, send_up, send_down, recv_up, recv_down):
        """send_up -> rank-1 (lands in its recv_down), send_down -> rank+1 (lands in its recv_up).
        Any of the tensors may be None at the outer borders. Returns when the receives have completed
        (stream-ordered for NCCL)."""
        d, ops = self.dist, []
        if self.rank > 0:
            ops.append(d.P2POp(d.isend, send_up, self.rank - 1))
            ops.append(d.P2POp(d.irecv, recv_up, self.rank - 1))
        if self.rank < self.world - 1:
            ops.append(d.P2POp(d.isend, send_down, self.rank + 1))
            ops.append(d.P2POp(d.irecv, recv_down, self.rank + 1))
        if not ops:
            return
        for w in d.batch_isend_irecv(ops):
            w.wait()


def connect_row_neighbours(dist, grid, rank: int, world: int) -> bool:
    """Fused halo exchange (cxb_grid_p2p_*): every rank publishes the CUDA IPC handles of its halo buffer and sweep
    counters, opens its row neighbours' and from then on `grid.sweep()` stores the cut-edge messages straight into the
    neighbour GPU's memory over NVLink — no separate exchange call. Returns False (and connects nothing) when any rank
    cannot open a neighbour's handle; the caller then keeps using `HaloExchanger` (NCCL)."""
    if world == 1:
        return True
    handles = [None] * world
    dist.all_gather_object(handles, grid.p2p_export())
    ok = 1
    try:
        if rank > 0:
            grid.p2p_connect_ipc(0, handles[rank - 1])
        if rank < world - 1:
            grid.p2p_connect_ipc(1, handles[rank + 1])
    except Exception:  # no peer access between the two GPUs
        ok = 0
    oks = [None] * world
    dist.all_gather_object(oks, ok)
    return all(oks)


def device_tensor(ptr: int, n_elems: int, device_index: int, typestr: str = "<f4"):
    """Zero-copy torch view of a device buffer owned by the CUDA library (for NCCL)."""
    import torch

    class _Arr:
        pass

    a = _Arr()
    a.__cuda_array_interface__ = {"shape": (int(n_elems),), "typestr": typestr, "data": (int(ptr), False), "version": 2}
    return torch.as_tensor(a, device=f"cuda:{device_index}")
