"""Cost of per-edge couplings on the Potts sweep at the benchmarked size (8192^2, K = 16, fp32): a uniform grid (one beta,
the path bench.py times) against a grid with contrast-sensitive couplings beta_ij = lam * exp(-|I_i - I_j|^2 / 2 <|I_i - I_j|^2>)
of a smooth random image I, beta in [0, lam], lam = 1.5 (cxb_grid_set_couplings). Both grids live side by side (60 GB each)
and are timed alternately, `rounds` rounds of one window each: a window is WINDOW_SWEEPS sweeps (>= 1 s) between two CUDA
events on the library's stream, after 3 x 50 warm-up sweeps; last_kernel_ms (the library's own events around one sweep)
over 10 sweeps follows each window. Each round also times the m2v and marginal rebuilds (k_potts_m2v) of both grids with
torch.profiler. Before the timing, a bit-identity check at 2048^2: per-edge couplings all equal to the create-time beta
against the uniform grid, every message plane and the marginals after 3 sweeps.
Usage: python profiles/time_potts_couplings.py [N] [rounds]"""
import gc
import os
import statistics
import subprocess
import sys

import numpy as np
import torch
from scipy.ndimage import gaussian_filter

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import load_package  # noqa: E402

C = load_package()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 4
K, BETA, LAM, WARMUP, WINDOW_SWEEPS = 16, 0.7, 1.5, 150, 200

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                     text=True).stdout.strip(), flush=True)


def evidence(n):
    rng = np.random.Generator(np.random.PCG64(1234))  # the evidence of bench.py's potts_grid record
    u = np.empty((n, n, K), dtype=np.float32)
    for i in range(0, n, 256):
        e = rng.standard_exponential((min(256, n - i), n, K), dtype=np.float32)
        u[i:i + 256] = e / e.sum(axis=-1, keepdims=True)
    return u


def contrast_couplings(n, seed=7):
    img = gaussian_filter(np.random.Generator(np.random.PCG64(seed)).random((n, n)), 4.0)
    img = (img - img.min()) / (img.max() - img.min())
    dh, dv = img[:, 1:] - img[:, :-1], img[1:, :] - img[:-1, :]
    s2 = 2 * np.mean(np.concatenate([dh.ravel() ** 2, dv.ravel() ** 2]))
    return LAM * np.exp(-dh ** 2 / s2), LAM * np.exp(-dv ** 2 / s2)


# ---- bit identity: equal per-edge couplings == the uniform grid ----------------------------------------------------------------
n = 2048
u = evidence(n)
grids = []
for per_edge in (False, True):
    g = C.PottsGrid(n, n, K, BETA, dtype=C.capi.F32)
    if per_edge:
        g.set_couplings(np.full((n, n - 1), BETA), np.full((n + 1, n), BETA))
    g.set_unary(u)
    g.reset_messages()
    for _ in range(3):
        g.sweep()
    grids.append(g)
same = all(np.array_equal(grids[0].get_messages(w), grids[1].get_messages(w)) for w in range(8)) and \
    np.array_equal(grids[0].get_marginals(), grids[1].get_marginals())
print(f"bit identity at {n}^2, K = {K}, 3 sweeps, per-edge couplings all = beta vs the uniform grid, 8 planes + marginals: "
      f"{'identical' if same else 'DIFFERENT'}", flush=True)
del grids, g, u
gc.collect()
if not same:
    sys.exit(1)

# ---- timing ---------------------------------------------------------------------------------------------------------------------
unary = evidence(N)
hz, vt = contrast_couplings(N)
print(f"couplings: {hz.size + vt.size} edges, beta in [{min(hz.min(), vt.min()):.3f}, {max(hz.max(), vt.max()):.3f}], "
      f"mean {np.mean(np.concatenate([hz.ravel(), vt.ravel()])):.3f}", flush=True)
# bytes per sweep, counted as bench.py does: 64 B per K-vector read or written; m2v = existing (pixel, direction) pairs
pix = N * N
m2v = 2 * (N - 1) * N * 2
bytes_uniform = 64 * ((m2v + pix) + m2v)  # 576 B per interior pixel: reads 4 m2f + unary, writes 4 m2f
bytes_coupled = bytes_uniform + 4 * (N * N + (N + 1) * N)  # + the two coupling planes, each weight from DRAM once: 584 B
bytes_rb_marg = 64 * ((m2v + pix) + pix)
bytes_rb_m2v = 64 * 2 * m2v

grid = {}
for per_edge in (False, True):
    g = C.PottsGrid(N, N, K, BETA, dtype=C.capi.F32)
    g.set_unary(unary)
    if per_edge:
        g.set_couplings(*C.shard_couplings(hz, vt, 0, N))
    g.reset_messages()
    grid[per_edge] = g
del unary, hz, vt
gc.collect()


def rebuild_ms(g, read):
    """device time of the k_potts_m2v launch that read(g), the first read after a sweep, enqueues"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        read(g)
    us = [e.time_range.elapsed_us() for e in prof.events() if "k_potts_m2v" in e.name]
    return us[0] / 1e3 if us else float("nan")


def window(g, sweeps):
    ext = torch.cuda.ExternalStream(g.stream)
    ext.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(sweeps):
        g.sweep()
    e1.record(ext)
    e1.synchronize()
    return e0.elapsed_time(e1)


for g in grid.values():
    window(g, WARMUP)
res = {False: [], True: []}
for r in range(ROUNDS):
    for per_edge in (False, True):
        g = grid[per_edge]
        total = window(g, WINDOW_SWEEPS)
        kms = []
        for _ in range(10):
            g.sweep()
            kms.append(g.last_kernel_ms())
        rb_marg = rebuild_ms(g, lambda x: x.get_marginals())
        g.sweep()
        rb_m2v = rebuild_ms(g, lambda x: x.get_messages(0))
        res[per_edge].append((total / WINDOW_SWEEPS, statistics.mean(kms), rb_marg, rb_m2v))
        ms = total / WINDOW_SWEEPS
        print(f"round {r} {'per-edge' if per_edge else 'uniform':8s}: {ms:.3f} ms per sweep ({WINDOW_SWEEPS} sweeps, {total / 1e3:.2f} s), "
              f"last_kernel_ms {statistics.mean(kms):.3f}; rebuild of the marginals {rb_marg:.3f} ms, of the m2v planes {rb_m2v:.3f} ms",
              flush=True)

print(f"{N}^2, K = {K}: bytes per sweep, uniform {bytes_uniform / 1e9:.2f} GB (576 B per pixel), per-edge {bytes_coupled / 1e9:.2f} GB "
      f"(584 B per pixel, predicted ratio {bytes_coupled / bytes_uniform:.4f})")
for per_edge, nb in ((False, bytes_uniform), (True, bytes_coupled)):
    ev = [x[0] for x in res[per_edge]]
    kk = [x[1] for x in res[per_edge]]
    mean = statistics.mean(ev)
    rm, rv = statistics.mean(x[2] for x in res[per_edge]), statistics.mean(x[3] for x in res[per_edge])
    print(f"{'per-edge' if per_edge else 'uniform':8s}: {mean:.3f} ms per sweep (events), spread {min(ev):.3f} .. {max(ev):.3f} "
          f"({(max(ev) - min(ev)) / mean * 100:.2f} %); last_kernel_ms {statistics.mean(kk):.3f} ({min(kk):.3f} .. {max(kk):.3f}); "
          f"{nb / (mean * 1e6):.0f} GB/s on its byte count; rebuild of the marginals {rm:.3f} ms "
          f"({bytes_rb_marg / (rm * 1e6):.0f} GB/s), of the m2v planes {rv:.3f} ms ({bytes_rb_m2v / (rv * 1e6):.0f} GB/s)")
ratio = [b[0] / a[0] for a, b in zip(res[False], res[True])]
print(f"per-edge / uniform per sweep: {statistics.mean(ratio):.4f} (rounds: {', '.join(f'{x:.4f}' for x in ratio)}); "
      f"rebuilds: marginals {statistics.mean(b[2] / a[2] for a, b in zip(res[False], res[True])):.4f}, "
      f"m2v {statistics.mean(b[3] / a[3] for a, b in zip(res[False], res[True])):.4f}")
