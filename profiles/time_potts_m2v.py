"""A/B of the Potts sweep at the benchmarked size (8192^2, K = 16, fp32): every m2v plane and every marginal stored each
sweep (CXB_GRID_EAGER_M2V=1) against the default, where a sweep stores the m2v and the marginals of its first and last rows
only and the first read of an m2v plane or of the marginals rebuilds the others (k_potts_m2v). The two grids take 60 GB
each, so they are created one after the other, alternating, for `rounds` rounds. Per arm: 3 x 50 warm-up sweeps, 50 sweeps
timed with CUDA events on the library's stream, then last_kernel_ms over 10 sweeps; the lazy arm also times the two rebuilds
(marginals, then m2v planes) with torch.profiler.
Usage: python profiles/time_potts_m2v.py [N] [rounds]"""
import gc
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import load_package  # noqa: E402

C = load_package()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 3
K, BETA, SWEEPS = 16, 0.7, 50

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                     text=True).stdout.strip(), flush=True)
rng = np.random.Generator(np.random.PCG64(1234))  # the evidence of bench.py's potts_grid record
unary = np.empty((N, N, K), dtype=np.float32)
for i in range(0, N, 256):
    e = rng.standard_exponential((min(256, N - i), N, K), dtype=np.float32)
    unary[i:i + 256] = e / e.sum(axis=-1, keepdims=True)
# bytes per sweep, counted as bench.py does: 64 B per K-vector read or written; m2v = existing (pixel, direction) pairs
pix = N * N
m2v = 2 * (N - 1) * N * 2
bytes_all = 64 * ((m2v + pix) + (2 * m2v + pix))  # 896 B per interior pixel: reads 4 m2f + unary, writes 4 m2v + 4 m2f + marginal
bytes_lazy = 64 * ((m2v + pix) + m2v)  # 576 B per interior pixel: without the m2v and marginal stores
bytes_rb_marg = 64 * ((m2v + pix) + pix)  # marginal rebuild: reads 4 m2f + unary, writes the marginal
bytes_rb_m2v = 64 * 2 * m2v  # m2v rebuild: reads 4 m2f, writes 4 m2v


def rebuild_ms(g, read):
    """device time of the k_potts_m2v launch that read(g), the first read after a sweep, enqueues"""
    try:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            read(g)
        us = [e.time_range.elapsed_us() for e in prof.events() if "k_potts_m2v" in e.name]
        return us[0] / 1e3 if us else None
    except Exception as ex:  # noqa: BLE001 - the A/B numbers do not depend on it
        print(f"rebuild not timed: {type(ex).__name__}: {ex}", flush=True)
        return None


def arm(eager):
    os.environ["CXB_GRID_EAGER_M2V"] = "1" if eager else "0"
    g = C.PottsGrid(N, N, K, BETA, dtype=C.capi.F32)
    g.set_unary(unary)
    g.reset_messages()
    ext = torch.cuda.ExternalStream(g.stream)
    for _ in range(3 * SWEEPS):
        g.sweep()
    ext.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(SWEEPS):
        g.sweep()
    e1.record(ext)
    e1.synchronize()
    ms = e0.elapsed_time(e1) / SWEEPS
    kms = []
    for _ in range(10):
        g.sweep()
        kms.append(g.last_kernel_ms())
    rb = None if eager else (rebuild_ms(g, lambda x: x.get_marginals()), rebuild_ms(g, lambda x: x.get_messages(0)))
    del g
    gc.collect()
    return ms, statistics.mean(kms), rb


res = {True: [], False: []}
for r in range(ROUNDS):
    for eager in (True, False):
        ms, kms, rb = arm(eager)
        res[eager].append((ms, kms))
        name = "eager (every value stored)" if eager else "lazy (rebuilt on read)"
        extra = ""
        for what, t, nb in zip(("marginals", "m2v planes"), rb or (), (bytes_rb_marg, bytes_rb_m2v)):
            if t:
                extra += f", rebuild of the {what} {t:.3f} ms = {nb / (t * 1e6):.0f} GB/s"
        print(f"round {r} {name:26s}: {ms:.3f} ms per sweep (events, {SWEEPS} sweeps), last_kernel_ms {kms:.3f}{extra}", flush=True)
print(f"{N}^2, K = {K}: bytes per sweep {bytes_all / 1e9:.2f} GB (896 B per pixel) / {bytes_lazy / 1e9:.2f} GB (576 B per pixel)")
for eager in (True, False):
    ev = [m for m, _ in res[eager]]
    kk = [k for _, k in res[eager]]
    mean = statistics.mean(ev)
    print(f"{'eager' if eager else 'lazy':5s}: {mean:.3f} ms per sweep (events), spread {min(ev):.3f} .. {max(ev):.3f} "
          f"({(max(ev) - min(ev)) / mean * 100:.2f} %); last_kernel_ms {statistics.mean(kk):.3f} "
          f"({min(kk):.3f} .. {max(kk):.3f}); {bytes_all / (mean * 1e6):.0f} GB/s on the 896-B count, "
          f"{bytes_lazy / (mean * 1e6):.0f} GB/s on the 576-B count")
ratio = [a[0] / b[0] for a, b in zip(res[True], res[False])]
print(f"eager / lazy per sweep: {statistics.mean(ratio):.3f} (rounds: {', '.join(f'{x:.3f}' for x in ratio)})")
