#!/usr/bin/env python
"""bench.py — message-updates/sec of the update_marginals! hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload potts_grid|gauss_chains|hmm64|hmm512|powerlaw|powerlaw_engine|chain1k|chains_engine]
    python bench.py --impl reference ...     # the CPU oracle port of the reference, on the host cores
    python bench.py ... --dump-outputs DIR   # also write the marginals of the last timed step as DIR/<workload>_marginals.npy

One "step" = one pass of the hot path over one batch of synthetic input:
  potts_grid  (default at every N, BASELINE configs[3]): 50 synchronous sweeps of the 8192^2, K=16 grid, row-sharded over the
              N GPUs with the halo exchange fused into the sweep kernel (strong scaling: the north star's 1 -> 8 target);
  gauss_chains (configs[1]): update_marginals! over 65,536 chains x T=1,024 per GPU (fp32 / fp64);
  hmm64 / hmm512 (configs[2]): scaled forward-backward of 1,024 HMMs x T=1e5, batch-sharded (K=512: 1,024/N chains per GPU,
              at most 128: the marginal planes of more do not fit one GPU);
  powerlaw    (configs[4]): one protocol-B sweep of the fused CSR engine on a 10M-variable Chung-Lu graph;
  powerlaw_engine / chain1k (configs[0]) / chains_engine: the same models through cxb_graph_build + cxb_update_marginals (the
              reference's single entry point; memoised schedules and closed-form plans behind it).
The default run prints ONE JSON line (rank 0): the potts_grid record, with one sub-record per other config under "others".
It runs on the tree build() left (the CUDA library and the CPU oracle) and writes nothing there: the tree may be read-only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # no __pycache__ in the tree
import __graft_entry__ as entry  # noqa: E402

METRIC, UNIT = "message_updates_per_sec", "updates/s"
DUMP_BYTES = 60 * 2**20  # --dump-outputs writes at most this much (64 MB in all with the .npy headers)


def dump_rows(n_rows, row_bytes):
    """Indices of the rows of an output that --dump-outputs writes: all of them when they fit DUMP_BYTES, else a fixed, seeded
    sample (the same for the same arguments, so that two builds can be compared output for output)."""
    k = max(1, DUMP_BYTES // row_bytes)
    if n_rows <= k:
        return np.arange(n_rows)
    return np.sort(np.random.default_rng(0).choice(n_rows, k, replace=False))


def dump_output(args, name, rows):
    """Write one output of the last timed step (rows chosen by dump_rows) as <DIR>/<workload>_<name>.npy."""
    out = Path(args.dump_outputs)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / f"{args.workload}_{name}.npy", np.ascontiguousarray(rows))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)", d
    return 6650.0, "fallback (B200_PROFILING.md)", {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx, self.rows, self.proc = device_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
def dist_setup(n_gpus):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


NUMA_NOTE = {}


def bind_to_gpu_numa_node(local):
    """Run this rank (and first-touch its pinned buffers) on the CPU cores of the NUMA node its GPU hangs off
    (/sys/bus/pci/devices/<bdf>/local_cpulist): on an 8-GPU box the host side of the host<->device copies of all ranks
    otherwise ends up behind one memory controller / PCIe root (round 1: per-GPU e2e fell 4.9x from 1 to 8 GPUs)."""
    import torch

    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        path = Path("/sys/bus/pci/devices") / bdf / "local_cpulist"
        cpus = set()
        for part in path.read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            node = (Path("/sys/bus/pci/devices") / bdf / "numa_node").read_text().strip()
            NUMA_NOTE.update({"gpu": local, "pci": bdf, "numa_node": int(node), "cpus": len(cpus)})
    except Exception as e:  # noqa: BLE001 - binding is an optimisation; say why it did not happen
        NUMA_NOTE.update({"gpu": local, "unbound": repr(e)[:120]})


def barrier(world):
    import torch
    import torch.distributed as dist

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world, local):
    import torch
    import torch.distributed as dist

    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, world, local):
    import torch
    import torch.distributed as dist

    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


class DevArr:
    def __init__(self, ptr, n, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def timed(stream_ptr, fn, steps, warmup, world, local, min_ms=0.0):
    """W warm-up + K timed steps on the library's stream; returns the elapsed ms (max over ranks). With min_ms the step
    count is raised until the timed region is at least that long (sub-records: >= 1 s, so that the clock sampler sees
    the region); the count actually timed is left in timed.last_steps."""
    import torch

    ext = torch.cuda.ExternalStream(stream_ptr, device=local)
    for _ in range(warmup):
        fn()
    ext.synchronize()
    while True:
        barrier(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        for _ in range(steps):
            fn()
        e1.record(ext)
        e1.synchronize()
        barrier(world)
        ms = max_over_ranks(e0.elapsed_time(e1), world, local)
        if ms >= min_ms or steps >= 1 << 20:
            timed.last_steps = steps
            return ms
        steps = int(min(1 << 20, max(steps * 2, steps * 1.25 * min_ms / max(ms, 1e-3)))) + 1


# ---------------------------------------------------------------------------------------------------------------
def cpu_baseline_chain(T=1024, budget_s=12.0):
    """The reference CPU path = oracle port (explicit Signal graph, sequential update_marginals!), 1 core."""
    from tests import models
    from tests._pkg import ORACLE_LIB, pkg

    api = pkg.CApi(ORACLE_LIB, "cxo_")
    rng = np.random.Generator(np.random.PCG64(1234))
    e, x, y, lik, tr = models.make_ssm_model(T, api, form="canon", q=1.0, r=1.0)
    data = np.cumsum(rng.standard_normal(T)) + rng.standard_normal(T)
    sig = [pkg.get_connection_message_to_factor(e, y[i], lik[i]) for i in range(T)]
    ids = np.ascontiguousarray([s.sid for s in sig], dtype=np.int64)
    vals = np.zeros((T, 2))
    vals[:, 0] = data
    xs = np.ascontiguousarray(x, dtype=np.int64)
    cap = pkg.capi

    def one():
        api.set_values(e.store.h, T, ids.ctypes.data_as(cap.i64p), vals.ctypes.data_as(cap.f64p), 2)
        st = cap.UpdateStats()
        import ctypes

        api.update_marginals_seq(e.store.h, T, xs.ctypes.data_as(cap.i64p), ctypes.byref(st))
        return st.updates

    one()
    t0, n, reps = time.perf_counter(), 0, 0
    while time.perf_counter() - t0 < budget_s:
        n += one()
        reps += 1
    dt = time.perf_counter() - t0
    return n / dt, f"1 chain x T={T} explicit Signal graph, sequential update_marginals!, {reps} repetitions in {dt:.1f} s"


def _timed_updates(one, budget_s):
    """Repeat `one()` (returns the number of updates it performed) for about budget_s seconds -> (updates/s, reps, seconds)."""
    one()
    t0, n, reps = time.perf_counter(), 0, 0
    while time.perf_counter() - t0 < budget_s:
        n += one()
        reps += 1
    dt = time.perf_counter() - t0
    return n / dt, reps, dt


def cpu_baseline_workload(workload, budget_s=12.0):
    """The oracle port (explicit Signal graph, sequential update_marginals!, 1 core) on a BOUNDED sample of the same
    workload: the full-size graphs of configs 3-5 cannot be built on the host (SURVEY 8d), so the sample is a reduced
    instance of the same family, rules and protocol; the size is stated in the returned text."""
    if workload in ("gauss_chains", "chain1k", "chains_engine"):
        return cpu_baseline_chain(1024 if workload == "gauss_chains" else 1000, budget_s)
    from tests import models
    from tests._pkg import ORACLE_LIB, pkg

    api = pkg.CApi(ORACLE_LIB, "cxo_")
    rng = np.random.Generator(np.random.PCG64(1234))
    if workload == "potts_grid":
        H = W = 64
        K = 16
        e, pix, un, pair = models.make_grid_model(H, W, K, 0.7, api, rule="potts", link=True)
        vs = [v for row in pix for v in row]
        models.protocol_b_init(e, vs, K)
        usig = [pkg.get_connection_message_to_variable(e, pix[i][j], un[i][j]) for i in range(H) for j in range(W)]
        unary = rng.dirichlet(np.ones(K), size=H * W)
        v, reps, dt = _timed_updates(lambda: models.protocol_b_sweep(e, vs, usig, unary, schedule="seq").updates, budget_s)
        return v, f"Potts grid {H}x{W}, K={K}, protocol-B sweeps on the explicit Signal graph, {reps} sweeps in {dt:.1f} s"
    if workload in ("hmm64", "hmm512"):
        K, M = (512, 32) if workload == "hmm512" else (64, 32)
        T = 64 if K == 512 else 512
        A = rng.dirichlet(np.ones(K), size=K)
        E = rng.dirichlet(np.ones(K), size=M).T * K
        e, z, y, prior, em, tr = models.make_hmm_model(T, K, M, A, E, api)
        obs = rng.integers(0, M, size=T)

        def one():
            models.hmm_set_data(e, z, y, prior, em, obs, K)
            return pkg.update_marginals(e, z, schedule="seq").updates

        v, reps, dt = _timed_updates(one, budget_s)
        return v, f"1 HMM chain, K={K}, M={M}, T={T}, explicit Signal graph, sequential update_marginals!, {reps} repetitions in {dt:.1f} s"
    if workload in ("powerlaw", "powerlaw_engine"):
        n = 20000
        e, vs, un, pair, unary, tables, ttype = models.make_powerlaw_model(n, 2 * n, 8, api)
        models.protocol_b_init(e, vs, 8)
        usig = [pkg.get_connection_message_to_variable(e, vs[i], un[i]) for i in range(n)]
        v, reps, dt = _timed_updates(lambda: models.protocol_b_sweep(e, vs, usig, unary, schedule="seq").updates, budget_s)
        return v, (f"Chung-Lu power-law graph, {n} variables, {2 * n} pairwise factors, K=8, protocol-B sweeps on the explicit Signal "
                   f"graph, {reps} sweeps in {dt:.1f} s")
    raise ValueError(workload)


def _ref_worker(args):
    workload, budget = args
    v, _ = cpu_baseline_workload(workload, budget)
    return v


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (= the oracle port; Julia is absent from the
    image) on the host cores. The reference is single-threaded, so 'all host threads' = independent replicas."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    cores = os.cpu_count() or 1
    per_step_budget = max(1.0, min(10.0, 75.0 / max(1, args.steps + args.warmup)))
    _, what = cpu_baseline_workload(args.workload, 0.2)  # the sample's description (and a warm build of the graph code paths)
    vals = []
    with mp.get_context("spawn").Pool(cores) as pool:
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            v = sum(pool.map(_ref_worker, [(args.workload, per_step_budget)] * cores))
            if s >= args.warmup:
                vals.append((v, time.perf_counter() - t0))
    value = statistics.mean(v for v, _ in vals)
    sample = (f"SAMPLED: {cores} independent replicas (one per core; the reference is single-threaded), each: {what.split(', explicit')[0]}, "
              f"explicit Signal graph, sequential schedule, ~{per_step_budget:.1f} s of work per step (ms_per_step is that time budget, not "
              f"the time of the full-size workload)")
    cfg = workload_config(args, max(1, args.gpus))  # the GPU arm's config; what the CPU actually ran is in "sampled" / cpu_baseline.sample
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(t for _, t in vals), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "sampled": what.split(", explicit")[0] + " per core (the full-size explicit Signal graph does not fit / build on the host)",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(args, world):
    if args.workload == "gauss_chains":
        return {"workload": f"batch of {args.chains} independent linear-Gaussian chains per GPU, T={args.chain_steps}, "
                            f"canonical-form forward-backward (BASELINE configs[1])", "chains_per_gpu": args.chains,
                "T": args.chain_steps, "l2": "inputs exceed L2 (4.3 GB touched per step)", "parallelism": f"batch-shard x{world}"}
    if args.workload == "potts_grid":
        return {"workload": f"2D Potts grid {args.grid}x{args.grid}, K=16, {args.sweeps} synchronous sweeps (protocol B) per step, "
                            f"row-sharded (BASELINE configs[3])", "grid": args.grid, "K": 16, "sweeps_per_step": args.sweeps,
                "l2": "inputs exceed L2 (60 GB touched per sweep)",
                "parallelism": f"row-shard x{world}" + (", halo exchange of the cut-edge messages every sweep (transport: see comm)" if world > 1 else ""),
                "e2e_step": "per job: unary evidence pinned host->device, the sweeps, marginals device->pinned host (each rank its rows); "
                            "consecutive jobs are pipelined over three streams (cxb_grid_infer_host), messages carry over"}
    if args.workload in ("hmm64", "hmm512"):
        k = 512 if args.workload == "hmm512" else 64
        cfg = {"workload": f"{args.hmm_chains} HMMs per GPU, K={k}, M=32, T={args.hmm_steps} (BASELINE configs[2] K={k})",
               "l2": "inputs exceed L2", "parallelism": f"batch-shard x{world}",
               "e2e_result": "observations in (all T), marginals of the last min(T, 256) time steps out (the full plane is "
                             f"{args.hmm_chains * args.hmm_steps * k * 4 / 1e9:.0f} GB; fetch any window with cxb_hmm_get_marginals)"}
        if k == 512 and args.hmm_chains < 1024:
            cfg["batch_tile"] = (f"BASELINE names 1,024 chains: at K=512 their forward and marginal planes are 2 x 210 GB, so the job runs "
                                 f"in batch tiles of {args.hmm_chains} chains per GPU (SURVEY 8d: '<= 256 chains per GPU, or 128 chains/GPU on "
                                 f"8 GPUs'); one tile is timed, the rate is the job's")
        return cfg
    if args.workload in ("powerlaw", "powerlaw_engine"):
        eng = "fused CSR sweep engine" if args.workload == "powerlaw" else "generic reactive engine"
        per = f"{args.pl_sweeps} protocol-B sweeps per step" if args.workload == "powerlaw" else "one protocol-B sweep per step"
        return {"workload": f"Chung-Lu power-law graph, {args.pl_vars} variables, {2 * args.pl_vars} pairwise factors, K=8, "
                            f"{per} on the {eng} (BASELINE configs[4])", "l2": "inputs exceed L2 at full size",
                "parallelism": "replicas only", "e2e_step": "unary evidence pinned host->device, the sweeps, marginals device->pinned host"}
    if args.workload == "chains_engine":
        return {"workload": f"{args.engine_chains} Gaussian random-walk chains x T=1000 as ONE explicit graph through cxb_graph_build + "
                            f"cxb_update_marginals (the reference's single entry point; cf. gauss_chains for the structured engine)",
                "l2": "inputs exceed L2", "parallelism": "replicas only"}
    return {"workload": "1-D Gaussian random-walk chain T=1000 through cxb_graph_build + cxb_update_marginals (BASELINE configs[0])",
            "l2": "fits L2 (latency config)", "parallelism": "replicas only"}


# ---------------------------------------------------------------------------------------------------------------
def bench_gauss_chains(args, pkg, rank, world, local):
    import torch

    cap = pkg.capi
    dtype = cap.F32 if args.dtype == "f32" else cap.F64
    B, T = args.chains, args.chain_steps
    npdt = np.float32 if dtype == cap.F32 else np.float64
    rng = np.random.Generator(np.random.PCG64(1234 + rank))
    q, r = rng.uniform(0.5, 2.0, B), rng.uniform(0.5, 2.0, B)
    y_host = torch.empty((T, B), dtype=torch.float32 if dtype == cap.F32 else torch.float64).pin_memory()
    ynp = y_host.numpy()
    x = np.zeros(B)
    for t in range(T):  # fp64 master data cast to the engine dtype (SURVEY §8d)
        x = x + rng.standard_normal(B) * np.sqrt(q)
        ynp[t] = (x + rng.standard_normal(B) * np.sqrt(r)).astype(npdt)
    out_host = torch.empty((T, B, 2), dtype=y_host.dtype).pin_memory()
    ch = pkg.GaussianChainBatch(B, T, dtype=dtype, device=local)
    ch.set_noise(q, r)
    ch.set_observations(ynp)
    n_upd = ch.n_updates
    kernel_ms = []

    def step():
        ch.update_marginals()

    # device-resident timing (value)
    for _ in range(args.warmup):
        step()
    ch.sync()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = pkg.default_api().kernel_launches()
    ms = timed(ch.stream, step, args.steps, 0, world, local, min_ms=args.min_ms)
    steps_timed = timed.last_steps
    launches = pkg.default_api().kernel_launches() - launches0
    if args.dump_outputs:
        marg = ch.get_marginals().reshape(T * B, 2)
        dump_output(args, "marginals", marg[dump_rows(T * B, marg[0].nbytes)])
    # per-launch kernel duration from the library's own CUDA events (same stream)
    for _ in range(min(args.steps, 10)):
        step()
        kernel_ms.append(ch.last_kernel_ms())
    # end to end: pinned host observations -> device -> update -> marginals back to pinned host memory
    def e2e_step():
        ch.infer_host(y_host.data_ptr(), out_host.data_ptr())

    e2e_ms = timed(ch.stream, e2e_step, max(2, min(args.steps, 5)), 1, world, local, min_ms=args.min_ms)
    e2e_steps = timed.last_steps
    clocks = sampler.stop()
    esz = 4 if dtype == cap.F32 else 8
    alg_bytes = B * T * (16 * esz)  # 64 B (fp32) / 128 B (fp64) per variable: SURVEY §8d config 2
    return {"ms": ms, "updates_per_step": n_upd, "kernel_ms": statistics.mean(kernel_ms), "alg_bytes": alg_bytes,
            "e2e_ms": e2e_ms, "e2e_steps": e2e_steps, "h2d": B * T * esz, "d2h": B * T * 2 * esz, "launches": launches,
            "clocks": clocks, "dtype": args.dtype, "kernel": "k_chains_fwd_bwd", "scaling": "weak", "steps_timed": steps_timed}


def bench_potts_grid(args, pkg, rank, world, local):
    import torch
    import torch.distributed as dist

    cap = pkg.capi
    N, K, beta = args.grid, 16, 0.7
    row0, rows, has_up, has_down = pkg.row_shard(N, world, rank)
    gr = pkg.PottsGrid(rows, N, K, beta, dtype=cap.F32, device=local, has_upper=has_up, has_lower=has_down)
    rng = np.random.Generator(np.random.PCG64(1234 + rank))
    unary_host = torch.empty((rows, N, K), dtype=torch.float32).pin_memory()
    un = unary_host.numpy()
    blk = 256
    for i in range(0, rows, blk):  # Dirichlet(1) rows = normalised exponentials
        e = rng.standard_exponential((min(blk, rows - i), N, K), dtype=np.float32)
        un[i:i + blk] = e / e.sum(axis=-1, keepdims=True)
    gr.set_unary(un)
    gr.reset_messages()
    ext = torch.cuda.ExternalStream(gr.stream, device=local)
    n = gr.halo_elems
    cache = {}

    def tens(ptr):
        if ptr not in cache:
            cache[ptr] = pkg.device_tensor(ptr, n, local)
        return cache[ptr]

    halo = pkg.HaloExchanger(dist, rank, world)
    upd = [0]
    # fused exchange: the sweep kernel stores the cut-edge messages into the neighbour GPU's halo buffer over NVLink
    # (cxb_grid_p2p_*); CXB_GRID_NCCL=1 (or GPUs without peer access) keeps the separate NCCL send/recv per sweep
    fused = world > 1 and os.environ.get("CXB_GRID_NCCL", "0") != "1" and pkg.connect_row_neighbours(dist, gr, rank, world)
    args.halo_transport = "peer stores fused in the sweep kernel (NVLink P2P)" if fused else "NCCL send/recv per sweep"
    if world > 1:
        gr.sync()
        dist.barrier()

    def sweep():
        upd[0] = gr.sweep()
        if world > 1 and not fused:
            with torch.cuda.stream(ext):  # NCCL orders itself after the sweep on the library's stream
                halo.exchange(tens(gr.halo_send_ptr(0)) if has_up else None, tens(gr.halo_send_ptr(1)) if has_down else None,
                              tens(gr.halo_recv_ptr(0)) if has_up else None, tens(gr.halo_recv_ptr(1)) if has_down else None)

    sweeps = args.sweeps

    def step():  # BASELINE configs[3]: 50 synchronous sweeps
        for _ in range(sweeps):
            sweep()

    for _ in range(args.warmup):
        step()
    gr.sync()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = pkg.default_api().kernel_launches()
    ms = timed(gr.stream, step, args.steps, 0, world, local)
    launches = pkg.default_api().kernel_launches() - launches0
    if args.dump_outputs:
        marg = gr.get_marginals().reshape(rows * N, K)
        dump_output(args, "marginals", marg[dump_rows(rows * N, marg[0].nbytes)])
        del marg
    kernel_ms = []
    for _ in range(10):
        sweep()
        kernel_ms.append(gr.last_kernel_ms())
    # end to end: evidence from pinned host memory, the 50 sweeps, marginals back to pinned host memory
    marg_host = torch.empty((rows, N, K), dtype=torch.float32).pin_memory()

    if world > 1 and not fused:  # NCCL transport: the exchange is a host-driven call per sweep, no pipelined entry point
        def e2e_step():
            gr.set_unary(un)
            step()
            gr.api.grid_get_marginals(gr.h, marg_host.data_ptr())
    else:
        def e2e_step():  # cxb_grid_infer_host: this job's sweeps overlap the next job's evidence upload and the previous download
            gr.infer_host(unary_host.data_ptr(), marg_host.data_ptr(), sweeps)

    e2e_steps = max(3, min(args.steps, 10))
    e2e_step()
    gr.sync()
    barrier(world)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    gr.sync()  # every copy of every job has landed
    e2e_ms = max_over_ranks(1e3 * (time.perf_counter() - t0), world, local)
    barrier(world)
    clocks = sampler.stop()
    total_updates = sum_over_ranks(upd[0], world, local) * sweeps
    pix = rows * N
    # 64 B x [(4 m2f + unary) reads + (4 m2v + 4 m2f + marginal) writes] for interior pixels; exact count from the updates
    m2v_local = (upd[0] - pix) // 2
    alg_bytes = 64 * ((m2v_local + pix) + (2 * m2v_local + pix))
    transport = None
    if world > 1:
        transport = {"kind": "peer stores over NVLink (CUDA IPC), fused in k_potts_sweep" if fused else "NCCL send/recv per sweep",
                     "bytes_per_boundary_per_sweep": 2 * N * K * 4, "boundaries": world - 1}
    return {"ms": ms, "updates_per_step": total_updates, "kernel_ms": statistics.mean(kernel_ms), "alg_bytes": alg_bytes,
            "e2e_ms": e2e_ms, "e2e_steps": e2e_steps, "h2d": pix * K * 4, "d2h": pix * K * 4, "launches": launches,
            "clocks": clocks, "dtype": "f32", "kernel": "k_potts_sweep", "scaling": "strong", "already_global": True,
            "comm": transport, "bytes_are_per_rank": world > 1}


def bench_hmm64(args, pkg, rank, world, local):
    import torch

    cap = pkg.capi
    B, T, K, M = args.hmm_chains, args.hmm_steps, (512 if args.workload == "hmm512" else 64), 32
    rng = np.random.Generator(np.random.PCG64(1234 + rank))
    A = rng.dirichlet(np.ones(K), size=K)
    E = rng.dirichlet(np.ones(K), size=M).T * K
    obs_host = torch.empty((T, B), dtype=torch.uint8).pin_memory()
    obs_host.numpy()[:] = rng.integers(0, M, size=(T, B), dtype=np.uint8)
    hm = pkg.HmmBatch(B, T, K, M, dtype=cap.F32, device=local)
    hm.set_tables(A, E)
    hm.set_observations(obs_host.numpy())

    def step():
        hm.update_marginals()

    for _ in range(args.warmup):
        step()
    hm.sync()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = pkg.default_api().kernel_launches()
    ms = timed(hm.stream, step, args.steps, 0, world, local, min_ms=args.min_ms)
    steps_timed = timed.last_steps
    launches = pkg.default_api().kernel_launches() - launches0
    if args.dump_outputs:  # rows = time steps (all chains), fetched one at a time: the full plane does not fit the host
        dump_output(args, "marginals", np.stack([hm.get_marginals(t, t + 1)[0] for t in dump_rows(T, B * K * 4)]))
    kernel_ms = []
    for _ in range(min(args.steps, 3)):
        step()
        kernel_ms.append(hm.last_kernel_ms())
    tail = min(T, 256)
    out_host = torch.empty((tail, B, K), dtype=torch.float32).pin_memory()

    def e2e_step():
        hm.set_observations(obs_host.numpy())
        step()
        hm.api.hmm_get_marginals(hm.h, T - tail, T, out_host.data_ptr())

    e2e_steps = 2
    e2e_ms = timed(hm.stream, e2e_step, e2e_steps, 1, world, local)
    clocks = sampler.stop()
    alg_bytes = B * T * (12 * K + 2)  # SURVEY §8d config 3: forward message + marginal contract
    out = {"ms": ms, "updates_per_step": hm.n_updates, "kernel_ms": statistics.mean(kernel_ms), "alg_bytes": alg_bytes,
           "e2e_ms": e2e_ms, "e2e_steps": e2e_steps, "h2d": B * T, "d2h": tail * B * K * 4, "launches": launches,
           "clocks": clocks, "dtype": "f32", "scaling": "weak", "steps_timed": steps_timed,
           "kernel": "k_hmm64_pass (forward launch + backward launch, one warp per chain)"}
    if K >= 128:
        # tensor-core path: each fp32 product is 6 bf16 MMAs (3-piece split operands, hmm_tc.cuh), 2 passes per time step
        pieces = 2 if os.environ.get("CXB_HMM_TC_PIECES") == "2" else 3
        mmas = 3 if pieces == 2 else 6
        out["kernel"] = "k_hmm_tc_step_pair (tcgen05 + TMEM; one launch per time step, forward and backward halves; wide-N piece products, two MMA issuers)"
        out["tensor"] = {"issued_flops": 2.0 * B * K * K * mmas * 2 * T, "fp32_equivalent_flops": 2.0 * B * K * K * 2 * T,
                         "note": f"{mmas} bf16 MMAs per fp32 product ({pieces}-piece split operands)"}
    return out


def bench_powerlaw(args, pkg, rank, world, local):
    """BASELINE configs[4] on the fused CSR sweep engine (cxb_pairwise_*): replicas only."""
    import torch
    from tests import models  # graph generator only (numpy); no oracle code is executed

    cap = pkg.capi
    n = args.pl_vars
    m, K = 2 * n, 8
    rng = np.random.Generator(np.random.PCG64(1235 + rank))
    edges = np.asarray(models.chung_lu_edges_fast(n, m), dtype=np.int64)
    ttype = rng.integers(0, 16, size=m).astype(np.int32)
    tables = np.exp(rng.standard_normal((16, K, K)))
    pw = pkg.PairwiseGraph(n, edges[:, 0], edges[:, 1], ttype, tables, dtype=cap.F32, device=local)
    unary_host = torch.empty((n, K), dtype=torch.float32).pin_memory()
    e = rng.standard_exponential((n, K), dtype=np.float32)
    unary_host.numpy()[:] = e / e.sum(axis=-1, keepdims=True)
    pw.set_unary(unary_host.numpy())
    pw.reset_messages()
    upd = [0]

    sweeps = args.pl_sweeps

    def sweep():
        upd[0] = pw.sweep()

    def step():  # BASELINE configs[4]: 10 sweeps of protocol B
        for _ in range(sweeps):
            sweep()

    for _ in range(args.warmup):
        step()
    pw.sync()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = pkg.default_api().kernel_launches()
    ms = timed(pw.stream, step, args.steps, 0, world, local, min_ms=args.min_ms)
    steps_timed = timed.last_steps
    launches = pkg.default_api().kernel_launches() - launches0
    if args.dump_outputs:
        marg = pw.get_marginals()
        dump_output(args, "marginals", marg[dump_rows(n, marg[0].nbytes)])
    kernel_ms = []
    for _ in range(10):
        sweep()
        kernel_ms.append(pw.last_kernel_ms())
    marg_host = torch.empty((n, K), dtype=torch.float32).pin_memory()

    def e2e_step():
        pw.api.pairwise_set_unary(pw.h, unary_host.data_ptr())
        step()
        pw.api.pairwise_get_marginals(pw.h, marg_host.data_ptr())

    e2e_ms = timed(pw.stream, e2e_step, max(2, min(args.steps, 5)), 1, world, local, min_ms=args.min_ms)
    e2e_steps = timed.last_steps
    clocks = sampler.stop()
    return {"ms": ms, "updates_per_step": upd[0] * sweeps, "kernel_ms": statistics.mean(kernel_ms), "alg_bytes": pw.algorithmic_bytes,
            "e2e_ms": e2e_ms, "e2e_steps": e2e_steps, "h2d": n * K * 4, "d2h": n * K * 4, "launches": launches,
            "clocks": clocks, "dtype": "f32", "kernel": "k_pw_exact_staged + k_pw_team + k_pw_hub_scan (one sweep)", "scaling": "weak",
            "steps_timed": steps_timed, "scatters": 2 * m}


def bench_engine_graph(args, pkg, rank, world, local, which):
    """Generic CSR engine: chain1k (one update_marginals!) or powerlaw (protocol-B sweeps)."""
    import ctypes

    import torch

    cap = pkg.capi
    api = pkg.default_api()
    if which in ("chain1k", "chains_engine"):
        # B chains of T steps as ONE explicit graph (ids time-major: x[t][b], y[t][b], likelihood[t][b], transition[t][b]):
        # chain1k = BASELINE configs[0] (B = 1, fp64, latency); chains_engine = a batch through the same single entry point
        T = 1000
        B = 1 if which == "chain1k" else args.engine_chains
        edt = cap.F64 if which == "chain1k" else cap.F32
        rng = np.random.Generator(np.random.PCG64(1234))
        nx = T * B
        n_ids = 3 * nx + (T - 1) * B
        is_factor = np.zeros(n_ids, dtype=np.uint8)
        is_factor[2 * nx:] = 1
        ftype = np.zeros(n_ids, dtype=np.int32)
        ftype[3 * nx:] = 1
        xid = np.arange(nx, dtype=np.int64)  # x[t][b] = t * B + b
        ev = np.concatenate([np.stack([nx + xid, xid], axis=1).ravel(), np.stack([xid[:nx - B], xid[B:]], axis=1).ravel()])
        ef = np.concatenate([np.repeat(2 * nx + xid, 2), np.repeat(3 * nx + xid[:nx - B], 2)])
        store = pkg.SignalStore(api, 2, cap.FAMILY_GAUSS_CANON, edt, local)
        ev, ef = np.ascontiguousarray(ev, dtype=np.int64), np.ascontiguousarray(ef, dtype=np.int64)
        store.check(api.graph_build(store.h, n_ids, is_factor.ctypes.data_as(cap.u8p), ftype.ctypes.data_as(cap.i32p), len(ev),
                                    ev.ctypes.data_as(cap.i64p), ef.ctypes.data_as(cap.i64p)))
        one = np.array([1.0])
        store.check(api.register_rule(store.h, 0, cap.RULE_GAUSS_OBS, one.ctypes.data_as(cap.f64p), 1))
        store.check(api.register_rule(store.h, 1, cap.RULE_GAUSS_RW, one.ctypes.data_as(cap.f64p), 1))
        store.check(api.resolve_dependencies(store.h, cap.RESOLVER_DEFAULT_BP))
        obs_sig = np.ascontiguousarray(2 * nx + 2 * (2 * xid) + 1, dtype=np.int64)  # m2f(y_i, likelihood_i) = n_var + 2c + 1, c = 2i, n_var = 2 nx
        assert int(obs_sig[5 % nx]) == api.signal_id(store.h, cap.KIND_M2F, nx + 5 % nx, 2 * nx + 5 % nx)
        vals = np.zeros((nx, 2))
        vals[:, 0] = (np.cumsum(rng.standard_normal((T, B)), axis=0) + rng.standard_normal((T, B))).ravel()
        xs = np.ascontiguousarray(xid)
        stats = cap.UpdateStats()

        in_sig, in_vals, vdim = obs_sig, vals, 2
        store.check(api.set_values(store.h, nx, obs_sig.ctypes.data_as(cap.i64p), vals.ctypes.data_as(cap.f64p), 2))
        store.check(api.update_marginals(store.h, nx, xs.ctypes.data_as(cap.i64p), ctypes.byref(stats)))
        upd = B * (6 * T - 4)
        assert stats.updates == upd, stats.updates
        # the same algorithmic bytes as the structured engine (64 B fp32 per variable, SURVEY 8d config 2); the index arrays of
        # the plan kernel come on top
        alg_bytes, dtype = (0, "f64") if which == "chain1k" else (nx * 64, "f32")
        unary = vals
    else:
        from tests import models  # graph generator only (numpy); no oracle code is executed

        n = args.pl_vars
        m, K = 2 * n, 8
        rng = np.random.Generator(np.random.PCG64(1235))
        edges = np.asarray(models.chung_lu_edges_fast(n, m), dtype=np.int64)
        ttype = rng.integers(0, 16, size=m)
        tables = np.exp(rng.standard_normal((16, K, K)))
        n_ids = 2 * n + m
        is_factor = np.zeros(n_ids, dtype=np.uint8)
        is_factor[n:] = 1
        ftype = np.zeros(n_ids, dtype=np.int32)
        ftype[n:2 * n] = 16  # unary
        ftype[2 * n:] = ttype
        ev = np.concatenate([np.arange(n), edges.ravel()]).astype(np.int64)
        ef = np.concatenate([n + np.arange(n), np.repeat(2 * n + np.arange(m), 2)]).astype(np.int64)
        store = pkg.SignalStore(api, K, cap.FAMILY_CATEGORICAL, cap.F32, local)
        store.check(api.graph_build(store.h, n_ids, is_factor.ctypes.data_as(cap.u8p), ftype.ctypes.data_as(cap.i32p), len(ev),
                                    ev.ctypes.data_as(cap.i64p), ef.ctypes.data_as(cap.i64p)))
        for t in range(16):
            tb = np.ascontiguousarray(tables[t].ravel())
            store.check(api.register_rule(store.h, t, cap.RULE_CAT_TABLE, tb.ctypes.data_as(cap.f64p), tb.size))
        store.check(api.resolve_dependencies(store.h, cap.RESOLVER_DEFAULT_BP))
        # protocol B: link + initialise every pairwise m2f, evidence = unary m2v
        pair_m2f = n + 2 * (n + np.arange(2 * m)) + 1  # sid of m2f(connection c) = n_var + 2c + 1, pair connections c >= n
        lv = np.ascontiguousarray(ev[n:n + 2 * m], dtype=np.int64)
        ls = np.ascontiguousarray(pair_m2f, dtype=np.int64)
        store.check(api.link_signals(store.h, 2 * m, lv.ctypes.data_as(cap.i64p), ls.ctypes.data_as(cap.i64p)))
        init = np.full((2 * m, K), 1.0 / K)
        pm = np.ascontiguousarray(pair_m2f, dtype=np.int64)
        store.check(api.set_values(store.h, 2 * m, pm.ctypes.data_as(cap.i64p), init.ctypes.data_as(cap.f64p), K))
        unary_sig = np.ascontiguousarray(n + 2 * np.arange(n), dtype=np.int64)
        unary = rng.dirichlet(np.ones(K), size=n)
        xs = np.arange(n, dtype=np.int64)
        stats = cap.UpdateStats()

        in_sig, in_vals, vdim = unary_sig, unary, K
        store.check(api.set_values(store.h, n, unary_sig.ctypes.data_as(cap.i64p), unary.ctypes.data_as(cap.f64p), K))
        store.check(api.update_marginals(store.h, n, xs.ctypes.data_as(cap.i64p), ctypes.byref(stats)))
        upd = int(stats.updates)
        deg = np.bincount(edges.ravel(), minlength=n)
        n_prod = int(np.sum(np.where(deg + 1 > 5, deg - 1, 0)))
        alg_bytes = 32 * (int(np.sum((deg + 1) + (2 * deg + 1))) + 3 * n_prod)  # SURVEY §8d config 5
        dtype = "f32"
    # "prepare once, run many": the evidence list, the request and the marginal list are validated and uploaded once
    # (cxb_prepare_signals / cxb_prepare_request); per step the evidence is re-asserted (set_value! + notification), the request
    # runs, and - end to end - the marginals come back. `value`: evidence already on the device; `e2e`: pinned host buffers.
    tdt = torch.float32 if dtype == "f32" else torch.float64
    n_in, n_req = len(in_sig), len(xs)
    ev_list = api.prepare_signals(store.h, n_in, in_sig.ctypes.data_as(cap.i64p))
    marg_list = api.prepare_signals(store.h, n_req, np.ascontiguousarray(np.arange(n_req), dtype=np.int64).ctypes.data_as(cap.i64p))
    req = api.prepare_request(store.h, n_req, xs.ctypes.data_as(cap.i64p))
    assert ev_list >= 0 and marg_list >= 0 and req >= 0
    host_in = torch.from_numpy(np.ascontiguousarray(in_vals)).to(tdt).pin_memory()
    host_out = torch.empty((n_req, vdim), dtype=tdt).pin_memory()
    dev_in = host_in.to(f"cuda:{local}")
    torch.cuda.synchronize()

    def step():  # device-resident
        store.check(api.set_values_prepared(store.h, ev_list, ctypes.c_void_p(dev_in.data_ptr()), 1))
        store.check(api.update_marginals_prepared(store.h, req, ctypes.byref(stats)))

    def e2e_step():
        store.check(api.set_values_prepared(store.h, ev_list, ctypes.c_void_p(host_in.data_ptr()), 0))
        store.check(api.update_marginals_prepared(store.h, req, ctypes.byref(stats)))
        store.check(api.get_values_prepared(store.h, marg_list, ctypes.c_void_p(host_out.data_ptr()), 0))

    def wall(fn, steps):
        while True:
            barrier(world)
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            ms = max_over_ranks(1e3 * (time.perf_counter() - t0), world, local)
            if ms >= args.min_ms or steps >= 1 << 16:
                return ms, steps
            steps = int(max(steps * 2, steps * 1.25 * args.min_ms / max(ms, 1e-3))) + 1

    launches0 = api.kernel_launches()
    for _ in range(args.warmup):
        step()
        e2e_step()
    torch.cuda.synchronize()
    assert int(stats.updates) == upd
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = api.kernel_launches()
    ms, steps = wall(step, args.steps)
    launches = api.kernel_launches() - launches0
    if args.dump_outputs:
        store.check(api.get_values_prepared(store.h, marg_list, ctypes.c_void_p(host_out.data_ptr()), 0))
        marg = host_out.numpy()
        dump_output(args, "marginals", marg[dump_rows(n_req, marg[0].nbytes)])
    e2e_ms, e2e_steps = wall(e2e_step, max(2, min(args.steps, 5)))
    clocks = sampler.stop()
    ran = {1: "level schedule", 2: "sequential executor", 3: "memoised level schedule (replay)", 4: "closed-form plan"}.get(
        int(api.last_schedule(store.h)), "?")
    return {"ms": ms, "updates_per_step": upd, "kernel_ms": ms / steps, "alg_bytes": alg_bytes, "e2e_ms": e2e_ms, "steps_timed": steps,
            "e2e_steps": e2e_steps, "h2d": int(host_in.numel() * host_in.element_size()), "d2h": int(host_out.numel() * host_out.element_size()),
            "launches": launches, "clocks": clocks, "dtype": dtype, "answered_by": ran,
            "kernel": "cxb_set_values_prepared + cxb_update_marginals_prepared: k_write_values, k_apply_list, k_state_differs, "
                      "k_chain_plan / k_replay_resident / k_rule_* (memoised; first run: k_bfs, k_apply)", "scaling": "weak",
            "timer": "host wall clock around the ABI calls (cxb_update_marginals_prepared ends with a stream sync)"}


# ---------------------------------------------------------------------------------------------------------------
WORKLOADS = ["potts_grid", "gauss_chains", "hmm64", "hmm512", "powerlaw", "powerlaw_engine", "chain1k", "chains_engine"]
BENCH_FN = {"gauss_chains": bench_gauss_chains, "potts_grid": bench_potts_grid, "hmm64": bench_hmm64, "hmm512": bench_hmm64,
            "powerlaw": bench_powerlaw, "powerlaw_engine": lambda *a: bench_engine_graph(*a, "powerlaw"),
            "chain1k": lambda *a: bench_engine_graph(*a, "chain1k"), "chains_engine": lambda *a: bench_engine_graph(*a, "chains_engine")}


def run_workload(args, name, pkg, rank, world, local, main_record):
    """One workload -> its record (the bench line without the keys that only the top-level line carries)."""
    import copy
    import gc

    import torch

    a = copy.copy(args)
    a.workload = name
    a.min_ms = 0.0 if main_record else 1000.0  # the main record times exactly --steps; sub-records run for >= 1 s
    if name == "hmm512":  # the forward + marginal planes of 1,024 x 1e5 x 512 are 2 x 210 GB: batch tiles of <= 256 chains per GPU (SURVEY 8d)
        a.hmm_chains = min(args.hmm_chains, max(1, min(256, 1024 // world)))
    elif name == "hmm64":
        a.hmm_chains = min(args.hmm_chains, max(1, 1024 // world)) if world > 1 else args.hmm_chains
    if not main_record:
        a.dump_outputs = None  # only the main record's timed path is dumped
        a.steps, a.warmup = min(args.steps, 3), 3
        if name == "powerlaw_engine":
            a.pl_vars = min(args.pl_vars, 1000000)  # the explicit Signal graph of 10M variables takes minutes to build on the host
    r = BENCH_FN[name](a, pkg, rank, world, local)
    peak, peak_src, _ = measured_peaks()
    steps = r.get("steps_timed", a.steps)
    ms_per_step = r["ms"] / steps
    total_updates = r["updates_per_step"] if r.get("already_global") else r["updates_per_step"] * world
    value = total_updates / (ms_per_step * 1e-3)
    e2e_value = total_updates / (r["e2e_ms"] / r["e2e_steps"] * 1e-3)
    achieved = r["alg_bytes"] / (r["kernel_ms"] * 1e-3) / 1e9 if r["alg_bytes"] else None
    rec = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": a.warmup,
           "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": r["scaling"], "vs_baseline": None,
           "dtype": r["dtype"], "data": "synthetic", "config": workload_config(a, world),
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(sum_over_ranks(r["h2d"], world, local)),
                   "d2h_bytes_per_step": int(sum_over_ranks(r["d2h"], world, local)), "steps": r["e2e_steps"],
                   "ms_per_step": r["e2e_ms"] / r["e2e_steps"]},
           "gpu_launches": int(r["launches"]), "clocks": r["clocks"],
           "roofline": {"bound": "hbm", "kernel": r["kernel"], "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": (achieved / peak) if achieved else None, "traffic": None, "peak_source": peak_src,
                        "kernel_ms": r["kernel_ms"], "algorithmic_bytes_per_launch": r["alg_bytes"]}}
    for k in ("timer", "comm", "answered_by"):
        if r.get(k) is not None:
            rec[k] = r[k]
    if "tensor" in r:  # K = 512 HMM: tensor-pipe utilisation beside the HBM figure (north star: "or tensor-pipe utilisation against peak")
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
        tpeak = float(peaks.get("bf16_tflops_sustained", 1410.1))
        tf = r["tensor"]["issued_flops"] / (r["kernel_ms"] * 1e-3) / 1e12
        rec["roofline_tensor"] = {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak,
                                  "fp32_equivalent_tflops": r["tensor"]["fp32_equivalent_flops"] / (r["kernel_ms"] * 1e-3) / 1e12,
                                  "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16 8192^3, dense)",
                                  "note": r["tensor"]["note"]}
    if name == "gauss_chains" and achieved:
        # profiles/micro/stream_mix.cu (profiles/r02_stream_mix.log): a plain grid-stride kernel that reads 1 and writes 4 planes of
        # 8-byte elements - the chain kernel's 12 B : 52 B mix - streams at 5.57 TB/s on a B200 (1 : 6: 5.72, 2 : 3: 5.92), the
        # 1 : 1 copy that defines `peak` at 5.8 - 6.5: write-heavy streams do not reach the copy bandwidth.
        rec["roofline"]["access_pattern_ceiling"] = {
            "model": "streaming kernel with the same read : write mix (1 : 4 planes of 8-byte elements), measured",
            "ceiling_gbs": 5574.7, "frac_of_ceiling": achieved / 5574.7,
            "source": "profiles/r02_stream_mix.log (profiles/micro/stream_mix.cu)"}
    if name == "powerlaw" and r.get("scatters"):
        # What the memory system gives to THIS access pattern (profiles/micro/scatter_bw.cu on a B200, profiles/r02_scatter_bw.log):
        # random 32-byte sector scatters run at 35.1 G/s whatever else is going on (1.14 ms for the 40 M messages of a sweep),
        # streams at 6.4 TB/s, and the two ADD (a kernel that streams 64 B and scatters 32 B per slot takes the sum of both
        # times). The copy bandwidth above is therefore not reachable by a sweep that scatters one message per directed edge.
        stream_gbs, scatter_gps = 6404.0, 35.1
        stream_bytes = r["alg_bytes"] - 32 * r["scatters"] + 5 * r["scatters"]  # + the opp / tsel index streams
        floor_ms = stream_bytes / (stream_gbs * 1e6) + r["scatters"] / (scatter_gps * 1e6)
        rec["roofline"]["access_pattern_ceiling"] = {
            "model": "streamed bytes / 6404 GB/s + scattered 32-byte messages / 35.1 G/s (measured, additive)",
            "floor_ms_per_sweep": floor_ms, "frac_of_ceiling": floor_ms / r["kernel_ms"],
            "source": "profiles/r02_scatter_bw.log (profiles/micro/scatter_bw.cu)"}
    traffic_file = ROOT / "profiles" / f"traffic_{name}.json"
    if traffic_file.exists():
        try:
            tj = json.loads(traffic_file.read_text())
            rec["roofline"]["traffic"] = tj.get("dram_bytes_per_launch")
            if rec["roofline"]["traffic"] and tj.get("algorithmic_bytes_per_launch") and r["alg_bytes"]:
                # the capture was taken on the full single-GPU launch: scale to this launch (a row shard moves its share)
                rec["roofline"]["traffic"] = rec["roofline"]["traffic"] * r["alg_bytes"] / tj["algorithmic_bytes_per_launch"]
            if "dram_bytes_per_chain_step" in tj:  # HMM workloads: the ncu capture ran fewer time steps
                rec["roofline"]["traffic"] = tj["dram_bytes_per_chain_step"] * a.hmm_chains * a.hmm_steps
        except Exception:
            pass
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, sample = cpu_baseline_workload(name, 12.0 if main_record else 5.0)
        rec["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                               "host_cores_available": os.cpu_count()}
    del r
    gc.collect()
    torch.cuda.synchronize()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="potts_grid", choices=WORKLOADS)
    ap.add_argument("--others", default=None, help="comma-separated sub-records to attach (default: every other config when the "
                                                   "default workload runs; 'none' to skip)")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--chains", type=int, default=65536)
    ap.add_argument("--chain-steps", type=int, default=1024)
    ap.add_argument("--grid", type=int, default=8192)
    ap.add_argument("--sweeps", type=int, default=50)
    ap.add_argument("--hmm-chains", type=int, default=1024)
    ap.add_argument("--hmm-steps", type=int, default=100000)
    ap.add_argument("--pl-vars", type=int, default=10000000)
    ap.add_argument("--pl-sweeps", type=int, default=10)
    ap.add_argument("--engine-chains", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the main record, write the marginals its last step computed as "
                         "DIR/<workload>_marginals.npy (a fixed, seeded sample of rows when larger than 60 MiB); one GPU only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    pkg = entry.load_package()
    rank, world, local = dist_setup(args.gpus)
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs runs on one GPU (each rank holds only its shard of the outputs)")
    line = run_workload(args, args.workload, pkg, rank, world, local, main_record=True)
    if NUMA_NOTE:
        line["host_binding"] = dict(NUMA_NOTE)
    if args.others is None:
        others = [w for w in WORKLOADS if w != "potts_grid"] if args.workload == "potts_grid" else []
        if world > 1:  # the batch-sharded configs only; the single-GPU ones are on the N = 1 line
            others = [w for w in others if w in ("gauss_chains", "hmm64", "hmm512")]
    else:
        others = [w for w in args.others.split(",") if w and w != "none"]
    if others:
        line["others"] = {}
        for name in others:
            try:
                line["others"][name] = run_workload(args, name, pkg, rank, world, local, main_record=False)
            except Exception as e:  # noqa: BLE001 - a failing sub-record must not take the main record down; it is reported
                line["others"][name] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
