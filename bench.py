#!/usr/bin/env python
"""bench.py -- Bellman cell-updates/s of the MDP value-iteration hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                  [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...        (N > 1: one rank per GPU, NCCL)

K is the number of timed steps of the headline and of e2e (the syn16k and
QV-tree sections keep their own fixed counts, so that their checksums and
medians stay comparable between runs).

--dump-outputs DIR writes, after the timed steps, what they computed in their
last step (inputs are seeded, so two builds can be compared file for file):
mdp_cost / mdp_action (the whole grid, gathered to rank 0, at the cells listed
in mdp_sample_index), mdp_residual, e2e_cost / e2e_action (rank 0's rows as
the host received them in the last step of the e2e run that downloads J, same
cells), qv_actions / qv_values (rank 0's queries of the last timed QV batch).
With --impl reference, each step is then a whole main-arm step (100 sweeps)
instead of a timing-sized sample, and mdp_sweeps holds the sweep count.

Workload (BASELINE.json configs[2], SURVEY.md section 8d): synthetic 4096 x
4096 grid per GPU, i.i.d. 20 % occupied (numpy PCG64 seed 12345), goal at the
centre forced free, 9 actions, gamma = 0.95f.  N > 1 stacks N such tiles
vertically (rows = 4096*N, weak scaling) and row-shards them, ghost rows over
NCCL every 2 sweeps, MAX all-reduce of the residual every 100.
A "step" is one convergence-check period of the reference
(src/mdp/path_planning_2d.cu:226-251): 100 Jacobi sweeps of the whole grid +
the inf-norm residual.  value = cells * 100 * K / t (device time, max over
ranks).  e2e = the same work through the public API with HOST buffers: map
upload, 100 sweeps, residual, download of J and the action grid.

--impl reference: the reference has no CPU solver (SURVEY.md section 0); the
arm times the oracle port of its kernel arithmetic (oracle/mdp_oracle.c,
OpenMP over all host cores) on a bounded sample of the same grid.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

TILE = 4096
SWEEPS_PER_STEP = 100
ALGO_BYTES_PER_CELL_UPDATE = 10   # SURVEY.md section 8d
DUMP_CELLS = 1 << 20              # --dump-outputs: cells sampled per grid (~24 MB written)
METRIC = "bellman_cell_updates_per_sec"
UNIT = "cell-updates/s"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,"
         "clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                 "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no_samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx),
                "reasons": sorted(reasons), "samples": len(sm)}


def make_grid(n_tiles):
    import cases
    h, w = TILE * n_tiles, TILE
    grid, goal = cases.synthetic_map(h, w, 0.20, seed=12345,
                                     goal=(w // 2, TILE // 2))
    return grid, goal


def dump_sample(cells):
    """The cells --dump-outputs keeps: a fixed, seeded sample, sorted."""
    return np.sort(np.random.default_rng(0).choice(cells, min(cells, DUMP_CELLS),
                                                   replace=False))


def write_dump(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# --------------------------------------------------------------------------
def host_cores():
    return len(os.sched_getaffinity(0))


def cpu_port_throughput(grid, goal, gamma, budget_s=12.0, sample=2048):
    """Oracle port on the top-left sample x sample crop: OpenMP on all host
    cores (thread count set explicitly and read back), plus the 1-thread
    figure on a smaller sample."""
    import oracle_py
    crop = np.ascontiguousarray(grid[:sample, :sample])
    g = goal if (goal[0] < sample and goal[1] < sample) else None
    if g is None or crop[g[1], g[0]]:
        free = np.argwhere(crop == 0)[0]
        g = (int(free[1]), int(free[0]))
    threads = oracle_py.set_threads(host_cores())
    ora = oracle_py.OracleMdp(crop, g, gamma)
    ora.sweeps(2)                                   # warm-up + calibration
    t0 = time.perf_counter()
    ora.sweeps(2)
    per = (time.perf_counter() - t0) / 2
    n = max(2, min(200, int(budget_s / max(per, 1e-6))))
    t0 = time.perf_counter()
    ora.sweeps(n)
    dt = time.perf_counter() - t0
    oracle_py.set_threads(1)
    t0 = time.perf_counter()
    ora.sweeps(2)
    one = crop.size * 2 / (time.perf_counter() - t0)
    oracle_py.set_threads(threads)
    return {"value": crop.size * n / dt, "unit": UNIT, "cores": threads,
            "kind": "port", "value_1_thread": one,
            "sample": f"{n} sweeps of the {sample}x{sample} top-left crop of the "
                      f"workload grid, oracle/mdp_oracle.c with OpenMP on {threads} threads "
                      f"(1-thread figure: 2 sweeps of the same crop)"}


def run_reference_arm(args):
    """The reference's CPU side of the path: it has no CPU solver (SURVEY.md
    section 0), so this is the oracle port of its kernel arithmetic, OpenMP
    over ALL host cores of the box (set explicitly: torchrun exports
    OMP_NUM_THREADS=1), on the SAME grid and goal as the main arm's per-GPU
    tile.  A step is a bounded sample of the main arm's step: S <= 100 sweeps
    of the whole 4096 x 4096 grid, S sized so that the run ends in ~2 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import cases
    import oracle_py
    grid, goal = make_grid(1)
    threads = oracle_py.set_threads(host_cores())
    ora = oracle_py.OracleMdp(grid, goal, cases.GAMMA)
    ora.sweeps(1)
    t0 = time.perf_counter()
    ora.sweeps(1)
    per = time.perf_counter() - t0
    total_steps = max(1, args.steps + args.warmup)
    sweeps_per_step = max(1, min(SWEEPS_PER_STEP, int(100.0 / total_steps / max(per, 1e-6))))
    if args.dump_outputs:
        # the dumped solution must not depend on a timing: whole main-arm steps
        sweeps_per_step = SWEEPS_PER_STEP
    for _ in range(args.warmup):
        ora.sweeps(sweeps_per_step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ora.sweeps(sweeps_per_step)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        sample = dump_sample(grid.size)
        write_dump(args.dump_outputs, {
            "mdp_sample_index": sample.astype(np.float64),
            "mdp_cost": ora.cost.reshape(-1)[sample].astype(np.float32),
            "mdp_action": ora.act.reshape(-1)[sample].astype(np.float32),
            "mdp_sweeps": np.array([ora.n], np.float64)})
    value = grid.size * sweeps_per_step * args.steps / dt
    sample_txt = (f"each step = {sweeps_per_step} of the 100 sweeps of a main-arm step, on the "
                  f"whole {TILE}x{TILE} per-GPU grid with the main arm's goal {goal}; "
                  f"OpenMP threads used: {threads} of {host_cores()} host cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"syn4k x{args.gpus}: {TILE}x{TILE} per GPU, i.i.d. 20% "
                               f"occupied (PCG64 seed 12345), goal {goal}, 9 actions, "
                               "gamma 0.95f, J0 = 0; " + sample_txt,
                   "note": "the reference has no CPU value-iteration path; this is "
                           "the oracle port of its CUDA kernel arithmetic; the metric is "
                           "per cell-update, so the per-GPU tile stands for the N-tile grid"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads,
                         "kind": "port", "sample": sample_txt},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    args.emit(json.dumps(line))


# --------------------------------------------------------------------------
def reference_cuda_on_this_gpu(grid, goal, gamma):
    """The reference's own kernels (oracle/_ref) on the same B200, if built."""
    so = os.path.join(ROOT, "oracle", "_ref", "libpp2d_ref_mdp.so")
    if not os.path.exists(so):
        return None
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import ctypes
        import make_golden
        lib = make_golden.ref_lib()
        ms = ctypes.c_float()
        h, w = grid.shape
        lib.ref_mdp_time_sweeps(h, w, grid.ctypes.data, goal[0], goal[1], gamma,
                                20, 4, ctypes.byref(ms))
        return {"value": h * w * 20 / (ms.value * 1e-3), "unit": UNIT,
                "what": "unmodified reference kernels (oracle/_ref, sm_100a, "
                        "--use_fast_math), 20 sweeps, same grid, same GPU"}
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


def syn16k_section(rank, world, barrier, steps=5):
    """BASELINE.json configs[3]: ONE synthetic 16384 x 16384 grid, row-sharded
    over the N GPUs of the run (strong scaling: 16384/N rows each; N = 1 keeps
    the whole grid on one GPU).  Same step as the headline: 100 sweeps + the
    residual, ghost rows through the fused kernel's peer stores."""
    import torch
    import torch.distributed as dist
    import cases
    from path_planning_2d_b200.distributed import ShardedValueIteration
    n = 16384
    grid, goal = cases.synthetic_map(n, n, 0.20, seed=12345, goal=(n // 2, 2048))
    vi = ShardedValueIteration(grid, goal, cases.GAMMA, rank=rank, world_size=world)

    def step():
        vi.sweeps(SWEEPS_PER_STEP - 2, want_action=False)
        vi.sweeps(2, want_action=True)
        r = vi.shard.residual_tensor()
        if world > 1:
            dist.all_reduce(r, op=dist.ReduceOp.MAX)
        return r

    for _ in range(3):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    rows = vi.rows[1] - vi.rows[0]
    # Evidence that the shards computed what one GPU computes (BASELINE.md
    # config 4): a partition-invariant checksum of J and the action grid after
    # the (3 + steps) x 100 sweeps every run of this section performs; it must
    # print the same number for every N.  download() also fails the section if a
    # peer-to-peer hand-shake timed out anywhere in the loop.
    t0 = time.perf_counter()
    checksum = vi.checksum()
    checksum_s = time.perf_counter() - t0
    sweeps_done = vi.n_sweeps
    vi.close()
    return {"cell_updates_per_sec": n * n * SWEEPS_PER_STEP * steps / (ms * 1e-3),
            "solution_checksum": f"{checksum:016x}", "checksum_after_sweeps": sweeps_done,
            "checksum_what": "sum over rows of crc32(J row) * (2r+1) + crc32(action row) * "
                             "(2r+2) * 0x9E3779B1 mod 2^64 (distributed.grid_checksum); "
                             "identical for every --gpus N iff the row shards are "
                             "bit-identical to the single-GPU solve",
            "checksum_seconds": checksum_s,
            "ms_per_step": ms / steps, "steps": steps, "scaling": "strong",
            "workload": f"syn16k: 16384x16384 grid, i.i.d. 20% occupied (PCG64 seed 12345), "
                        f"goal {goal}, row-sharded over {world} GPU(s), {rows} rows per GPU",
            "hbm_gbs_algorithmic_per_gpu": n * n * SWEEPS_PER_STEP * steps / (ms * 1e-3)
            * ALGO_BYTES_PER_CELL_UPDATE / 1e9 / world}


def qv_tree_section(rank, world, with_cpu, dump=None):
    """BASELINE.json configs[4]: batched QV-Tree Search, 1250 queries per GPU
    (10 000 on 8 GPUs), sharded independently, no collective on the data path.
    dump: dict that receives this rank's actions and values of the last batch."""
    import torch
    import torch.distributed as dist
    import cases
    import pomdp_fixtures as pf
    from path_planning_2d_b200 import PomdpPathPlanning2d
    per_gpu = 1250
    grid = cases.load_bundled("sparse_map_100x40")
    goal = (95, 34)
    beliefs = pf.gaussian_beliefs(grid, per_gpu * world, sigma=2.0, seed=0)
    mine = beliefs[rank * per_gpu:(rank + 1) * per_gpu]
    with PomdpPathPlanning2d(grid, goal, cases.GAMMA) as p:
        # offline part of PomdpPathPlanning2d::initialize (untimed, as in the
        # reference where it runs once at start-up): FIB upper-bound and PBVI
        # lower-bound alpha vectors from the GPU solvers, replicated per rank
        free = (grid.reshape(-1) == 0).astype(np.float32)
        b0 = free / free.sum(dtype=np.float32)
        t0 = time.perf_counter()
        fib, fa, fib_sweeps = p.fastInformedBound()
        _, pbvi, pa = p.pointBasedValueIteration(b0, 500, rand_seed=1)
        offline_s = time.perf_counter() - t0
        p.set_alphas(fib, pbvi, fa, pa)
        p.plan_batch(mine[:64])
        p.plan_batch(mine)                      # warm-up at full size
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        # three timed batches, the median counts (a batch is ~50 ms of host
        # threads and device in lock-step: one descheduled thread shows)
        times = []
        for _ in range(3):
            w0 = p.work_counters()
            t0 = time.perf_counter()
            acts, vals, stats = p.plan_batch(mine, with_stats=True)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
            w1 = p.work_counters()
        dt = torch.tensor([sorted(times)[1]], dtype=torch.float64, device="cuda")
        p_live = p.live_cells()
    if dump is not None:
        dump["qv_actions"] = np.asarray(acts, np.float32)
        dump["qv_values"] = np.asarray(vals, np.float32)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt.item())
    out = {"plans_per_sec": per_gpu * world / dt, "queries": per_gpu * world,
           "seconds": dt, "seconds_of_3_batches": times,
           "v_nodes_per_plan": float(stats[:, 0].mean()),
           "offline_solve_seconds": offline_s,
           "config": "sparse_map_100x40, goal (95,34), Gaussian start beliefs "
                     "(sigma 2 cells), 9 FIB + 500 PBVI alpha vectors from the GPU "
                     "offline solvers (untimed; FIB bit-identical to the reference's, PBVI "
                     "per the contract of DESIGN.md 7a, tests/test_pbvi_gpu.py), depth cap "
                     "50, 15 expansions, 50 samples "
                     "per Q node; host beliefs in, actions out; queries sharded per "
                     "GPU, no data-path collective",
           "parity": "actions, bounds and tree shapes bit-identical to the oracle and to "
                     "the reference's own SearchTree (tests/test_pomdp_gpu.py, "
                     "tests/test_tree_pin_gpu.py)"}
    # FP32 roofline of the batch (BASELINE.md config 5 asks for plans/s AND FP32
    # GFLOP/s).  The dominant kernel, pomdp_values_kernel, evaluates per V node
    # the 9 FIB + 9 reward + 500 PBVI inner products of the reference as
    # separately rounded multiplies and adds (no FMA: the reference's host code
    # is x86-64 without contraction), i.e. 2 floating-point INSTRUCTIONS per
    # multiply-add; the bound is the FP32 instruction issue rate, 128 lanes x
    # 148 SMs x SM clock (an FMUL or an FADD is one flop each).  Algorithmic
    # flops = V nodes x HW cells x (9 + n_pbvi) columns x 2; the kernel executes
    # fewer: cells no probability mass can enter are skipped exactly, and every
    # tile of 128 beliefs walks only the cells on which one of them is non-zero
    # (also exact) -- `executed` counts the belief x cell products really done
    # (pp2d_pomdp_work_counters), this rank's.
    hw = grid.size
    vnodes = float(stats[:, 0].sum()) * world
    ncols = 9 + pbvi.shape[0]
    live = int(p_live)
    sm_hz = 1.965e9
    try:
        sm_hz = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"]) * 1e6
    except Exception:
        pass
    peak = 128 * 148 * sm_hz * world / 1e12
    algo = vnodes * hw * ncols * 2 / dt / 1e12
    out["roofline"] = {
        "bound": "fp32_issue", "unit": "TFLOP/s (separately rounded FMUL + FADD)",
        "achieved": algo, "peak": peak, "frac": algo / peak,
        "executed": float(w1[2] - w0[2]) * world * ncols * 2 / dt / 1e12,
        "frac_executed": float(w1[2] - w0[2]) * world * ncols * 2 / dt / 1e12 / peak,
        "note": "achieved = the reference's dense count (every V node x every cell x every "
                "alpha vector); it can exceed the peak because most of those multiply-adds are "
                "provably +-0 and are skipped bit-exactly (cells no mass can enter; per tile of "
                "64 beliefs the cells where all of them are zero) -- executed is what the GPU "
                "really did, over the whole batch time, like roofline.traffic for the sweeps",
        "live_cells": live, "cells": hw,
        "cells_walked_per_belief": float(w1[2] - w0[2]) / max(1, w1[0] - w0[0]),
        "peak_what": "128 FP32 lanes x 148 SMs x SM clock x GPUs, one flop per instruction "
                     "(tools/ubench/fma_pipes.cu measures 109-119 of the 128 lanes/clk/SM "
                     "for scalar FP32 streams, profiles/r01_ubench_fma_pipes.txt)",
        "what": "bounds of all V nodes of the batch over the whole batch time (host tree "
                "logic, sampling, Bayes updates included in the time)"}
    if with_cpu and rank == 0:
        import concurrent.futures
        import pomdp_oracle_py as po
        m = po.Model(grid, goal)
        po.lib()                                 # load before the threads start

        def one(i):
            t = po.Tree(m, cases.GAMMA, fib, pbvi, pf.uniforms(), mine[i], fa, pa)
            a, r, st, rc = t.plan(50, 15)
            t.close()
            return a == acts[i] and np.float32(r) == vals[i]

        t0 = time.perf_counter()
        same1 = all(one(i) for i in range(4))
        one_thread = 4 / (time.perf_counter() - t0)
        # the trees of different queries are independent: one oracle tree per
        # host thread (the C oracle runs outside the GIL)
        cores = host_cores()
        k = 2 * cores
        t0 = time.perf_counter()
        with concurrent.futures.ThreadPoolExecutor(cores) as ex:
            same = all(ex.map(one, range(4, 4 + k)))
        out["cpu_baseline"] = {"value": k / (time.perf_counter() - t0), "unit": "plans/s",
                               "cores": cores, "kind": "port", "value_1_thread": one_thread,
                               "sample": f"queries 4..{4 + k - 1}, one oracle/pomdp_oracle.c tree "
                                         f"per thread on {cores} threads; 1-thread figure: "
                                         "queries 0..3",
                               "same_actions_and_values_as_gpu": bool(same and same1)}
        if not (same and same1):
            raise RuntimeError("QV-tree batch disagrees with the CPU oracle")
    return out


def run_main_arm(args):
    import torch
    import torch.distributed as dist
    import cases
    from path_planning_2d_b200 import MdpPathPlanning2d, _lib
    from path_planning_2d_b200.distributed import ShardedValueIteration

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.load()
    gamma = cases.GAMMA
    grid, goal = make_grid(world)
    H, W = grid.shape
    cells = H * W

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    vi = ShardedValueIteration(grid, goal, gamma, rank=rank, world_size=world)
    rows = vi.rows[1] - vi.rows[0]

    def step(ev=None):
        # 98 value-only sweeps = 49 launches of the fused 2-sweep kernel
        if ev is not None:
            ev[0].record()
        vi.sweeps(SWEEPS_PER_STEP - 2, want_action=False)
        if ev is not None:
            ev[1].record()
        vi.sweeps(2, want_action=True)
        r = vi.shard.residual_tensor()
        if world > 1:
            dist.all_reduce(r, op=dist.ReduceOp.MAX)
        return r

    for _ in range(max(args.warmup, 3)):
        r_first = step().clone()     # (also loads torch's copy kernel before the timed region)
    barrier()
    # the timed steps start from J = 0 again (same map): they do the work of
    # the reference's first check periods, not sweeps of a converged grid
    vi.reset(grid, goal)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.pp2d_kernel_launches()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(args.steps)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for i in range(args.steps):
        r = step(evs[i])
        if i == 0:
            r_first.copy_(r)
    end.record()
    barrier()
    launches = lib.pp2d_kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if vi.p2p and vi.shard.p2p_timed_out():
        raise SystemExit("peer-to-peer ghost-row hand-shake timed out inside the timed "
                         "region: no valid number")
    ms = start.elapsed_time(end)
    fused_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([ms, fused_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, fused_ms = t.tolist()
    value = cells * SWEEPS_PER_STEP * args.steps / (ms * 1e-3)
    residual = float(r.item())
    residual_first = float(r_first.item())

    # roofline of the dominant kernel (fused 2-sweep kernel), per launch
    n_fused = (SWEEPS_PER_STEP - 2) // 2 * args.steps
    launch_s = fused_ms * 1e-3 / n_fused
    algo_bytes = rows * W * 2 * ALGO_BYTES_PER_CELL_UPDATE
    peak, which = peaks()
    achieved = algo_bytes / launch_s / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None,
                "kernel": "mdp_sweep_kernel<T=2> (2 fused sweeps per launch)",
                "launch_ms": launch_s * 1e3, "peak_source": which,
                "algorithmic_bytes_per_launch": algo_bytes}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            roofline["traffic"] = json.load(open(prof)).get("dram_bytes_per_launch")
        except Exception:
            pass

    # what the timed steps computed: the whole J and action grid after the last
    # step, sampled at fixed cells (the same cells for every run of a grid size)
    dump = None
    if args.dump_outputs:
        dump = {}
        cost, action = vi.gather()
        sample = dump_sample(cells)
        if rank == 0:
            dump["mdp_sample_index"] = sample.astype(np.float64)
            dump["mdp_cost"] = cost.reshape(-1)[sample].astype(np.float32)
            dump["mdp_action"] = action.reshape(-1)[sample].astype(np.float32)
            dump["mdp_residual"] = np.array([residual], np.float32)

    # e2e: public API, host buffers, copies inside the timed region
    p2p_used = vi.p2p
    vi.close()
    del vi
    from path_planning_2d_b200.distributed import partition_rows
    bounds = partition_rows(H, world)[rank]
    # two page-locked map buffers (same content: every step solves the same
    # problem, so the results can be verified): while step i is being solved,
    # the map of step i+1 already travels to the device (pp2d_mdp_stage_map)
    pinned_maps = [torch.from_numpy(grid).pin_memory() for _ in range(2)]
    maps_np = [t.numpy() for t in pinned_maps]
    n_own = (bounds[1] - bounds[0]) * W
    # two sets of page-locked result buffers: the download of step i overlaps
    # the re-solve of step i+1 (pp2d_mdp_download_begin / _wait), as a planner
    # that re-plans on every new map would run it
    cost_host = [torch.empty(n_own, dtype=torch.float32).pin_memory() for _ in range(2)]
    act_host = [torch.empty(n_own, dtype=torch.uint8).pin_memory() for _ in range(2)]
    v = ShardedValueIteration(maps_np[0], goal, gamma, rank=rank, world_size=world)
    mdp_handle = v.shard.mdp
    stage = not args.no_stage

    trace = [] if os.environ.get("PP2D_E2E_TRACE") else None   # host time per phase (debugging aid)

    def e2e_step(i, with_cost=True):
        t = [time.perf_counter()]
        v.reset(maps_np[i % 2], goal)  # map rows on the device (staged by step i-1, or H2D here), codes, J = 0
        t.append(time.perf_counter())
        v.sweeps(SWEEPS_PER_STEP)
        if stage:
            v.stage_map(maps_np[(i + 1) % 2])    # H2D of the next step's map, under this solve
        t.append(time.perf_counter())
        res = v.residual()             # D2H scalar (+ all-reduce)
        t.append(time.perf_counter())
        if i > 0:
            mdp_handle.download_wait()           # step i-1's J and actions are on the host
        t.append(time.perf_counter())
        mdp_handle.download_begin(cost_host[i % 2].data_ptr() if with_cost else None,
                                  act_host[i % 2].data_ptr())
        t.append(time.perf_counter())
        if trace is not None and with_cost:
            trace.append([round((b - a) * 1e3, 3) for a, b in zip(t, t[1:])])
        return res

    e2e_step(0)
    mdp_handle.download_wait()
    first = (cost_host[0].clone(), act_host[0].clone())
    e2e_steps = args.steps   # (the drain of the last download is inside the timed region)

    def e2e_run(with_cost):
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            e2e_step(i, with_cost)
        mdp_handle.download_wait()
        barrier()
        sec = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        # every step solved the same problem: all downloads must hold the same bits
        for k in range(min(2, e2e_steps)):
            if not ((not with_cost or
                     torch.equal(cost_host[k].view(torch.int32), first[0].view(torch.int32)))
                    and torch.equal(act_host[k], first[1])):
                raise SystemExit("e2e: overlapped downloads disagree")
        return cells * SWEEPS_PER_STEP * e2e_steps / float(sec.item())

    e2e_val = e2e_run(True)
    if dump is not None and rank == 0:
        # this rank's rows as the host received them in the last step
        own = sample[sample < n_own]
        last = (e2e_steps - 1) % 2
        dump["e2e_cost"] = cost_host[last].numpy()[own].astype(np.float32)
        dump["e2e_action"] = act_host[last].numpy()[own].astype(np.float32)
    if trace is not None:
        print(f"rank {rank} e2e ms per phase [reset, enqueue sweeps, residual, download_wait, "
              f"download_begin]: {trace[1:]}", file=sys.stderr)
    # the same pipeline for a planner that only needs the policy (beliefCallback
    # reads optimal_action only; the reference's host copy of J feeds RViz
    # markers, src/mdp/path_planning_2d.cu:380-393): pp2d_mdp_download_begin(cost = NULL)
    for t_ in act_host:
        t_.zero_()
    e2e_policy_val = e2e_run(False)
    occ_rows = min(H, bounds[1] + 3) - max(0, bounds[0] - 3)
    e2e = {"value": e2e_val, "unit": UNIT,
           "h2d_bytes_per_step": occ_rows * W,
           "d2h_bytes_per_step": (bounds[1] - bounds[0]) * W * 5 + 4,
           "steps": e2e_steps,
           "policy_only": {"value": e2e_policy_val, "unit": UNIT,
                           "d2h_bytes_per_step": (bounds[1] - bounds[0]) * W + 4,
                           "what": "the same pipeline with pp2d_mdp_download_begin(cost = NULL): "
                                   "only the action grid travels back (all a planner's "
                                   "beliefCallback reads); NOT the headline e2e"},
           "map_upload": "staged (pp2d_mdp_stage_map, under the previous solve)" if stage
                         else "inside pp2d_mdp_reset",
           "what": "pp2d_mdp_reset(map from pinned host) + 100 sweeps + residual "
                   "+ download of J f32 and action u8 to pinned host per step, on a handle "
                   "created once; software-pipelined like a planner that re-plans on a stream "
                   "of maps: the map of step i+1 is uploaded while step i is solved "
                   "(pp2d_mdp_stage_map, own upload stream) and the download of step i "
                   "(pp2d_mdp_download_begin/_wait, device snapshot + copy stream) overlaps "
                   "the solve of step i+1; every step's copies happen inside the timed region, "
                   "the last download is waited for in it; all downloads verified equal"}
    v.close()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {
                "workload": f"syn4k x{world}: {H}x{W} grid ({TILE}x{TILE} per GPU), "
                            "i.i.d. 20% occupied (PCG64 seed 12345), goal "
                            f"{goal}, 9 actions, gamma 0.95f, J0 = 0",
                "step": "100 Jacobi sweeps + inf-norm residual (one reference "
                        "check period)",
                "parallelism": f"rows{world}" if world > 1 else "single",
                "l2": "working set (2 x J + codes, ~164 MiB per GPU) exceeds the "
                      "126 MB L2; no explicit flush",
                "hbm_gbs_algorithmic": value * ALGO_BYTES_PER_CELL_UPDATE / 1e9 / world,
            },
            "roofline": roofline,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "residual_after_first_timed_step": residual_first,
            "residual_after_timed_steps": residual,
            "p2p_ghost_rows": bool(p2p_used),
        }
        ref_cuda = reference_cuda_on_this_gpu(grid[:TILE], goal, gamma) \
            if world == 1 and not args.no_ref_cuda else None
        if ref_cuda:
            line["reference_cuda_same_gpu"] = ref_cuda
        if world == 1 and not args.no_cpu:
            try:
                line["cpu_baseline"] = cpu_port_throughput(grid, goal, gamma)
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"error": repr(e)}
    # the side sections must never cost the headline line
    syn16k = qv = None
    try:
        syn16k = None if args.no_syn16k else syn16k_section(rank, world, barrier)
    except Exception as e:  # pragma: no cover
        syn16k = {"error": repr(e)}
    if rank == 0 and syn16k:
        line["syn16k"] = syn16k
    try:
        qv = None if args.no_qv else qv_tree_section(rank, world, world == 1 and not args.no_cpu,
                                                       dump)
    except Exception as e:  # pragma: no cover
        qv = {"error": repr(e)}
    if rank == 0:
        if qv:
            line["qv_tree"] = qv
        if dump is not None:
            write_dump(args.dump_outputs, dump)
        args.emit(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


class StdoutGuard:
    """Only the final JSON line may reach stdout: anything libraries print to
    fd 1 meanwhile (NCCL's version banner, the reference's printf) goes to
    stderr."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.saved, (text + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    # Several ranks share the node's cores: there the OpenMP workers of the
    # QV-tree host code sleep between parallel regions instead of spinning
    # (must be set before libgomp is loaded).  A single rank keeps the default
    # (spinning workers wake up faster: ~7 % more plans/s).
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip cpu_baseline")
    ap.add_argument("--no-qv", action="store_true", help="skip the QV-tree section")
    ap.add_argument("--no-syn16k", action="store_true",
                    help="skip the 16384x16384 strong-scaling section")
    ap.add_argument("--no-stage", action="store_true",
                    help="e2e: upload each step's map inside pp2d_mdp_reset instead of "
                         "staging it under the previous solve (A/B)")
    ap.add_argument("--no-ref-cuda", action="store_true",
                    help="skip the reference-kernels-on-this-GPU line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what they computed as DIR/<name>.npy "
                         "(float32, J and action at a fixed sample of 2^20 cells, sample "
                         "indices as float64), for comparing two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    with StdoutGuard() as out:
        args.emit = out.emit
        if args.impl == "reference":
            run_reference_arm(args)
        else:
            run_main_arm(args)


if __name__ == "__main__":
    main()
