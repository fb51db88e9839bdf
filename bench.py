#!/usr/bin/env python3
"""Headline benchmark: Newton-solved sweep states per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--instances I] [--impl reference] [--single-process]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the configuration the metric's target is quoted on):
mirrored double-wishbone axle with pushrod-rocker coilovers and U-bar ARB (reference
tests/data/axle_geometry_rocker.yaml + coilover points, SURVEY.md section 8d "C3"), 21-step
roll sweep +-20 mm with the rack held, I hardpoint-perturbed instances per GPU (sigma 0.5 mm
on the left + centre points, right side mirrored; seeded).  One bench "step" = one pass of the
hot path over the whole batch = I x 21 solved states per GPU.  Only ACCEPTED states count.

Own arm   : CUDA path.  `e2e` (the headline, SURVEY.md section 8d "wall = kernel + H2D + D2H of the
            requested outputs") = the public Python API, ``BatchSolver.solve`` on page-locked NumPy
            buffers it allocates itself (``pinned=True`` / ``out=``), which calls ``okin_solve_batch``
            through ctypes; every step copies the hardpoints to the device and the results back.
            Reported for three result sets (`e2e.variants`): every point of every state (what the
            reference's solve returns; this one is `e2e.value`), moving points per state + the fixed
            points once per instance (same information, packed), and the metric table only.
            `value` = the same metric with inputs and outputs resident in HBM (device entry point of
            the C ABI, CUDA events on the launch stream): the number the roofline explains.
            `parity_max_mm`: the 256 reference-solved instances of tests/golden/batch256_c3 pushed
            through the benchmarked solver object in this run.
Reference : `--impl reference` times the UNMODIFIED reference (baseline/_ref, its public
            build_suspension / solve_sweep API, one process per host core) over a bounded sample of
            the same workload; if baseline/_ref is missing, the oracle port (oracle/solve.py).
Multi-GPU : torchrun, one rank per GPU, instance ranges sharded with no data-path collective
            (weak scaling); timing = max over ranks.  `--single-process`: one process drives all
            N devices through okin_solve_batch's own instance-range split (one host thread per device).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "solved_sweep_states_per_sec"
UNIT = "states/s"
WORKLOAD = "c3_rocker_ubar_coilover_axle_roll21"
N_STEPS_SWEEP = 21
SIGMA_MM = 0.5


def workload_case():
    """Geometry + sweep of the flagship workload from the committed golden inputs (the GPU box
    has no /root/reference)."""
    from helpers import build_case, load_golden
    meta, _ = load_golden("c3_rocker_ubar_coilover_roll")
    return build_case(meta)


def perturbation_mask(program) -> tuple:
    """(index arrays) so that left + centre points get independent noise and every right point
    mirrors its left twin (y -> -y), as the reference mirrors omitted right sides (build.py:344-354)."""
    from open_kinematics_b200.core.primitives.point_ref import PointRef, Side
    slot = {k: i for i, k in enumerate(program.in_keys)}
    own = [i for k, i in slot.items() if k.side in (Side.LEFT, Side.CENTER)]
    pairs = [(slot[PointRef(Side.LEFT, k.point)], i) for k, i in slot.items() if k.side is Side.RIGHT]
    return np.array(own), np.array(pairs)


def make_hardpoints_numpy(nominal: np.ndarray, program, n: int, seed: int) -> np.ndarray:
    own, pairs = perturbation_mask(program)
    rng = np.random.default_rng(seed)
    hp = np.repeat(nominal[None, :].reshape(1, -1, 3), n, axis=0)
    hp[:, own, :] += rng.normal(0.0, SIGMA_MM, size=(n, own.size, 3))
    hp[:, pairs[:, 1], :] = hp[:, pairs[:, 0], :] * np.array([1.0, -1.0, 1.0])
    return hp.reshape(n, -1)


def algorithmic_flops_per_state(stats: dict, mean_iters: float, n_targets: int) -> float:
    """Executed-sparse flop model (DESIGN.md section 5): per linear solve 2*(assembly + update
    + triangular solves) FMAs + ~row evaluation; plus the tangent solves per state."""
    eval_flops = 60.0 * stats["n_rows"]                     # ~45 flops per distance row + a few heavy rows
    per_iter = 2.0 * (stats["asm_fma"] + stats["g_fma"] + stats["update_fma"] + stats["solve_fma"]) \
        + 11.0 * stats["scale_tasks"] + 40.0 * stats["n_free"] + eval_flops   # row scalings + 3x3 Choleskys
    lin_solves = max(mean_iters - 1.0, 1.0)                 # nfev counts one residual-only evaluation
    return lin_solves * per_iter + eval_flops + n_targets * 2.0 * stats["solve_fma"]


def bind_to_gpu_numa_node(index: int) -> int:
    """Pin this process to the CPUs NVML reports as local to GPU ``index`` so that the pinned host
    buffers of the end-to-end path are first-touched on the GPU's own NUMA node (with 8 ranks the
    D2H stream otherwise crosses the socket interconnect).  Returns the CPU count, 0 if unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
        cpus = {64 * w + b for w, word in enumerate(mask) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:  # noqa: BLE001 - affinity is an optimisation only
        return 0


def rank_seed(rank: int) -> int:
    """Perturbation seed of a rank: config index (2) + rank, so ranks draw disjoint streams."""
    return 2 + rank


def reduce_max_ms(values, device, world: int) -> list:
    """Max over ranks of per-rank timings (the job is as slow as its slowest rank)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(list(values), device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


def job_throughput(units_per_rank: float, world: int, ms: float) -> float:
    """Whole-job units per second with per-rank work fixed (weak scaling)."""
    return world * units_per_rank / (ms * 1e-3)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if v > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REF_DIR, "kinematics"))


def perturbed_geometry(seed: int) -> tuple:
    """(geometry mapping, sweep mapping) of one instance: sigma on every left / centre hardpoint,
    right side mirrored by the reference itself (right block omitted, build.py:344-354)."""
    import copy
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "c3_rocker_ubar_coilover_roll.json")))
    geom = copy.deepcopy(meta["geometry"])
    rng = np.random.default_rng(seed)
    for side in ("left", "center"):
        block = geom["hardpoints"].get(side) or {}
        for name in sorted(block):
            for ax in "xyz":
                block[name][ax] = float(block[name][ax]) + float(rng.normal(0.0, SIGMA_MM))
    return geom, meta["sweep"]


def reference_instance_worker(args):
    """One perturbed instance through the reference's own public API (runs in a worker process):
    build_suspension + build_sweep (model build) then solve_sweep.  Returns (accepted states,
    build seconds, solve seconds)."""
    seed, = args
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    from kinematics.core.input import build_suspension, build_sweep
    from kinematics.core.sweep import solve_sweep
    geom, sweep = perturbed_geometry(seed)
    t0 = time.perf_counter()
    sus = build_suspension(geom)
    cfg = build_sweep(sweep, sus)
    t1 = time.perf_counter()
    try:
        states, _ = solve_sweep(sus, cfg)
        solved = len(states)
    except RuntimeError:
        solved = 0
    return solved, t1 - t0, time.perf_counter() - t1


def oracle_instance_worker(args):
    """Solve one perturbed instance with the oracle port (runs in a worker process)."""
    seed, = args
    from helpers import authored_positions, oracle_problem
    sus, sweep = workload_case()
    problem, values = oracle_problem(sus, sweep)
    from open_kinematics_b200.core.primitives.point_ref import Side
    from oracle.solve import solve_sweep
    rng = np.random.default_rng(seed)
    auth = authored_positions(sus)
    pert = {}
    for k, v in auth.items():
        if k.side in (Side.LEFT, Side.CENTER):
            pert[k] = v + rng.normal(0.0, SIGMA_MM, 3)
    for k, v in auth.items():
        if k.side is Side.RIGHT:
            twin = type(k)(Side.LEFT, k.point)
            pert[k] = pert[twin] * np.array([1.0, -1.0, 1.0]) if twin in pert else v
    t0 = time.perf_counter()
    out = solve_sweep(problem, pert, values)
    return int(out["status"] == 0) * values.shape[1], 0.0, time.perf_counter() - t0


def cpu_worker():
    return reference_instance_worker if reference_available() else oracle_instance_worker


def cpu_kind() -> tuple:
    if reference_available():
        return "reference", ("nickmccleery/open-kinematics itself (baseline/_ref, unmodified): build_suspension + "
                             "build_sweep + solve_sweep per instance, SciPy MINPACK LM at its default tolerances")
    return "port", "oracle/solve.py (SciPy MINPACK LM on the restated residual/Jacobian callbacks, default tolerances)"


def cpu_baseline(sample_instances: int, processes: int) -> dict:
    """The reference's CPU path timed on the host cores over a bounded sample of the workload."""
    seeds = [(1000 + i,) for i in range(sample_instances)]
    worker = cpu_worker()
    t0 = time.perf_counter()
    if processes <= 1:
        recs = [worker(s) for s in seeds]
    else:
        import multiprocessing as mp
        with mp.get_context("spawn").Pool(processes) as pool:
            recs = pool.map(worker, seeds, chunksize=1)
    dt = time.perf_counter() - t0
    solved = sum(r[0] for r in recs)
    build_s, solve_s = sum(r[1] for r in recs), sum(r[2] for r in recs)
    kind, what = cpu_kind()
    return {"value": solved / dt, "unit": UNIT, "cores": processes, "kind": kind,
            "value_without_model_build": solved / solve_s * processes if solve_s > 0 else None,
            "sample": f"{sample_instances} perturbed instances x {N_STEPS_SWEEP} steps of {WORKLOAD}, {what}, "
                      f"{dt:.1f} s wall ({build_s:.1f} s of it model build)"}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = max(cores, 4)
    worker = cpu_worker()
    kind, what = cpu_kind()
    # warm-up (imports, process pool start) then K timed steps of `per_step` instances each
    warmup = min(args.warmup, 1)              # one warm-up step is enough for a CPU pool
    times, solved, solve_s = [], 0, 0.0
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(cores) as pool:
        for step in range(warmup + args.steps):
            seeds = [(5000 + step * per_step + i,) for i in range(per_step)]
            t0 = time.perf_counter()
            recs = pool.map(worker, seeds, chunksize=1)
            dt = time.perf_counter() - t0
            if step >= warmup:
                times.append(dt)
                solved += sum(r[0] for r in recs)
                solve_s += sum(r[2] for r in recs)
    value = solved / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": warmup, "ms_per_step": 1e3 * float(np.mean(times)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "instances_per_step": per_step, "sweep_steps": N_STEPS_SWEEP,
                   "sigma_mm": SIGMA_MM},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "value_without_model_build": solved / solve_s * cores if solve_s > 0 else None,
                         "sample": f"{per_step} instances x {N_STEPS_SWEEP} steps per bench step, "
                                   f"multiprocessing.Pool({cores}), {what}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
def accepted_states(status, failed_step, n_steps: int) -> int:
    """States that were solved AND accepted: all steps of an ok instance, the steps before the
    first failed one otherwise."""
    failed = np.asarray(failed_step)
    return int(np.where(np.asarray(status) == 0, n_steps, np.maximum(failed, 0)).sum())


def parity_check(solver) -> dict:
    """The 256 reference-solved instances of tests/golden/batch256_c3 (generated by the reference
    itself at ftol = xtol = gtol = 1e-15) through the benchmarked solver object, lean kernel."""
    from helpers import key_from_name, load_golden
    from test_batches import batch_inputs
    meta, arr = load_golden("batch256_c3")
    prog = solver.program
    hp, _ = batch_inputs(meta, arr, prog, range(arr["hardpoints"].shape[0]))
    res = solver.solve(hp)
    order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    got = res.positions[:, arr["steps"]][:, :, order]
    return {"parity_max_mm": float(np.abs(got - arr["positions_tight"]).max()),
            "parity_instances": int(hp.shape[0]), "parity_flags_identical": bool(
                np.array_equal(res.status, arr["status"]) and np.array_equal(res.failed_step, arr["failed_step"])),
            "parity_source": "tests/golden/batch256_c3 (reference tight run), steps "
                             + str([int(v) for v in arr["steps"]])}


DUMP_BYTES = 60_000_000     # --dump-outputs stays below 64 MB in all


def dump_outputs(out_dir: str, t: dict) -> None:
    """Write the outputs of the device-resident path's last launch as float64 ``.npy`` files: all
    instances if they fit in DUMP_BYTES, else a fixed seeded sample of instances (sorted; their
    indices in ``instance_index.npy``).  The inputs are seeded, so two builds run with the same
    arguments can be compared file for file."""
    import torch
    names = {"positions": "pos", "status": "status", "failed_step": "failed", "iters": "iters",
             "max_residual": "maxres"}
    n_inst = t["pos"].shape[0]
    per_inst = 8 * (1 + sum(t[key][0].numel() for key in names.values()))
    k = min(n_inst, DUMP_BYTES // per_inst)
    index = np.sort(np.random.default_rng(0).choice(n_inst, k, replace=False)) if k < n_inst else np.arange(n_inst)
    rows = torch.from_numpy(index).to(t["pos"].device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instance_index.npy"), index.astype(np.float64))
    for name, key in names.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[key][rows].double().cpu().numpy())


def moving_point_keys(solver) -> list:
    """Output subset for the packed result: points that move during a sweep (free + derived)."""
    prog = solver.program
    derived = set(solver.suspension.derived_spec().functions)
    free = set(prog.free_order)
    return [k for k in prog.point_keys if k in free or k in derived]


def run_cuda(args) -> None:
    import ctypes

    import torch
    import torch.distributed as dist

    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.sweep import BatchSolver

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    single = bool(args.single_process) and world == 1 and args.gpus > 1
    devices = list(range(args.gpus)) if single else [local]
    n_dev = len(devices)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    _lib.require_device()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    local_cpus = bind_to_gpu_numa_node(local) if world > 1 else 0

    sus, sweep = workload_case()
    solver = BatchSolver(sus, sweep, tune_layout=True)     # bank-conflict-aware block placement (compile time)
    prog, topo = solver.program, solver.topology
    n_inst, S = args.instances, N_STEPS_SWEEP
    nin3, nout3, nt, n = 3 * prog.n_in, 3 * prog.n_out, len(prog.target_points), prog.n_unknowns
    lib = _lib.load()
    cfg = _lib.default_cfg()
    parity = parity_check(solver) if rank == 0 else {}

    # ---- device-resident inputs and outputs (value), one set per device --------------------
    own, pairs = perturbation_mask(prog)

    def device_set(index: int, seed: int):
        d = torch.device("cuda", index)
        gen = torch.Generator(device=d)
        gen.manual_seed(seed)
        nominal = torch.tensor(solver.nominal_hardpoints(), device=d, dtype=torch.float64).reshape(-1, 3)
        hp = nominal.unsqueeze(0).repeat(n_inst, 1, 1)
        hp[:, torch.tensor(own, device=d), :] += SIGMA_MM * torch.randn(
            (n_inst, own.size, 3), device=d, dtype=torch.float64, generator=gen)
        flip = torch.tensor([1.0, -1.0, 1.0], device=d, dtype=torch.float64)
        hp[:, torch.tensor(pairs[:, 1], device=d), :] = hp[:, torch.tensor(pairs[:, 0], device=d), :] * flip
        t = {"hp": hp.reshape(n_inst, nin3).contiguous(),
             "tv": torch.tensor(solver.values, device=d, dtype=torch.float64).contiguous(),
             "pos": torch.empty((n_inst, S, nout3), device=d, dtype=torch.float64),
             "status": torch.empty(n_inst, device=d, dtype=torch.int32),
             "failed": torch.empty(n_inst, device=d, dtype=torch.int32),
             "iters": torch.empty((n_inst, S), device=d, dtype=torch.int32),
             "maxres": torch.empty((n_inst, S), device=d, dtype=torch.float64)}
        t["io"] = _lib.BatchIO.of(hardpoints=t["hp"].data_ptr(), target_values=t["tv"].data_ptr(),
                                  positions=t["pos"].data_ptr(), status=t["status"].data_ptr(),
                                  failed_step=t["failed"].data_ptr(), iters=t["iters"].data_ptr(),
                                  max_residual=t["maxres"].data_ptr())
        t["stream"] = torch.cuda.Stream(device=d)
        return t

    sets = {index: device_set(index, rank_seed(rank if not single else index)) for index in devices}

    def launch():
        for index, t in sets.items():
            _lib.check(lib.okin_solve_batch_device(
                topo.handle, ctypes.byref(cfg), index, ctypes.c_void_p(t["stream"].cuda_stream), n_inst, S,
                ctypes.byref(t["io"])), "okin_solve_batch_device")

    def barrier():
        if world > 1:
            dist.barrier()
        for index in devices:
            torch.cuda.synchronize(index)

    for _ in range(max(args.warmup, 3)):
        launch()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # CUDA events on the stream the kernels are launched on, per device
    ev = {index: [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)] for index in devices}
    for index, t in sets.items():
        ev[index][0].record(t["stream"])
    for k in range(args.steps):
        launch()
        for index, t in sets.items():
            ev[index][k + 1].record(t["stream"])
    barrier()
    kernel_ms = [max(ev[i][k].elapsed_time(ev[i][k + 1]) for i in devices) for k in range(args.steps)]
    total_ms = max(ev[i][0].elapsed_time(ev[i][-1]) for i in devices)
    clocks = sampler.stop() if rank == 0 else None

    first = sets[devices[0]]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, first)
    status_np, failed_np = first["status"].cpu().numpy(), first["failed"].cpu().numpy()
    ok_frac = float((status_np == 0).mean())
    solved_frac = accepted_states(status_np, failed_np, S) / float(n_inst * S)
    mean_iters = float(first["iters"].double().mean().item())
    states_per_launch = n_inst * S * solved_frac            # accepted states per device per launch

    # ---- end to end through the public Python API (BatchSolver.solve on page-locked buffers) ------
    import psutil
    avail = psutil.virtual_memory().available
    bytes_per_inst_out = S * nout3 * 8 + S * 12 + 8
    budget = min(30e9 * n_dev, 0.25 * avail / max(world, 1))
    if single:
        budget = min(budget, 64e9)          # one process page-locks every buffer itself: keep that bounded
    e2e_inst = int(min(n_inst * n_dev, max(4096, budget // bytes_per_inst_out)))
    host_hp = solver.pinned_hardpoints(e2e_inst, devices[0])
    per = (e2e_inst + n_dev - 1) // n_dev
    for k, index in enumerate(devices):
        lo, hi = k * per, min((k + 1) * per, e2e_inst)
        host_hp[lo:hi] = sets[index]["hp"][: hi - lo].cpu().numpy()
    e2e_steps = args.steps

    def time_e2e(label, slv, rows, **want):
        """K calls of BatchSolver.solve on the same page-locked buffers (allocated by the first call)."""
        res = slv.solve(host_hp[:rows], devices=devices, pinned=True, **want)
        res = slv.solve(host_hp[:rows], devices=devices, out=res, **want)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            res = slv.solve(host_hp[:rows], devices=devices, out=res, **want)      # returns after the last D2H copy
        barrier()
        seconds = (time.perf_counter() - t0) / e2e_steps
        d2h = sum(a.nbytes for a in res.buffers().values() if isinstance(a, np.ndarray))
        return {"label": label, "seconds": seconds, "rows": rows, "accepted": accepted_states(res.status, res.failed_step, S),
                "h2d_bytes_per_step": int(rows * nin3 * 8 + nt * S * 8), "d2h_bytes_per_step": int(d2h)}

    runs = [time_e2e("all_points", solver, e2e_inst)]
    if not args.e2e_all_points_only:
        moving = BatchSolver(sus, sweep, output_points=moving_point_keys(solver), tune_layout=True)
        runs.append(time_e2e("moving_points_per_state+fixed_points_per_instance", moving, e2e_inst, want_design=True))
        moving.close()
        runs.append(time_e2e("metrics_only", solver, min(e2e_inst, n_inst * n_dev), want_positions=False, want_metrics=True))

    # ---- reduce over ranks (max time) ------------------------------------------------------
    reduced = reduce_max_ms([total_ms] + [r["seconds"] for r in runs], dev, world)
    total_ms_max = reduced[0]
    for r, sec in zip(runs, reduced[1:]):
        r["seconds_max_over_ranks"] = sec

    if rank == 0:
        jobs = world * n_dev if not single else n_dev        # devices in the whole job
        ms_per_step = total_ms_max / args.steps
        value = jobs * states_per_launch / (ms_per_step * 1e-3)
        variants = {}
        for r in runs:
            scale = world if not single else 1               # a single process already covers all devices
            variants[r["label"]] = {
                "value": scale * r["accepted"] / r["seconds_max_over_ranks"], "unit": UNIT,
                "instances_per_call": r["rows"], "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                "d2h_bytes_per_step": r["d2h_bytes_per_step"],
                "d2h_gb_per_s": scale * r["d2h_bytes_per_step"] / r["seconds_max_over_ranks"] / 1e9}
        head = variants["all_points"]
        peak = ctypes.c_double(0.0)
        _lib.check(lib.okin_fp64_peak(local, ctypes.byref(peak)), "okin_fp64_peak")
        model_flops_state = algorithmic_flops_per_state(prog.stats, mean_iters, 0)   # lean kernel: no tangent solves
        k_ms = float(np.mean(kernel_ms))
        executed, flops_src = None, None
        try:
            fj = json.load(open(os.path.join(ROOT, "profiles", "fp64_flops.json")))
            executed, flops_src = fj["executed_fp64_flops_per_state"], fj.get("source")
        except (OSError, KeyError):
            pass
        # SURVEY.md section 8(d): a kernel that exploits the sparsity reports executed flops (ncu
        # 2*dfma + dmul + dadd per state, profiles/fp64_flops.json); the structural model is the fallback
        flops_state = executed if executed else model_flops_state
        achieved_tflops = flops_state * n_inst * S / (k_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        alg_bytes_state = nout3 * 8 + 12 + (nin3 * 8 + 8) / S
        hbm_achieved = alg_bytes_state * n_inst * S / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
            traffic = tj["dram_bytes_per_state"] * n_inst * S
            traffic_src = tj["source"]
        except (OSError, KeyError):
            pass
        smem_pipe = None
        try:
            smem_pipe = json.load(open(os.path.join(ROOT, "profiles", "smem_pipe.json")))
        except OSError:
            pass
        geo = topo.launch_geometry(n_inst, local)
        base = cpu_baseline(sample_instances=args.cpu_sample, processes=1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": jobs, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": WORKLOAD, "instances_per_gpu": n_inst, "sweep_steps": S, "sigma_mm": SIGMA_MM,
                "n_unknowns": n, "n_rows": prog.stats["n_rows"], "ok_fraction": ok_frac,
                "accepted_state_fraction": solved_frac,
                "mean_nfev_per_state": mean_iters, "outputs": "positions(all points)+nfev+max_residual+status",
                "value_is": "device-resident (inputs and outputs in HBM); e2e is the wall-clock metric of SURVEY.md 8(d)",
                "l2_policy": f"inputs+outputs per launch {n_inst * (nin3 * 8 + S * nout3 * 8) / 1e9:.2f} GB >> 126 MB L2",
                "launch": geo, "lean_kernel_family": topo.lean_calibration(local),
                "layout_tuning": prog.stats.get("layout_tuning"), "numa_local_cpus": local_cpus,
                "process_model": "one process, okin_solve_batch splits the instance range over the devices "
                                 "(one host thread each)" if single else "one process per GPU (torchrun)",
                "e2e_api": "BatchSolver.solve(hardpoints, devices=..., out=previous result) on page-locked NumPy "
                           "buffers (okin_host_alloc), ctypes -> okin_solve_batch",
                **parity,
            },
            "e2e": {"value": head["value"], "unit": UNIT, "h2d_bytes_per_step": head["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": head["d2h_bytes_per_step"], "variants": variants},
            "gpu_launches": args.steps * n_dev,
            "clocks": clocks,
            "roofline": {
                "bound": "fp64", "achieved": achieved_tflops, "peak": peak.value, "unit": "TFLOP/s",
                "frac": achieved_tflops / peak.value if peak.value else None, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": "okin_fp64_peak DFMA microbenchmark measured in this run (MEASURED_PEAKS.json has no fp64 entry)",
                "flops_per_state": flops_state,
                "flops_source": (f"from file profiles/fp64_flops.json (ncu executed 2*dfma+dmul+dadd per state; {flops_src})"
                                 if executed else "structural model (bench.py::algorithmic_flops_per_state)"),
                "model_flops_per_state": model_flops_state,
                "dense_lu_equivalent_flops_per_state": float(prog.stats["dense_lu_flops"]) * max(mean_iters - 1.0, 1.0),
                "kernel_ms": k_ms,
                # the unit ncu shows closest to its peak is the shared-memory data pipe, not FP64 (from file)
                "shared_memory_pipe_ncu": smem_pipe,
                "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
                        "algorithmic_bytes_per_state": alg_bytes_state,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650"},
            },
            "cpu_baseline": base,
        }
        print(json.dumps(line))
    solver.close()
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--instances", type=int, default=1 << 20, help="perturbed instances per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=8, help="instances in the CPU-baseline sample")
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--single-process", action="store_true",
                    help="with --gpus N > 1 and no torchrun: one process drives all N devices")
    ap.add_argument("--e2e-all-points-only", action="store_true", help="skip the packed / metrics-only e2e variants")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last device-resident launch "
                         "(rank 0, first device) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl cuda)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
