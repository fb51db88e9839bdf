#!/usr/bin/env python3
"""BASELINE.json configs[3] and configs[4] at their stated sizes, as tolerance studies
(``BatchSolver.study``: inputs generated and statistics reduced on the device).

    python tools/config_scale.py --config c4 [--instances 10000000] [--steps 101] [--devices 0,1,...]
    python tools/config_scale.py --config c5 --arm both --repeats 2

c4: double-wishbone axle with torsion bars, T-bar ARB, rocker-to-rocker heave link and camber shims,
    101-step bump (or roll) sweep, 1e7 Monte-Carlo tolerance instances: every left / centre hardpoint
    coordinate normal with sigma 0.25 mm (right points mirror their left twins, centre-line y held),
    every shim set-up thickness uniform on +-0.5 mm.
c5: DoE sensitivity sweep over a hardpoint grid: 1e8 instance-steps (4 761 905 instances x 21 steps of
    the flagship axle, each instance one node of a 13-level, 6-factor full factorial on +-2 mm) with
    every metric column evaluated on the device.

Arms, run alternately in one call (``--arm both``):
  study   ``BatchSolver.study`` end to end (generation, sweep kernel, reduction, host fold), timed on
          the host clock around the call; the result has arrived on the host when it returns.
  kernel  the device-resident sweep kernel alone (``okin_solve_batch_device``) on the same chunks of
          the same inputs, timed with CUDA events around each launch (inputs are regenerated per chunk
          outside the timed window; needs torch and a single device).
One JSON line per arm and repeat.  ``--memory`` samples free device memory while the study runs.
``--profile`` runs the study arm once more under torch.profiler and reports the device time of the
sweep kernel, the generator (``okin_study_generate``) and the reduction (``okin_study_reduce`` +
``okin_study_merge``).
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
from helpers import build_case, load_golden  # noqa: E402
from open_kinematics_b200 import _lib  # noqa: E402
from open_kinematics_b200.core.study import Sampling  # noqa: E402
from open_kinematics_b200.core.sweep import BatchSolver  # noqa: E402

# the metric columns whose ranges the c5 line reports
C5_RANGE_COLUMNS = ("roll_center_z", "camber_left", "deriv_damper_length_wrt_hub_z_left",
                    "deriv_arb_twist_wrt_hub_z_left")


def c4_sampling(solver) -> Sampling:
    smp = Sampling(solver, mirror_right=True).normal("all", 0.25)
    return smp.uniform([n for n in solver.program.param_names if n.endswith("setup_thickness")], 0.5)


def c5_sampling(solver) -> tuple:
    """(sampling, factor coordinates): six left / centre hardpoint coordinates on a 13-level grid of
    +-2 mm, the first factor varying fastest; right points mirror their left twins."""
    own, _ = bench.perturbation_mask(solver.program)
    coords = [3 * int(own[k % own.size]) + k % 3 for k in range(0, 6 * 5, 5)]
    smp = Sampling(solver, mirror_right=True)
    for c in coords:
        smp.grid((solver.program.in_keys[c // 3], c % 3), 2.0, 13)
    return smp, coords


def case(args):
    if args.config == "c4":
        from open_kinematics_b200.core.input import build_sweep
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from config_throughput import axle_sweep
        meta, _ = load_golden("c4_tbar_heave_shim_bump")
        sus, _ = build_case(meta)
        steps = args.steps or 101
        sweep = build_sweep(axle_sweep(steps, 50.0, args.mode == "roll"), sus)
        solver = BatchSolver(sus, sweep, tune_layout=True)
        return (solver, c4_sampling(solver), args.instances or 10_000_000,
                f"c4_tbar_heave_shim_{args.mode}{steps}_montecarlo", dict(points="all", solver_quantities=(
                    "solver_nfev",)))
    meta, _ = load_golden("c3_rocker_ubar_coilover_roll")
    sus, sweep = build_case(meta)
    solver = BatchSolver(sus, sweep, tune_layout=True)
    total = args.instances or -(-100_000_000 // sweep.n_steps)      # 1e8 instance-steps
    return (solver, c5_sampling(solver)[0], total, "c5_doe_grid_c3_axle_roll21_all_metrics",
            dict(metrics="all", solver_quantities=("solver_nfev",)))


class MemorySampler:
    """Smallest free device memory seen while running (cudaMemGetInfo through torch)."""

    def __init__(self, device: int):
        import torch
        self.torch, self.device = torch, device
        self.min_free = self.free()
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def free(self) -> int:
        return int(self.torch.cuda.mem_get_info(self.device)[0])

    def _run(self):
        while not self._stop.wait(0.05):
            self.min_free = min(self.min_free, self.free())

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join()


def study_arm(solver, smp, total, kw, devices, seed, memory) -> dict:
    sampler = MemorySampler(devices[0]) if memory else None
    before = sampler.free() if sampler else None
    t0 = time.perf_counter()
    if sampler:
        with sampler:
            res = solver.study(smp, total, seed=seed, devices=devices, **kw)
    else:
        res = solver.study(smp, total, seed=seed, devices=devices, **kw)
    seconds = time.perf_counter() - t0
    nfev = res.quantities.index("solver_nfev")
    accepted = float(res.count[:, nfev].sum())
    line = {"arm": "study", "seconds": seconds, "accepted_states": accepted, "states_per_s": accepted / seconds,
            "ok_fraction": float(res.status_counts[0]) / total, "status_counts": res.status_counts.tolist(),
            "mean_nfev_per_state": float((res.mean[:, nfev] * res.count[:, nfev]).sum()) / max(accepted, 1.0)}
    if kw.get("metrics"):
        line["metric_ranges"] = {c: [float(np.nanmin(res.min[:, res.quantities.index(c)])),
                                     float(np.nanmax(res.max[:, res.quantities.index(c)]))]
                                 for c in C5_RANGE_COLUMNS if c in res.quantities}
    if sampler:
        line["device_free_bytes_before"] = before
        line["device_used_bytes_during_peak"] = before - sampler.min_free
    return line


def kernel_arm(solver, smp, total, want_metrics, seed, device) -> dict:
    """The sweep kernel alone on the study's chunks: inputs regenerated per chunk (okin_study_sample)
    and uploaded outside the timed window."""
    import torch
    prog, topo = solver.program, solver.topology
    S, nout3, nm = solver.values.shape[1], 3 * prog.n_out, len(prog.metric_names)
    chunk = 65536
    dev = torch.device("cuda", device)
    hp = torch.empty((chunk, 3 * prog.n_in), device=dev, dtype=torch.float64)
    par = torch.empty((chunk, len(prog.param_names)), device=dev, dtype=torch.float64) if prog.param_names else None
    tv = torch.tensor(solver.values, device=dev, dtype=torch.float64).contiguous()
    pos = None if want_metrics else torch.empty((chunk, S, nout3), device=dev, dtype=torch.float64)
    met = torch.empty((chunk, S, nm), device=dev, dtype=torch.float64) if want_metrics else None
    status = torch.empty(chunk, device=dev, dtype=torch.int32)
    failed = torch.empty(chunk, device=dev, dtype=torch.int32)
    iters = torch.empty((chunk, S), device=dev, dtype=torch.int32)
    maxres = torch.empty((chunk, S), device=dev, dtype=torch.float64)
    io = _lib.BatchIO.of(hardpoints=hp.data_ptr(), params=par.data_ptr() if par is not None else None,
                         target_values=tv.data_ptr(), positions=pos.data_ptr() if pos is not None else None,
                         metrics=met.data_ptr() if met is not None else None, status=status.data_ptr(),
                         failed_step=failed.data_ptr(), iters=iters.data_ptr(), max_residual=maxres.data_ptr())
    lib, cfg = _lib.load(), _lib.default_cfg()
    from open_kinematics_b200.core.study import study_request
    _, _, _, desc = study_request(solver, smp, seed, None, None, ("solver_nfev",), None, 0)
    stream = torch.cuda.current_stream(dev)
    kernel_ms, accepted, n_ok = 0.0, 0, 0
    for lo in range(0, total, chunk):
        c = min(chunk, total - lo)
        h, p = topo.study_sample(desc, np.arange(lo, lo + c), device)
        hp[:c].copy_(torch.from_numpy(h))
        if par is not None:
            par[:c].copy_(torch.from_numpy(p))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        _lib.check(lib.okin_solve_batch_device(topo.handle, ctypes.byref(cfg), device,
                                               ctypes.c_void_p(stream.cuda_stream), c, S, ctypes.byref(io)), "kernel arm")
        e1.record(stream)
        e1.synchronize()
        kernel_ms += e0.elapsed_time(e1)
        ok = status[:c] == 0
        n_ok += int(ok.sum())
        accepted += int(torch.where(ok, torch.full_like(failed[:c], S), failed[:c].clamp(min=0)).sum())
    return {"arm": "kernel", "kernel_seconds": kernel_ms * 1e-3, "accepted_states": float(accepted),
            "states_per_s": accepted / (kernel_ms * 1e-3), "ok_fraction": n_ok / total}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", choices=["c4", "c5"], required=True)
    ap.add_argument("--instances", type=int, default=None)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--mode", default="bump", choices=["bump", "roll"], help="c4 sweep kind")
    ap.add_argument("--arm", default="study", choices=["study", "kernel", "both"])
    ap.add_argument("--repeats", type=int, default=1)
    ap.add_argument("--devices", default="0", help="comma-separated device ids of the study arm")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--memory", action="store_true", help="sample device memory during the study arm")
    ap.add_argument("--profile", action="store_true", help="kernel-time split of one study run")
    args = ap.parse_args()
    _lib.require_device()
    devices = [int(d) for d in args.devices.split(",")]
    solver, smp, total, label, kw = case(args)
    arms = ["kernel", "study"] if args.arm == "both" else [args.arm]
    if "kernel" in arms and len(devices) != 1:
        raise SystemExit("the kernel arm runs on a single device")
    # warm-up of both arms on one chunk (module load, lean-family calibration)
    solver.study(smp, 65536, seed=args.seed, devices=devices, **kw)
    base = {"config": label, "instances_total": total, "sweep_steps": int(solver.values.shape[1]),
            "instance_steps_total": total * int(solver.values.shape[1]), "devices": devices,
            "n_metric_columns": len(solver.program.metric_names) if kw.get("metrics") else 0,
            "n_unknowns": solver.program.n_unknowns}
    for rep in range(args.repeats):
        for arm in arms:
            if arm == "study":
                line = study_arm(solver, smp, total, kw, devices, args.seed, args.memory)
            else:
                line = kernel_arm(solver, smp, total, bool(kw.get("metrics")), args.seed, devices[0])
            print(json.dumps(dict(base, repeat=rep, **line)), flush=True)
    if args.profile:
        print(json.dumps(dict(base, **profile_study(solver, smp, total, kw, devices, args.seed))), flush=True)
    solver.close()


def profile_study(solver, smp, total, kw, devices, seed) -> dict:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        solver.study(smp, total, seed=seed, devices=devices, **kw)
    us = {"sweep_kernel": 0.0, "generate": 0.0, "reduce": 0.0, "other": 0.0}
    for ev in prof.key_averages():
        t = float(getattr(ev, "device_time_total", 0.0) or getattr(ev, "cuda_time_total", 0.0))
        if "okin_sweep_kernel" in ev.key:
            us["sweep_kernel"] += t
        elif "okin_study_generate" in ev.key:
            us["generate"] += t
        elif "okin_study_reduce" in ev.key or "okin_study_merge" in ev.key:
            us["reduce"] += t
        else:
            us["other"] += t
    return {"arm": "profile", "device_us": us,
            "generate_plus_reduce_over_sweep_kernel": (us["generate"] + us["reduce"]) / max(us["sweep_kernel"], 1e-9)}


if __name__ == "__main__":
    main()
