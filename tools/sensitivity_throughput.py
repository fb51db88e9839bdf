#!/usr/bin/env python3
"""Cost of the hardpoint sensitivities on the device: accepted states per second of the full-output
kernel (positions + tangents) with and without the sensitivity output, all input coordinates and six
selected ones, for C1 (double-wishbone corner, 36-step bump) and C3 (rocker / U-bar coilover axle).

    python tools/sensitivity_throughput.py [--out FILE]

Device buffers (okin_solve_batch_device on torch tensors), timed with CUDA events after one warm-up
launch of each shape, median of five launches.  Inputs: authored hardpoints + N(0, 0.5 mm).  Prints one
JSON line with the card name and power limit read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import authored_positions, build_case, load_golden  # noqa: E402
from open_kinematics_b200 import _lib  # noqa: E402
from open_kinematics_b200.core.solver import sweep_target_values  # noqa: E402
from open_kinematics_b200.core.topology import compile_suspension  # noqa: E402

CASES = [("C1", "c1_dw_corner_bump", 16384), ("C3", "c3_rocker_ubar_coilover_roll", 4096)]


def time_launches(topo, prog, hp, values, sens: bool, reps: int = 5) -> tuple:
    dev = torch.device("cuda:0")
    n, S = hp.shape[0], values.shape[1]
    t_hp, t_tv = torch.tensor(hp, device=dev), torch.tensor(values, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    failed = torch.empty(n, dtype=torch.int32, device=dev)
    pos = torch.empty((n, S, prog.n_out, 3), dtype=torch.float64, device=dev)
    tan = torch.empty((n, S, len(prog.target_points), prog.n_unknowns), dtype=torch.float64, device=dev)
    bufs = dict(hardpoints=t_hp.data_ptr(), target_values=t_tv.data_ptr(), status=status.data_ptr(),
                failed_step=failed.data_ptr(), positions=pos.data_ptr(), tangents=tan.data_ptr())
    if sens:
        out = torch.empty((n, S, len(prog.sensitivity_inputs), prog.n_out, 3), dtype=torch.float64, device=dev)
        bufs["hardpoint_sensitivity"] = out.data_ptr()
    io = _lib.BatchIO.of(**bufs)
    cfg = _lib.default_cfg()
    stream = torch.cuda.current_stream(dev)

    def launch():
        _lib.check(_lib.load().okin_solve_batch_device(topo.handle, ctypes.byref(cfg), 0,
                                                       ctypes.c_void_p(stream.cuda_stream), n, S, ctypes.byref(io)),
                   "okin_solve_batch_device")
    launch()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        launch()
        e1.record(stream)
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    st, fs = status.cpu().numpy(), failed.cpu().numpy()
    accepted = int(np.where(fs < 0, S, fs).sum())
    return float(np.median(times)), accepted


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True).stdout.strip()
    result = {"device": torch.cuda.get_device_name(0), "power_limit": power, "cases": []}
    for label, golden, n in CASES:
        meta, _ = load_golden(golden)
        sus, sweep = build_case(meta)
        _, values = sweep_target_values(sweep)
        values = np.asarray(values, dtype=np.float64)
        full = compile_suspension(sus, sweep, with_shims=False)
        six = compile_suspension(sus, sweep, with_shims=False,
                                 sensitivity_inputs=full.sensitivity_inputs[::max(1, len(full.sensitivity_inputs) // 6)][:6])
        auth = authored_positions(sus)
        nominal = np.concatenate([auth[k] for k in full.in_keys])
        hp = nominal + np.random.default_rng(7).normal(0.0, 0.5, (n, nominal.size))
        row = {"config": label, "instances": n, "steps": int(values.shape[1])}
        for name, prog, sens in (("full_outputs", full, False), ("sens_all", full, True), ("sens_6", six, True)):
            topo = _lib.DeviceTopology(prog)
            try:
                sec, accepted = time_launches(topo, prog, hp, values, sens)
            finally:
                topo.close()
            row[name] = {"n_sens": len(prog.sensitivity_inputs) if sens else 0, "seconds": sec,
                         "accepted_states": accepted, "states_per_s": accepted / sec}
        result["cases"].append(row)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
