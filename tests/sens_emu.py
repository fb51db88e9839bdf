"""Lane-emulation build of the hardpoint-sensitivity instantiation of the device core (tests only;
the product never loads it): ``emu_solve_sens`` is ``helpers.emu_solve`` with the
``hardpoint_sensitivity`` output ``[n, n_steps, n_sens, n_out, 3]`` added."""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from helpers import ROOT

_LIB = None


def emu_sens_lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(ROOT, "tests", "emu", "okin_emu_sens.cpp")
        out = os.path.join(ROOT, "tests", "emu", "libokin_emu_sens.so")
        csrc = os.path.join(ROOT, "open-kinematics_b200", "csrc")
        deps = [src, os.path.join(ROOT, "include", "okin.h")]
        deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".cuh"))]
        if not os.path.exists(out) or os.path.getmtime(out) < max(map(os.path.getmtime, deps)):
            subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", f"-I{csrc}", "-o", out, src], check=True)
        lib = ctypes.CDLL(out)
        lib.okin_emu_sens_sweep.restype = ctypes.c_int
        lib.okin_emu_sens_sweep.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_long, ctypes.c_int] + [ctypes.c_void_p] * 2
        _LIB = lib
    return _LIB


class UsageError(RuntimeError):
    """The library would return OKIN_ERR_USAGE (a topology with camber-shim records)."""


def emu_solve_sens(program, hardpoints: np.ndarray, values: np.ndarray, want_health=False, **cfg) -> dict:
    from open_kinematics_b200._lib import BatchIO, SolverCfg
    hp = np.ascontiguousarray(hardpoints, dtype=np.float64).reshape(-1, 3 * program.n_in)
    tv = np.ascontiguousarray(values, dtype=np.float64)
    n_inst, n_steps, nt, n = hp.shape[0], tv.shape[1], tv.shape[0], program.n_unknowns
    out = {
        "positions": np.zeros((n_inst, n_steps, program.n_out, 3)), "iters": np.zeros((n_inst, n_steps), np.int32),
        "max_residual": np.zeros((n_inst, n_steps)), "tangents": np.zeros((n_inst, n_steps, nt, n)),
        "velocities": np.zeros((n_inst, n_steps, nt, program.n_out, 3)),
        "tangent_health": np.zeros((n_inst, n_steps, 2)) if want_health else None,
        "status": np.zeros(n_inst, np.int32), "failed_step": np.zeros(n_inst, np.int32),
        "metrics": np.zeros((n_inst, n_steps, len(program.metric_names))) if program.metric_names else None,
        "design": np.zeros((n_inst, program.n_out, 3)),
        "diagnostics": np.zeros((n_inst, n_steps, len(program.diagnostic_names))) if program.diagnostic_names else None,
        "jumps": np.zeros((n_inst, n_steps, n // 3)) if program.diagnostic_names else None,
        "worst_row": np.zeros(n_inst, np.int32),
        "hardpoint_sensitivity": np.zeros((n_inst, n_steps, len(program.sensitivity_inputs), program.n_out, 3)),
    }
    settings = dict(step_tol=1e-6, coarse_tol=1e-3, fine_tol=1e-4, residual_tol=1e-3, mu_init=1e-3, max_iter=50,
                    use_predictor=4)
    settings.update(cfg)
    c = SolverCfg(**settings)
    hdr = np.ascontiguousarray(program.hdr)
    io = BatchIO.of(hardpoints=hp, target_values=tv, **out)
    rc = emu_sens_lib().okin_emu_sens_sweep(hdr.ctypes.data, program.iblob.ctypes.data, program.fblob.ctypes.data,
                                            n_inst, n_steps, ctypes.byref(c), ctypes.byref(io))
    if rc == -3:
        raise UsageError("hardpoint sensitivities are not available on a topology with camber-shim records")
    assert rc == 0, rc
    if out["metrics"] is None:
        out["metrics"] = np.zeros((n_inst, n_steps, 1))
    return out
