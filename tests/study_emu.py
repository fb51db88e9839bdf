"""Lane-emulation build of the tolerance-study pipeline (tests only; the product never loads it):
``emu_study`` runs the generator, the sweep and the reduction order of ``okin_study`` with a chosen
chunk size and number of emulated devices; ``emu_study_inputs`` is its ``okin_study_sample``."""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from helpers import ROOT

_LIB = None


def emu_study_lib():
    global _LIB
    if _LIB is None:
        src = os.path.join(ROOT, "tests", "emu", "okin_emu_study.cpp")
        out = os.path.join(ROOT, "tests", "emu", "libokin_emu_study.so")
        csrc = os.path.join(ROOT, "open-kinematics_b200", "csrc")
        deps = [src, os.path.join(ROOT, "include", "okin.h")]
        deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".cuh"))]
        if not os.path.exists(out) or os.path.getmtime(out) < max(map(os.path.getmtime, deps)):
            subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", f"-I{csrc}", "-o", out, src], check=True)
        lib = ctypes.CDLL(out)
        lib.okin_emu_study.restype = ctypes.c_int
        lib.okin_emu_study.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_longlong, ctypes.c_int] + \
            [ctypes.c_void_p] * 4 + [ctypes.c_longlong, ctypes.c_int]
        lib.okin_emu_study_sample.restype = ctypes.c_int
        lib.okin_emu_study_sample.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong] + [ctypes.c_void_p] * 3
        lib.okin_emu_philox.restype = None
        lib.okin_emu_philox.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        _LIB = lib
    return _LIB


def emu_philox(ctr, key) -> list:
    c = np.array(ctr, dtype=np.uint32)
    k = np.array(key, dtype=np.uint32)
    emu_study_lib().okin_emu_philox(c.ctypes.data, k.ctypes.data)
    return [int(x) for x in c]


def emu_study_inputs(solver, sampling, seed: int, ids) -> tuple:
    from open_kinematics_b200.core.study import study_request
    _, _, arrays, desc = study_request(solver, sampling, seed, None, None, ("solver_nfev",), None, 0)
    prog = solver.program
    ids = np.ascontiguousarray(ids, dtype=np.int64).reshape(-1)
    hp = np.zeros((ids.size, 3 * prog.n_in))
    par = np.zeros((ids.size, max(len(prog.param_names), 1)))
    hdr = np.ascontiguousarray(prog.hdr)
    emu_study_lib().okin_emu_study_sample(hdr.ctypes.data, ctypes.byref(desc), ids.size, ids.ctypes.data,
                                          hp.ctypes.data, par.ctypes.data)
    return hp, par[:, :len(prog.param_names)]


def emu_study(solver, sampling, n_instances: int, seed: int = 0, points=None, metrics=None, solver_quantities=(),
              histograms=None, bins: int = 64, chunk: int = 64, n_devices: int = 1, **cfg):
    """``BatchSolver.study`` in the lane emulation; ``cfg`` overrides ``okin_solver_cfg`` fields."""
    from open_kinematics_b200._lib import SolverCfg, StudyOut
    from open_kinematics_b200.core.study import StudyResult, study_request
    names, units, arrays, desc = study_request(solver, sampling, seed, points, metrics, solver_quantities,
                                               histograms, bins)
    prog = solver.program
    S, Q, nb = solver.values.shape[1], len(names), desc.n_bins
    out = {n: np.zeros((S, Q), np.int64 if n in ("count", "nonfinite", "argmin", "argmax") else np.float64)
           for n in StudyOut.FIELDS[:8]}
    out["histogram"] = np.zeros((S, Q, nb + 2), np.int64) if nb else None
    out["status_counts"] = np.zeros(4, np.int64)
    out["failed_at_step"] = np.zeros(S, np.int64)
    o = StudyOut(**{k: (v.ctypes.data if v is not None else None) for k, v in out.items()})
    settings = dict(step_tol=1e-6, coarse_tol=1e-3, fine_tol=1e-4, residual_tol=1e-3, mu_init=1e-3, max_iter=50,
                    use_predictor=4)
    settings.update(cfg)
    c = SolverCfg(**settings)
    hdr = np.ascontiguousarray(prog.hdr)
    tv = np.ascontiguousarray(solver.values, dtype=np.float64)
    rc = emu_study_lib().okin_emu_study(hdr.ctypes.data, prog.iblob.ctypes.data, prog.fblob.ctypes.data,
                                        int(n_instances), S, tv.ctypes.data, ctypes.byref(c), ctypes.byref(desc),
                                        ctypes.byref(o), int(chunk), int(n_devices))
    assert rc == 0, rc
    return StudyResult.from_out(names, units, out, arrays["hist_lo"], arrays["hist_hi"])
