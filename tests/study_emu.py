"""Lane-emulated tolerance-study pipeline (tests only; the product never loads it): ``emu_study``
runs the generator, the sweep and the reduction order of ``okin_study`` with a chosen chunk size
and number of emulated devices; ``emu_study_inputs`` is its ``okin_study_sample``."""

from __future__ import annotations

import ctypes

import numpy as np

from helpers import emu_cfg, emu_lib


def emu_philox(ctr, key) -> list:
    c = np.array(ctr, dtype=np.uint32)
    k = np.array(key, dtype=np.uint32)
    emu_lib().okin_emu_philox(c.ctypes.data, k.ctypes.data)
    return [int(x) for x in c]


def emu_study_inputs(solver, sampling, seed: int, ids) -> tuple:
    from open_kinematics_b200.core.study import study_request
    _, _, arrays, desc = study_request(solver, sampling, seed, None, None, ("solver_nfev",), None, 0)
    prog = solver.program
    ids = np.ascontiguousarray(ids, dtype=np.int64).reshape(-1)
    hp = np.zeros((ids.size, 3 * prog.n_in))
    par = np.zeros((ids.size, max(len(prog.param_names), 1)))
    hdr = np.ascontiguousarray(prog.hdr)
    emu_lib().okin_emu_study_sample(hdr.ctypes.data, ctypes.byref(desc), ids.size, ids.ctypes.data,
                                    hp.ctypes.data, par.ctypes.data)
    return hp, par[:, :len(prog.param_names)]


def emu_study(solver, sampling, n_instances: int, seed: int = 0, points=None, metrics=None, solver_quantities=(),
              histograms=None, bins: int = 64, chunk: int = 64, n_devices: int = 1, **cfg):
    """``BatchSolver.study`` in the lane emulation; ``cfg`` overrides ``okin_solver_cfg`` fields."""
    from open_kinematics_b200._lib import StudyOut
    from open_kinematics_b200.core.study import StudyResult, study_request
    names, units, arrays, desc = study_request(solver, sampling, seed, points, metrics, solver_quantities,
                                               histograms, bins)
    prog = solver.program
    S = solver.values.shape[1]
    out, o = StudyOut.allocate(S, len(names), desc.n_bins)
    hdr = np.ascontiguousarray(prog.hdr)
    tv = np.ascontiguousarray(solver.values, dtype=np.float64)
    rc = emu_lib().okin_emu_study(hdr.ctypes.data, prog.iblob.ctypes.data, prog.fblob.ctypes.data,
                                  int(n_instances), S, tv.ctypes.data, ctypes.byref(emu_cfg(**cfg)),
                                  ctypes.byref(desc), ctypes.byref(o), int(chunk), int(n_devices))
    assert rc == 0, rc
    return StudyResult.from_out(names, units, out, arrays["hist_lo"], arrays["hist_hi"])
