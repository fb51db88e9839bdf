"""Tolerance studies on the device: every study equals numpy statistics of ``BatchSolver.solve`` on
``study_inputs`` of all its instances (exact fields exact, moments within 1e-13 of the column's
scale), across several chunks including a partial one; device-generated inputs against the numpy
restatement; repeatability, seeds, device lists; and the linearised spread at n = 65536."""

from __future__ import annotations

import numpy as np
import pytest

import study_reference as ref
from test_study import EXACT, solver_of

pytestmark = pytest.mark.gpu
CHUNK = 65536


def device_count() -> int:
    from open_kinematics_b200 import _lib
    return _lib.device_count()


def check_study(solver, smp, n, seed, want_metrics, **kw):
    res = solver.study(smp, n, seed=seed, **kw)
    values, status, failed = [], [], []
    for lo in range(0, n, CHUNK):
        ids = np.arange(lo, min(n, lo + CHUNK))
        hp, par = solver.study_inputs(smp, seed, ids)
        per = solver.solve(hp, params=par if par.shape[1] else None, want_metrics=want_metrics)
        values.append(ref.quantity_values(solver, res.quantities, per))
        status.append(per.status)
        failed.append(per.failed_step)
    values, status, failed = np.concatenate(values), np.concatenate(status), np.concatenate(failed)
    nb = 0 if res.histogram is None else res.histogram.shape[-1] - 2
    want = ref.statistics(values, status, failed, res.hist_lo, res.hist_hi, nb)
    for name in EXACT:
        if want[name] is None:
            assert getattr(res, name) is None
            continue
        assert np.array_equal(getattr(res, name), want[name], equal_nan=True), name
    scale = np.fmax(np.abs(want["mean"]), np.nan_to_num(want["std"]))
    for name in ("mean", "std"):
        got, exp = getattr(res, name), want[name]
        assert np.array_equal(np.isnan(got), np.isnan(exp)), name
        ok = ~np.isnan(exp)
        assert (np.abs(got[ok] - exp[ok]) <= 1e-13 * scale[ok]).all(), name
    return res


def test_study_c1_lean():
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c1_dw_corner_bump")
    try:
        smp = Sampling(solver).normal("all", 0.5)
        names = [f"{k.name.lower()}_{a}" for k in solver.program.out_keys for a in "xyz"] + ["solver_nfev"]
        hist = {n: (-1e3, 1e3) for n in names}
        hist["solver_nfev"] = (0.0, 12.0)
        res = check_study(solver, smp, 2 * CHUNK + 4321, 11, False, points="all", solver_quantities=("solver_nfev",),
                          histograms=hist, bins=24)
        assert res.status_counts.sum() == 2 * CHUNK + 4321
    finally:
        solver.close()


def test_study_flagship_full():
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c3_rocker_ubar_coilover_roll")
    try:
        smp = Sampling(solver, mirror_right=True).normal("all", 0.5)
        res = check_study(solver, smp, 2 * CHUNK + 777, 3, True, metrics="all",
                          points=[solver.program.out_keys[0]], solver_quantities=("solver_max_residual", "solver_nfev"))
        assert res.count.sum() > 0
    finally:
        solver.close()


def test_study_tbar_uniform_shims():
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c4_tbar_heave_shim_bump")
    try:
        prog = solver.program
        smp = Sampling(solver, mirror_right=True).normal("all", 0.25)
        smp.uniform([n for n in prog.param_names if n.endswith("setup_thickness")], 0.5)
        check_study(solver, smp, CHUNK + 999, 5, False, points=prog.out_keys[:6], solver_quantities=("solver_nfev",))
    finally:
        solver.close()


def test_device_inputs_match_restatement():
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c4_tbar_heave_shim_bump")
    try:
        prog = solver.program
        keys = prog.in_keys
        smp = Sampling(solver, mirror_right=True).normal(keys[:4], 0.3).uniform(keys[4], 0.2)
        smp.grid([(keys[5], 0), (keys[6], 2)], 2.0, 7)
        smp.uniform([n for n in prog.param_names if n.endswith("setup_thickness")], 0.5)
        ids = np.concatenate([np.arange(5000), [2 ** 32 + 3, 2 ** 45 + 1]])
        for seed in (0, 2 ** 33 + 5):
            hp, par = solver.study_inputs(smp, seed, ids)
            want = ref.inputs(smp.tables(), seed, ids)
            assert np.abs(np.concatenate([hp, par], axis=1) - want).max() <= 1e-12
    finally:
        solver.close()


def test_repeatable_and_seeded():
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c1_dw_corner_bump")
    try:
        smp = Sampling(solver).normal("all", 0.5)
        runs = [solver.study(smp, CHUNK + 100, seed=s, points="all", metrics="all") for s in (1, 1, 2)]
        for f in ("count", "mean", "std", "min", "max", "argmin", "argmax"):
            assert getattr(runs[0], f).tobytes() == getattr(runs[1], f).tobytes(), f
        assert not np.array_equal(runs[0].mean, runs[2].mean)
    finally:
        solver.close()


@pytest.mark.skipif("device_count() < 2")
def test_device_lists_bit_identical():
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c1_dw_corner_bump")
    try:
        smp = Sampling(solver).normal("all", 0.5)
        names = [f"{k.name.lower()}_{a}" for k in solver.program.out_keys for a in "xyz"]
        runs = [solver.study(smp, 4 * CHUNK + 17, seed=9, points="all", devices=d,
                             histograms={n: (-1e3, 1e3) for n in names}, bins=16) for d in ([0], [0, 1], [1, 0])]
        for other in runs[1:]:
            for f in ("count", "nonfinite", "mean", "std", "min", "max", "argmin", "argmax", "histogram",
                      "status_counts", "failed_at_step"):
                assert getattr(runs[0], f).tobytes() == getattr(other, f).tobytes(), f
    finally:
        solver.close()


def test_linearised_spread_65536():
    """sigma = 0.01 mm on every hardpoint coordinate of C1, n = 65536: the study's std within 3 % of
    the first-order spread of the nominal instance's hardpoint sensitivities wherever that exceeds
    1e-4 mm (sampling error of a std at this n: 0.3 %)."""
    from open_kinematics_b200.core.sensitivity import linearised_std
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c1_dw_corner_bump")
    try:
        smp = Sampling(solver).normal("all", 0.01)
        res = solver.study(smp, CHUNK, seed=5, points="all")
        sens = solver.solve(solver.nominal_hardpoints()[None], want_hardpoint_sensitivity=True)
        prog = solver.program
        sig = np.array([0.01 if smp.source[3 * prog.in_keys.index(k) + a] >= 0 else 0.0
                        for k, a in sens.sensitivity_inputs])
        lin = linearised_std(sens.hardpoint_sensitivity, sig)[0].reshape(solver.values.shape[1], -1)
        mask = lin > 1e-4
        assert mask.sum() > 100
        assert np.abs(res.std[mask] / lin[mask] - 1.0).max() < 0.03
    finally:
        solver.close()
