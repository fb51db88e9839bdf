"""Scrambled Sobol' studies on the device: device-generated inputs against the numpy restatement,
studies against numpy statistics of ``BatchSolver.solve`` on the same instances, bit-identity
across device lists, and the variance reduction over Philox sampling on C1."""

from __future__ import annotations

import json

import numpy as np
import pytest

import sobol_reference as sref
from test_study import solver_of
from test_study_gpu import CHUNK, check_study, device_count
from test_study_sobol import mixed_sobol_sampling

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["c1_dw_corner_bump", "c4_tbar_heave_shim_bump"])
def test_device_inputs_match_restatement(name):
    solver = solver_of(name)
    try:
        smp = mixed_sobol_sampling(solver, mirror_right=name.startswith("c4"))
        ids = np.concatenate([np.arange(5000), [2 ** 32 + 3, 2 ** 45 + 1, 3 * 2 ** 52 - 1]])
        kind = np.asarray(smp.variate_kind)
        normal = (smp.source >= 0) & np.isin(kind[np.maximum(smp.source, 0)], (0, 4))
        for seed in (0, 2 ** 33 + 5):
            hp, par = solver.study_inputs(smp, seed, ids)
            got = np.concatenate([hp, par], axis=1)
            want = sref.inputs(smp.tables(), seed, ids)
            assert np.array_equal(got[:, ~normal], want[:, ~normal])
            assert np.abs(got[:, normal] - want[:, normal]).max() <= 1e-12
    finally:
        solver.close()


def c1_sobol_study(solver) -> tuple:
    from open_kinematics_b200.core.study import Sampling
    smp = Sampling(solver).normal("all", 0.5, sequence="sobol")
    names = [f"{k.name.lower()}_{a}" for k in solver.program.out_keys for a in "xyz"] + ["solver_nfev"]
    hist = {n: (-1e3, 1e3) for n in names}
    hist["solver_nfev"] = (0.0, 12.0)
    return smp, 2 * CHUNK + 4321, 11, dict(points="all", solver_quantities=("solver_nfev",), histograms=hist, bins=24)


def tbar_sobol_study(solver) -> tuple:
    from open_kinematics_b200.core.study import Sampling
    prog = solver.program
    smp = Sampling(solver, mirror_right=True).normal("all", 0.25, sequence="sobol")
    smp.uniform([n for n in prog.param_names if n.endswith("setup_thickness")], 0.5, sequence="sobol")
    return smp, CHUNK + 999, 5, dict(points=prog.out_keys[:6], solver_quantities=("solver_nfev",))


def test_study_c1_lean_sobol():
    solver = solver_of("c1_dw_corner_bump")
    try:
        smp, n, seed, kw = c1_sobol_study(solver)
        res = check_study(solver, smp, n, seed, False, **kw)
        assert res.status_counts.sum() == n
    finally:
        solver.close()


def test_study_tbar_shims_sobol():
    solver = solver_of("c4_tbar_heave_shim_bump")
    try:
        smp, n, seed, kw = tbar_sobol_study(solver)
        check_study(solver, smp, n, seed, False, **kw)
        # mixed with a grid factor: a crossed design, also against numpy
        mixed = mixed_sobol_sampling(solver, mirror_right=True)
        check_study(solver, mixed, CHUNK + 3 * 111, 6, False, **kw)
    finally:
        solver.close()


@pytest.mark.skipif("device_count() < 2")
@pytest.mark.parametrize("name,study", [("c1_dw_corner_bump", c1_sobol_study),
                                        ("c4_tbar_heave_shim_bump", tbar_sobol_study)])
def test_device_lists_bit_identical(name, study):
    solver = solver_of(name)
    try:
        smp, _, seed, kw = study(solver)
        runs = [solver.study(smp, 4 * CHUNK + 17, seed=seed, devices=d, **kw) for d in ([0], [0, 1], [1, 0])]
        for other in runs[1:]:
            for f in ("count", "nonfinite", "mean", "std", "min", "max", "argmin", "argmax", "status_counts",
                      "failed_at_step"):
                assert getattr(runs[0], f).tobytes() == getattr(other, f).tobytes(), f
    finally:
        solver.close()


def test_variance_reduction_c1():
    """C1 lean, sigma = 0.5 mm on every hardpoint coordinate, N = 2^14, 8 seeds per sequence: the
    across-seed variance of the study mean and std of every position column, Sobol' over Philox.
    The bars (median ratio <= 1/16 for the mean, <= 1/4 for the std) are loose on purpose; the
    measured ratios are printed as one JSON line."""
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("c1_dw_corner_bump")
    try:
        out = {}
        for seq in ("philox", "sobol"):
            smp = Sampling(solver).normal("all", 0.5, sequence=seq)
            runs = [solver.study(smp, 2 ** 14, seed=1000 + s, points="all") for s in range(8)]
            assert all(r.status_counts[0] == 2 ** 14 for r in runs)
            out[seq] = {f: np.var(np.stack([getattr(r, f) for r in runs]), axis=0, ddof=1) for f in ("mean", "std")}
        ratio = {f: out["sobol"][f] / out["philox"][f] for f in ("mean", "std")}
        live = out["philox"]["std"] > 0
        med = {f: float(np.median(ratio[f][live])) for f in ratio}
        print(json.dumps({"variance_ratio_sobol_over_philox": {
            f: {"median": med[f], "p10": float(np.percentile(ratio[f][live], 10)),
                "p90": float(np.percentile(ratio[f][live], 90)), "max": float(ratio[f][live].max())} for f in ratio},
            "columns": int(live.sum()), "n": 2 ** 14, "seeds": 8}))
        assert med["mean"] <= 1 / 16 and med["std"] <= 1 / 4, med
    finally:
        solver.close()
