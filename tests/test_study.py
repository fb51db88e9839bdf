"""Tolerance studies on the CPU: the sampling contract against its numpy restatement
(tests/study_reference.py), the lane-emulated study pipeline (tests/emu/okin_emu_study.cpp: the
library's generator and reduction order with a small chunk size) against numpy statistics of the
emulation's own per-instance outputs, shard-split invariance, the linearised spread of the hardpoint
sensitivities, and every usage error of the C ABI."""

from __future__ import annotations

import ctypes
import os
import sys

import numpy as np
import pytest

import study_reference as ref
from helpers import ROOT, build_case, emu_solve, load_golden
from sens_emu import emu_solve_sens
from study_emu import emu_philox, emu_study, emu_study_inputs

PHILOX_KAT = [
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
]
EXACT = ("count", "nonfinite", "min", "max", "argmin", "argmax", "histogram", "status_counts", "failed_at_step")


def solver_of(name: str):
    from open_kinematics_b200.core.sweep import BatchSolver
    meta, _ = load_golden(name)
    sus, sweep = build_case(meta)
    return BatchSolver(sus, sweep)


@pytest.fixture(scope="module")
def c1():
    s = solver_of("c1_dw_corner_bump")
    yield s
    s.close()


@pytest.fixture(scope="module")
def axle():
    s = solver_of("c4_tbar_heave_shim_bump")
    yield s
    s.close()


@pytest.mark.parametrize("ctr,key,expect", PHILOX_KAT)
def test_philox_known_answers(ctr, key, expect):
    assert emu_philox(ctr, key) == expect
    assert [int(x[0]) for x in ref.philox4x32_10([np.array([c]) for c in ctr], key)] == expect


def mixed_sampling(solver):
    from open_kinematics_b200.core.study import Sampling
    keys = solver.program.in_keys
    smp = Sampling(solver)
    smp.normal(keys[0], 0.7).uniform([keys[1], (keys[2], "z")], [0.3, 0.2, 0.1, 0.05])
    smp.grid([(keys[3], 0), (keys[4], "y")], 2.0, 5).grid((keys[5], 2), 1.5, 3)
    smp.uniform("camber_shim.setup_thickness", 0.5)
    return smp


def test_generator_matches_restatement(c1):
    smp = mixed_sampling(c1)
    tables = smp.tables()
    ids = np.concatenate([np.arange(300), np.array([2 ** 32 - 1, 2 ** 32, 2 ** 40 + 12345, 2 ** 62 + 7])])
    for seed in (0, 12345, 2 ** 40 + 99):
        hp, par = emu_study_inputs(c1, smp, seed, ids)
        got = np.concatenate([hp, par], axis=1)
        want = ref.inputs(tables, seed, ids)
        kind = np.asarray(smp.variate_kind)
        src = smp.source
        normal = (src >= 0) & (kind[np.maximum(src, 0)] == 0)
        assert np.array_equal(got[:, ~normal], want[:, ~normal])
        # normal variates within 4 ulp of z, carried through nominal + scale * z
        z = (want[:, normal] - smp.nominal[normal]) / smp.scale[normal]
        tol = 4 * np.spacing(np.abs(z)) * np.abs(smp.scale[normal]) + np.spacing(np.abs(want[:, normal]))
        assert (np.abs(got[:, normal] - want[:, normal]) <= tol).all()
        assert normal.sum() == 3 and np.abs(z).max() > 2.0


def test_grid_nodes_match_doe_levels():
    """The ported c5 DoE visits the nodes the torch driver's ``doe_levels`` visited, bit for bit:
    column f = (idx % 13) / 12 * 2 - 1 of idx written in base 13, added as nominal + 2 * column."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from config_scale import c5_sampling
    solver = solver_of("c3_rocker_ubar_coilover_roll")
    try:
        smp, factor_coords = c5_sampling(solver)
        ids = np.concatenate([np.arange(0, 4000), np.arange(4_826_000, 4_826_809)])
        hp, _ = emu_study_inputs(solver, smp, 0, ids)
        expect = np.repeat(solver.nominal_hardpoints()[None, :], ids.size, axis=0)
        idx = ids.copy()
        for c in factor_coords:
            col = (idx % 13).astype(np.float64) / (13 - 1) * 2.0 - 1.0
            idx = idx // 13
            expect[:, c] += 2.0 * col
        right = smp.source[:expect.shape[1]] >= 0
        assert np.array_equal(hp[:, right & np.isin(np.arange(expect.shape[1]), factor_coords)],
                              expect[:, right & np.isin(np.arange(expect.shape[1]), factor_coords)])
        # the mirrored right twins carry the same node with y negated
        for c in factor_coords:
            twins = np.nonzero((smp.source == smp.source[c]) & (np.arange(smp.source.size) != c))[0]
            for t in twins:
                sign = -1.0 if c % 3 == 1 else 1.0
                assert np.array_equal(hp[:, t] - smp.nominal[t], sign * (hp[:, c] - smp.nominal[c]))
    finally:
        solver.close()


def test_sampling_tables(axle):
    from open_kinematics_b200.core.primitives.point_ref import PointRef, Side
    from open_kinematics_b200.core.study import Sampling
    prog = axle.program
    smp = Sampling(axle, mirror_right=True).normal("all", 0.25)
    slot = {k: i for i, k in enumerate(prog.in_keys)}
    n_in3 = 3 * prog.n_in
    for k, i in slot.items():
        if k.side is Side.RIGHT and PointRef(Side.LEFT, k.point) in slot:
            j = slot[PointRef(Side.LEFT, k.point)]
            assert list(smp.source[3 * i: 3 * i + 3]) == list(smp.source[3 * j: 3 * j + 3])
            assert list(smp.scale[3 * i: 3 * i + 3]) == [0.25, -0.25, 0.25]
        elif k.side is Side.CENTER and abs(smp.nominal[3 * i + 1]) < 1e-9:
            assert smp.source[3 * i + 1] == -1 and smp.source[3 * i] >= 0
    assert (smp.source[n_in3:] == -1).all()                          # params are not part of "all"
    assert len(smp.variate_kind) == (smp.source[:n_in3] >= 0).sum() - sum(
        3 for k in slot if k.side is Side.RIGHT and PointRef(Side.LEFT, k.point) in slot)
    thick = [n for n in prog.param_names if n.endswith("setup_thickness")]
    smp.uniform(thick, 0.5)
    for n in thick:
        c = n_in3 + prog.param_names.index(n)
        assert smp.scale[c] == 0.5 and smp.variate_kind[smp.source[c]] == 1
    right = next(k for k in slot if k.side is Side.RIGHT)
    with pytest.raises(ValueError, match="follows its left twin"):
        Sampling(axle, mirror_right=True).normal(right, 1.0)
    with pytest.raises(ValueError, match="assigned twice"):
        smp.normal((prog.in_keys[0], "x"), 1.0)
    with pytest.raises(ValueError, match="assigned twice"):
        Sampling(axle).normal([prog.in_keys[0], (prog.in_keys[0], 2)], 1.0)
    with pytest.raises(ValueError, match="at least 2 levels"):
        Sampling(axle).grid(prog.in_keys[0], 1.0, 1)
    # grid ordering: first grid coordinate named varies fastest
    g = Sampling(axle).grid([(prog.in_keys[0], 0), (prog.in_keys[1], 0)], 1.0, 3)
    hp, _ = emu_study_inputs(axle, g, 0, np.arange(9))
    d0 = np.round(hp[:, 0] - g.nominal[0], 12)
    d1 = np.round(hp[:, 3] - g.nominal[3], 12)
    assert list(d0) == [-1, 0, 1] * 3 and list(d1) == [-1] * 3 + [0] * 3 + [1] * 3


def check_against_numpy(solver, smp, seed, n, res, want_metrics, **emu_kw):
    hp, par = emu_study_inputs(solver, smp, seed, np.arange(n))
    per = emu_solve(solver.program, hp, solver.values, params=par, lean=not want_metrics, **emu_kw)
    values = ref.quantity_values(solver, res.quantities, per)
    want = ref.statistics(values, per["status"], per["failed_step"], res.hist_lo, res.hist_hi,
                          0 if res.histogram is None else res.histogram.shape[-1] - 2)
    for name in EXACT:
        got = getattr(res, name)
        if want[name] is None:
            assert got is None
            continue
        assert np.array_equal(got, want[name], equal_nan=True), name
    # relative to the column's scale: a near-constant column (std ~ 1e-14 about a mean of 180) has
    # its std defined only to ~eps |mean|, and a mean near 0 to ~eps std
    scale = np.fmax(np.abs(want["mean"]), np.nan_to_num(want["std"]))
    for name in ("mean", "std"):
        got, exp = getattr(res, name), want[name]
        assert np.array_equal(np.isnan(got), np.isnan(exp)), name
        ok = ~np.isnan(exp)
        assert (np.abs(got[ok] - exp[ok]) <= 1e-13 * scale[ok]).all(), name
    return per


def histogram_ranges(solver, names, n=16):
    """(lo, hi) per quantity from a small emulated batch: the values mostly inside, some outside."""
    from open_kinematics_b200.core.study import Sampling
    hp = np.repeat(solver.nominal_hardpoints()[None], 1, axis=0)
    per = emu_solve(solver.program, hp, solver.values)
    v = ref.quantity_values(solver, names, per)[0]
    mid = np.nanmedian(np.where(np.isfinite(v), v, np.nan), axis=0)
    mid = np.where(np.isfinite(mid), mid, 0.0)
    half = np.maximum(np.abs(mid) * 0.02, 1e-3)
    return {name: (mid[q] - half[q], mid[q] + half[q]) for q, name in enumerate(names)}


def test_emulated_study_matches_numpy_c1(c1):
    from open_kinematics_b200.core.study import Sampling, study_quantities
    smp = Sampling(c1).normal("all", 0.5)
    kw = dict(points=[c1.program.out_keys[0], c1.program.out_keys[-1]], metrics="all",
              solver_quantities=("solver_max_residual", "solver_nfev"))
    names = study_quantities(c1.program, **kw)[0]
    hist = histogram_ranges(c1, names)
    res = emu_study(c1, smp, 200, seed=7, histograms=hist, bins=16, chunk=64, **kw)
    per = check_against_numpy(c1, smp, 7, 200, res, want_metrics=True)
    assert res.count.sum() > 0 and (res.histogram[..., 0].sum() + res.histogram[..., -1].sum()) > 0
    assert res.status_counts.sum() == 200 and (per["status"] == 0).all()
    # lean family (positions only)
    res_lean = emu_study(c1, smp, 150, seed=8, points="all", chunk=64)
    check_against_numpy(c1, smp, 8, 150, res_lean, want_metrics=False)


def test_emulated_study_matches_numpy_failing_c1():
    """C1 on the long failure-batch sweep.  At sigma = 10 mm no instance of it fails, so the batch is
    drawn with sigma = 30 mm: residual-rejected instances, failed steps and None metric columns."""
    from open_kinematics_b200.core.study import Sampling
    solver = solver_of("fail256_c1")
    try:
        smp = Sampling(solver).normal("all", 30.0)
        res = emu_study(solver, smp, 256, seed=22, points="all", metrics="all", solver_quantities=("solver_nfev",),
                        chunk=48)
        per = check_against_numpy(solver, smp, 22, 256, res, want_metrics=True)
        assert (per["status"] != 0).sum() >= 2 and res.failed_at_step.sum() == (per["failed_step"] >= 0).sum()
        assert res.nonfinite.sum() > 0          # metric columns with None (NaN) among accepted states
    finally:
        solver.close()


def test_shard_splits_bit_identical(c1):
    from open_kinematics_b200.core.study import Sampling
    smp = Sampling(c1).normal("all", 1.0).uniform("camber_shim.setup_thickness", 0.5)
    names = ["solver_nfev"]
    hist = {"solver_nfev": (0.0, 40.0)}
    runs = [emu_study(c1, smp, 170, seed=3, points="all", solver_quantities=names, histograms=dict(
        hist, **{f"{k.name.lower()}_{a}": (-1e3, 1e3) for k in c1.program.out_keys for a in "xyz"}), bins=8,
        chunk=32, n_devices=g) for g in (1, 2, 3)]
    for other in runs[1:]:
        for field in ("count", "nonfinite", "mean", "std", "min", "max", "argmin", "argmax", "histogram",
                      "status_counts", "failed_at_step"):
            a, b = getattr(runs[0], field), getattr(other, field)
            assert a.tobytes() == b.tobytes(), field


def test_linearised_spread_c1(c1):
    """sigma = 0.01 mm on every hardpoint coordinate: the study's std of every output coordinate is
    within 20 % of the first-order spread of the nominal instance's hardpoint sensitivities wherever
    that exceeds 1e-4 mm (n = 512: sampling error of a std about 3 %)."""
    from open_kinematics_b200.core.sensitivity import linearised_std
    from open_kinematics_b200.core.study import Sampling
    from test_hardpoint_sensitivity import compile_case
    smp = Sampling(c1).normal("all", 0.01)
    res = emu_study(c1, smp, 512, seed=5, points="all", chunk=128)
    prog, hp, values = compile_case("c1_dw_corner_bump")
    assert prog.in_keys == c1.program.in_keys and prog.out_keys == c1.program.out_keys
    sens = emu_solve_sens(prog, hp, values)["hardpoint_sensitivity"]
    sig = np.array([0.01 if smp.source[3 * prog.in_keys.index(k) + a] >= 0 else 0.0 for k, a in prog.sensitivity_inputs])
    lin = linearised_std(sens, sig)[0].reshape(values.shape[1], -1)
    mask = lin > 1e-4
    assert mask.sum() > 100
    ratio = res.std[mask] / lin[mask]
    assert np.abs(ratio - 1.0).max() < 0.2, np.abs(ratio - 1.0).max()


# ---- usage errors of the C ABI (validated before any device work) ----------------------------------
def call_study(solver, arrays, n_bins=0, n=10, out_fields=None, seed=0, n_steps=None):
    from open_kinematics_b200 import _lib
    desc = _lib.StudyDesc.of(arrays, seed=seed, n_bins=n_bins)
    S, Q = solver.values.shape[1], max(desc.n_quantities, 1)
    bufs = {f: np.zeros((S, Q) if f not in ("status_counts", "failed_at_step", "histogram") else
                        {"status_counts": 4, "failed_at_step": S, "histogram": S * Q * (n_bins + 2)}[f])
            for f in _lib.StudyOut.FIELDS}
    o = _lib.StudyOut(**{f: (None if out_fields is not None and f not in out_fields else b.ctypes.data)
                         for f, b in bufs.items()})
    tv = np.ascontiguousarray(solver.values)
    rc = _lib.load().okin_study(solver.topology.handle, ctypes.byref(_lib.default_cfg()), n,
                                S if n_steps is None else n_steps, tv.ctypes.data,
                                ctypes.byref(desc), ctypes.byref(o), None, 0)
    return rc, _lib.last_error()


def base_arrays(solver):
    from open_kinematics_b200.core.study import Sampling, study_quantities
    t = Sampling(solver).normal((solver.program.in_keys[0], 0), 1.0).grid((solver.program.in_keys[1], 0), 1.0, 3) \
        .tables()
    _, _, kinds, idx = study_quantities(solver.program, points=[solver.program.out_keys[0]], metrics=["camber"]
                                        if "camber" in solver.program.metric_names else [solver.program.metric_names[0]])
    return dict(t, quantity_kind=kinds, quantity_index=idx, hist_lo=np.zeros(kinds.size), hist_hi=np.ones(kinds.size))


def test_usage_errors(c1):
    from open_kinematics_b200 import _lib
    a = base_arrays(c1)

    def expect(arrays, match, **kw):
        rc, msg = call_study(c1, arrays, **kw)
        assert rc == -1 and match in msg, (rc, msg)

    expect(dict(a, nominal=a["nominal"][:-1].copy(), source=a["source"][:-1].copy(), scale=a["scale"][:-1].copy()),
           "n_coords")
    expect(a, "negative size", n=-1)
    rc, msg = call_study(c1, a, n_steps=0)
    assert rc == -1 and "at least one sweep step" in msg, msg
    for bad in (-2, 2):
        src = a["source"].copy()
        src[0] = bad
        expect(dict(a, source=src), "source out of range")
    for kind, index, match in ((0, 3 * c1.program.n_out, "position quantity out of range"),
                               (1, len(c1.program.metric_names), "metric quantity out of range"),
                               (7, 0, "unknown study quantity kind")):
        expect(dict(a, quantity_kind=np.array([kind], np.int32), quantity_index=np.array([index], np.int32),
                    hist_lo=np.zeros(1), hist_hi=np.ones(1)), match)
    expect(dict(a, quantity_kind=np.zeros(0, np.int32), quantity_index=np.zeros(0, np.int32)), "at least one quantity")
    lv = a["grid_levels"].copy()
    lv[1] = 1
    expect(dict(a, grid_levels=lv), "at least 2 levels")
    vk = a["variate_kind"].copy()
    vk[0] = 5
    expect(dict(a, variate_kind=vk), "unknown variate kind")
    for field in ("nominal", "scale"):
        for v in (np.nan, np.inf):
            arr = a[field].copy()
            arr[0] = v
            expect(dict(a, **{field: arr}), "non-finite")
    expect(dict(a, hist_lo=np.ones(2), hist_hi=np.ones(2)), "lo < hi", n_bins=4)
    expect(dict(a, hist_lo=np.array([0.0, np.nan]), hist_hi=np.ones(2)), "lo < hi", n_bins=4)
    for nb in (-1, 4097):
        expect(a, "n_bins", n_bins=nb)
    expect(a, "null study output", out_fields=("count",))
    expect(a, "null study output", n_bins=4, out_fields=tuple(f for f in _lib.StudyOut.FIELDS if f != "histogram"))
    # a metric quantity on a topology compiled without a metric program
    from open_kinematics_b200.core.topology import compile_topology
    from helpers import generic_mechanism
    from open_kinematics_b200.core.solver import sweep_target_values
    state, cons, sweep, manager, _, _ = generic_mechanism()
    heads, values = sweep_target_values(sweep)
    prog = compile_topology(state, cons, manager.spec, heads)
    topo = _lib.DeviceTopology(prog)
    try:
        class Bare:
            pass
        bare = Bare()
        bare.topology, bare.values, bare.program = topo, np.asarray(values, dtype=np.float64), prog
        nc = 3 * prog.n_in
        arrays = dict(variate_kind=np.zeros(0, np.int32), grid_levels=np.zeros(0, np.int32),
                      nominal=np.zeros(nc), source=np.full(nc, -1, np.int32), scale=np.zeros(nc),
                      quantity_kind=np.array([1], np.int32), quantity_index=np.array([0], np.int32))
        rc, msg = call_study(bare, arrays)
        assert rc == -1 and "without a metric program" in msg, msg
    finally:
        topo.close()
    # okin_study_sample: same generator checks, and ids
    desc = _lib.StudyDesc.of(dict(a, source=np.full_like(a["source"], 9)))
    hp = np.zeros((1, 3 * c1.program.n_in))
    par = np.zeros((1, len(c1.program.param_names)))
    ids = np.array([0], np.int64)
    rc = _lib.load().okin_study_sample(c1.topology.handle, ctypes.byref(desc), 1, ids.ctypes.data, hp.ctypes.data,
                                       par.ctypes.data, 0)
    assert rc == -1 and "source out of range" in _lib.last_error()
    desc = _lib.StudyDesc.of(a)
    ids = np.array([-1], np.int64)
    rc = _lib.load().okin_study_sample(c1.topology.handle, ctypes.byref(desc), 1, ids.ctypes.data, hp.ctypes.data,
                                       par.ctypes.data, 0)
    assert rc == -1 and "negative instance id" in _lib.last_error()


def test_python_usage_errors(c1):
    from open_kinematics_b200.core.study import Sampling, StudyResult
    smp = Sampling(c1).normal("all", 0.1)
    with pytest.raises(ValueError, match="at least one quantity"):
        emu_study(c1, smp, 4)
    with pytest.raises(ValueError, match="Unknown metric"):
        emu_study(c1, smp, 4, metrics=["no_such_metric"])
    with pytest.raises(ValueError, match="Unknown solver quantity"):
        emu_study(c1, smp, 4, solver_quantities=("nfev",))
    with pytest.raises(ValueError, match="every quantity"):
        emu_study(c1, smp, 4, solver_quantities=("solver_nfev", "solver_max_residual"),
                  histograms={"solver_nfev": (0, 10)})
    with pytest.raises(ValueError, match="Unknown study coordinate"):
        Sampling(c1).normal("no_such_point", 1.0)
    # quantile: linear inside a bin, NaN in the under- / overflow bins
    h = np.zeros((1, 1, 6), np.int64)
    h[0, 0] = [1, 2, 2, 0, 4, 1]
    r = StudyResult(["q"], [""], *([None] * 8), h, None, None, np.array([0.0]), np.array([4.0]))
    assert np.isnan(r.quantile(0.05)[0, 0]) and np.isnan(r.quantile(0.95)[0, 0])
    assert r.quantile(0.2)[0, 0] == pytest.approx(0.5)
    assert r.quantile(0.7)[0, 0] == pytest.approx(3.5)
