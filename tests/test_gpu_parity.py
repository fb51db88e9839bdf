"""Parity of the CUDA path (through the C ABI) against the reference golden vectors and the
oracle.  Runs on the B200 box: ``pytest -m gpu``."""

import json
import os

import numpy as np
import pytest

from helpers import (GOLDEN, SWEEP_CASES, authored_positions, build_case, key_from_name, load_golden,
                     oracle_problem, perturbed_hardpoints)
from test_emu_core import POS_TOL_MM, _nominal, _program, check_failure_flags

pytestmark = pytest.mark.gpu


def gpu_solve(prog, hardpoints, values, **cfg):
    from open_kinematics_b200 import _lib
    topo = _lib.DeviceTopology(prog)
    try:
        out = topo.solve_batch(hardpoints, values, _lib.default_cfg(**cfg), want_tangents=True,
                               want_metrics=bool(prog.metric_names))
    finally:
        topo.close()
    return out


@pytest.mark.parametrize("case", SWEEP_CASES)
def test_positions_match_reference_tight_run(case):
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    out = gpu_solve(prog, _nominal(sus, prog), values)
    assert out["status"][0] == 0 and out["failed_step"][0] == -1
    order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    diff = np.abs(out["positions"][0][:, order] - arr["positions_tight"]).max()
    assert diff <= POS_TOL_MM, diff
    scale = max(1.0, np.abs(arr["tangents"]).max())
    assert np.abs(out["tangents"][0] - arr["tangents"]).max() <= 1e-7 * scale
    assert out["max_residual"].max() < 1e-5


@pytest.mark.parametrize("case", SWEEP_CASES)
def test_metric_rows_match_reference(case):
    """State, mechanism and derivative metrics evaluated on the device vs the reference's
    compute_sweep_metrics rows (angles within 1e-9 rad)."""
    from open_kinematics_b200.core.topology import compile_suspension
    from test_emu_metrics import check_metrics
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    assert prog.metric_names == meta["metric_names"]
    out = gpu_solve(prog, _nominal(sus, prog), arr["sweep_values"])
    assert out["status"][0] == 0
    check_metrics(prog.metric_names, out["metrics"][0], arr["metrics"])


@pytest.mark.parametrize("batch,case", [("batch_c1", "c1_dw_corner_bump"), ("batch_c2", "c2_macpherson_bump_steer"),
                                        ("batch_c3", "c3_rocker_ubar_coilover_roll")])
def test_perturbed_instances_match_reference(batch, case):
    meta, _ = load_golden(case)
    bmeta, barr = load_golden(batch)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    out = gpu_solve(prog, perturbed_hardpoints(bmeta, prog), values)
    assert (out["status"] == 0).all()
    order = [prog.out_keys.index(key_from_name(n)) for n in bmeta["point_keys"]]
    assert np.abs(out["positions"][:, :, order] - barr["positions_tight"]).max() <= POS_TOL_MM


def test_failure_flags_match_reference():
    cases = json.load(open(os.path.join(GOLDEN, "failures.json")))
    check_failure_flags(lambda prog, hp, values: gpu_solve(prog, hp, values), cases)


def test_reference_boundary_solve_suspension_sweep():
    """Boundary B1 with the reference's own call shape (tests/core/test_solver.py:156-208 style)."""
    from open_kinematics_b200.core.points.derived.manager import DerivedPointsManager
    from open_kinematics_b200.core.solver import SolverInfo, solve_suspension_sweep
    from open_kinematics_b200.core.sweep import solve_sweep

    meta, arr = load_golden("c1_dw_corner_bump")
    sus, sweep = build_case(meta)
    initial = sus.initial_state()
    before = {k: p.data.copy() for k, p in initial.positions.items()}
    states, stats = solve_suspension_sweep(initial, sus.constraints(), sweep, DerivedPointsManager(sus.derived_spec()))
    assert len(states) == len(stats) == sweep.n_steps
    assert all(isinstance(s, SolverInfo) and s.converged and s.max_residual < 1e-3 for s in stats)
    assert all(np.array_equal(before[k], initial.positions[k].data) for k in before)  # inputs not mutated
    keys = [key_from_name(n) for n in meta["point_keys"]]
    got = np.array([[st.positions[k].data for k in keys] for st in states])
    assert np.abs(got - arr["positions_tight"]).max() <= POS_TOL_MM
    states2, _ = solve_sweep(sus, sweep)
    assert np.abs(np.array([[st.positions[k].data for k in keys] for st in states2]) - got).max() < 1e-9


def test_reference_boundary_errors():
    """Infeasible target -> RuntimeError naming the step (tests/core/test_solver.py:223-244);
    underdetermined system -> ValueError (tests/core/test_solver.py:211-220)."""
    from open_kinematics_b200.core.sweep import solve_sweep
    cases = json.load(open(os.path.join(GOLDEN, "failures.json")))
    rec = cases["dw_corner_rocker_bump_-60_+80"]
    sus, sweep = build_case(rec)
    with pytest.raises(RuntimeError, match=r"sweep step 3[456] did not reach an acceptable residual"):
        solve_sweep(sus, sweep)


def test_large_batch_properties():
    """Size-independent properties at batch scale (2e4 perturbed C3 instances):
    every accepted state satisfies the rigid-link lengths of its own instance, repeated
    instances give bit-identical answers, and instance order does not matter."""
    meta, _ = load_golden("c3_rocker_ubar_coilover_roll")
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    rng = np.random.default_rng(11)
    nominal = _nominal(sus, prog)[0]
    n = 20000
    hp = nominal[None, :] + rng.normal(0.0, 0.25, size=(n, nominal.size))
    hp[n // 2:] = hp[: n // 2]                      # duplicates
    out = gpu_solve(prog, hp, values)
    ok = out["status"] == 0
    assert ok.mean() > 0.99
    assert np.array_equal(out["positions"][: n // 2][ok[: n // 2]], out["positions"][n // 2:][ok[n // 2:]])
    perm = rng.permutation(n)
    out2 = gpu_solve(prog, hp[perm], values)
    assert np.array_equal(out2["positions"][np.argsort(perm)][ok], out["positions"][ok])
    # link lengths: |p_a - p_b| constant over the sweep for every distance row (softnorm bias 1e-6)
    from open_kinematics_b200.core.constraints import DistanceConstraint
    pos = out["positions"][ok]
    for c in sus.constraints():
        if isinstance(c, DistanceConstraint):
            a, b = prog.out_keys.index(c.p1), prog.out_keys.index(c.p2)
            ia, ib = prog.in_keys.index(c.p1), prog.in_keys.index(c.p2)
            design = np.linalg.norm(hp[ok][:, 3 * ia: 3 * ia + 3] - hp[ok][:, 3 * ib: 3 * ib + 3], axis=1)
            length = np.linalg.norm(pos[:, :, a] - pos[:, :, b], axis=2)
            assert np.abs(length - design[:, None]).max() < 1e-4
    assert out["max_residual"][ok].max() <= 1e-3


def test_empty_batch_and_zero_steps():
    meta, _ = load_golden("c1_dw_corner_bump")
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    out = gpu_solve(prog, np.zeros((0, 3 * prog.n_in)), values)
    assert out["positions"].shape[0] == 0 and out["status"].shape == (0,)
    out = gpu_solve(prog, _nominal(sus, prog), values[:, :0])
    assert out["status"][0] == 0 and out["positions"].shape[1] == 0


def test_invalid_geometry_is_flagged_not_propagated():
    """A NaN / collapsed instance must not poison its warp-mates."""
    meta, arr = load_golden("c1_dw_corner_bump")
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    hp = np.repeat(_nominal(sus, prog), 8, axis=0)
    hp[3, :] = np.nan
    hp[5, :] = 0.0
    out = gpu_solve(prog, hp, values)
    assert out["status"][3] != 0 and out["status"][5] != 0
    good = [0, 1, 2, 4, 6, 7]
    assert (out["status"][good] == 0).all()
    assert np.abs(out["positions"][good] - out["positions"][0]).max() == 0.0


from helpers import SHIM_CASES  # noqa: E402


@pytest.mark.parametrize("case", SHIM_CASES)
def test_camber_shim_presolve_matches_reference(case):
    """Setup pose from the on-device shim assembly pre-solve, the sweep solved from it and its
    metric rows vs the reference; also the host model's initial_state(), which asks the device
    for the setup pose (no host-side shim arithmetic)."""
    from open_kinematics_b200.core.topology import compile_suspension
    from test_emu_metrics import check_metrics
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    out = gpu_solve(prog, _nominal(sus, prog), arr["sweep_values"])
    assert out["status"][0] == 0
    order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    assert np.abs(out["positions"][0][:, order] - arr["positions_tight"]).max() <= POS_TOL_MM
    check_metrics(prog.metric_names, out["metrics"][0], arr["metrics"])
    state = sus.initial_state()
    got = np.array([state.positions[key_from_name(n)].data for n in meta["point_keys"]])
    assert np.abs(got - arr["design_positions"]).max() <= POS_TOL_MM
    # single-instance boundary on the shimmed model
    from open_kinematics_b200.core.sweep import solve_sweep
    states, _ = solve_sweep(sus, sweep)
    got = np.array([[st.positions[key_from_name(n)].data for n in meta["point_keys"]] for st in states])
    assert np.abs(got - arr["positions_tight"]).max() <= POS_TOL_MM


def test_per_instance_shim_thickness_batch():
    """Monte-Carlo over shim thickness (BASELINE configs[3]): each instance's setup pose is
    solved on the device; thickness == design reproduces the un-shimmed sweep."""
    from open_kinematics_b200.core.sweep import BatchSolver
    meta, arr = load_golden("c4_tbar_heave_shim_roll")
    sus, sweep = build_case(meta)
    solver = BatchSolver(sus, sweep)
    prog = solver.program
    n = 64
    hp = np.repeat(solver.nominal_hardpoints()[None, :], n, axis=0)
    params = np.repeat(prog.param_default[None, :], n, axis=0)
    setup_cols = [i for i, name in enumerate(prog.param_names) if name.endswith("setup_thickness")]
    rng = np.random.default_rng(4)
    params[:, setup_cols] = rng.uniform(29.5, 30.5, size=(n, len(setup_cols)))
    params[0, setup_cols] = 31.0      # the golden instance (left shim; the mirrored right follows)
    params[1, setup_cols] = 30.0      # no-op shim
    res = solver.solve(hp, params=params)
    assert (res.status == 0).all()
    order = [prog.out_keys.index(key_from_name(k)) for k in meta["point_keys"]]
    assert np.abs(res.positions[0][:, order] - arr["positions_tight"]).max() <= POS_TOL_MM
    meta0, arr0 = load_golden("c4_tbar_roll")      # same T-bar axle without heave link / shim
    cam = prog.metric_names.index("camber_left")
    met = solver.solve(hp, params=params, want_metrics=True).metrics
    # camber at the design step is a monotone function of the shim thickness
    mid = arr["sweep_values"].shape[1] // 2
    # (instances within 0.01 mm of the design thickness are left out: below a 1e-6 rad upright
    # rotation the reference skips the attachment rotation, double_wishbone.py:554)
    far = np.abs(params[:, setup_cols[0]] - 30.0) > 0.01
    order_t = np.argsort(params[:, setup_cols[0]])
    order_t = order_t[far[order_t]]
    steps = np.diff(met[order_t, mid, cam])
    assert np.all(steps > 0) or np.all(steps < 0)
    assert abs(met[order_t[-1], mid, cam] - met[order_t[0], mid, cam]) > 0.1
    solver.close()


# ---------------------------------------------------------------------------------------------
# Boundaries B2 (compute_state_tangents) and B3 (compute_state_metrics) and the sweep facade,
# called with the reference's own call shapes on states built from the golden tight run.
# ---------------------------------------------------------------------------------------------
def _golden_states(sus, meta, arr, steps):
    from open_kinematics_b200.core.primitives.geometry import Point3
    from open_kinematics_b200.core.state import SuspensionState
    keys = [key_from_name(n) for n in meta["point_keys"]]
    free = set(sus.initial_state().free_points)
    return [SuspensionState(positions={k: Point3(arr["positions_tight"][s, i]) for i, k in enumerate(keys)},
                            free_points=set(free)) for s in steps], keys


@pytest.mark.parametrize("case", ["c1_dw_corner_bump_steer", "c3_rocker_ubar_coilover_roll"])
def test_reference_boundary_compute_state_tangents(case):
    from open_kinematics_b200.core.points.derived.manager import DerivedPointsManager
    from open_kinematics_b200.core.sensitivity import TangentField, TangentSolveInfo, compute_state_tangents
    from open_kinematics_b200.core.solver import convert_targets_to_absolute
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    steps = [0, sweep.n_steps // 2, sweep.n_steps - 1]
    states, keys = _golden_states(sus, meta, arr, steps)
    initial, constraints = sus.initial_state(), sus.constraints()
    manager = DerivedPointsManager(sus.derived_spec())
    for s, state in zip(steps, states):
        before = {k: p.data.copy() for k, p in state.positions.items()}
        targets = convert_targets_to_absolute([dim[s] for dim in sweep.target_sweeps], initial)
        fields, info = compute_state_tangents(state, constraints, manager, targets)
        assert all(np.array_equal(before[k], state.positions[k].data) for k in before)
        assert isinstance(info, TangentSolveInfo) and not info.rank_deficient
        assert info.n_variables == meta["n_unknowns"] == info.rank
        assert abs(info.smallest_singular_value / arr["tangent_sigma_min"][s] - 1) <= 1e-5
        assert abs(info.condition_number / arr["tangent_cond"][s] - 1) <= 1e-5
        assert len(fields) == len(targets) and all(isinstance(f, TangentField) for f in fields)
        for j, f in enumerate(fields):
            assert f.target_index == j and f.target == targets[j]
            got = np.array([f.velocity(k) for k in keys])
            assert np.abs(got - arr["velocities"][s, j]).max() <= 1e-7 * max(1.0, np.abs(arr["velocities"]).max())
    assert compute_state_tangents(states[0], constraints, manager, []) == (
        [], TangentSolveInfo(n_variables=0, rank=0, smallest_singular_value=0.0, condition_number=1.0))


@pytest.mark.parametrize("case", ["c1_dw_corner_bump_steer", "c4_tbar_heave_shim_roll"])
def test_reference_boundary_metrics_of_solved_states(case):
    """compute_sweep_metrics / compute_sweep_tangents / compute_state_metrics on given states."""
    from open_kinematics_b200.core.metrics.main import AxleMetricRows
    from open_kinematics_b200.core.sweep import compute_sweep_metrics, compute_sweep_tangents
    from test_emu_metrics import check_metrics
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    states, keys = _golden_states(sus, meta, arr, range(sweep.n_steps))
    result = compute_sweep_metrics(sus, sweep, states)
    assert result.derivative_error is None and len(result.rows) == sweep.n_steps
    assert all(not info.rank_deficient for info in result.tangent_solve_infos)
    flat = [row.flat_row() if isinstance(row, AxleMetricRows) else row for row in result.rows]
    assert isinstance(result.rows[0], AxleMetricRows) == sus.is_axle
    assert all(list(r.keys()) == meta["metric_names"] for r in flat)
    got = np.array([[np.nan if r[k] is None else r[k] for k in meta["metric_names"]] for r in flat])
    check_metrics(meta["metric_names"], got, arr["metrics"])

    tangents = compute_sweep_tangents(sus, sweep, states)
    assert len(tangents.per_step) == len(tangents.solve_infos) == sweep.n_steps
    s = sweep.n_steps - 1
    vel = np.array([[f.velocity(k) for k in keys] for f in tangents.per_step[s]])
    assert np.abs(vel - arr["velocities"][s]).max() <= 1e-7 * max(1.0, np.abs(arr["velocities"]).max())

    # one state, with and without tangents (derivative columns only with tangents)
    row = sus.compute_state_metrics(states[s], tangents.per_step[s])
    flat_row = row.flat_row() if isinstance(row, AxleMetricRows) else row
    got1 = np.array([[np.nan if flat_row[k] is None else flat_row[k] for k in meta["metric_names"]]])
    check_metrics(meta["metric_names"], got1, arr["metrics"][s:s + 1])
    bare = sus.compute_state_metrics(states[s])
    bare = bare.flat_row() if isinstance(bare, AxleMetricRows) else bare
    assert list(bare.keys()) == [k for k in meta["metric_names"] if not k.startswith("deriv_")]
    assert all(bare[k] == flat_row[k] or abs(bare[k] - flat_row[k]) <= 1e-9 * max(1.0, abs(flat_row[k]))
               for k in bare if flat_row[k] is not None)


def test_sweep_diagnostics_match_reference():
    """diagnose_sweep issue for issue, continuity thresholds and U-bar quantities against the
    reference on sweeps with an uneven step (tests/golden/diagnostics.*), plus the batch arrays."""
    from open_kinematics_b200.core.diagnostics import DiagnosticCategory, diagnose_sweep
    from open_kinematics_b200.core.sweep import BatchSolver, solve_evaluated_sweep, solve_sweep
    from open_kinematics_b200.csrc_defs import D
    cases = json.load(open(os.path.join(GOLDEN, "diagnostics.json")))
    arrays = np.load(os.path.join(GOLDEN, "diagnostics.npz"))
    for label, rec in cases.items():
        sus, sweep = build_case(rec)
        states, stats = solve_sweep(sus, sweep)
        report = diagnose_sweep(sus, states, stats)
        got = [(i.step, str(i.category.value), str(i.severity.value), i.message) for i in report.issues]
        ref = [(i["step"], i["category"], i["severity"], i["message"]) for i in rec["issues"]]
        assert got == ref, label
        for i, r in zip(report.issues, rec["issues"]):
            assert abs(i.value - r["value"]) <= 1e-6 * max(1.0, abs(r["value"]))
        assert report.ok == (not any(r["severity"] == "error" for r in rec["issues"]))

        # batch arrays: the nominal instance twice
        solver = BatchSolver(sus, sweep)
        try:
            hp = np.repeat(solver.nominal_hardpoints()[None, :], 2, axis=0)
            res = solver.solve(hp, want_diagnostics=True)
        finally:
            solver.close()
        prog = solver.program
        assert res.diagnostics.shape == (2, sweep.n_steps, len(prog.diagnostic_names))
        assert np.array_equal(res.diagnostics[0], res.diagnostics[1], equal_nan=True)
        thresholds = np.array([rec["thresholds"][k.name.lower()] for k in prog.free_order])
        assert np.abs(res.jumps[0, 0] - thresholds).max() <= 1e-6
        jump_steps = sorted({r["step"] for r in rec["issues"] if r["category"] == "jump"})
        flagged = [s for s in range(sweep.n_steps) if int(res.diagnostics[0, s, 0]) & D["OKIN_DIAG_JUMP"]]
        assert flagged == jump_steps
        for s in jump_steps:
            n_ref = sum(1 for r in rec["issues"] if r["category"] == "jump" and r["step"] == s)
            worst = max(r["value"] for r in rec["issues"] if r["category"] == "jump" and r["step"] == s)
            assert res.diagnostics[0, s, 1] == n_ref and abs(res.diagnostics[0, s, 2] - worst) <= 1e-6
        if "column_names" in rec:
            cols = [prog.diagnostic_names.index(n) for n in rec["column_names"]]
            ref_cols = arrays[label + "_columns"]
            got_cols = res.diagnostics[0][:, cols]
            assert np.abs(got_cols - ref_cols).max() <= 1e-6 * max(1.0, np.abs(ref_cols).max())
    # facade: solve + metrics + diagnostics in one call
    sus, sweep = build_case(cases["c1_uneven_bump"])
    evaluated = solve_evaluated_sweep(sus, sweep)
    assert len(evaluated.states) == len(evaluated.metrics.rows) == sweep.n_steps
    assert [i.category for i in evaluated.diagnostics] == [DiagnosticCategory.JUMP] * 5


def test_generic_family_mechanism_matches_reference():
    """Boundary B1 / B2 on a linkage written with the generic constraint families no shipped topology
    uses (SURVEY.md section 8 row f4): positions vs the reference's tight run, velocities vs
    compute_state_tangents."""
    from helpers import generic_mechanism
    from open_kinematics_b200.core.sensitivity import compute_state_tangents
    from open_kinematics_b200.core.solver import convert_targets_to_absolute, solve_suspension_sweep
    state, cons, sweep, manager, spec, arr = generic_mechanism()
    states, stats = solve_suspension_sweep(state, cons, sweep, manager)
    keys = [key_from_name(n) for n in spec["point_keys"]]
    got = np.array([[st.positions[k].data for k in keys] for st in states])
    assert np.abs(got - arr["positions_tight"]).max() <= POS_TOL_MM
    assert max(s.max_residual for s in stats) < 1e-6
    for s in (0, len(states) - 1):
        targets = convert_targets_to_absolute([dim[s] for dim in sweep.target_sweeps], state)
        fields, info = compute_state_tangents(states[s], cons, manager, targets)
        assert not info.rank_deficient
        vel = np.array([[f.velocity(k) for k in keys] for f in fields])
        assert np.abs(vel - arr["velocities"][s]).max() <= 1e-7 * max(1.0, np.abs(arr["velocities"]).max())


def test_result_files_match_reference(tmp_path):
    """Wide-form sweep file against the reference's own CSV for the same inputs (reference e2e test,
    tests/e2e/test_e2e.py:203-213: same columns in the same order, values at atol=rtol=1e-3 with the
    solver columns excluded -- here 1e-4 absolute on a 1e-5 mm reference), same unit metadata;
    CSV and Parquet carry the same table; batch table has the same columns per (instance, step)."""
    import csv

    import pyarrow.parquet as pq

    from open_kinematics_b200.core.sweep import BatchSolver
    from open_kinematics_b200.io.results_writer import (METADATA_KEY, batch_table, metric_unit, run_sweep,
                                                        write_batch_parquet)
    info = json.load(open(os.path.join(GOLDEN, "result_files.json")))
    for name, unit in info["metric_units"].items():
        assert metric_unit(name) == unit, name
    ref_lines = open(os.path.join(GOLDEN, "e2e_c1_bump_steer.csv")).read().splitlines()
    ref_units = json.loads(next(ln for ln in ref_lines if ln.startswith("# column_units: "))[len("# column_units: "):])
    ref_rows = list(csv.reader(ln for ln in ref_lines if not ln.startswith("#")))

    meta, arr = load_golden(info["case"])
    sus, sweep = build_case(meta)
    run_sweep(sus, sweep, tmp_path / "out.csv")
    run_sweep(sus, sweep, tmp_path / "out.parquet")
    lines = (tmp_path / "out.csv").read_text().splitlines()
    assert lines[0] == "# format_version: 3"
    units = json.loads(next(ln for ln in lines if ln.startswith("# column_units: "))[len("# column_units: "):])
    assert units == ref_units
    rows = list(csv.reader(ln for ln in lines if not ln.startswith("#")))
    assert rows[0] == ref_rows[0] and len(rows) == len(ref_rows)
    solver_cols = {"solver_converged", "solver_max_residual", "solver_nfev"}
    for got, ref in zip(rows[1:], ref_rows[1:]):
        for name, g, r in zip(rows[0], got, ref):
            if name in solver_cols:
                continue
            assert (g == "") == (r == ""), name
            if g != "":
                assert abs(float(g) - float(r)) <= 1e-4 * max(1.0, abs(float(r))), (name, g, r)

    table = pq.read_table(tmp_path / "out.parquet")
    assert table.column_names == rows[0]
    assert json.loads(table.schema.metadata[METADATA_KEY])["format_version"] == "3"
    assert table.schema.field("camber").metadata[b"unit"] == b"deg"
    assert table.schema.field("wheel_center_z").metadata[b"unit"] == b"mm"
    col = table.column("wheel_center_z").to_pylist()
    assert all(abs(v - float(r[rows[0].index("wheel_center_z")])) < 1e-9 for v, r in zip(col, rows[1:]))

    solver = BatchSolver(sus, sweep, output_points=list(sus.output_points()))
    try:
        hp = np.repeat(solver.nominal_hardpoints()[None, :], 3, axis=0)
        res = solver.solve(hp, want_metrics=True)
    finally:
        solver.close()
    bt = batch_table(res)
    assert bt.column_names == ["instance_index"] + rows[0]
    assert bt.num_rows == 3 * sweep.n_steps
    assert np.allclose(bt.column("camber").to_numpy()[:sweep.n_steps], table.column("camber").to_numpy(), atol=1e-9)
    write_batch_parquet(tmp_path / "batch.parquet", res, instances_per_row_group=2)
    back = pq.read_table(tmp_path / "batch.parquet")
    assert back.num_rows == bt.num_rows and back.column_names == bt.column_names
    assert back.column("instance_index").to_pylist()[-1] == 2


@pytest.mark.parametrize("case", ["c1_dw_corner_bump_steer", "c3_rocker_ubar_coilover_roll", "c4_tbar_roll"])
def test_analyze_sweep_matches_reference(case):
    """analyze_sweep (reference core/analysis.py:219-316): frame / key structure, sweep parameters,
    the named positions of the frames incl. the presentation points (rocker-pickup axis projections,
    T-bar midpoint; presentation.py:295-348) and the solved setup-reference pose with its metric rows."""
    from open_kinematics_b200.core.analysis import analyze_sweep
    ref = json.load(open(os.path.join(GOLDEN, "result_files.json")))["analysis"][case]
    meta, _ = load_golden(case)
    sus, sweep = build_case(meta)
    res = analyze_sweep(sus, sweep)
    assert res.steps == ref["steps"] and res.locations == ref["locations"]
    assert res.metric_keys == ref["metric_keys"] and res.corner_metric_keys == ref["corner_metric_keys"]
    assert [[p.point, p.axis, p.side] for p in res.sweep_parameters] == ref["sweep_parameters"]
    assert [[d.step, str(d.category.value)] for d in res.diagnostics] == ref["diagnostics"]
    setup = res.references["setup"]
    assert setup.label == "Setup"
    # every name the reference lists (physical, projected, midpoint) is produced, with its value
    assert set(res.point_keys) == set(ref["point_keys"]) == set(setup.positions) == set(res.frames[-1].positions)
    derived = [n for n in ref["point_keys"] if "_axis_projection_" in n or n.endswith("_t_bar_midpoint")]
    assert res.point_keys[-len(derived):] == derived if derived else True
    for name, xyz in ref["setup_positions"].items():
        assert np.abs(np.array(setup.positions[name]) - np.array(xyz)).max() <= 1e-4, name
    for name, xyz in ref["last_frame_positions"].items():
        assert np.abs(np.array(res.frames[-1].positions[name]) - np.array(xyz)).max() <= 1e-4, name

    def check_row(got, want, label):
        assert list(got) == list(want), label
        for key, value in want.items():
            assert (got[key] is None) == (value is None), (label, key)
            if value is not None:
                assert abs(got[key] - value) <= 1e-4 * max(1.0, abs(value)), (label, key, got[key], value)

    check_row(setup.metrics, ref["setup_metrics"], "setup")
    assert list(setup.corner_metrics) == list(ref["setup_corner_metrics"])
    for side, row in ref["setup_corner_metrics"].items():
        check_row(setup.corner_metrics[side], row, side)
    check_row(res.frames[-1].metrics, ref["last_frame_metrics"], "last frame")


def test_c2_macpherson_batch_properties():
    """BASELINE config 2 at its full size: 1e5 hardpoint-perturbed MacPherson corners, coordinated
    bump + steer sweep.  Size-independent properties: every accepted state keeps its own link
    lengths and keeps the strut bottom on the ball-joint -> strut-top line at its clamp offset; a
    random subsample matches the oracle (SciPy LM, tight) on the same inputs."""
    from oracle.solve import solve_sweep as oracle_sweep
    meta, _ = load_golden("c2_macpherson_bump_steer")
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    rng = np.random.default_rng(2)
    nominal = _nominal(sus, prog)[0].reshape(-1, 3)
    n = 100000
    hp = nominal[None] + rng.normal(0.0, 0.5, size=(n,) + nominal.shape)
    from open_kinematics_b200.core.enums import PointID as P
    i_lbj, i_top, i_sb = (prog.in_keys.index(k) for k in (P.LOWER_WISHBONE_OUTBOARD, P.STRUT_TOP, P.STRUT_BOTTOM))
    axis0 = nominal[i_top] - nominal[i_lbj]
    frac = float((nominal[i_sb] - nominal[i_lbj]) @ axis0 / (axis0 @ axis0))
    hp[:, i_sb] = hp[:, i_lbj] + frac * (hp[:, i_top] - hp[:, i_lbj])      # validator (SURVEY App. F)
    out = gpu_solve(prog, hp.reshape(n, -1), values)
    ok = out["status"] == 0
    assert ok.mean() > 0.999
    pos = out["positions"][ok]
    from open_kinematics_b200.core.constraints import DistanceConstraint
    for c in sus.constraints():
        if isinstance(c, DistanceConstraint) and c.p1 in prog.in_keys and c.p2 in prog.in_keys:
            ia, ib = prog.in_keys.index(c.p1), prog.in_keys.index(c.p2)
            design = np.linalg.norm(hp[ok][:, ia] - hp[ok][:, ib], axis=1)
            length = np.linalg.norm(pos[:, :, prog.out_keys.index(c.p1)] - pos[:, :, prog.out_keys.index(c.p2)], axis=2)
            assert np.abs(length - design[:, None]).max() < 1e-4
    lbj, top, sb = (pos[:, :, prog.out_keys.index(k)] for k in (P.LOWER_WISHBONE_OUTBOARD, P.STRUT_TOP, P.STRUT_BOTTOM))
    u = (top - lbj) / np.linalg.norm(top - lbj, axis=2, keepdims=True)
    off_line = (sb - lbj) - np.sum((sb - lbj) * u, axis=2, keepdims=True) * u
    assert np.abs(off_line).max() < 1e-4
    clamp = np.sum((sb - lbj) * u, axis=2)
    assert np.abs(clamp - clamp[:, :1]).max() < 1e-4
    problem, _ = oracle_problem(sus, sweep)
    for i in rng.choice(np.flatnonzero(ok), 3, replace=False):
        inst = {k: hp[i, j] for j, k in enumerate(prog.in_keys)}
        ref = oracle_sweep(problem, inst, values, ftol=1e-15, xtol=1e-15, gtol=1e-15)
        order = [prog.out_keys.index(k) for k in ref["keys"]]
        assert np.abs(out["positions"][i][:, order] - ref["positions"]).max() <= POS_TOL_MM


def test_c5_doe_grid_metrics_consistency():
    """BASELINE config 5 in small: full-factorial grid over 6 hardpoint coordinates of the C3 axle
    (3^6 instances) with metrics on.  Derivative metrics, obtained on the device from the tangent
    solves, must agree with central differences of the state metrics along the sweep."""
    from open_kinematics_b200.core.sweep import BatchSolver
    meta, _ = load_golden("c3_rocker_ubar_coilover_roll")
    sus, sweep = build_case(meta)
    solver = BatchSolver(sus, sweep)
    try:
        nominal = solver.nominal_hardpoints()
        rng = np.random.default_rng(5)
        coords = rng.choice(np.flatnonzero(np.abs(nominal) > 1.0), 6, replace=False)
        levels = np.array(np.meshgrid(*[[-1.0, 0.0, 1.0]] * 6, indexing="ij")).reshape(6, -1).T
        hp = np.repeat(nominal[None, :], len(levels), axis=0)
        hp[:, coords] += levels
        res = solver.solve(hp, want_metrics=True)
    finally:
        solver.close()
    ok = res.status == 0
    assert ok.mean() > 0.95
    names = res.metric_names
    m = res.metrics[ok]
    col = {n: i for i, n in enumerate(names)}
    checked = 0
    for side in ("left", "right"):
        travel = m[:, :, col[f"wheel_travel_{side}"]]
        for response in ("camber", "roadwheel_angle", "caster", "kpi", "half_track"):
            value = m[:, :, col[f"{response}_{side}"]]
            deriv = m[:, :, col[f"deriv_{response}_wrt_hub_z_{side}"]]
            # Central difference of the response against the own hub's travel along the roll sweep.
            # The other hub moves too, but it reaches this corner only through the U-bar arm, which
            # does not load the wheel carrier kinematically: the cross term is below the tolerance.
            fd = (value[:, 2:] - value[:, :-2]) / (travel[:, 2:] - travel[:, :-2])
            err = np.abs(fd - deriv[:, 1:-1])
            scale = np.maximum(np.abs(deriv[:, 1:-1]), 1e-3)
            if response in ("camber", "roadwheel_angle", "half_track"):   # O(h^2) difference error: 2 %
                assert np.nanmedian(err / scale) < 0.02, (response, side, np.nanmedian(err / scale))
                checked += 1
    assert checked == 6
    assert np.isfinite(m[:, :, col["roll_center_z"]]).mean() > 0.9


def test_optional_outputs_are_independent():
    """Every optional output can be requested on its own (the host path allocates device scratch
    for what the kernels need but the caller did not ask for), long sweeps included."""
    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.topology import compile_suspension
    meta, arr = load_golden("c4_tbar_heave_shim_bump")      # 31 steps, shimmed axle
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    hp = np.repeat(_nominal(sus, prog), 5, axis=0)
    sv = arr["sweep_values"]
    values = np.concatenate([sv, sv[:, ::-1], sv, sv[:, ::-1]], axis=1)   # 124 steps: up, down, up, down
    topo = _lib.DeviceTopology(prog)
    try:
        full = topo.solve_batch(hp, values, want_metrics=True, want_velocities=True, want_health=True,
                                want_diagnostics=True, want_tangents=True, want_design=True)
        assert (full["status"] == 0).all()
        only_diag = topo.solve_batch(hp, values, want_positions=False, want_diagnostics=True)
        assert only_diag["positions"] is None
        # (a different set of outputs takes a different code path: equal to rounding, not bit for bit)
        assert np.allclose(only_diag["diagnostics"], full["diagnostics"], rtol=0, atol=1e-9, equal_nan=True)
        assert np.allclose(only_diag["jumps"], full["jumps"], rtol=0, atol=1e-9)
        only_metrics = topo.solve_batch(hp, values, want_positions=False, want_metrics=True)
        assert np.allclose(only_metrics["metrics"], full["metrics"], rtol=1e-9, atol=1e-9, equal_nan=True)
        lean = topo.solve_batch(hp, values)
        assert np.abs(lean["positions"] - full["positions"]).max() <= 1e-9
        # the sweep retraces itself: same states on the way back, no jump flags
        n = sv.shape[1]
        assert np.abs(full["positions"][:, :n] - full["positions"][:, 2 * n - 1:n - 1:-1]).max() <= 1e-7
        assert (full["diagnostics"][:, :, 0] == 0).all()
    finally:
        topo.close()


# ---------------------------------------------------------------------------------------------
# Round 2: launch-shape robustness, in-process multi-device split, page-locked result reuse,
# per-instance target tables, worst-residual-row reporting, tuned layout on the device.
# ---------------------------------------------------------------------------------------------
def _solver(case, **kw):
    from open_kinematics_b200.core.sweep import BatchSolver
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    return BatchSolver(sus, sweep, **kw), meta, arr


def _perturbed(solver, n, sigma=0.5, seed=5):
    rng = np.random.default_rng(seed)
    nominal = solver.nominal_hardpoints()
    return nominal[None, :] + rng.normal(0.0, sigma, size=(n, nominal.size)) * (nominal != 0)[None, :]


def test_interleaved_topologies_keep_their_launch_shape():
    """Two live topologies with very different shared-memory sizes used alternately (the dynamic
    shared-memory attribute belongs to the kernel function, not to a topology: round-1 ADVICE)."""
    big, _, _ = _solver("c3_rocker_ubar_coilover_roll")
    small, _, _ = _solver("c1_dw_corner_bump")
    try:
        hb, hs = _perturbed(big, 600), _perturbed(small, 600)
        first = big.solve(hb)
        s1 = small.solve(hs)
        again = big.solve(hb)
        s2 = small.solve(hs, want_metrics=True)      # full instantiation of the small one
        third = big.solve(hb, want_metrics=True)
        assert (first.status == 0).all() and (s1.status == 0).all()
        assert np.array_equal(first.positions, again.positions)
        assert np.abs(s1.positions - s2.positions).max() <= 1e-9      # lean vs full instantiation
        assert np.abs(first.positions - third.positions).max() <= 1e-9
    finally:
        big.close()
        small.close()


@pytest.mark.parametrize("case", ["c3_rocker_ubar_coilover_roll", "c1_dw_corner_bump", "c4_tbar_heave_shim_roll"])
def test_tuned_layout_matches_reference_on_device(case):
    """The configuration bench.py runs (tune_layout=True) against the reference's tight run."""
    solver, meta, arr = _solver(case, tune_layout=True)
    try:
        res = solver.solve(solver.nominal_hardpoints()[None, :], want_tangents=True, want_metrics=True)
        assert res.status[0] == 0
        prog = solver.program
        order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
        assert np.abs(res.positions[0][:, order] - arr["positions_tight"]).max() <= POS_TOL_MM
        assert np.abs(res.tangents[0] - arr["tangents"]).max() <= 1e-7 * max(1.0, np.abs(arr["tangents"]).max())
        from test_emu_metrics import check_metrics
        check_metrics(prog.metric_names, res.metrics[0], arr["metrics"])
    finally:
        solver.close()


def test_multi_device_split_matches_single_device():
    """okin_solve_batch(device_ids, n > 1): instance ranges per device, one host thread each; the
    result is bit-identical to the single-device call (needs >= 2 visible devices)."""
    from open_kinematics_b200 import _lib
    n_dev = _lib.device_count()
    if n_dev < 2:
        pytest.skip("one visible device")
    solver, _, _ = _solver("c3_rocker_ubar_coilover_roll")
    try:
        hp = _perturbed(solver, 70001)               # odd count: uneven shards, several chunks per device
        one = solver.solve(hp, devices=[0])
        for devices in ([0, 1], list(range(n_dev)), [n_dev - 1, 0]):
            many = solver.solve(hp, devices=devices, pinned=True)
            assert np.array_equal(one.status, many.status) and np.array_equal(one.failed_step, many.failed_step)
            assert np.array_equal(one.positions, many.positions, equal_nan=True)
            assert np.array_equal(one.nfev, many.nfev)
        with pytest.raises(RuntimeError, match="twice"):
            solver.solve(hp[:10], devices=[0, 0])
    finally:
        solver.close()


def test_pinned_result_is_reused():
    solver, _, _ = _solver("c1_dw_corner_bump")
    try:
        a = _perturbed(solver, 5000, seed=1)
        b = _perturbed(solver, 5000, seed=2)
        hp = solver.pinned_hardpoints(5000)
        hp[:] = a
        first = solver.solve(hp, pinned=True, want_metrics=True)
        plain = solver.solve(a, want_metrics=True)
        assert np.array_equal(first.positions, plain.positions) and np.array_equal(first.metrics, plain.metrics, equal_nan=True)
        keep = first.positions
        hp[:] = b
        second = solver.solve(hp, out=first, want_metrics=True)
        assert second.positions is keep and second.metrics is first.metrics     # overwritten in place
        assert np.array_equal(second.positions, solver.solve(b).positions)
    finally:
        solver.close()


def test_per_instance_target_tables():
    """instance_targets[n_instances][n_targets][n_steps] replaces the shared table (Monte Carlo over
    the sweep itself): each instance must equal a plain solve with its own table."""
    from open_kinematics_b200.core.sweep import BatchSolver
    solver, meta, arr = _solver("c1_dw_corner_bump_steer")
    try:
        values = solver.values
        scales = np.array([1.0, 0.5, -0.25, 0.8])
        tables = values[None, :, :] * scales[:, None, None]
        hp = np.repeat(solver.nominal_hardpoints()[None, :], len(scales), axis=0)
        res = solver.solve(hp, instance_targets=tables, want_tangents=True)
        assert (res.status == 0).all()
        for i, sc in enumerate(scales):
            solver.values = values * sc
            single = solver.solve(hp[:1], want_tangents=True)
            assert np.array_equal(single.positions[0], res.positions[i])
            assert np.array_equal(single.tangents[0], res.tangents[i])
        solver.values = values
        if type(solver.topology).__name__ == "DeviceTopology":      # shape validation of the ctypes binding
            with pytest.raises(ValueError, match="instance_targets"):
                solver.solve(hp, instance_targets=tables[:, :, :-1])
    finally:
        solver.close()


def test_worst_residual_row_is_reported():
    """The rejection message names the same row as the reference (solver.py:640-651, :738-747)."""
    from open_kinematics_b200.core.sweep import BatchSolver, solve_sweep
    rec = json.load(open(os.path.join(GOLDEN, "failures.json")))["dw_corner_rocker_bump_-60_+80"]
    sus, sweep = build_case(rec)
    with pytest.raises(RuntimeError) as err:
        solve_sweep(sus, sweep)
    ref_row = rec["message"].split("Worst residual row: ")[1].split(". The mechanism")[0]
    assert f"Worst residual row: {ref_row}." in str(err.value), (str(err.value), ref_row)
    # batch form: the row index maps through program.row_source
    solver = BatchSolver(sus, sweep)
    try:
        res = solver.solve(solver.nominal_hardpoints()[None, :], want_worst_row=True)
        assert res.status[0] == 2 and res.worst_row[0] >= 0
        _, constraints = sus.structure()
        assert res.describe_worst_residual(0, constraints, solver.heads) == ref_row
        ok = solver.solve(solver.nominal_hardpoints()[None, :], want_worst_row=True,
                          instance_targets=solver.values[None, :, :] * 0.5)
        assert ok.status[0] == 0 and ok.worst_row[0] == -1
    finally:
        solver.close()


def test_vectors_parallel_and_spherical_families_solve_like_the_reference():
    """The two generic families no shipped topology and no other golden uses in a solve
    (VectorsParallelConstraint, SphericalJointConstraint; reference core/constraints.py:137-200,
    :311-400) through boundary B1, against the reference's tight run of the same linkage
    (tests/golden/generic_parallel_spherical.*).  The closed spherical joint is a row whose gradient
    vanishes at the solution: positions of the joint's free end are determined to second order only,
    so it is checked through the joint gap; everything else at the position bar."""
    from open_kinematics_b200.core import constraints as PC
    from open_kinematics_b200.core.enums import Axis, PointID as P, TargetPositionMode
    from open_kinematics_b200.core.points.derived.manager import DerivedPointsManager, DerivedPointsSpec
    from open_kinematics_b200.core.primitives.geometry import Direction3, Point3
    from open_kinematics_b200.core.solver import solve_suspension_sweep
    from open_kinematics_b200.core.state import SuspensionState
    from open_kinematics_b200.core.targeting import PointTarget, PointTargetAxis, SweepConfig
    meta = json.load(open(os.path.join(GOLDEN, "generic_parallel_spherical.json")))
    arr = np.load(os.path.join(GOLDEN, "generic_parallel_spherical.npz"))
    a, d, b, c, e = (P.LOWER_WISHBONE_INBOARD_FRONT, P.UPPER_WISHBONE_INBOARD_FRONT, P.LOWER_WISHBONE_OUTBOARD,
                     P.UPPER_WISHBONE_OUTBOARD, P.WHEEL_CENTER)
    pts = {a: [0, 0, 0], d: [100, 0, 0], b: [0, 0, 100], c: [100, 0, 100], e: [100, 0, 100]}
    state = SuspensionState(positions={k: Point3(np.array(v, float)) for k, v in pts.items()}, free_points={b, c, e})
    y0 = (Point3(np.zeros(3)), Direction3(np.array([0.0, 1.0, 0.0])))
    cons = [PC.DistanceConstraint(a, b, 100.0), PC.DistanceConstraint(b, c, 100.0), PC.DistanceConstraint(d, c, 100.0),
            PC.VectorsParallelConstraint(a, b, d, c), PC.PointOnPlaneConstraint(b, *y0), PC.PointOnPlaneConstraint(c, *y0),
            PC.SphericalJointConstraint(c, e), PC.FixedAxisConstraint(e, Axis.Y, 0.0), PC.DistanceConstraint(d, e, 100.0)]
    sweep = SweepConfig([[PointTarget(b, PointTargetAxis(Axis.X), float(v), TargetPositionMode.RELATIVE)
                          for v in arr["values"]]])
    manager = DerivedPointsManager(DerivedPointsSpec(functions={}, dependencies={}))
    states, stats = solve_suspension_sweep(state, cons, sweep, manager)
    assert len(states) == len(arr["values"]) and all(s.converged and s.max_residual <= 1e-3 for s in stats)
    keys = [key_from_name(n) for n in meta["point_keys"]]
    got = np.array([[st.positions[k].data for k in keys] for st in states])
    firm = [i for i, k in enumerate(keys) if k != e]
    assert np.abs(got[:, firm] - arr["positions_tight"][:, firm]).max() <= POS_TOL_MM
    gap = np.linalg.norm(got[:, keys.index(e)] - got[:, keys.index(c)], axis=1)
    assert gap.max() <= 1e-4, gap       # the reference accepts any gap below ~4.5e-5 mm (softnorm, tolerance 1e-3)


def test_lean_kernel_families_are_bit_identical_and_calibrated(monkeypatch):
    """The lean kernel exists in a 128- and a 168-register family (same source; csrc/okin_abi.cu); the
    first large batch of a topology times both and keeps the faster.  Pinned to either family
    (OKIN_LEAN_REGS, read when the topology is made resident) the results are bit-identical, and a
    calibrated solver reports which family it chose."""
    from open_kinematics_b200.core.sweep import BatchSolver
    meta, _ = load_golden("c3_rocker_ubar_coilover_roll")
    sus, sweep = build_case(meta)
    results = {}
    hp = None
    for regs in ("128", "168", None):
        if regs is None:
            monkeypatch.delenv("OKIN_LEAN_REGS", raising=False)
        else:
            monkeypatch.setenv("OKIN_LEAN_REGS", regs)
        solver = BatchSolver(sus, sweep)
        try:
            if hp is None:
                hp = _perturbed(solver, 40000, seed=9)
            results[regs] = solver.solve(hp)
            cal = solver.topology.lean_calibration(0)
            if regs is None:
                assert cal["registers"] in (128, 168) and cal["ms_128"] > 0.0 and cal["ms_168"] > 0.0
            else:
                assert cal["registers"] == int(regs)
        finally:
            solver.close()
    for other in ("168", None):
        assert np.array_equal(results["128"].positions, results[other].positions, equal_nan=True)
        assert np.array_equal(results["128"].nfev, results[other].nfev)
        assert np.array_equal(results["128"].status, results[other].status)
