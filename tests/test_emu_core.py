"""The device core (csrc/okin_core.cuh) executed lane-by-lane on the CPU against the reference
golden vectors and the oracle.  Exercises the exact kernel source without a GPU; the product
never loads this emulation build."""

import json
import os

import numpy as np
import pytest

from helpers import (GOLDEN, SWEEP_CASES, authored_positions, build_case, emu_solve, key_from_name, load_golden,
                     oracle_problem, perturbed_hardpoints)
from open_kinematics_b200.core.solver import sweep_target_values
from open_kinematics_b200.core.topology import compile_topology
from oracle.solve import solve_sweep

# North-star parity bar: positions within 1e-6 mm of the tight-tolerance reference run.
POS_TOL_MM = 1e-6


def _program(sus, sweep, design_rules=True):
    from open_kinematics_b200.core.shim_program import shim_records
    heads, values = sweep_target_values(sweep)
    state, constraints = sus.structure() if design_rules else (sus.initial_state(), sus.constraints())
    prog = compile_topology(state, constraints, sus.derived_spec(), heads, design_rules=design_rules,
                            shims=shim_records(sus) if design_rules else None)
    return prog, values


def _nominal(sus, prog):
    auth = authored_positions(sus)
    return np.concatenate([auth[k] for k in prog.in_keys])[None, :]


@pytest.mark.parametrize("case", SWEEP_CASES)
@pytest.mark.parametrize("design_rules", [True, False])
def test_positions_match_reference_tight_run(case, design_rules):
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep, design_rules)
    if design_rules:
        hp = _nominal(sus, prog)
    else:  # boundary B1: explicit constants, inputs are the initial state's positions
        st = sus.initial_state()
        hp = np.concatenate([st.positions[k].data for k in prog.in_keys])[None, :]
    out = emu_solve(prog, hp, values)
    assert out["status"][0] == 0 and out["failed_step"][0] == -1
    keys = [key_from_name(n) for n in meta["point_keys"]]
    order = [prog.out_keys.index(k) for k in keys]
    diff = np.abs(out["positions"][0][:, order] - arr["positions_tight"]).max()
    assert diff <= POS_TOL_MM, diff
    assert out["max_residual"].max() < 1e-5
    assert out["iters"].max() <= 10


@pytest.mark.parametrize("case", ["c1_dw_corner_bump", "c2_macpherson_bump_steer", "c3_rocker_ubar_coilover_roll",
                                  "c4_tbar_roll"])
def test_tangents_match_reference(case):
    """dq/dt_j from the Cholesky factor vs compute_state_tangents (lstsq on [J; pins])."""
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    out = emu_solve(prog, _nominal(sus, prog), values)
    scale = np.abs(arr["tangents"]).max()
    assert np.abs(out["tangents"][0] - arr["tangents"]).max() <= 1e-7 * max(1.0, scale)


@pytest.mark.parametrize("case", ["c1_dw_corner_bump_steer", "c2_macpherson_bump_steer", "c3_rocker_ubar_coilover_roll",
                                  "c4_tbar_heave_shim_bump"])
def test_point_velocities_and_tangent_health_match_reference(case):
    """TangentField.velocities of every point (free, fixed, derived) and TangentSolveInfo."""
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    out = emu_solve(prog, _nominal(sus, prog), values, want_health=True)
    order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    vel = out["velocities"][0][:, :, order]
    assert np.abs(vel - arr["velocities"]).max() <= 1e-7 * max(1.0, np.abs(arr["velocities"]).max())
    # Within 1e-5 relative: the bound okin_tangent_health's stopping rule guarantees (the states
    # themselves differ from the reference's by up to 1e-6 mm).
    smin, cond = out["tangent_health"][0, :, 0], out["tangent_health"][0, :, 1]
    assert np.abs(smin / arr["tangent_sigma_min"] - 1).max() <= 1e-5
    assert np.abs(cond / arr["tangent_cond"] - 1).max() <= 1e-5


def test_predictor_does_not_change_the_answer():
    meta, arr = load_golden("c3_rocker_ubar_coilover_roll")
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    hp = _nominal(sus, prog)
    a = emu_solve(prog, hp, values, use_predictor=1)
    b = emu_solve(prog, hp, values, use_predictor=0)
    assert np.abs(a["positions"] - b["positions"]).max() < 1e-8
    assert a["iters"].sum() < b["iters"].sum()


@pytest.mark.parametrize("batch,case", [("batch_c1", "c1_dw_corner_bump"), ("batch_c2", "c2_macpherson_bump_steer"),
                                        ("batch_c3", "c3_rocker_ubar_coilover_roll")])
def test_perturbed_instances_match_reference(batch, case):
    """Per-instance design constants recomputed on the 'device' from perturbed hardpoints."""
    meta, _ = load_golden(case)
    bmeta, barr = load_golden(batch)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    hp = perturbed_hardpoints(bmeta, prog)
    out = emu_solve(prog, hp, values)
    assert (out["status"] == 0).all()
    order = [prog.out_keys.index(key_from_name(n)) for n in bmeta["point_keys"]]
    diff = np.abs(out["positions"][:, :, order] - barr["positions_tight"]).max()
    assert diff <= POS_TOL_MM, diff


def reference_root_checker(sus, sweep, prog, hardpoints=None, setup_pose=None):
    """``max_residual(positions_row, values_column)``: max|r| of the *reference's* residuals (oracle
    restatement, pinned to the reference's rows by tests/test_oracle_golden.py) at a device state.
    ``setup_pose``: for camber-shimmed models, the setup pose of the input points ({key: xyz}, the
    solver's own ``design`` output, itself checked against the reference's shim solve in
    test_camber_shim_presolve_matches_reference); the design constants are taken there."""
    from oracle.solve import ResidualComputer, design_setup, target_bases
    problem, _ = oracle_problem(sus, sweep, structure_only=setup_pose is not None)
    authored = setup_pose if setup_pose is not None else (authored_positions(sus) if hardpoints is None else hardpoints)
    pos0, consts = design_setup(problem, authored)
    rc = ResidualComputer(problem, pos0, consts)
    bases = target_bases(problem, pos0)

    def max_residual(row, column):
        x = np.concatenate([row[prog.out_keys.index(k)] for k in problem.free_order])
        return float(np.abs(rc.compute(x, bases + column)).max())
    return max_residual


def check_flag_contract(label, ref_status, ref_failed, dev_status, dev_failed, positions, values, max_residual,
                        tol=1e-3) -> str:
    """The flag contract against the reference, one sweep (shared by the CPU and GPU tests and by
    tools/failure_confusion.py).  Returns the cell of the confusion matrix the sweep falls in.

    * reference ok (0)                    -> device ok on every step;
    * reference residual rejection (2)    -> device residual rejection at the SAME step (solver.py:735-747:
      the optimiser converged to a least-squares compromise of an unreachable target);
    * reference "failed to converge" (1)  is MINPACK running out of its 100*n evaluation budget while it
      still crawls towards a root (measured: 1500-1800 evaluations, cost still falling, tests/golden/
      generate_batches.py) -- a statement about the optimiser, not about the mechanism.  The device
      iteration pins the rank-deficient point-on-line rows and converges there in a handful of steps.
      Contract: the device never fails EARLIER than the reference, and every state it accepts from the
      reference's failed step on is verified to be a root of the reference's own residual function
      (max|r| <= the acceptance tolerance), i.e. a state the reference would have accepted had MINPACK
      reached it.
    """
    n_steps = values.shape[1]
    if ref_status == 0:
        assert dev_status == 0 and dev_failed == -1, (label, dev_status, dev_failed)
        return "ok/ok"
    accepted_to = n_steps if dev_status == 0 else dev_failed
    assert np.isfinite(positions[:accepted_to]).all() and np.isnan(positions[accepted_to:]).all(), label
    if ref_status == 2:
        assert (dev_status, dev_failed) == (2, ref_failed), (label, dev_status, dev_failed, ref_failed)
        return "rejected/rejected same step"
    assert ref_status == 1, (label, ref_status)
    assert accepted_to >= ref_failed, (label, "device failed earlier than the reference", dev_failed, ref_failed)
    for s in range(ref_failed, accepted_to):
        r = max_residual(positions[s], values[:, s])
        assert r <= tol, (label, s, r)
    if dev_status == 0:
        return "not converged/ok (all extra states verified roots)"
    kind = "not converged" if dev_status == 1 else "rejected"
    return f"not converged/{kind} " + ("same step" if dev_failed == ref_failed else
                                        f"+{dev_failed - ref_failed} steps (extra states verified roots)")


def check_failure_flags(solve, cases: dict) -> dict:
    cells = {}
    for label, rec in cases.items():
        sus, sweep = build_case(rec)
        prog, values = _program(sus, sweep)
        out = solve(prog, _nominal(sus, prog), values)
        cell = check_flag_contract(label, rec["status"], rec["failed_step"], int(out["status"][0]),
                                   int(out["failed_step"][0]), out["positions"][0], values,
                                   reference_root_checker(sus, sweep, prog))
        cells[label] = cell
    return cells


def test_failure_flags_match_reference():
    cases = json.load(open(os.path.join(GOLDEN, "failures.json")))
    check_failure_flags(emu_solve, cases)


def test_oracle_and_core_agree_on_random_instance():
    """Same seeded perturbed inputs through the oracle (SciPy LM, tight) and the core."""
    meta, _ = load_golden("c1_dw_corner_bump")
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    problem, _ = oracle_problem(sus, sweep)
    rng = np.random.default_rng(7)
    auth = authored_positions(sus)
    for _ in range(3):
        pert = {k: v + rng.normal(0, 0.5, 3) for k, v in auth.items()}
        hp = np.concatenate([pert[k] for k in prog.in_keys])[None, :]
        out = emu_solve(prog, hp, values)
        ref = solve_sweep(problem, pert, values, ftol=1e-15, xtol=1e-15, gtol=1e-15)
        assert out["status"][0] == 0 and ref["status"] == 0
        order = [prog.out_keys.index(k) for k in ref["keys"]]
        assert np.abs(out["positions"][0][:, order] - ref["positions"]).max() <= POS_TOL_MM


from helpers import SHIM_CASES  # noqa: E402


@pytest.mark.parametrize("case", SHIM_CASES)
def test_camber_shim_presolve_matches_reference(case):
    """Setup pose (config/shims.py assembly solve + double_wishbone.py:546-571 application) and the
    sweep solved from it, positions and metric rows vs the reference."""
    from open_kinematics_b200.core.topology import compile_suspension
    from test_emu_metrics import check_metrics
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    assert prog.param_names and prog.metric_names == meta["metric_names"]
    out = emu_solve(prog, _nominal(sus, prog), arr["sweep_values"])
    assert out["status"][0] == 0
    order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    assert np.abs(out["design"][0][order] - arr["design_positions"]).max() <= POS_TOL_MM
    assert np.abs(out["positions"][0][:, order] - arr["positions_tight"]).max() <= POS_TOL_MM
    check_metrics(prog.metric_names, out["metrics"][0], arr["metrics"])
    # the same answer when the shim parameters arrive per instance instead of as defaults
    out2 = emu_solve(prog, _nominal(sus, prog), arr["sweep_values"], params=prog.param_default[None, :])
    assert np.array_equal(out2["positions"], out["positions"])
    # a no-op shim (setup == design) leaves the authored pose untouched
    par = prog.param_default.copy()
    for i, name in enumerate(prog.param_names):
        if name.endswith("setup_thickness"):
            par[i] = par[i - 1]
    out3 = emu_solve(prog, _nominal(sus, prog), arr["sweep_values"][:, :1], params=par[None, :])
    auth = authored_positions(sus)
    for k, v in auth.items():
        assert np.array_equal(out3["design"][0][prog.out_keys.index(k)], v)


def test_generated_family_rows_match_reference():
    """Every generated constraint family (csrc/okin_gen_constraints.cuh, all 12) against the rows the
    reference's own residual()/jac_*() produced (tests/golden/families.json)."""
    from helpers import emu_family
    from open_kinematics_b200.core.topology import FAMILY_CODE
    recs = json.load(open(os.path.join(GOLDEN, "families.json")))
    assert set(recs) == set(FAMILY_CODE) - {"target"}
    for fam, rec in recs.items():
        for pts, consts, res, jac in zip(rec["points"], rec["consts"], rec["residual"], rec["jacobian"]):
            pts, jac = np.array(pts), np.array(jac)
            got, got_only, grad = emu_family(FAMILY_CODE[fam], pts, consts)
            scale = max(1.0, abs(res))
            assert abs(got - res) <= 1e-11 * scale and abs(got_only - res) <= 1e-11 * scale, fam
            assert np.abs(grad - jac).max() <= 1e-11 * max(1.0, np.abs(jac).max()), fam


def test_generic_family_mechanism_matches_reference(emu_device):
    """Boundary B1 / B2 on a linkage written with the generic families no shipped topology uses
    (three-point angle, equal distance, vectors perpendicular, fixed axis, point on plane, coplanar)."""
    import test_gpu_parity as G
    G.test_generic_family_mechanism_matches_reference()


@pytest.mark.parametrize("case", ["c3_rocker_ubar_coilover_roll", "c2_macpherson_bump_steer"])
def test_tuned_block_placement_keeps_the_answer(case):
    """Bank-conflict-aware placement of the factor blocks (core/layout_tuning.py) only permutes
    storage: fewer modelled wavefronts, same positions and tangents."""
    from open_kinematics_b200.core.topology import compile_suspension
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    plain = compile_suspension(sus, sweep)
    tuned = compile_suspension(sus, sweep, tune_layout=True)
    info = tuned.stats["layout_tuning"]
    assert info["wavefronts_ideal"] <= info["wavefronts_after"] <= info["wavefronts_before"]
    assert plain.stats["layout_tuning"] is None
    a = emu_solve(plain, _nominal(sus, plain), arr["sweep_values"])
    b = emu_solve(tuned, _nominal(sus, tuned), arr["sweep_values"])
    assert (b["status"] == 0).all()
    assert np.abs(a["positions"] - b["positions"]).max() <= 1e-9
    assert np.abs(a["tangents"] - b["tangents"]).max() <= 1e-9
    order = [tuned.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    assert np.abs(b["positions"][0][:, order] - arr["positions_tight"]).max() <= POS_TOL_MM


# ---------------------------------------------------------------------------------------------
# Lean kernel instantiation (positions + solver statistics only): its own predictor (extrapolation
# of the solution history, no tangents carried through the factorisation) and the short slice.
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", SWEEP_CASES + ["c1_shim_plus2mm", "c4_tbar_heave_shim_roll", "c4_tbar_heave_shim_bump"])
def test_lean_instantiation_matches_reference_tight_run(case):
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog, values = _program(sus, sweep)
    out = emu_solve(prog, _nominal(sus, prog), values, lean=True)
    assert out["status"][0] == 0 and out["failed_step"][0] == -1
    order = [prog.out_keys.index(key_from_name(n)) for n in meta["point_keys"]]
    assert np.abs(out["positions"][0][:, order] - arr["positions_tight"]).max() <= POS_TOL_MM
    assert out["max_residual"].max() < 1e-5
    # the predictor pays off: fewer evaluations than the plain warm start, same answer
    plain = emu_solve(prog, _nominal(sus, prog), values, lean=True, use_predictor=0)
    assert np.abs(plain["positions"] - out["positions"]).max() < 1e-8
    assert out["iters"].sum() < plain["iters"].sum()


def test_lean_instantiation_failure_flags_match_reference():
    cases = json.load(open(os.path.join(GOLDEN, "failures.json")))
    check_failure_flags(lambda prog, hp, values: emu_solve(prog, hp, values, lean=True), cases)
