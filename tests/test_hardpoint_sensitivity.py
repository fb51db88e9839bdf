"""Hardpoint sensitivities (d position / d hardpoint coordinate at every accepted state).

CPU tests run the lane emulation of the device core; ``-m gpu`` tests run the C ABI on a device.

Checks:
- the device's own finite differences: Richardson-extrapolated central differences of positions
  solved at p +- h e_k, p +- 2h e_k with tightened tolerances, against the sensitivity at p;
- invariants: fixed output points give exactly e_k; on topologies whose targets are all relative and
  whose explicit constants do not depend on where the mechanism sits, a common translation of every
  hardpoint translates every output point; failed steps are NaN;
- requesting the output leaves every other output bit-identical, and a sensitivity-row subset
  reproduces the corresponding rows of the full set bit for bit.
"""

from __future__ import annotations

import numpy as np
import pytest

from helpers import SWEEP_CASES, UsageError, authored_positions, build_case, emu_solve, generic_mechanism, load_golden
from test_batches import batch_inputs, compile_batch

# Shim-free sweeps plus the C1 corners, whose camber shim sits at its design thickness (solved without
# the shim records, as BatchSolver does).
CASES = [c for c in SWEEP_CASES if not c.startswith("c4_tbar_heave")]
FULL_OUTPUTS = ("positions", "status", "failed_step", "iters", "max_residual", "tangents", "velocities",
                "tangent_health", "metrics", "design", "diagnostics", "jumps", "worst_row")


def compile_case(name: str, sensitivity_inputs=None):
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_suspension
    meta, _ = load_golden(name)
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep, with_shims=False, sensitivity_inputs=sensitivity_inputs)
    auth = authored_positions(sus)
    hp = np.concatenate([auth[k] for k in prog.in_keys])[None]
    _, values = sweep_target_values(sweep)
    return prog, hp, np.asarray(values, dtype=np.float64)


def generic_case():
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_topology
    state, cons, sweep, manager, _, _ = generic_mechanism()
    heads, values = sweep_target_values(sweep)
    prog = compile_topology(state, cons, manager.spec, heads)
    hp = np.concatenate([state.positions[k].data for k in prog.in_keys])[None]
    return prog, hp, np.asarray(values, dtype=np.float64)


def richardson_fd(prog, hp, values, coords, h):
    """d positions / d p_k by Richardson extrapolation of central differences at h and 2h, solved
    at tightened tolerances: [n_steps, len(coords), n_out, 3]."""
    rows = []
    for k in coords:
        for d in (h, -h, 2 * h, -2 * h):
            q = hp[0].copy()
            q[k] += d
            rows.append(q)
    out = emu_solve(prog, np.array(rows), values, step_tol=1e-13, coarse_tol=1e-3, fine_tol=1e-10,
                    want_health=False)
    assert (out["status"] == 0).all()
    p = out["positions"].reshape(len(coords), 4, *out["positions"].shape[1:])
    d1 = (p[:, 0] - p[:, 1]) / (2 * h)
    d2 = (p[:, 2] - p[:, 3]) / (4 * h)
    return ((4 * d1 - d2) / 3).transpose(1, 0, 2, 3)


# Bar per entry, relative to max(1, |S|).  Richardson leaves a truncation error of order
# h^4 |d^5 x/dp^5| / 30 (below 1e-9 at h = 1e-2 mm: the result moves by less than 2e-10 between h = 2.5e-3
# and 4e-2); the tightened solve leaves every position within ~1e-12 mm of the root, which the difference
# amplifies by 1/h -> 1e-10.  The Gauss-Newton sensitivity drops sum_i r_i Hess(r_i): where the
# least-squares rows are not all zero at the solution (the softnorm rows leave |r| ~ 1e-6 on overdetermined
# systems) the exact derivative differs from it by a term proportional to max|r|; with row curvatures of
# order 1/mm that is <= max|r| x 1/mm.  Bar: FD_FLOOR + max|r| of the state (1/mm).
FD_STEP_MM = 1e-2
FD_FLOOR = 2e-9


def check_fd(prog, hp, values, n_coords=8):
    out = emu_solve(prog, hp, values, want_hardpoint_sensitivity=True)
    assert (out["status"] == 0).all()
    sens = out["hardpoint_sensitivity"][0]
    k_all = len(prog.sensitivity_inputs)
    coords = sorted(set(np.linspace(0, k_all - 1, n_coords).round().astype(int)))
    fd = richardson_fd(prog, hp, values, coords, FD_STEP_MM)
    got = sens[:, coords]
    err = np.abs(got - fd) / np.maximum(1.0, np.abs(fd))
    bar = FD_FLOOR + out["max_residual"][0][:, None, None, None]
    assert np.isfinite(got).all()
    assert (err <= bar).all(), ((err / bar).max(), np.unravel_index((err / bar).argmax(), err.shape))
    return (err / bar).max()


@pytest.mark.parametrize("name", CASES)
def test_matches_finite_differences_emu(name):
    prog, hp, values = compile_case(name)
    check_fd(prog, hp, values)


def test_generic_mechanism_matches_finite_differences_emu():
    prog, hp, values = generic_case()
    check_fd(prog, hp, values, n_coords=12)


def translation_invariant(prog) -> bool:
    """Every target relative and every explicit constant independent of where the mechanism sits."""
    from open_kinematics_b200.core.topology import D, FAMILY_CODE
    rows = prog.section("OKIN_S_ROW").reshape(-1, D["OKIN_ROW_STRIDE"])
    placed = {FAMILY_CODE[f] for f in ("linear_point", "midpoint_on_plane", "point_on_line", "target")}
    return not any(r[D["OKIN_R_RULE"]] == D["OKIN_RULE_EXPLICIT"] and r[D["OKIN_R_FAM"]] in placed for r in rows)


# The T-bar axles place rows with explicit absolute constants (fixed-axis / plane rows).
QUALIFY = set(CASES) - {"c4_tbar_roll", "c4_tbar_bump"}


@pytest.mark.parametrize("name", CASES)
def test_invariants_emu(name):
    prog, hp, values = compile_case(name)
    out = emu_solve(prog, hp, values, want_hardpoint_sensitivity=True)
    sens = out["hardpoint_sensitivity"][0]          # [S, K, n_out, 3]
    from open_kinematics_b200.core.topology import D
    kind = prog.section("OKIN_S_POINT_KIND")
    pidx = {k: i for i, k in enumerate(prog.point_keys)}
    for o, key in enumerate(prog.out_keys):
        if kind[pidx[key]] != D["OKIN_PT_FIXED"]:
            continue
        for k, (ikey, axis) in enumerate(prog.sensitivity_inputs):
            expect = np.zeros(3)
            if ikey == key:
                expect[axis] = 1.0
            assert (sens[:, k, o] == expect).all(), (name, key, k)
    assert translation_invariant(prog) == (name in QUALIFY), name
    if translation_invariant(prog):
        for axis in range(3):
            rows = [k for k, (_, a) in enumerate(prog.sensitivity_inputs) if a == axis]
            total = sens[:, rows].sum(axis=1)
            expect = np.zeros(3)
            expect[axis] = 1.0
            assert np.abs(total - expect).max() <= 1e-12, (name, axis, np.abs(total - expect).max())


def test_failed_steps_are_nan_emu():
    from open_kinematics_b200.core.solver import sweep_target_values
    meta, arr = load_golden("fail256_c3")
    sus, sweep, prog = compile_batch(meta)
    hp, par = batch_inputs(meta, arr, prog, range(48))
    _, values = sweep_target_values(sweep)
    out = emu_solve(prog, hp, values, want_hardpoint_sensitivity=True)
    failed = np.flatnonzero(out["status"] != 0)
    assert failed.size > 0
    sens = out["hardpoint_sensitivity"]
    for i in range(len(hp)):
        f = int(out["failed_step"][i])
        ok = sens[i] if f < 0 else sens[i, :f]
        assert np.isfinite(ok).all()
        if f >= 0:
            assert np.isnan(sens[i, f:]).all()


@pytest.mark.parametrize("name", CASES + ["generic"])
def test_other_outputs_unchanged_emu(name):
    prog, hp, values = generic_case() if name == "generic" else compile_case(name)
    rng = np.random.default_rng(3)
    hp = hp + rng.normal(0.0, 0.3, (4, hp.shape[1]))
    base = emu_solve(prog, hp, values, want_health=True)
    with_sens = emu_solve(prog, hp, values, want_health=True, want_hardpoint_sensitivity=True)
    for key in FULL_OUTPUTS:
        a, b = base[key], with_sens[key]
        if a is None:
            assert b is None
            continue
        assert np.array_equal(a, b, equal_nan=True), (name, key)


def test_sensitivity_input_subset_emu():
    prog, hp, values = compile_case("c3_rocker_ubar_coilover_roll")
    pick = [prog.sensitivity_inputs[k] for k in (5, 0, 40, 77, 13, 2)]
    sub, _, _ = compile_case("c3_rocker_ubar_coilover_roll", sensitivity_inputs=pick)
    assert sub.sensitivity_inputs == pick
    full = emu_solve(prog, hp, values, want_hardpoint_sensitivity=True)["hardpoint_sensitivity"]
    part = emu_solve(sub, hp, values, want_hardpoint_sensitivity=True)["hardpoint_sensitivity"]
    assert np.array_equal(part, full[:, :, [5, 0, 40, 77, 13, 2]])
    with pytest.raises(ValueError):
        compile_case("c3_rocker_ubar_coilover_roll", sensitivity_inputs=[(prog.in_keys[0], 3)])


def test_shim_topology_is_refused_emu():
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_suspension
    meta, _ = load_golden("c4_tbar_heave_shim_roll")
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    assert prog.param_names
    hp = np.concatenate([authored_positions(sus)[k] for k in prog.in_keys])[None]
    _, values = sweep_target_values(sweep)
    with pytest.raises(UsageError):
        emu_solve(prog, hp, values, want_hardpoint_sensitivity=True)


def test_linearised_std():
    from open_kinematics_b200.core.sensitivity import linearised_std
    s = np.zeros((1, 2, 3, 1, 3))
    s[0, :, 0, 0, 0] = 2.0
    s[0, :, 1, 0, 0] = 1.0
    got = linearised_std(s, [0.5, 1.0, 7.0])
    assert np.allclose(got[0, :, 0, 0], np.sqrt(2.0))
    assert (got[..., 1:] == 0).all()
