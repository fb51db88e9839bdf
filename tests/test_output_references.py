"""Every per-state output beyond positions and metric rows -- tangent health, tangents, point
velocities, sweep diagnostics -- against plain references at the device's own solved states:

* tangent health and tangents: ``oracle.solve.state_tangents`` (SVD least squares on [J; pins]);
* velocities: the oracle's tangents, through ``update_derived(..., jac=True)`` for derived points;
* diagnostics: a numpy restatement of the reference's continuity check and topology columns,
  itself pinned to the reference's own report (tests/golden/diagnostics.*).

The CPU tests run the lane emulation of the device core on perturbed and failing golden batches;
the GPU tests run the same checks through the C ABI, plus properties of the batch machinery: a
multi-chunk host-buffer call with per-instance parameters and target tables, the device-buffer
entry point (calibration inside the call, no output cell left unwritten) and launch-shape
invariance."""

import json
import os

import numpy as np
import pytest

from helpers import (GOLDEN, authored_positions, build_case, build_suspension, emu_solve, key_from_name, load_golden,
                     oracle_problem)
from open_kinematics_b200.core.solver import sweep_target_values
from open_kinematics_b200.csrc_defs import D
from oracle.solve import ResidualComputer, design_setup, state_tangents, target_bases
from test_batches import batch_geometry, batch_inputs, compile_batch
from test_emu_core import POS_TOL_MM, check_flag_contract, reference_root_checker

# Tangent health stops its subspace iterations once the residual of the Ritz pair is below 1e-5 of
# the Ritz value (okin_tangent_health): the eigenvalue of A = J^T J is then within 1e-5 relative,
# so sigma_min is within 5e-6 and cond within 1e-5.  (Measured: below 1e-9 on every batch here.)
HEALTH_TOL = 1e-5
TANGENT_TOL = 1e-9      # tangents and velocities, relative to the largest entry of the state
DIAG_TOL = 1e-12        # diagnostic columns: a pure function of the position rows
REF_BATCHES = ["batch256_c1", "batch256_c2", "batch256_c3", "batch64_c4_roll"]
FAIL_BATCHES = ["fail256_c1", "fail256_c3", "fail128_c4_roll"]
GEOM_EPS = 1e-6         # csrc/okin_metrics.cuh OKIN_GEOM_EPS (the reference's degenerate-geometry guard)


# ---------------------------------------------------------------------------------------------
# Oracle at device states
# ---------------------------------------------------------------------------------------------
class StateOracle:
    """The reference's residual system of one instance, design constants from ``setup`` (authored
    pose; for a camber-shimmed model the setup pose the device solved, as reference_root_checker)."""

    def __init__(self, sus, sweep, prog, setup: dict, shimmed: bool):
        self.problem, _ = oracle_problem(sus, sweep, structure_only=shimmed)
        pos0, consts = design_setup(self.problem, setup)
        self.rc = ResidualComputer(self.problem, pos0, consts)
        self.bases = target_bases(self.problem, pos0)
        self.prog = prog
        self.cols = [prog.out_keys.index(k) for k in self.problem.free_order]

    def check_state(self, row, column, tangents, velocities, health) -> dict:
        """Errors of one accepted state's outputs (``row``: positions [n_out, 3]; ``column``: its
        target values) against the oracle; asserts the bars and returns the relative errors."""
        x = row[self.cols].reshape(-1)
        ref = state_tangents(self.problem, self.rc, x, self.bases + column)
        assert ref["rank"] == self.problem.n
        err = {}
        if health is not None:
            err["health"] = max(abs(health[0] / ref["smallest_singular_value"] - 1.0),
                                abs(health[1] / ref["condition_number"] - 1.0))
            assert err["health"] <= HEALTH_TOL, (health, ref["smallest_singular_value"], ref["condition_number"])
        t_ref = ref["tangents"]
        scale = max(1.0, np.abs(t_ref).max())
        if tangents is not None:
            err["tangents"] = np.abs(tangents - t_ref).max() / scale
            assert err["tangents"] <= TANGENT_TOL, err
        if velocities is not None:
            v_ref = self.velocities(x, t_ref)
            vscale = max(1.0, np.abs(v_ref).max())
            err["velocities"] = np.abs(velocities - v_ref).max() / vscale
            assert err["velocities"] <= TANGENT_TOL, err
        return err

    def velocities(self, x, t_ref) -> np.ndarray:
        """[n_targets, n_out, 3]: free points from the tangent columns, fixed points zero, derived
        points through the chain rule of the derived-point ops."""
        blocks = self.rc._refresh(x, jac=True)
        pb = self.problem
        out = np.zeros((t_ref.shape[0], len(self.prog.out_keys), 3))
        for i, key in enumerate(self.prog.out_keys):
            if key in pb.col:
                out[:, i] = t_ref[:, pb.col[key]: pb.col[key] + 3]
            elif key in blocks:
                for base, b in blocks[key].items():
                    out[:, i] += t_ref[:, pb.col[base]: pb.col[base] + 3] @ b.T
        return out


def check_instance(oracle, out, k, values, steps) -> dict:
    """Health, tangents and velocities of instance ``k`` of a batch result at ``steps`` (accepted
    states only); returns the worst relative error per output."""
    n_ok = values.shape[1] if out["status"][k] == 0 else int(out["failed_step"][k])
    worst = {}
    for s in steps:
        if s >= n_ok:
            continue
        health = None if out.get("tangent_health") is None else out["tangent_health"][k, s]
        err = oracle.check_state(out["positions"][k, s], values[:, s], out["tangents"][k, s],
                                 out["velocities"][k, s], health)
        for name, e in err.items():
            worst[name] = max(worst.get(name, 0.0), e)
    return worst


def sample_steps(n_steps: int) -> list:
    """First, middle, last and every third step in between."""
    return sorted(set(range(0, n_steps, 3)) | {n_steps // 2, n_steps - 1})


def golden_oracle(meta, arr, i, sweep, prog, design=None) -> StateOracle:
    """Oracle of row ``i`` of a golden batch; ``design``: the device's design pose of the instance
    (used for camber-shimmed models only)."""
    sus_i = build_suspension(batch_geometry(meta, arr["hardpoints"][i]))
    if prog.param_names:
        setup = {k: design[prog.out_keys.index(k)] for k in prog.in_keys}
        return StateOracle(sus_i, sweep, prog, setup, shimmed=True)
    return StateOracle(sus_i, sweep, prog, authored_positions(sus_i), shimmed=False)


def _merge(worst: dict, err: dict) -> None:
    for name, e in err.items():
        worst[name] = max(worst.get(name, 0.0), e)


# ---------------------------------------------------------------------------------------------
# Diagnostics restated in numpy (reference core/diagnostics.py:176-226, axle/mechanisms.py:119-163,
# :432-549)
# ---------------------------------------------------------------------------------------------
def continuity_reference(free_slots: list, positions: np.ndarray, n_ok: int) -> tuple:
    """``(columns[n_steps, 4], jumps[n_steps, n_free])`` of one instance: columns = jump count, worst
    displacement, its output slot and its threshold per step; jumps row 0 = each free point's
    threshold, row s = displacement into step s where it exceeded the threshold."""
    n_steps, nf = positions.shape[0], len(free_slots)
    cols = np.zeros((n_steps, 4))
    cols[:, 2] = -1.0
    jumps = np.zeros((n_steps, nf))
    if n_ok < 2:
        return cols, jumps
    p = positions[:n_ok][:, free_slots]
    step = p[1:] - p[:-1]
    d = np.sqrt(step[..., 0] * step[..., 0] + step[..., 1] * step[..., 1] + step[..., 2] * step[..., 2])
    thr = np.empty(nf)
    for k in range(nf):
        moved = d[:, k][d[:, k] > 0.0]
        thr[k] = max(5.0, 4.0 * (float(np.median(moved)) if moved.size else 0.0))
    jumps[0] = thr
    over = d > thr[None, :]
    jumps[1:n_ok][over] = d[over]
    for t in range(n_ok - 1):
        ks = np.flatnonzero(over[t])
        if ks.size:
            w = ks[np.argmax(d[t, ks])]          # first point of the largest displacement
            cols[t + 1] = [ks.size, d[t, w], free_slots[w], thr[w]]
    return cols, jumps


def _stp(o, a, b, c):
    return float((a - o) @ np.cross(b - o, c - o))


def topology_reference(prog, row: np.ndarray, design: np.ndarray) -> tuple:
    """({column: value}, flag bits) of the topology checks at one state (U-bar chirality and
    transmission margins); ``row`` / ``design``: positions [n_out, 3] at the state / design pose."""
    from open_kinematics_b200.core.enums import PointID as P
    from open_kinematics_b200.core.primitives.point_ref import PointRef, Side
    at = {k: row[i] for i, k in enumerate(prog.out_keys)}
    dsn = {k: design[i] for i, k in enumerate(prog.out_keys)}
    cols, flags = {}, 0
    axis_a, axis_b = PointRef(Side.CENTER, P.ARB_U_BAR_AXIS_A), PointRef(Side.CENTER, P.ARB_U_BAR_AXIS_B)
    for kind, side, label, col in prog.diagnostic_checks:
        key = lambda p: PointRef(side, p)   # noqa: E731
        if kind == "chirality":
            branch = [axis_a, axis_b, key(P.DROPLINK_ROCKER), key(P.DROPLINK_U_BAR)]
            a, b, r, u = (at[k] for k in branch)
            vol = _stp(a, b, r, u)
            scale = np.linalg.norm(b - a) * np.linalg.norm(r - a) * np.linalg.norm(u - a)
            margin = 0.0 if scale <= GEOM_EPS else vol / scale
            design_vol = _stp(*(dsn[k] for k in branch))
            code = 1.0 if abs(margin) <= GEOM_EPS else (2.0 if np.sign(vol) != np.sign(design_vol) else 0.0)
            flags |= {0.0: 0, 1.0: D["OKIN_DIAG_CHIRALITY_BOUNDARY"], 2.0: D["OKIN_DIAG_CHIRALITY_INVERTED"]}[code]
            cols.update({col: vol, col + 1: margin, col + 2: code})
        else:
            driver, joint, link_end = {
                "droplink @ DROPLINK_U_BAR": (key(P.DROPLINK_U_BAR), (axis_a, axis_b), key(P.DROPLINK_ROCKER)),
                "pushrod @ PUSHROD_INBOARD": (key(P.PUSHROD_INBOARD), (key(P.ROCKER_AXIS_A), key(P.ROCKER_AXIS_B)),
                                              key(P.PUSHROD_OUTBOARD)),
                "droplink @ DROPLINK_ROCKER": (key(P.DROPLINK_ROCKER), (key(P.ROCKER_AXIS_A), key(P.ROCKER_AXIS_B)),
                                               key(P.DROPLINK_U_BAR)),
            }[label]
            a, b = at[joint[0]], at[joint[1]]
            link = at[link_end] - at[driver]
            axis = b - a
            margin = np.nan
            if np.linalg.norm(axis) != 0.0 and np.linalg.norm(link) != 0.0:
                axis = axis / np.linalg.norm(axis)
                radius = at[driver] - a
                radius = radius - axis * (radius @ axis)
                tangent = np.cross(axis, radius)
                if np.linalg.norm(tangent) != 0.0:
                    margin = abs(link @ tangent) / (np.linalg.norm(link) * np.linalg.norm(tangent))
            if margin < 0.15:
                flags |= D["OKIN_DIAG_TRANSMISSION"]
            cols[col] = margin
    return cols, flags


def diagnostics_reference(prog, positions, design, status: int, failed: int) -> tuple:
    """``(diagnostics[n_steps, n_diag], jumps[n_steps, n_free])`` of one instance from its position
    rows, design pose and (status, failed step)."""
    n_steps = positions.shape[0]
    n_ok = n_steps if status == 0 else failed
    free_slots = [prog.out_keys.index(k) for k in prog.free_order]
    cont, jumps = continuity_reference(free_slots, positions, n_ok)
    diag = np.full((n_steps, len(prog.diagnostic_names)), np.nan)
    diag[:, 1:5] = cont
    for s in range(n_steps):
        flags = D["OKIN_DIAG_JUMP"] if cont[s, 0] > 0 else 0
        if s < n_ok:
            cols, topo_flags = topology_reference(prog, positions[s], design)
            for c, v in cols.items():
                diag[s, c] = v
            flags |= topo_flags
        elif s == failed:
            flags |= D["OKIN_DIAG_RESIDUAL"] if status == D["OKIN_STATUS_RESIDUAL_REJECTED"] else D["OKIN_DIAG_NOT_CONVERGED"]
        diag[s, 0] = flags
    return diag, jumps


def check_diagnostics(prog, out, k) -> float:
    """Device diagnostics / jumps of instance ``k`` against the restatement on its own position rows;
    returns the worst relative error of the value columns (counts, slots, codes, flags: exact)."""
    ref, ref_jumps = diagnostics_reference(prog, out["positions"][k], out["design"][k], int(out["status"][k]),
                                           int(out["failed_step"][k]))
    got = out["diagnostics"][k]
    assert np.array_equal(np.isnan(got), np.isnan(ref)), k
    exact = [0, 1, 3] + [c + 2 for kind, _, _, c in prog.diagnostic_checks if kind == "chirality"]
    assert np.array_equal(got[:, exact], ref[:, exact], equal_nan=True), (k, got[:, exact], ref[:, exact])
    fin = np.isfinite(ref)
    err = np.abs(got[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))
    jerr = np.abs(out["jumps"][k] - ref_jumps) / np.maximum(1.0, np.abs(ref_jumps))
    worst = float(max(err.max(initial=0.0), jerr.max(initial=0.0)))
    assert worst <= DIAG_TOL, (k, worst)
    return worst


def test_diagnostics_restatement_matches_reference_report():
    """The numpy restatement on the reference's own states reproduces the reference's thresholds,
    jump issues and U-bar columns (tests/golden/diagnostics.*)."""
    from open_kinematics_b200.core.topology import compile_suspension
    cases = json.load(open(os.path.join(GOLDEN, "diagnostics.json")))
    arrays = np.load(os.path.join(GOLDEN, "diagnostics.npz"))
    for label, rec in cases.items():
        sus, sweep = build_case(rec)
        prog = compile_suspension(sus, sweep)
        keys = [key_from_name(n) for n in rec["point_keys"]]
        ref_pos = arrays[label + "_positions"]
        positions = np.full((ref_pos.shape[0], len(prog.out_keys), 3), np.nan)
        for j, k in enumerate(keys):
            positions[:, prog.out_keys.index(k)] = ref_pos[:, j]
        auth = authored_positions(sus)
        design = np.array([auth.get(k, np.full(3, np.nan)) for k in prog.out_keys])
        diag, jumps = diagnostics_reference(prog, positions, design, 0, -1)
        thresholds = np.array([rec["thresholds"][k.name.lower()] for k in prog.free_order])
        assert np.abs(jumps[0] - thresholds).max() <= 1e-12 * thresholds.max(), label
        got = sorted((int(s), float(jumps[s, k])) for s, k in zip(*np.nonzero(jumps[1:] > 0.0)) for s in [s + 1])
        ref = sorted((i["step"], i["value"]) for i in rec["issues"] if i["category"] == "jump")
        assert [s for s, _ in got] == [s for s, _ in ref], label
        assert all(abs(v - rv) <= 1e-12 * rv for (_, v), (_, rv) in zip(got, ref)), label
        flagged = [s for s in range(len(diag)) if int(diag[s, 0]) & D["OKIN_DIAG_JUMP"]]
        assert flagged == sorted({i["step"] for i in rec["issues"] if i["category"] == "jump"}), label
        for cat, bit in (("chirality", D["OKIN_DIAG_CHIRALITY_BOUNDARY"] | D["OKIN_DIAG_CHIRALITY_INVERTED"]),
                         ("transmission", D["OKIN_DIAG_TRANSMISSION"])):
            steps = [s for s in range(len(diag)) if int(diag[s, 0]) & bit]
            assert steps == sorted({i["step"] for i in rec["issues"] if i["category"] == cat}), (label, cat)
        if "column_names" in rec:
            cols = [prog.diagnostic_names.index(n) for n in rec["column_names"]]
            ref_cols = arrays[label + "_columns"]
            assert np.abs(diag[:, cols] - ref_cols).max() <= 1e-12 * max(1.0, np.abs(ref_cols).max()), label


# ---------------------------------------------------------------------------------------------
# CPU: the lane emulation of the device core
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", REF_BATCHES)
def test_health_tangents_velocities_match_oracle_emu(name):
    """sigma_min / cond of the tangent system, dq/dt and every point velocity at the emulated
    device states of perturbed reference instances."""
    meta, arr = load_golden(name)
    sus, sweep, prog = compile_batch(meta)
    n = arr["hardpoints"].shape[0]
    rows = sorted({0, n // 3, n // 2, n - 1} | set(range(7, n, n // 6)))
    hp, par = batch_inputs(meta, arr, prog, rows)
    _, values = sweep_target_values(sweep)
    out = emu_solve(prog, hp, values, params=par, want_health=True)
    assert (out["status"] == 0).all()
    worst = {}
    for k, i in enumerate(rows):
        oracle = golden_oracle(meta, arr, i, sweep, prog, out["design"][k])
        _merge(worst, check_instance(oracle, out, k, values, sample_steps(values.shape[1])))
    assert set(worst) == {"health", "tangents", "velocities"}
    print(name, "worst relative error", worst)


def _emu_diagnostics(prog, hp, values, par=None):
    out = emu_solve(prog, hp, values, params=par)
    assert out["diagnostics"] is not None
    return out


@pytest.mark.parametrize("name", FAIL_BATCHES)
def test_diagnostics_match_restatement_on_failure_batches_emu(name):
    """Failing instances (n_ok < n_steps): continuity on the accepted prefix, status flag at the failed
    step, NaN topology columns after it."""
    meta, arr = load_golden(name)
    sus, sweep, prog = compile_batch(meta)
    n = arr["hardpoints"].shape[0]
    hp, par = batch_inputs(meta, arr, prog, range(n))
    _, values = sweep_target_values(sweep)
    out = _emu_diagnostics(prog, hp, values, par)
    worst = max(check_diagnostics(prog, out, k) for k in range(n))
    print(name, "worst diagnostics error", worst)


def _perturbed_rows(sus, prog, n, sigma=0.5, seed=3):
    from test_emu_core import _nominal
    nominal = _nominal(sus, prog)[0]
    rng = np.random.default_rng(seed)
    hp = nominal[None, :] + rng.normal(0.0, sigma, (n, nominal.size)) * (nominal != 0)[None, :]
    hp[0] = nominal
    return hp


@pytest.mark.parametrize("label", ["c1_uneven_bump", "c3_uneven_roll", "c3_roll_pm45"])
def test_diagnostics_match_restatement_on_uneven_sweeps_emu(label):
    from open_kinematics_b200.core.topology import compile_suspension
    rec = json.load(open(os.path.join(GOLDEN, "diagnostics.json")))[label]
    sus, sweep = build_case(rec)
    prog = compile_suspension(sus, sweep)
    _, values = sweep_target_values(sweep)
    out = _emu_diagnostics(prog, _perturbed_rows(sus, prog, 12), values)
    assert (out["status"] == 0).all()
    if rec["issues"]:
        assert (out["diagnostics"][:, :, 1] > 0).any()     # the uneven step is flagged
    print(label, "worst diagnostics error", max(check_diagnostics(prog, out, k) for k in range(12)))


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
ALL_OUTPUTS = dict(want_positions=True, want_tangents=True, want_velocities=True, want_health=True,
                   want_metrics=True, want_design=True, want_diagnostics=True, want_worst_row=True)


def gpu_all_outputs(prog, hp, values, params=None, instance_targets=None, topo=None, **kw):
    from open_kinematics_b200 import _lib
    own = topo is None
    topo = _lib.DeviceTopology(prog) if own else topo
    try:
        want = dict(ALL_OUTPUTS, want_metrics=bool(prog.metric_names), want_diagnostics=bool(prog.diagnostic_names))
        want.update(kw)
        return topo.solve_batch(hp, values, params=params, instance_targets=instance_targets, **want)
    finally:
        if own:
            topo.close()


def _assert_same(a: dict, b: dict, label) -> None:
    for name, x in a.items():
        if x is None:
            assert b[name] is None, (label, name)
            continue
        assert np.array_equal(x, b[name], equal_nan=True), (label, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", REF_BATCHES)
def test_health_tangents_velocities_match_oracle_gpu(name):
    meta, arr = load_golden(name)
    sus, sweep, prog = compile_batch(meta)
    n = arr["hardpoints"].shape[0]
    rows = sorted({0, n // 3, n // 2, n - 1} | set(range(7, n, n // 6)))
    hp, par = batch_inputs(meta, arr, prog, rows)
    _, values = sweep_target_values(sweep)
    out = gpu_all_outputs(prog, hp, values, params=par)
    assert (out["status"] == 0).all()
    worst = {}
    for k, i in enumerate(rows):
        _merge(worst, check_instance(golden_oracle(meta, arr, i, sweep, prog, out["design"][k]), out, k, values,
                                     sample_steps(values.shape[1])))
        if prog.diagnostic_names:
            worst["diagnostics"] = max(worst.get("diagnostics", 0.0), check_diagnostics(prog, out, k))
    print(name, "worst relative error", worst)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAIL_BATCHES)
def test_diagnostics_match_restatement_on_failure_batches_gpu(name):
    meta, arr = load_golden(name)
    sus, sweep, prog = compile_batch(meta)
    n = arr["hardpoints"].shape[0]
    hp, par = batch_inputs(meta, arr, prog, range(n))
    _, values = sweep_target_values(sweep)
    out = gpu_all_outputs(prog, hp, values, params=par)
    print(name, "worst diagnostics error", max(check_diagnostics(prog, out, k) for k in range(n)))


@pytest.mark.gpu
@pytest.mark.parametrize("n_steps,n_inst", [(None, 12), (301, 2500), (701, 1500)])
def test_diagnostics_match_restatement_on_long_sweeps_gpu(n_steps, n_inst):
    """The uneven C3 roll refined to ~300 / ~700 steps: the continuity pass runs with 2-warp and 1-warp
    CTAs, and with more instances than its grid has warps (grid-stride loop)."""
    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.topology import compile_suspension
    rec = json.load(open(os.path.join(GOLDEN, "diagnostics.json")))["c3_uneven_roll"]
    sus, sweep = build_case(rec)
    prog = compile_suspension(sus, sweep)
    _, values = sweep_target_values(sweep)
    if n_steps is not None:
        u = np.linspace(0.0, values.shape[1] - 1, n_steps)
        values = np.array([np.interp(u, np.arange(values.shape[1]), v) for v in values])
    hp = _perturbed_rows(sus, prog, n_inst)
    topo = _lib.DeviceTopology(prog)
    try:
        out = topo.solve_batch(hp, values, want_design=True, want_diagnostics=True)
        if n_steps is not None:
            # the CTA shape the continuity launch picks for this sweep length (okin_abi.cu launch())
            per_warp = (32 * ((n_steps - 1) | 1) + 64) * 8
            assert 4 * per_warp > 227 * 1024 and (2 * per_warp <= 227 * 1024) == (n_steps < 400)
            assert n_inst > 148 * 8 * (2 if n_steps < 400 else 1)
    finally:
        topo.close()
    assert (out["status"] == 0).mean() > 0.9
    rng = np.random.default_rng(1)
    rows = sorted({0, n_inst - 1} | set(rng.choice(n_inst, min(n_inst, 40), replace=False).tolist()))
    print(n_steps, "worst diagnostics error", max(check_diagnostics(prog, out, k) for k in rows))


CHUNK = 32768
BOUNDARY_ROWS = [0, CHUNK - 1, CHUNK, 2 * CHUNK - 1, 2 * CHUNK, 3 * CHUNK - 1, 3 * CHUNK]


def _c4_batch_scale_inputs():
    """N = 3 chunks + 123 shimmed C4 roll instances, each with its own params and target table; the
    reference-solved instances of batch64_c4_roll / fail128_c4_roll, a NaN row and a collapsed row
    planted at the chunk boundaries and at random rows."""
    meta_b, arr_b = load_golden("batch64_c4_roll")
    meta_f, arr_f = load_golden("fail128_c4_roll")
    sus, sweep, prog = compile_batch(meta_b)
    _, values = sweep_target_values(sweep)
    assert meta_f["geometry"] == meta_b["geometry"] and meta_f["hp_names"] == meta_b["hp_names"]
    _, values_f = sweep_target_values(compile_batch(meta_f)[1])
    n = 3 * CHUNK + 123
    rng = np.random.default_rng(17)
    from test_emu_core import _nominal
    nominal = _nominal(sus, prog)[0]
    hp = nominal[None, :] + rng.normal(0.0, 0.5, (n, nominal.size)) * (nominal != 0)[None, :]
    params = np.repeat(prog.param_default[None, :], n, axis=0)
    setup_cols = [j for j, name in enumerate(prog.param_names) if name.endswith("setup_thickness")]
    params[:, setup_cols] = rng.uniform(29.5, 30.5, (n, len(setup_cols)))
    tables = values[None, :, :] * rng.uniform(0.6, 1.0, (n, 1, 1))
    hp_b, par_b = batch_inputs(meta_b, arr_b, prog, range(arr_b["hardpoints"].shape[0]))
    hp_f, _ = batch_inputs(meta_f, arr_f, prog, range(arr_f["hardpoints"].shape[0]))   # default shim
    plant = ([("batch", i, hp_b[i], par_b[i], values) for i in range(len(hp_b))]
             + [("fail", i, hp_f[i], prog.param_default, values_f) for i in range(len(hp_f))])
    free = np.setdiff1d(np.arange(n), BOUNDARY_ROWS + [n - 1])
    where = BOUNDARY_ROWS + [n - 1] + rng.choice(free, len(plant) + 2 - 8, replace=False).tolist()
    planted = {}
    for row, (kind, i, h, p, v) in zip(where, plant):
        hp[row], params[row], tables[row] = h, p, v
        planted[row] = (kind, i)
    nan_row, zero_row = where[len(plant)], where[len(plant) + 1]
    hp[nan_row] = np.nan
    hp[zero_row] = 0.0
    return dict(meta_b=meta_b, arr_b=arr_b, meta_f=meta_f, arr_f=arr_f, sus=sus, sweep=sweep, prog=prog,
                hp=hp, params=params, tables=tables, planted=planted, nan_row=nan_row, zero_row=zero_row, rng=rng)


@pytest.mark.gpu
def test_multi_chunk_batch_with_per_instance_params_and_targets_gpu():
    """The full kernel over more than three pipeline chunks with every output requested: planted
    reference instances meet the position and flag-contract bars wherever they sit, every planted
    instance and a random sample are bit-identical to the instance solved alone, and a sample
    passes the health / tangent / velocity / diagnostics references."""
    from open_kinematics_b200 import _lib
    b = _c4_batch_scale_inputs()
    prog, hp, params, tables = b["prog"], b["hp"], b["params"], b["tables"]
    n = hp.shape[0]
    topo = _lib.DeviceTopology(prog)
    try:
        out = gpu_all_outputs(prog, hp, tables[0], params=params, instance_targets=tables, topo=topo)
        assert out["status"][b["nan_row"]] != 0 and out["status"][b["zero_row"]] != 0
        assert (out["status"] == 0).mean() > 0.9
        # planted reference instances
        order = [prog.out_keys.index(key_from_name(k)) for k in b["meta_b"]["point_keys"]]
        for row, (kind, i) in b["planted"].items():
            if kind == "batch":
                arr = b["arr_b"]
                assert out["status"][row] == 0, row
                got = out["positions"][row][arr["steps"]][:, order]
                assert np.abs(got - arr["positions_tight"][i]).max() <= POS_TOL_MM, (row, i)
            else:
                arr, meta = b["arr_f"], b["meta_f"]
                checker = None
                if arr["status"][i] == 1:
                    sus_i = build_suspension(batch_geometry(meta, arr["hardpoints"][i]))
                    setup = {k: out["design"][row][prog.out_keys.index(k)] for k in prog.in_keys}
                    checker = reference_root_checker(sus_i, b["sweep"], prog, authored_positions(sus_i), setup)
                check_flag_contract(f"fail128_c4_roll[{i}]@{row}", int(arr["status"][i]), int(arr["failed_step"][i]),
                                    int(out["status"][row]), int(out["failed_step"][row]), out["positions"][row],
                                    tables[row], checker)
        # every planted instance and ~300 random ones, solved alone
        rng = b["rng"]
        alone_rows = sorted(set(b["planted"]) | {b["nan_row"], b["zero_row"]} | set(rng.choice(n, 300, replace=False).tolist()))
        for row in alone_rows:
            one = gpu_all_outputs(prog, hp[row:row + 1], tables[row], params=params[row:row + 1],
                                  instance_targets=tables[row:row + 1], topo=topo)
            _assert_same(one, {name: (None if x is None else x[row:row + 1]) for name, x in out.items()}, row)
    finally:
        topo.close()
    # health / tangents / velocities / diagnostics on a sample
    worst = {}
    sample = sorted({BOUNDARY_ROWS[1], BOUNDARY_ROWS[2], n - 1} | set(rng.choice(n, 47, replace=False).tolist()))
    for row in sample:
        if out["status"][row] == 3:
            continue
        setup = {k: out["design"][row][prog.out_keys.index(k)] for k in prog.in_keys}
        oracle = StateOracle(b["sus"], b["sweep"], prog, setup, shimmed=True)
        _merge(worst, check_instance(oracle, out, row, tables[row], sample_steps(tables.shape[2])))
        worst["diagnostics"] = max(worst.get("diagnostics", 0.0), check_diagnostics(prog, out, row))
    print("batch scale worst relative error", worst)


@pytest.mark.gpu
def test_multi_device_split_of_multi_chunk_batch_gpu():
    from open_kinematics_b200 import _lib
    if _lib.device_count() < 2:
        pytest.skip("one visible device")
    b = _c4_batch_scale_inputs()
    prog = b["prog"]
    topo = _lib.DeviceTopology(prog)
    try:
        kw = dict(params=b["params"], instance_targets=b["tables"], topo=topo)
        one = gpu_all_outputs(prog, b["hp"], b["tables"][0], devices=[0], **kw)
        two = gpu_all_outputs(prog, b["hp"], b["tables"][0], devices=[0, 1], **kw)
    finally:
        topo.close()
    _assert_same(one, two, "devices [0, 1]")


SENTINEL = -7.0e300


@pytest.mark.gpu
@pytest.mark.parametrize("full", [False, True])
def test_device_buffer_entry_point_writes_every_cell(full, monkeypatch):
    """okin_solve_batch_device on torch tensors, as bench.py calls it, on a fresh topology whose lean
    family is calibrated inside the call: no output cell keeps its sentinel, and the result equals the
    host-buffer path bit for bit."""
    import ctypes

    import torch

    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.sweep import BatchSolver
    monkeypatch.delenv("OKIN_LEAN_REGS", raising=False)
    meta, _ = load_golden("c3_rocker_ubar_coilover_roll")
    sus, sweep = build_case(meta)
    solver = BatchSolver(sus, sweep, tune_layout=True)
    prog, topo = solver.program, solver.topology
    try:
        n = 1 << 16
        nominal = solver.nominal_hardpoints()
        rng = np.random.default_rng(8)
        hp = nominal[None, :] + rng.normal(0.0, 0.5, (n, nominal.size)) * (nominal != 0)[None, :]
        values = solver.values
        nt, S = values.shape
        dev = torch.device("cuda", 0)
        shapes = {"positions": ((n, S, prog.n_out, 3), torch.float64), "status": ((n,), torch.int32),
                  "failed_step": ((n,), torch.int32), "iters": ((n, S), torch.int32),
                  "max_residual": ((n, S), torch.float64), "design": ((n, prog.n_out, 3), torch.float64),
                  "worst_row": ((n,), torch.int32)}
        if full:
            shapes.update({"tangents": ((n, S, nt, prog.n_unknowns), torch.float64),
                           "velocities": ((n, S, nt, prog.n_out, 3), torch.float64),
                           "tangent_health": ((n, S, 2), torch.float64),
                           "metrics": ((n, S, len(prog.metric_names)), torch.float64),
                           "diagnostics": ((n, S, len(prog.diagnostic_names)), torch.float64),
                           "jumps": ((n, S, prog.n_unknowns // 3), torch.float64)})
        bufs = {name: torch.full(shape, SENTINEL if dt == torch.float64 else -12345, dtype=dt, device=dev)
                for name, (shape, dt) in shapes.items()}
        d_hp = torch.tensor(hp, device=dev)
        d_tv = torch.tensor(values, device=dev)
        io = _lib.BatchIO.of(hardpoints=d_hp.data_ptr(), target_values=d_tv.data_ptr(),
                             **{name: t.data_ptr() for name, t in bufs.items()})
        stream = torch.cuda.Stream(device=dev)
        cfg = _lib.default_cfg()
        _lib.check(_lib.load().okin_solve_batch_device(topo.handle, ctypes.byref(cfg), 0,
                                                       ctypes.c_void_p(stream.cuda_stream), n, S, ctypes.byref(io)),
                   "okin_solve_batch_device")
        stream.synchronize()
        if not full:
            assert topo.lean_calibration(0)["registers"] in (128, 168)     # calibrated inside the call
        got = {name: t.cpu().numpy() for name, t in bufs.items()}
        del bufs
        for name, x in got.items():
            assert not (x == (SENTINEL if x.dtype == np.float64 else -12345)).any(), name
        assert (got["status"] == 0).mean() > 0.99
        host = topo.solve_batch(hp, values, want_positions=True, want_design=True, want_worst_row=True,
                                want_tangents=full, want_velocities=full, want_health=full, want_metrics=full,
                                want_diagnostics=full)
        for name, x in got.items():
            assert np.array_equal(x, host[name], equal_nan=True), name
    finally:
        solver.close()


@pytest.mark.gpu
@pytest.mark.parametrize("full", [False, True])
def test_launch_shape_does_not_change_results(full, monkeypatch):
    """A heterogeneous batch (failing instances + sigma = 0.5 perturbations) solved with 1-, 3- and
    5-warp CTAs gives the default shape's results bit for bit."""
    from open_kinematics_b200 import _lib
    meta, arr = load_golden("fail256_c3")
    sus, sweep, prog = compile_batch(meta)
    hp_f, _ = batch_inputs(meta, arr, prog, range(arr["hardpoints"].shape[0]))
    hp = np.concatenate([hp_f, _perturbed_rows(sus, prog, 744, seed=12)])
    _, values = sweep_target_values(sweep)
    want = dict(ALL_OUTPUTS) if full else dict(want_positions=True, want_design=True, want_worst_row=True)

    def solve(warps):
        if warps is None:
            monkeypatch.delenv("OKIN_WARPS_PER_CTA", raising=False)
        else:
            monkeypatch.setenv("OKIN_WARPS_PER_CTA", str(warps))
        topo = _lib.DeviceTopology(prog)
        try:
            if warps is not None:
                assert topo.launch_geometry(len(hp))["block"] == 32 * warps
            return topo.solve_batch(hp, values, **want)
        finally:
            topo.close()
    base = solve(None)
    assert (base["status"] != 0).any()
    for warps in (1, 3, 5):
        _assert_same(solve(warps), base, warps)
