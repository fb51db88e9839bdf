"""Sweep orchestration (reference core/sweep.py:35-65) and its batched counterpart."""

from __future__ import annotations

from collections import OrderedDict
from dataclasses import dataclass

import numpy as np

from .. import _lib
from .metrics.main import rows_from_columns
from .points.derived.manager import DerivedPointsManager
from .sensitivity import (STATE_MATCH_TOL_MM, TangentField, TangentSolveInfo, fields_from_velocities,  # noqa: F401
                          measured_targets, solve_info_from_health)
from .solver import (SolverConfig, SolverInfo, convert_targets_to_absolute, solve_suspension_sweep,  # noqa: F401
                     sweep_target_values)
from .targeting import SweepConfig, validate_sweep_controls
from .topology import TopologyProgram, compile_topology


def solve_sweep(suspension, sweep_config: SweepConfig) -> tuple:
    """Single-instance sweep: same call and results as reference ``solve_sweep``."""
    validate_sweep_controls(sweep_config, suspension.actuator_dofs())
    manager = DerivedPointsManager(suspension.derived_spec())
    return solve_suspension_sweep(
        initial_state=suspension.initial_state(),
        constraints=suspension.constraints(),
        sweep_config=sweep_config,
        derived_manager=manager,
    )


@dataclass
class BatchSweepResult:
    """Arrays for a batch of hardpoint-perturbed instances of one topology.

    positions    [n_instances, n_steps, n_out_points, 3]  (NaN from the failed step on)
    status       [n_instances]  0 ok | 1 not converged | 2 residual rejected | 3 invalid geometry
    failed_step  [n_instances]  -1 or first failed step
    nfev         [n_instances, n_steps]
    max_residual [n_instances, n_steps]
    tangents     [n_instances, n_steps, n_targets, n_unknowns] or None
    metrics      [n_instances, n_steps, n_metrics] or None; columns = ``metric_names`` (the
                 reference's flat export order), NaN where the reference yields None
    """

    program: TopologyProgram
    positions: np.ndarray | None
    status: np.ndarray
    failed_step: np.ndarray
    nfev: np.ndarray
    max_residual: np.ndarray
    tangents: np.ndarray | None
    metrics: np.ndarray | None = None
    velocities: np.ndarray | None = None       # [n_instances, n_steps, n_targets, n_out_points, 3]
    tangent_health: np.ndarray | None = None   # [n_instances, n_steps, 2] (sigma_min, cond)
    diagnostics: np.ndarray | None = None      # [n_instances, n_steps, n_diagnostics]; ``diagnostic_names``
    jumps: np.ndarray | None = None            # [n_instances, n_steps, n_free]; row 0 = thresholds
    worst_row: np.ndarray | None = None        # [n_instances] device row owning max|r| at the failed step, or -1
    design: np.ndarray | None = None           # [n_instances, n_out_points, 3] design (setup) pose
    # [n_instances, n_steps, n_sens, n_out_points, 3] d position / d hardpoint coordinate; row k is
    # ``sensitivity_inputs[k]`` = (input point key, axis)
    hardpoint_sensitivity: np.ndarray | None = None
    sensitivity_inputs: list | None = None

    _BUFFERS = (("positions", "positions"), ("status", "status"), ("failed_step", "failed_step"), ("nfev", "iters"),
                ("max_residual", "max_residual"), ("tangents", "tangents"), ("metrics", "metrics"),
                ("velocities", "velocities"), ("tangent_health", "tangent_health"), ("diagnostics", "diagnostics"),
                ("jumps", "jumps"), ("worst_row", "worst_row"), ("design", "design"),
                ("hardpoint_sensitivity", "hardpoint_sensitivity"))

    def buffers(self) -> dict:
        """The arrays keyed like ``DeviceTopology.solve_batch``'s result (for ``solve(out=...)`` reuse)."""
        return {abi: getattr(self, field) for field, abi in self._BUFFERS}

    def describe_worst_residual(self, instance: int, constraints: list, heads: list) -> str | None:
        """Text of the reference's "Worst residual row" (describe_worst_residual, solver.py:640-651)
        for a failed instance; None when the instance did not fail or ``worst_row`` was not requested."""
        if self.worst_row is None or int(self.worst_row[instance]) < 0:
            return None
        source = self.program.row_source[int(self.worst_row[instance])]
        if source[0] == "target":
            head = heads[source[1]]
            return f"target on point '{getattr(head.point_id, 'name', str(head.point_id))}' (direction {head.direction})"
        from .solver import describe_constraint
        return f"constraint {describe_constraint(constraints[source[1]])}"

    @property
    def point_keys(self) -> list:
        return self.program.out_keys

    @property
    def metric_names(self) -> list:
        return self.program.metric_names

    @property
    def diagnostic_names(self) -> list:
        return self.program.diagnostic_names


class BatchSolver:
    """A topology compiled once and resident on the device(s); solves any number of
    hardpoint sets of that topology.  Design constants (link lengths, upright angle,
    signed volumes, rack line point, strut clamp offset) are recomputed per instance on
    the device from that instance's hardpoints (reference recomputes them in
    ``Suspension.constraints()``, core/sweep.py:58-63)."""

    def __init__(self, suspension, sweep_config: SweepConfig, output_points=None, tune_layout: bool = False,
                 sensitivity_inputs=None):
        """``tune_layout``: spend a few seconds at compile time placing the factor blocks so that the
        kernel's shared-memory accesses hit fewer bank conflicts (core/layout_tuning.py); worth it for
        large batches, results are unchanged.  ``sensitivity_inputs``: the ``(input point key, axis)``
        hardpoint coordinates ``solve(want_hardpoint_sensitivity=True)`` differentiates by (default all)."""
        validate_sweep_controls(sweep_config, suspension.actuator_dofs())
        self.suspension = suspension
        self.heads, self.values = sweep_target_values(sweep_config)
        from .diagnostics_program import build_diagnostic_program
        from .metrics_program import build_metric_program
        from .shim_program import shim_records
        state, constraints = suspension.structure()

        def compile_with(shims):
            return compile_topology(
                state, constraints, suspension.derived_spec(), self.heads,
                output_points=output_points, design_rules=True,
                metrics=(lambda pidx: build_metric_program(suspension, self.heads, pidx))
                if suspension.config is not None else None,
                shims=shims,
                diagnostics=lambda pidx, design_pts: build_diagnostic_program(suspension, pidx, design_pts),
                tune_layout=tune_layout, sensitivity_inputs=sensitivity_inputs,
            )

        shims = shim_records(suspension)
        self.program = compile_with(shims)
        self.topology = _lib.DeviceTopology(self.program)
        # Hardpoint sensitivities do not differentiate the camber-shim pre-solve.  A shim at its design
        # thickness leaves the design pose as authored (okin_shim_presolve skips a thickness change below
        # OKIN_GEOM_EPS = 1e-6 mm), so such a model is solved for sensitivities by the same topology without
        # its shim records.
        self._sens_shims_inactive = all(abs(sh["params"][9] - sh["params"][10]) < 1e-6 for sh in shims)
        self._compile_without_shims = lambda: compile_with(None)
        self._sens_topology = None

    def nominal_hardpoints(self) -> np.ndarray:
        """Authored positions of the input points, shape ``[n_in*3]`` (input slot order)."""
        authored = self.authored_positions()
        return np.array([authored[k].data for k in self.program.in_keys]).reshape(-1)

    def authored_positions(self) -> dict:
        sus = self.suspension
        if getattr(sus, "is_axle", False):
            from .enums import PointID
            from .primitives.point_ref import PointRef, Side
            out = {PointRef(side, k): p for side, corner in sus.corners.items() for k, p in corner.hardpoints.items()}
            for point, p in getattr(sus.anti_roll, "center_points", {}).items():
                out[PointRef(Side.CENTER, point)] = p
            for side, p in getattr(sus.anti_roll, "droplink_points", {}).items():
                arm = PointID.DROPLINK_U_BAR if PointRef(side, PointID.DROPLINK_U_BAR) in self.program.in_keys \
                    else PointID.DROPLINK_T_BAR
                out[PointRef(side, arm)] = p
            return out
        return dict(sus.hardpoints)

    def solve(self, hardpoints: np.ndarray, solver_config: SolverConfig = SolverConfig(), devices=None,
              want_positions: bool = True, want_tangents: bool = False,
              want_metrics: bool = False, params: np.ndarray | None = None, want_velocities: bool = False,
              want_health: bool = False, want_diagnostics: bool = False, want_design: bool = False,
              want_worst_row: bool = False, instance_targets: np.ndarray | None = None,
              out: BatchSweepResult | None = None, pinned: bool = False,
              want_hardpoint_sensitivity: bool = False) -> BatchSweepResult:
        """``params``: optional ``[n_instances, n_params]`` per-instance scalars in the order of
        ``program.param_names`` (camber-shim datums and thicknesses); default = the model's.
        ``instance_targets``: optional ``[n_instances, n_targets, n_steps]`` per-instance sweep tables
        (same meaning as the sweep's own values: relative displacement / absolute coordinate).
        ``devices``: CUDA device ids; the instance range is split evenly over them.
        ``out``: an earlier result of the same shape whose arrays are overwritten (no allocation);
        ``pinned``: allocate result arrays in page-locked host memory (slow to allocate, fast to fill:
        keep the result and pass it back as ``out``).
        ``want_hardpoint_sensitivity``: d position / d hardpoint coordinate of every output point at every
        state (``hardpoint_sensitivity``, rows named by ``sensitivity_inputs``), params held fixed; see
        DESIGN.md.  Not available with active camber shims (ValueError)."""
        cfg = _lib.default_cfg(residual_tol=float(solver_config.residual_tolerance))
        hp = np.asarray(hardpoints, dtype=np.float64)
        hp = hp.reshape(hp.shape[0], -1)
        topology = self.topology
        if want_hardpoint_sensitivity and self.program.param_names:
            if params is not None or not self._sens_shims_inactive:
                raise ValueError("Hardpoint sensitivities are not available with camber shims away from their "
                                 "design thickness (the shim pre-solve is not differentiated)")
            if self._sens_topology is None:
                self._sens_topology = _lib.DeviceTopology(self._compile_without_shims())
            topology = self._sens_topology
        res = topology.solve_batch(hp, self.values, cfg, devices=devices,
                                        want_positions=want_positions, want_tangents=want_tangents,
                                        want_metrics=want_metrics, params=params,
                                        want_velocities=want_velocities, want_health=want_health,
                                        want_diagnostics=want_diagnostics, want_design=want_design,
                                        want_worst_row=want_worst_row, instance_targets=instance_targets,
                                        out=out.buffers() if out is not None else None, pinned=pinned,
                                        **({"want_hardpoint_sensitivity": True} if want_hardpoint_sensitivity else {}))
        return BatchSweepResult(self.program, res["positions"], res["status"], res["failed_step"],
                                res["iters"], res["max_residual"], res["tangents"], res["metrics"],
                                res["velocities"], res["tangent_health"], res["diagnostics"], res["jumps"],
                                res.get("worst_row"), res.get("design"), res.get("hardpoint_sensitivity"),
                                list(self.program.sensitivity_inputs) if want_hardpoint_sensitivity else None)

    def study(self, sampling, n_instances: int, seed: int = 0, points=None, metrics=None, solver_quantities=(),
              histograms=None, bins: int = 64, solver_config: SolverConfig = SolverConfig(), devices=None):
        """Tolerance study (core/study.py): ``n_instances`` instances drawn by ``sampling``
        (a ``Sampling`` of this solver) from ``(seed, instance id)``, generated, solved and reduced on
        the device(s) ``devices`` (default ``[0]``).  Quantities: ``points`` (output point keys or
        names, or ``"all"``: ``<point>_{x,y,z}``), ``metrics`` (metric names or ``"all"``) and
        ``solver_quantities`` (``"solver_max_residual"``, ``"solver_nfev"``).  ``histograms``:
        optional ``{quantity: (lo, hi)}`` for every quantity, ``bins`` bins each.  Returns a
        ``StudyResult``; the result does not depend on ``devices``."""
        from .study import run_study
        return run_study(self, sampling, n_instances, seed, points, metrics, solver_quantities, histograms, bins,
                         solver_config, devices)

    def study_inputs(self, sampling, seed: int, ids, device: int = 0) -> tuple:
        """``(hardpoints [n, n_in*3], params [n, n_params])`` a study with ``sampling`` and ``seed``
        gives the instances ``ids``, ready for ``solve(hardpoints, params=params)``."""
        from .study import study_inputs
        return study_inputs(self, sampling, seed, ids, device)

    def pinned_hardpoints(self, n_instances: int, device: int = 0) -> np.ndarray:
        """Page-locked ``[n_instances, n_in*3]`` input array (fill it, pass it to ``solve``)."""
        return _lib.pinned_empty((n_instances, 3 * self.program.n_in), np.float64, device)

    def close(self) -> None:
        self.topology.close()
        if self._sens_topology is not None:
            self._sens_topology.close()


def solve_sweep_batch(suspension, sweep_config: SweepConfig, hardpoints: np.ndarray, **kwargs) -> BatchSweepResult:
    """One-shot batched solve (compile + solve + release)."""
    solver = BatchSolver(suspension, sweep_config, output_points=kwargs.pop("output_points", None))
    try:
        return solver.solve(hardpoints, **kwargs)
    finally:
        solver.close()


def compute_sweep_metrics_batch(suspension, sweep_config: SweepConfig, hardpoints: np.ndarray, **kwargs):
    """Batched counterpart of reference ``compute_sweep_metrics`` (core/sweep.py:144-173): solves
    the sweeps and returns ``(metric_names, metrics[n_instances, n_steps, n_metrics], result)``
    with tangents and derivative metrics evaluated on the device."""
    result = solve_sweep_batch(suspension, sweep_config, hardpoints, want_metrics=True, **kwargs)
    return result.metric_names, result.metrics, result


# ---------------------------------------------------------------------------------------------
# Single-instance facade: tangents, metrics and evaluation of already solved states
# (reference core/sweep.py:67-330).  The states are re-pinned on the device at their own target
# coordinates, so tangents and metrics are evaluated exactly where the reference evaluates them.
# ---------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class SweepTangents:
    per_step: list
    solve_infos: list


@dataclass(frozen=True)
class SweepMetricsResult:
    rows: list
    derivative_error: str | None = None
    tangent_solve_infos: list | None = None


@dataclass(frozen=True)
class EvaluatedSweep:
    states: list
    solver_stats: list
    metrics: SweepMetricsResult
    diagnostics: list

    def __post_init__(self) -> None:
        lengths = (len(self.states), len(self.solver_stats), len(self.metrics.rows))
        if len(set(lengths)) != 1:
            raise ValueError(
                "Evaluated sweep state, solver-stat, and metric counts must match: "
                f"{lengths[0]} states, {lengths[1]} solver stats, {lengths[2]} metric rows."
            )


def evaluate_states_on_device(suspension, heads: list, states: list, *, want_metrics: bool, ramp: int = 0):
    """Re-pin ``states`` on the device: a sweep whose targets (``heads``: point + direction) take the
    values the states themselves have.  ``ramp`` extra leading steps walk from the design pose to
    the first state (for isolated states far from design).  Returns ``(result, solver)`` with
    per-step arrays trimmed to ``len(states)``."""
    if not states:
        raise ValueError("No states to evaluate")
    pinned = [[measured_targets([h], st)[0] for st in states] for h in heads]
    if ramp:
        design = suspension.initial_state()
        base = measured_targets(heads, design)
        pinned = [[b._replace(value=b.value + (dim[0].value - b.value) * (k + 1) / (ramp + 1)) for k in range(ramp)]
                  + dim for b, dim in zip(base, pinned)]
    solver = BatchSolver(suspension, SweepConfig(pinned))
    try:
        res = solver.solve(solver.nominal_hardpoints()[None, :], want_velocities=True, want_health=True,
                           want_metrics=want_metrics and bool(solver.program.metric_names))
    finally:
        solver.close()
    if int(res.status[0]) != 0:
        raise RuntimeError(f"State evaluation failed at step {int(res.failed_step[0]) - ramp}: the states are not "
                           f"solutions of this suspension (device status {int(res.status[0])}).")
    out_keys = solver.program.out_keys
    for s, st in enumerate(states):
        given = np.array([st.positions[k].data for k in out_keys])
        drift = float(np.abs(res.positions[0, ramp + s] - given).max())
        if drift > STATE_MATCH_TOL_MM:
            raise RuntimeError(f"State evaluation failed: state {s} is {drift:.3g} mm away from the nearest "
                               "solution of this suspension.")
    return res, solver, ramp


def compute_sweep_tangents(suspension, sweep_config: SweepConfig, states: list) -> SweepTangents:
    """Tangent fields of every solved state (reference core/sweep.py:109-141)."""
    if not states:
        return SweepTangents(per_step=[], solve_infos=[])
    heads = [dim[0] for dim in sweep_config.target_sweeps]
    initial_state = suspension.initial_state()
    res, solver, ramp = evaluate_states_on_device(suspension, heads, states, want_metrics=False)
    prog = solver.program
    per_step, infos = [], []
    for s in range(len(states)):
        step_targets = convert_targets_to_absolute([dim[s] for dim in sweep_config.target_sweeps], initial_state)
        per_step.append(fields_from_velocities(res.velocities[0, ramp + s], step_targets, prog.out_keys))
        infos.append(solve_info_from_health(res.tangent_health[0, ramp + s], prog.n_unknowns, prog.stats["n_rows"]))
    return SweepTangents(per_step=per_step, solve_infos=infos)


def compute_sweep_metrics(suspension, sweep_config: SweepConfig, states: list) -> SweepMetricsResult:
    """All sweep metrics of already solved states (reference core/sweep.py:144-173).  State,
    mechanism and derivative metrics come out of one device pass together with the tangents they
    are built on, so there is no separate derivative failure mode: ``derivative_error`` stays
    ``None`` and undefined values are ``None`` in the rows."""
    if suspension.config is None:
        return SweepMetricsResult(rows=[OrderedDict() for _ in states])
    if not states:
        return SweepMetricsResult(rows=[], tangent_solve_infos=[])
    heads = [dim[0] for dim in sweep_config.target_sweeps]
    res, solver, ramp = evaluate_states_on_device(suspension, heads, states, want_metrics=True)
    prog = solver.program
    rows = [rows_from_columns(res.metrics[0, ramp + s], prog.metric_locations, suspension.is_axle)
            for s in range(len(states))]
    infos = [solve_info_from_health(res.tangent_health[0, ramp + s], prog.n_unknowns, prog.stats["n_rows"])
             for s in range(len(states))]
    return SweepMetricsResult(rows=rows, derivative_error=None, tangent_solve_infos=infos)


def _derivative_issues(result: SweepMetricsResult) -> list:
    """Tangent-computation health as advisory diagnostics (reference core/sweep.py:176-219)."""
    from .diagnostics import DiagnosticCategory, DiagnosticIssue, DiagnosticSeverity
    issues = []
    if result.derivative_error is not None:
        issues.append(DiagnosticIssue(
            None, DiagnosticCategory.DERIVATIVES, DiagnosticSeverity.WARNING,
            "Derivative metrics unavailable: tangent computation failed "
            f"({result.derivative_error}); derivative columns are omitted.", None))
    infos = result.tangent_solve_infos or []
    deficient = [step for step, info in enumerate(infos) if info.rank_deficient]
    if deficient:
        first = deficient[0]
        min_sv = min(infos[step].smallest_singular_value for step in deficient)
        issues.append(DiagnosticIssue(
            first, DiagnosticCategory.DERIVATIVES, DiagnosticSeverity.WARNING,
            f"Tangent system rank-deficient at {len(deficient)} of {len(infos)} steps (first at step {first}, "
            f"rank {infos[first].rank}/{infos[first].n_variables}, smallest singular value {min_sv:.3g}); "
            "derivative values may not be unique.", min_sv))
    return issues


def evaluate_solved_sweep(suspension, sweep_config: SweepConfig, states: list, solver_stats: list) -> EvaluatedSweep:
    """Metrics and diagnostics of an already solved sweep (reference core/sweep.py:222-262)."""
    from .diagnostics import DiagnosticCategory, DiagnosticIssue, DiagnosticSeverity, diagnose_sweep
    if len(states) != len(solver_stats):
        raise ValueError("Solved state and solver-stat counts must match: "
                         f"{len(states)} states, {len(solver_stats)} solver stats.")
    metrics = compute_sweep_metrics(suspension, sweep_config, states)
    try:
        diagnostics = list(diagnose_sweep(suspension, states, solver_stats).issues)
    except Exception as error:  # noqa: BLE001 - diagnostics are advisory
        diagnostics = [DiagnosticIssue(
            None, DiagnosticCategory.DIAGNOSTICS, DiagnosticSeverity.WARNING,
            f"Sweep diagnostics unavailable: diagnostic evaluation failed ({type(error).__name__}: {error}).", None)]
    diagnostics.extend(_derivative_issues(metrics))
    return EvaluatedSweep(states=states, solver_stats=solver_stats, metrics=metrics, diagnostics=diagnostics)


def solve_evaluated_sweep(suspension, sweep_config: SweepConfig) -> EvaluatedSweep:
    """Solve one sweep and compute its metrics and advisory diagnostics
    (reference core/sweep.py:265-279)."""
    states, solver_stats = solve_sweep(suspension, sweep_config)
    return evaluate_solved_sweep(suspension, sweep_config, states, solver_stats)
