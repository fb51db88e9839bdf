"""Solution-manifold tangents behind the reference's boundary B2.

``compute_state_tangents`` has the signature and return types of reference
``core/sensitivity.py:57-143``.  The reference solves ``[J; pins] V = E`` by SVD least squares on
the host; here the state is handed to the device as a one-step sweep whose targets sit at the
state's own target coordinates, and the tangents come out of the Cholesky factor of the pinned
normal equations (``okin_solve_batch`` with ``velocities`` / ``tangent_health``).
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np

from .. import _lib
from .enums import TargetPositionMode
from .points.derived.manager import DerivedPointsManager
from .state import SuspensionState
from .targeting import PointTarget, resolve_target
from .topology import compile_topology

# A state handed in for evaluation must be a solution of the constraints it is evaluated with.  The
# bound is the accuracy of states the reference itself produces and accepts: its default-tolerance
# solves sit 0.6-2.3e-5 mm from the tight solution (tests/golden, positions_default vs
# positions_tight) and it accepts any state with max|r| <= SOLVE_ACCEPT_RESIDUAL = 1e-3
# (primitives/constants.py:20); tangents and metrics move by (their derivative) x (that distance).
STATE_MATCH_TOL_MM = 1e-3


@dataclass(frozen=True)
class TangentField:
    """First-order response of every point position to one sweep target
    (reference sensitivity.py:26-39)."""

    target_index: int
    target: PointTarget
    velocities: dict

    def velocity(self, point_id) -> np.ndarray:
        velocity = self.velocities.get(point_id)
        if velocity is None:
            return np.zeros(3, dtype=np.float64)
        return velocity


@dataclass(frozen=True)
class TangentSolveInfo:
    """Numerical health of one state's tangent solve (reference sensitivity.py:42-55).

    ``smallest_singular_value`` and ``condition_number`` are the device's power / inverse
    iteration estimates for the pinned Jacobian; ``rank`` is ``n_variables`` unless the smallest
    singular value falls below LAPACK's ``eps * max(m, n) * sigma_max`` cut-off (then
    ``n_variables - 1``: deficient, multiplicity not resolved)."""

    n_variables: int
    rank: int
    smallest_singular_value: float
    condition_number: float

    @property
    def rank_deficient(self) -> bool:
        return self.rank < self.n_variables


def measured_targets(targets: Sequence[PointTarget], state: SuspensionState) -> list:
    """The same targets, absolute, valued at the coordinates ``state`` actually has."""
    out = []
    for t in targets:
        d = resolve_target(t.direction).data
        out.append(PointTarget(t.point_id, t.direction, float(np.dot(state.positions[t.point_id].data, d)),
                               TargetPositionMode.ABSOLUTE))
    return out


def solve_info_from_health(health: np.ndarray, n_variables: int, n_rows: int) -> TangentSolveInfo:
    smin, cond = float(health[0]), float(health[1])
    cutoff = np.finfo(np.float64).eps * max(n_rows, n_variables)
    deficient = not np.isfinite(cond) or smin <= 0.0 or 1.0 / cond <= cutoff
    return TangentSolveInfo(n_variables=n_variables, rank=n_variables - 1 if deficient else n_variables,
                            smallest_singular_value=smin if np.isfinite(smin) else 0.0,
                            condition_number=cond if np.isfinite(cond) else float("inf"))


def fields_from_velocities(velocities: np.ndarray, targets: Sequence[PointTarget], out_keys: list) -> list:
    """``velocities`` [n_targets, n_out, 3] -> one ``TangentField`` per target."""
    return [TangentField(target_index=j, target=t,
                         velocities={k: velocities[j, i].copy() for i, k in enumerate(out_keys)})
            for j, t in enumerate(targets)]


def compute_state_tangents(state: SuspensionState, constraints: list, derived_manager: DerivedPointsManager,
                           step_targets: Sequence[PointTarget]) -> tuple:
    """One tangent field per target plus solve health (reference sensitivity.py:57-143).

    ``state`` must satisfy ``constraints`` (it is a solved sweep state); the inputs are not
    mutated.  Raises ``RuntimeError`` if the device finds no solution at the state."""
    if not step_targets:
        return [], TangentSolveInfo(n_variables=0, rank=0, smallest_singular_value=0.0, condition_number=1.0)
    pinned = measured_targets(step_targets, state)
    program = compile_topology(state, constraints, derived_manager.spec, pinned, design_rules=False)
    topo = _lib.DeviceTopology(program)
    try:
        hardpoints = np.array([state.positions[k].data for k in program.in_keys]).reshape(1, -1)
        values = np.array([[t.value] for t in pinned], dtype=np.float64)
        out = topo.solve_batch(hardpoints, values, _lib.default_cfg(), want_velocities=True, want_health=True)
    finally:
        topo.close()
    if int(out["status"][0]) != 0:
        raise RuntimeError("Tangent computation failed: the state is not a solution of the given constraints "
                           f"(device status {int(out['status'][0])}).")
    given = np.array([state.positions[k].data for k in program.out_keys])
    drift = float(np.abs(out["positions"][0, 0] - given).max())
    if drift > STATE_MATCH_TOL_MM:
        raise RuntimeError(f"Tangent computation failed: the state is {drift:.3g} mm away from the nearest "
                           "solution of the given constraints.")
    fields = fields_from_velocities(out["velocities"][0, 0], list(step_targets), program.out_keys)
    info = solve_info_from_health(out["tangent_health"][0, 0], program.n_unknowns, program.stats["n_rows"])
    return fields, info


def linearised_std(hardpoint_sensitivity: np.ndarray, sigma) -> np.ndarray:
    """First-order standard deviation of every output coordinate, ``[n, n_steps, n_out, 3]``, for
    independent hardpoint coordinates with standard deviations ``sigma`` (a scalar or one value per
    sensitivity row): ``sqrt(sum_k S_k^2 sigma_k^2)`` over the rows ``S_k`` of
    ``BatchSweepResult.hardpoint_sensitivity`` ``[n, n_steps, n_sens, n_out, 3]``.  Valid while the
    tolerances are small against the curvature of the response (no second-order terms)."""
    s = np.asarray(hardpoint_sensitivity, dtype=np.float64)
    sig = np.broadcast_to(np.asarray(sigma, dtype=np.float64), (s.shape[2],))
    return np.sqrt(np.einsum("nsk...,k->ns...", s * s, sig * sig))
