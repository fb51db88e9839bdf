"""Shared test helpers: golden loading, product-model -> oracle-problem adapter,
lane-emulation build of the device core."""

from __future__ import annotations

import ctypes
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

from open_kinematics_b200.core import constraints as PC  # noqa: E402
from open_kinematics_b200.core.enums import PointID  # noqa: E402
from open_kinematics_b200.core.input import build_suspension, build_sweep  # noqa: E402
from open_kinematics_b200.core.primitives.point_ref import PointRef, Side  # noqa: E402
from open_kinematics_b200.core.solver import sweep_target_values  # noqa: E402
from open_kinematics_b200.core.targeting import resolve_target  # noqa: E402
from open_kinematics_b200.core.enums import TargetPositionMode  # noqa: E402
from oracle.solve import OracleConstraint, OracleDerived, OracleProblem, OracleTarget  # noqa: E402

SWEEP_CASES = [
    "c1_dw_corner_bump", "c1_dw_corner_bump_steer", "c2_macpherson_bump_steer", "c3_rocker_ubar_roll_shipped",
    "c3_rocker_ubar_coilover_roll", "c4_tbar_roll", "c4_tbar_bump", "dw_axle_direct", "macpherson_axle",
    "dw_corner_coilover_direct", "dw_corner_rocker",
]
# Configurations with a camber shim whose setup thickness differs from design: the pre-solve runs
# on the device, so the host model's initial_state() needs a GPU; CPU tests use structure().
SHIM_CASES = ["c1_shim_plus2mm", "c4_tbar_heave_shim_roll", "c4_tbar_heave_shim_bump"]


def load_golden(name: str):
    meta = json.load(open(os.path.join(GOLDEN, name + ".json")))
    arrays = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    return meta, arrays


def key_name(key) -> str:
    return key.name.lower()


def key_from_name(name: str):
    for side in (Side.LEFT, Side.RIGHT, Side.CENTER):
        prefix = side.name.lower() + "_"
        if name.startswith(prefix) and name[len(prefix):].upper() in PointID.__members__:
            return PointRef(side, PointID[name[len(prefix):].upper()])
    return PointID[name.upper()]


def authored_positions(suspension) -> dict:
    """Authored (un-derived, un-shimmed) position of every input point, keyed like a solved state."""
    if getattr(suspension, "is_axle", False):
        out = {PointRef(side, k): p.data.copy() for side, c in suspension.corners.items()
               for k, p in c.hardpoints.items()}
        arb = suspension.anti_roll
        for point, p in getattr(arb, "center_points", {}).items():
            out[PointRef(Side.CENTER, point)] = p.data.copy()
        arm = PointID.DROPLINK_U_BAR if type(arb).__name__ == "ArbUBar" else PointID.DROPLINK_T_BAR
        for side, p in getattr(arb, "droplink_points", {}).items():
            out[PointRef(side, arm)] = p.data.copy()
        return out
    return {k: p.data.copy() for k, p in suspension.hardpoints.items()}


_FAMILY = {
    PC.DistanceConstraint: "distance", PC.SphericalJointConstraint: "spherical", PC.AngleConstraint: "angle",
    PC.ThreePointAngleConstraint: "three_point_angle", PC.VectorsParallelConstraint: "vectors_parallel",
    PC.VectorsPerpendicularConstraint: "vectors_perpendicular", PC.EqualDistanceConstraint: "equal_distance",
    PC.PointOnLineConstraint: "point_on_line", PC.PointOnPlaneConstraint: "linear_point",
    PC.MidpointOnPlaneConstraint: "midpoint_on_plane", PC.ScalarTripleProductConstraint: "scalar_triple",
    PC.CoplanarPointsConstraint: "coplanar", PC.FixedAxisConstraint: "linear_point",
}


def oracle_problem(suspension, sweep_config, from_design: bool = True, structure_only: bool = False) -> OracleProblem:
    """Describe a built product model to the oracle (declarations only; no product arithmetic).
    ``structure_only``: take points and constraint declarations from ``structure()`` (authored pose, no
    camber-shim pre-solve, which needs the device); every design constant must then come from
    ``design_setup`` (``from_design``)."""
    if structure_only:
        assert from_design
        state, constraints = suspension.structure()
    else:
        state, constraints = suspension.initial_state(), suspension.constraints()
    heads, values = sweep_target_values(sweep_config)
    return oracle_problem_of(state, constraints, suspension.derived_spec(), heads, from_design), values


def oracle_problem_of(state, constraints, spec, heads, from_design: bool = True) -> OracleProblem:
    """``(state, constraint declarations, derived spec, one PointTarget per sweep dimension)`` ->
    ``OracleProblem``: the mapping of ``oracle_problem`` for a linkage built without a suspension."""
    cons = []
    for c in constraints:
        fam = _FAMILY[type(c)]
        if fam == "distance":
            consts = [c.target_distance]
        elif fam in ("angle", "three_point_angle"):
            consts = [c.target_angle]
        elif fam == "scalar_triple":
            consts = [c.target_volume, 1.0 / c.scale]
        elif fam == "point_on_line":
            consts = [*c.line_point.data, *c.line_direction.data]
        elif isinstance(c, PC.FixedAxisConstraint):
            n = np.zeros(3)
            n[int(c.axis)] = 1.0
            consts = [*(n * c.value), *n]
        elif fam in ("linear_point", "midpoint_on_plane"):
            consts = [*c.plane_point.data, *c.plane_normal.data]
        else:
            consts = []
        design = from_design and fam in ("distance", "angle", "scalar_triple", "point_on_line")
        cons.append(OracleConstraint(fam, c.point_keys, list(map(float, consts)), design))
    from open_kinematics_b200.core.points.derived.manager import DerivedPointsManager
    derived = []
    for key in DerivedPointsManager(spec).update_order:
        fn = spec.functions[key]
        derived.append(OracleDerived(fn.OP, key, tuple(fn.inputs), float(fn.param),
                                     fn.design_projection if from_design else None))
    targets = [OracleTarget(h.point_id, resolve_target(h.direction).data.copy(),
                            TargetPositionMode(h.mode) == TargetPositionMode.RELATIVE) for h in heads]
    return OracleProblem(sorted(state.positions), list(state.free_points_order), cons, derived, targets)


def build_case(meta: dict):
    sus = build_suspension(meta["geometry"])
    sweep = build_sweep(meta["sweep"], sus)
    return sus, sweep


# ---------------------------------------------------------------------------
# Lane-emulation build of csrc/okin_core.cuh (tests only; the product never loads it).
# ---------------------------------------------------------------------------
_EMU = None
# okin_default_cfg
DEFAULT_CFG = dict(step_tol=1e-6, coarse_tol=1e-3, fine_tol=1e-4, residual_tol=1e-3, mu_init=1e-3, max_iter=50,
                   use_predictor=4)


def emu_lib():
    global _EMU
    if _EMU is None:
        src = os.path.join(ROOT, "tests", "emu", "okin_emu.cpp")
        out = os.path.join(ROOT, "tests", "emu", "libokin_emu.so")
        csrc = os.path.join(ROOT, "open-kinematics_b200", "csrc")
        deps = [src, os.path.join(ROOT, "include", "okin.h")]
        deps += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".cuh"))]
        if not os.path.exists(out) or os.path.getmtime(out) < max(map(os.path.getmtime, deps)):
            subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", f"-I{csrc}", "-o", out, src], check=True)
        lib = ctypes.CDLL(out)
        lib.okin_emu_sweep.restype = ctypes.c_int
        lib.okin_emu_sweep.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_long, ctypes.c_int] + [ctypes.c_void_p] * 2
        lib.okin_emu_family.restype = ctypes.c_int
        lib.okin_emu_family.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 5
        lib.okin_emu_study.restype = ctypes.c_int
        lib.okin_emu_study.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_longlong, ctypes.c_int] + \
            [ctypes.c_void_p] * 4 + [ctypes.c_longlong, ctypes.c_int]
        lib.okin_emu_study_sample.restype = ctypes.c_int
        lib.okin_emu_study_sample.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong] + [ctypes.c_void_p] * 3
        lib.okin_emu_philox.restype = None
        lib.okin_emu_philox.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        _EMU = lib
    return _EMU


def emu_cfg(**overrides):
    """``okin_solver_cfg`` of the default settings with ``overrides``."""
    from open_kinematics_b200._lib import SolverCfg
    return SolverCfg(**{**DEFAULT_CFG, **overrides})


def emu_family(fam_code: int, points: np.ndarray, consts) -> tuple:
    """(residual from okin_family_resgrad, residual from okin_family_res, gradient[n_points, 3])."""
    p = np.zeros(12)
    p[:points.size] = np.asarray(points, dtype=np.float64).reshape(-1)
    c = np.zeros(8)
    c[:len(consts)] = consts
    res, res_only, g = np.zeros(1), np.zeros(1), np.zeros(12)
    emu_lib().okin_emu_family(fam_code, p.ctypes.data, c.ctypes.data, res.ctypes.data, res_only.ctypes.data,
                              g.ctypes.data)
    return float(res[0]), float(res_only[0]), g[:points.size].reshape(-1, 3)


def generic_mechanism():
    """Mirror-class build of tests/golden/generic_mechanism.json (generic constraint families):
    ``(initial_state, constraints, sweep_config, derived_manager, spec, arrays)``."""
    from open_kinematics_b200.core.enums import Axis
    from open_kinematics_b200.core.points.derived.manager import DerivedPointsManager, DerivedPointsSpec
    from open_kinematics_b200.core.primitives.geometry import Direction3, Point3
    from open_kinematics_b200.core.state import SuspensionState
    from open_kinematics_b200.core.targeting import PointTarget, PointTargetAxis, SweepConfig
    spec = json.load(open(os.path.join(GOLDEN, "generic_mechanism.json")))
    arrays = np.load(os.path.join(GOLDEN, "generic_mechanism.npz"))
    key = lambda name: PointID[name.upper()]   # noqa: E731
    state = SuspensionState(positions={key(k): Point3(np.array(v, float)) for k, v in spec["points"].items()},
                            free_points={key(k) for k in spec["free"]})
    cons = []
    for c in spec["constraints"]:
        k = [key(n) for n in c["points"]]
        fam = c["family"]
        if fam == "distance":
            cons.append(PC.DistanceConstraint(k[0], k[1], c["value"]))
        elif fam == "point_on_plane":
            cons.append(PC.PointOnPlaneConstraint(k[0], Point3(np.array(c["plane_point"], float)),
                                                  Direction3(np.array(c["plane_normal"], float))))
        elif fam == "fixed_axis":
            cons.append(PC.FixedAxisConstraint(k[0], Axis(c["axis"]), c["value"]))
        elif fam == "equal_distance":
            cons.append(PC.EqualDistanceConstraint(*k))
        elif fam == "three_point_angle":
            cons.append(PC.ThreePointAngleConstraint(*k, c["value"]))
        elif fam == "coplanar":
            cons.append(PC.CoplanarPointsConstraint(*k))
        elif fam == "vectors_perpendicular":
            cons.append(PC.VectorsPerpendicularConstraint(*k))
        else:
            raise KeyError(fam)
    t = spec["target"]
    sweep = SweepConfig([[PointTarget(key(t["point"]), PointTargetAxis(Axis(t["axis"])), float(v),
                                      TargetPositionMode.RELATIVE) for v in t["values"]]])
    manager = DerivedPointsManager(DerivedPointsSpec(functions={}, dependencies={}))
    return state, cons, sweep, manager, spec, arrays


class UsageError(RuntimeError):
    """The library would return OKIN_ERR_USAGE (hardpoint sensitivities on a topology with camber-shim records)."""


def emu_solve(program, hardpoints: np.ndarray, values: np.ndarray, params=None, want_health=False,
              instance_targets=None, lean=False, want_hardpoint_sensitivity=False, **cfg) -> dict:
    """Run the lane-emulation build of the device core; ``cfg`` overrides ``okin_solver_cfg`` fields.
    ``lean``: no tangent / metric / diagnostic outputs, i.e. the lean kernel instantiation (its own
    predictor and the short slice).  ``want_hardpoint_sensitivity``: the sensitivity instantiation and
    its ``hardpoint_sensitivity`` output ``[n, n_steps, n_sens, n_out, 3]``."""
    from open_kinematics_b200._lib import BatchIO, batch_shapes
    hp = np.ascontiguousarray(hardpoints, dtype=np.float64).reshape(-1, 3 * program.n_in)
    tv = np.ascontiguousarray(values, dtype=np.float64)
    n_inst, n_steps = hp.shape[0], tv.shape[1]
    full = not lean
    want = {"tangents": full, "velocities": full, "tangent_health": full and want_health,
            "metrics": full and bool(program.metric_names), "diagnostics": full and bool(program.diagnostic_names),
            "jumps": full and bool(program.diagnostic_names), "hardpoint_sensitivity": want_hardpoint_sensitivity}
    out = {name: np.zeros(shape, dtype) if want.get(name, True) else None
           for name, (shape, dtype) in batch_shapes(program, n_inst, n_steps).items()}
    itv = None if instance_targets is None else np.ascontiguousarray(instance_targets, dtype=np.float64)
    par = None if params is None else np.ascontiguousarray(params, dtype=np.float64)
    hdr = np.ascontiguousarray(program.hdr)
    io = BatchIO.of(hardpoints=hp, params=par, target_values=tv, instance_targets=itv, **out)
    rc = emu_lib().okin_emu_sweep(
        hdr.ctypes.data, program.iblob.ctypes.data, program.fblob.ctypes.data, n_inst, n_steps,
        ctypes.byref(emu_cfg(**cfg)), ctypes.byref(io))
    if rc == -3:
        raise UsageError("hardpoint sensitivities are not available on a topology with camber-shim records")
    assert rc == 0, rc
    if out["metrics"] is None:
        out["metrics"] = np.zeros((n_inst, n_steps, 1))
    if not want_hardpoint_sensitivity:
        del out["hardpoint_sensitivity"]
    return out


def perturbed_hardpoints(meta_batch: dict, program) -> np.ndarray:
    """Hardpoint rows (input-slot order) for the perturbed geometries of a golden batch."""
    rows = []
    for geom in meta_batch["geometries"]:
        sus = build_suspension(geom)
        auth = authored_positions(sus)
        rows.append(np.concatenate([auth[k] for k in program.in_keys]))
    return np.array(rows)
