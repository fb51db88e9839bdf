"""Seeded corpus of generated linkages for the generic solver API.

Every linkage is built through the public declarations (``SuspensionState``, the constraint classes,
``DerivedPointsSpec``, ``PointTarget``) over the 102 side-qualified keys ``PointRef(side, PointID)``:

* a few fixed points, then free points added one at a time, each hung on three earlier points
  (fixed, free or derived) so that the linkage holds at the design pose by construction;
* the anchors choose the shape: ``chain`` (the last three points: one elimination level per point),
  ``star`` (fixed points only: one level as wide as the linkage), ``random`` (any earlier point);
* ``well`` places each new point so that the unit directions to its anchors have |det| > 0.4;
  ``ill`` squeezes them towards a plane, and ``random`` takes them as they come;
* families: a new point may swap one anchor distance for an angle, three-point angle, equal
  distance, perpendicular pair, point on plane, fixed axis, midpoint on plane, coplanar or scalar
  triple row, or be put on a line (two pins plus the report row) -- each made to hold at the
  design pose -- and identically satisfied spherical / parallel rows on derived points make the
  over-determined cases;
* a chain of four derived points (midpoint, along-line, contact-patch, along-line) anchors a later
  point, so the derived Jacobian runs through ``OKIN_MAX_CHAIN`` ops;
* each target drops the last constraint of a free point and drives that point along the dropped
  direction (relative or absolute); ``reach`` sweeps drive it past the end of its travel.

``CASES`` is a fixed list; a case name reproduces its linkage exactly.
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from open_kinematics_b200.core import constraints as PC
from open_kinematics_b200.core.enums import Axis, PointID, TargetPositionMode
from open_kinematics_b200.core.points.derived.definitions import ContactPatch, Midpoint, PointAlongLine
from open_kinematics_b200.core.points.derived.manager import DerivedPointsSpec
from open_kinematics_b200.core.primitives.geometry import Direction3, Point3
from open_kinematics_b200.core.primitives.point_ref import PointRef, Side
from open_kinematics_b200.core.state import SuspensionState
from open_kinematics_b200.core.targeting import PointTarget, PointTargetVector, SweepConfig

KEYS = [PointRef(side, pid) for side in Side for pid in PointID]      # 102 keys

# families a free point may use in place of one anchor distance ("line": two pins).  The coplanar
# row is unscaled (its gradient is an area, ~1e4 mm^2 here), so it only joins the ill-conditioned class.
SWAPS = ("angle", "three_point_angle", "equal_distance", "perpendicular", "plane", "fixed_axis",
         "midpoint_plane", "coplanar", "scalar_triple", "line")
SCALED = tuple(s for s in SWAPS if s != "coplanar")


@dataclass(frozen=True)
class Case:
    name: str
    seed: int
    n_free: int
    shape: str                  # chain | star | random
    cond: str                   # well | ill | random
    n_targets: int = 1
    relative: bool = True
    families: tuple = ()        # the families a new point may swap an anchor distance for
    derived: bool = False       # a four-op derived chain anchoring later points
    reach: bool = False         # drive the first target past the end of its travel
    steps: int = 5
    amplitude: float = 1.0      # mm, largest target displacement (reach: per unit of travel)


@dataclass
class Linkage:
    case: Case
    state: SuspensionState
    constraints: list
    spec: DerivedPointsSpec
    heads: list                 # one PointTarget per sweep dimension
    values: np.ndarray          # [T, S]
    design: dict                # key -> authored xyz of every point

    @property
    def sweep(self) -> SweepConfig:
        return SweepConfig([[PointTarget(h.point_id, h.direction, float(v), h.mode) for v in row]
                            for h, row in zip(self.heads, self.values)])

    def hardpoints(self, in_keys, sigma: float = 0.0, seed: int = 0) -> np.ndarray:
        """Hardpoint row in ``in_keys`` order; ``sigma`` > 0 perturbs every coordinate (mm)."""
        row = np.concatenate([self.design[k] for k in in_keys])
        if sigma > 0.0:
            row = row + np.random.default_rng(seed).normal(0.0, sigma, row.shape)
        return row


def _unit(v):
    return v / np.linalg.norm(v)


def _place(rng, anchors, cond: str):
    """A new point near its three anchors; ``well``: |det| of the unit directions > 0.4,
    ``ill``: directions squeezed towards a plane (|det| in 5e-3..2e-2)."""
    centre = np.mean(anchors, axis=0)
    spread = max(80.0, max(np.linalg.norm(a - centre) for a in anchors))
    for _ in range(2000):
        p = centre + rng.normal(0.0, 1.0, 3) * spread + _unit(rng.normal(size=3)) * 60.0
        if min(np.linalg.norm(p - a) for a in anchors) < 40.0:
            continue
        det = abs(np.linalg.det(np.array([_unit(p - a) for a in anchors])))
        if cond == "random":
            return p
        if cond == "well" and det > 0.4:
            return p
        if cond == "ill":
            # push p towards the plane through the anchors: the three directions flatten
            n = _unit(np.cross(anchors[1] - anchors[0], anchors[2] - anchors[0]))
            h = (p - anchors[0]) @ n
            for scale in (0.05, 0.02, 0.01, 0.005):
                q = p - h * (1 - scale) * n
                d = abs(np.linalg.det(np.array([_unit(q - a) for a in anchors])))
                if 5e-3 <= d <= 2e-2 and min(np.linalg.norm(q - a) for a in anchors) > 40.0:
                    return q
    return None


def _hang(kind: str, k, p, anchors, pos, rng):
    """The row that replaces the third anchor distance of a new point ``k`` near ``p``:
    ``(p moved onto the row's zero set where needed, constraint, the row's gradient direction at p)``."""
    a, b, c = (pos[q] for q in anchors)
    ka, kb, kc = anchors
    if kind == "plane":
        n = _unit(p - c + rng.normal(0.0, 20.0, 3))
        return p, PC.PointOnPlaneConstraint(k, Point3(p + np.cross(n, rng.normal(size=3)) * 10.0), Direction3(n)), n
    if kind == "fixed_axis":
        ax = int(np.argmax(np.abs(p - c)))
        return p, PC.FixedAxisConstraint(k, Axis(ax), float(p[ax])), np.eye(3)[ax]
    if kind == "midpoint_plane":
        n = _unit(p - c)
        return p, PC.MidpointOnPlaneConstraint(k, kc, Point3((p + c) / 2.0), Direction3(n)), n
    if kind == "coplanar":
        n = _unit(np.cross(b - a, c - a))
        return p - ((p - a) @ n) * n, PC.CoplanarPointsConstraint(ka, kb, kc, k), n
    if kind == "scalar_triple":
        v = float((b - a) @ np.cross(c - a, p - a))
        return p, PC.ScalarTripleProductConstraint(ka, kb, kc, k, v, abs(v)), np.cross(b - a, c - a)
    if kind in ("angle", "three_point_angle"):
        u, w = _unit(p - c), _unit(b - a if kind == "angle" else a - c)
        theta = float(np.arctan2(np.linalg.norm(np.cross(u, w)), u @ w))
        con = PC.AngleConstraint(kc, k, ka, kb, theta) if kind == "angle" else PC.ThreePointAngleConstraint(ka, kc, k, theta)
        return p, con, w - (w @ u) * u
    if kind == "equal_distance":      # |p - c| = |p - b|: p on the bisector plane of b and c
        n = _unit(c - b)
        p = p - ((p - (b + c) / 2.0) @ n) * n
        return p, PC.EqualDistanceConstraint(k, kc, k, kb), _unit(p - b) - _unit(p - c)
    if kind == "perpendicular":       # (p - a) . (c - b) = 0
        n = _unit(c - b)
        return p - ((p - a) @ n) * n, PC.VectorsPerpendicularConstraint(ka, k, kb, kc), n
    if kind == "line":                # two pins: the free direction along the line is d
        d = _unit(p - b + rng.normal(0.0, 30.0, 3))
        return p, PC.PointOnLineConstraint(k, Point3(p - 25.0 * d), Direction3(d)), d
    return p, PC.DistanceConstraint(k, kc, float(np.linalg.norm(p - c))), p - c


def build(case: Case) -> Linkage:
    rng = np.random.default_rng(case.seed)
    keys = iter(KEYS)
    pos: dict = {}
    fixed, free, order = [], [], []          # order: every point usable as an anchor, in creation order
    cons: list = []
    owner: dict = {}                         # free key -> indices of its constraints
    functions, deps = {}, {}

    def add_fixed(p):
        k = next(keys)
        pos[k] = np.asarray(p, float)
        fixed.append(k)
        order.append(k)
        return k

    for corner in ((1, 1, 1), (1, -1, -1), (-1, 1, -1), (-1, -1, 1)):     # a tetrahedron, jittered
        add_fixed(np.array(corner, float) * 100.0 + rng.normal(0.0, 20.0, 3))

    def add_derived(fn):
        k = next(keys)
        functions[k] = fn
        deps[k] = set(fn.inputs)
        pos[k] = fn({q: Point3(v) for q, v in pos.items()}).data.copy()
        return k

    chain_at = case.n_free // 3 if case.derived else -1
    for i in range(case.n_free):
        if i == chain_at:
            # four chained ops on two free points; the end of the chain becomes an anchor
            a, b = free[-1], free[-2]
            d1 = add_derived(Midpoint(a, b))
            d2 = add_derived(PointAlongLine(d1, b, 15.0))
            d3 = add_derived(ContactPatch(d2, a, b, 30.0))
            d4 = add_derived(PointAlongLine(d3, a, -12.0))
            order.append(d4)
            # identically satisfied rows (over-determined case): d4 stays on the line d3 -> a
            # (parallel), d2 on the line d1 -> b (spherical on a zero-offset copy)
            d5 = add_derived(PointAlongLine(d2, b, 0.0))
            cons.append(PC.VectorsParallelConstraint(d3, d4, d3, a))
            cons.append(PC.SphericalJointConstraint(d2, d5))
        if case.shape == "star":
            pool = fixed
        elif case.shape == "chain":
            pool = order[-3:]
        else:
            pool = order
        k = next(keys)
        kind = case.families[rng.integers(len(case.families))] if case.families and rng.random() < 0.5 else "distance"
        while True:
            p = None
            while p is None:        # a nearly collinear anchor triple leaves no placement: draw again
                idx = rng.choice(len(pool), 3, replace=False)
                anchors = [pool[j] for j in sorted(idx)]
                if case.shape == "chain" and i == chain_at:
                    anchors = [order[-1], order[-2], order[-4]]    # the chain end anchors the next point
                p = _place(rng, [pos[a] for a in anchors], case.cond)
            p, last, grad = _hang(kind, k, p, anchors, pos, rng)
            a, b, c = anchors
            if kind == "line":
                shape = abs(_unit(p - pos[a]) @ grad)
            else:
                shape = abs(np.linalg.det(np.array([_unit(p - pos[a]), _unit(p - pos[b]), _unit(grad)])))
            # well: the swapped row keeps the point's three gradient directions well apart
            if case.cond != "well" or shape > 0.3:
                break
        pos[k] = p
        mine = []
        if kind == "line":
            mine.append(len(cons))
            cons.append(PC.DistanceConstraint(k, a, float(np.linalg.norm(p - pos[a]))))
            mine.append(len(cons))
            cons.append(last)
            # the line takes two rows but counts as one constraint: a zero row keeps m >= n
            mid = add_derived(Midpoint(k, a))
            cons.append(PC.VectorsParallelConstraint(a, k, a, mid))
        else:
            for q in (a, b):
                mine.append(len(cons))
                cons.append(PC.DistanceConstraint(k, q, float(np.linalg.norm(p - pos[q]))))
            mine.append(len(cons))
            cons.append(last)
        free.append(k)
        order.append(k)
        owner[k] = (mine, kind, anchors)

    # targets: drop the last row of a distance-hung point and drive it along that row's direction
    eligible = [k for k in free if owner[k][1] == "distance"]
    tpoints = [eligible[j] for j in sorted(rng.choice(len(eligible), case.n_targets, replace=False))]
    drop, heads, values = set(), [], []
    ramp = np.linspace(0.0, 1.0, case.steps)
    for t, k in enumerate(tpoints):
        mine, _, anchors = owner[k]
        drop.add(mine[-1])
        d = _unit(pos[k] - pos[anchors[2]])
        mode = TargetPositionMode.RELATIVE if case.relative else TargetPositionMode.ABSOLUTE
        base = 0.0 if case.relative else float(pos[k] @ d)
        heads.append(PointTarget(k, PointTargetVector(Direction3(d)), 0.0, mode))
        if case.reach and t == 0:
            # travel of a point on two spheres along d is at most the circle's diameter
            values.append(base + ramp * case.amplitude * 400.0)
        else:
            values.append(base + np.sin(np.pi * ramp * (1 + t)) * case.amplitude * rng.uniform(0.5, 1.0))
    cons = [c for i, c in enumerate(cons) if i not in drop]
    state = SuspensionState(positions={k: Point3(v) for k, v in pos.items()}, free_points=set(free))
    spec = DerivedPointsSpec(functions=functions, dependencies=deps)
    design = {k: v.copy() for k, v in pos.items()}
    return Linkage(case, state, cons, spec, heads, np.array(values), design)


CASES = [
    # well conditioned: shapes, sizes on both sides of 32 / 64 / 96 free blocks, 1-4 targets
    Case("well_chain_31", 101, 31, "chain", "well", n_targets=2),
    Case("well_chain_33", 102, 33, "chain", "well", n_targets=1, relative=False),
    Case("well_star_40", 103, 40, "star", "well", n_targets=2),
    Case("well_star_65", 104, 65, "star", "well", n_targets=4),
    Case("well_random_63", 105, 63, "random", "well", n_targets=3),
    Case("well_random_95", 106, 95, "random", "well", n_targets=4, relative=False),
    Case("well_families_30", 107, 30, "random", "well", n_targets=2, families=SCALED, derived=True),
    Case("well_families_chain_34", 108, 34, "chain", "well", n_targets=1, families=SCALED, derived=True),
    Case("well_reach_12", 109, 12, "random", "well", n_targets=1, reach=True, steps=8),
    Case("well_reach_chain_20", 110, 20, "chain", "well", n_targets=2, reach=True, steps=8, relative=False),
    # ill conditioned and unfiltered placements
    Case("ill_random_20", 201, 20, "random", "ill", n_targets=2),
    Case("ill_chain_33", 202, 33, "chain", "ill", n_targets=1),
    Case("ill_families_24", 203, 24, "random", "ill", n_targets=3, families=SWAPS, derived=True),
    Case("random_60_4", 301, 60, "random", "random", n_targets=4),
    Case("random_29_2", 302, 29, "random", "random", n_targets=2),
    Case("random_reach_15", 303, 15, "random", "random", n_targets=1, reach=True, steps=8),
]
