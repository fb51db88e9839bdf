"""Topology compiler: suspension model -> flat device program.

Runs once per topology on the host (never per instance).  It lowers

* the point table (fixed / free / derived, reference ``core/state.py:50`` column order),
* the derived-point DAG (reference ``core/points/derived/manager.py:146-197``),
* the constraint list plus sweep targets into least-squares rows with the
  point-on-line rows replaced by two linear pins (reference
  ``core/sensitivity.py:146-174``; SURVEY.md section 0 fact 2),
* the gather lists that assemble the normal equations ``A = J^T J``, ``g = J^T r``
  from per-row gradients, and
* a symbolic 3x3-block sparse Cholesky of ``A`` (fill-reducing order, elimination
  tree levels, left-looking update lists, triangular-solve lists)

into the int32/double blobs described in ``csrc/okin_defs.h``.  The CUDA kernel
(``csrc/okin_core.cuh``) is an interpreter of that program, so one kernel serves
every topology the host can describe.
"""

from __future__ import annotations

import os
import re
from dataclasses import dataclass, field

import numpy as np

from .constraints import (
    AngleConstraint, Constraint, CoplanarPointsConstraint, DistanceConstraint, EqualDistanceConstraint,
    FixedAxisConstraint, MidpointOnPlaneConstraint, PointOnLineConstraint, PointOnPlaneConstraint,
    ScalarTripleProductConstraint, SphericalJointConstraint, ThreePointAngleConstraint,
    VectorsParallelConstraint, VectorsPerpendicularConstraint,
)
from .enums import TargetPositionMode
from .points.derived.manager import DerivedPointsManager, DerivedPointsSpec
from .schedule import Dest, schedule
from .targeting import resolve_target

_CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "csrc")


def _parse_defs() -> dict:
    """Read the integer constants of csrc/okin_defs.h (single source of truth)."""
    text = open(os.path.join(_CSRC, "okin_defs.h"), encoding="utf-8").read()
    text = re.sub(r"//[^\n]*", "", text)
    out: dict = {}
    for name, value in re.findall(r"#define\s+(OKIN_\w+)\s+(-?(?:0x[0-9a-fA-F]+|\d+))\s*$", text, re.M):
        out[name] = int(value, 0)
    for body in re.findall(r"enum\s+\w+\s*\{([^}]*)\}", text):
        nxt = 0
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, expr = (s.strip() for s in item.split("=", 1))
                nxt = int(eval(expr, {}, dict(out)))  # noqa: S307 - arithmetic on parsed constants
            else:
                name = item
            out[name] = nxt
            nxt += 1
    return out


D = _parse_defs()
assert D["OKIN_S_COUNT"] <= 64 and D["OKIN_F_COUNT"] <= 8 and D["OKIN_H_NGROW"] < D["OKIN_H_SEC0"]

FAMILY_CODE = {
    "distance": D["OKIN_FAM_DISTANCE"], "spherical": D["OKIN_FAM_SPHERICAL"], "angle": D["OKIN_FAM_ANGLE"],
    "three_point_angle": D["OKIN_FAM_THREE_POINT_ANGLE"], "vectors_parallel": D["OKIN_FAM_VECTORS_PARALLEL"],
    "vectors_perpendicular": D["OKIN_FAM_VECTORS_PERPENDICULAR"], "equal_distance": D["OKIN_FAM_EQUAL_DISTANCE"],
    "point_on_line": D["OKIN_FAM_POINT_ON_LINE"], "linear_point": D["OKIN_FAM_LINEAR_POINT"],
    "midpoint_on_plane": D["OKIN_FAM_MIDPOINT_ON_PLANE"], "coplanar": D["OKIN_FAM_COPLANAR"],
    "scalar_triple": D["OKIN_FAM_SCALAR_TRIPLE"], "target": D["OKIN_FAM_TARGET"],
}
_DOP_CODE = {"midpoint": D["OKIN_DOP_MIDPOINT"], "along_line": D["OKIN_DOP_ALONG_LINE"],
             "contact_patch": D["OKIN_DOP_CONTACT_PATCH"]}


def pin_normals(direction: np.ndarray) -> tuple:
    """Two unit normals spanning the plane perpendicular to a line direction
    (reference core/sensitivity.py:159-173)."""
    d = np.asarray(direction, dtype=np.float64)
    d = d / np.linalg.norm(d)
    least = np.zeros(3)
    least[int(np.argmin(np.abs(d)))] = 1.0
    n1 = np.cross(d, least)
    n1 /= np.linalg.norm(n1)
    return n1, np.cross(d, n1)


@dataclass
class _Row:
    fam: int
    points: list            # point indices (len <= 4)
    consts: list            # default constants (floats)
    rule: int
    source: tuple           # ("constraint", index) | ("pin", index, k) | ("target", index) | ("report", index)
    aux: int = 0
    eff: list = field(default_factory=list)        # effective free blocks (reference column block ids)
    slotmap: list = field(default_factory=list)
    cst_off: int = 0
    rg_off: int = 0
    fast: bool = False      # plain distance row evaluated by the dedicated fast path (stores u only)

    def grad_ref(self, e: int) -> tuple:
        """(rg offset, negate) of the gradient w.r.t. effective block ``e``.  A fast distance row
        stores the unit vector u = dR/dp2 once; dR/dp1 = -u."""
        if self.fast:
            return self.rg_off, self.eff_sign[e] < 0
        return self.rg_off + 3 * e, False


@dataclass
class TopologyProgram:
    hdr: np.ndarray
    iblob: np.ndarray
    fblob: np.ndarray
    point_keys: list          # index -> key
    free_order: list          # reference column order (sorted free keys)
    in_keys: list             # input slot -> key
    out_keys: list            # output slot -> key
    n_constraints: int
    row_source: list          # LS rows then report rows
    target_points: list
    stats: dict
    metric_names: list = field(default_factory=list)
    metric_locations: list = field(default_factory=list)
    diagnostic_names: list = field(default_factory=list)
    diagnostic_checks: list = field(default_factory=list)
    param_names: list = field(default_factory=list)
    param_default: np.ndarray = field(default_factory=lambda: np.zeros(0))
    sensitivity_inputs: list = field(default_factory=list)   # (input point key, axis) per sensitivity row

    @property
    def n_unknowns(self) -> int:
        return 3 * len(self.free_order)

    @property
    def n_in(self) -> int:
        return len(self.in_keys)

    @property
    def n_out(self) -> int:
        return len(self.out_keys)

    def section(self, name: str) -> np.ndarray:
        s = D[name]
        off, n = self.hdr[D["OKIN_H_SEC0"] + 2 * s], self.hdr[D["OKIN_H_SEC0"] + 2 * s + 1]
        return self.iblob[off: off + n]

    def fsection(self, name: str) -> np.ndarray:
        s = D[name]
        off, n = self.hdr[D["OKIN_H_FSEC0"] + 2 * s], self.hdr[D["OKIN_H_FSEC0"] + 2 * s + 1]
        return self.fblob[off: off + n]

    def spec_phases(self) -> list:
        """Task lists of the lean kernel's hot phases, in the phase order of ``csrc/okin_core.cuh``
        (OKIN_PH_*): per phase a list of ``(task word, [contribution words])``."""
        sec = lambda name: [int(w) & 0xFFFFFFFF for w in self.section(name)]   # noqa: E731
        h = self.hdr
        nat, nf, nlev = int(h[D["OKIN_H_NAT"]]), int(h[D["OKIN_H_NF"]]), int(h[D["OKIN_H_NLEV"]])
        aptr, atask, acon = sec("OKIN_S_ASM_PTR"), sec("OKIN_S_ASM_TASK"), sec("OKIN_S_ASM_CON")
        gptr, gcon = sec("OKIN_S_G_PTR"), sec("OKIN_S_G_CON")
        phases = [[(atask[t], acon[aptr[t]:aptr[t + 1]]) for t in range(nat)],
                  [(j, gcon[gptr[j]:gptr[j + 1]]) for j in range(nf)]]
        lev_upd, upd_mid = sec("OKIN_S_LEV_UPD"), sec("OKIN_S_LEV_UPD_MID")
        udst, uptr, ucon = sec("OKIN_S_UPD_DST"), sec("OKIN_S_UPD_PTR"), sec("OKIN_S_UPD_CON")
        lev_scl, scl_mid, scl = sec("OKIN_S_LEV_SCL"), sec("OKIN_S_LEV_SCL_MID"), sec("OKIN_S_SCL")
        lcp, lcol, doffs = sec("OKIN_S_LEV_COL_PTR"), sec("OKIN_S_LEV_COL"), sec("OKIN_S_DIAG_OFF")
        for lv in range(nlev):   # the lean kernel never carries tangent right-hand sides: up to the mid pointers
            phases.append([(udst[t], ucon[uptr[t]:uptr[t + 1]]) for t in range(lev_upd[lv], upd_mid[lv])])
            phases.append([(doffs[lcol[c]], []) for c in range(lcp[lv], lcp[lv + 1])])
            phases.append([(scl[t], []) for t in range(lev_scl[lv], scl_mid[lv])])
        slev, stask, scon = sec("OKIN_S_SOLVE_LEV"), sec("OKIN_S_SOLVE_TASK"), sec("OKIN_S_SOLVE_CON")
        assert max(doffs, default=0) < 1 << 16
        for p in list(range(nlev)) + [nlev + 1 + ph for ph in range(nlev)]:
            # solve task word: FIN | column, with the column's diagonal block offset in the high half
            phases.append([((stask[k] & 0xFFFF) | doffs[stask[k] & 0x7FFF] << 16,
                            scon[stask[k] >> 16:stask[k + 1] >> 16]) for k in range(slev[p], slev[p + 1])])
        # distance rows: one slot per task, in slot order (every task has two contributions, so the packing
        # keeps slot s in lane s % 32 of round s // 32, as the generic loop runs it)
        drow, ndrow = sec("OKIN_S_DROW"), int(h[D["OKIN_H_NDROW"]])
        phases.append([(drow[s], [drow[ndrow + s], drow[2 * ndrow + s]]) for s in range(ndrow)])
        # linear-model residuals: task = least-squares row, contributions = its JH_CON words in order
        jptr, jcon = sec("OKIN_S_JH_PTR"), sec("OKIN_S_JH_CON")
        phases.append([(t, jcon[jptr[t]:jptr[t + 1]]) for t in range(int(h[D["OKIN_H_NROW"]]))])
        # derived points, per dependency level: all ops, then the active ones only (okin_derived_update).
        # task = output point | op << 16, contributions = {a | b << 16, c | param << 16}, missing inputs = a
        dop = [self.section("OKIN_S_DOP")[k:k + D["OKIN_DOP_STRIDE"]]
               for k in range(0, len(self.section("OKIN_S_DOP")), D["OKIN_DOP_STRIDE"])]
        dlev = sec("OKIN_S_DOP_LEV")
        for active_only in (False, True):
            for lv in range(len(dlev) - 1):
                tasks = []
                for d in range(dlev[lv], dlev[lv + 1]):
                    op, o, ia, ib, ic, p = (int(v) for v in dop[d][:6])
                    if active_only and not dop[d][7]:
                        continue
                    ib, ic = ia if ib < 0 else ib, ia if ic < 0 else ic
                    assert max(o, ia, ib, ic, p) < 1 << 16
                    tasks.append((o | op << 16, [ia | ib << 16, ic | p << 16]))
                phases.append(tasks)
        return phases

    def spec_source(self) -> str:
        """C++ header ``okin_spec.h`` of this program for an OKIN_SPEC build of ``csrc/okin_core.cuh``:
        the header fields as constants, and every hot phase as lane rounds whose task and contribution
        words are packed lane-major into ``okin_spec_words``.  A round takes up to 32 tasks, longest
        contribution list first (a stable sort: tasks with equal-length lists keep their order), so the
        lanes holding slot s are always a prefix of the round."""
        words, phase_round, rounds, slot_lanes = [], [], [], []
        for tasks in self.spec_phases():
            phase_round.append(len(rounds))
            order = sorted(tasks, key=lambda tc: -len(tc[1]))
            for r0 in range(0, len(order), 32):
                chunk = order[r0:r0 + 32]
                width, slots = len(chunk), len(chunk[0][1])
                rounds.append((len(words), width, slots, len(slot_lanes)))
                words += [t for t, _ in chunk]
                for s in range(slots):
                    slot_lanes.append(sum(len(c) > s for _, c in chunk))
                    words += [c[s] if len(c) > s else 0 for _, c in chunk]
        phase_round.append(len(rounds))
        as_i32 = lambda w: str(int(np.int32(np.uint32(w))))   # noqa: E731
        arr = lambda name, vals: (f"constexpr int32_t {name}[] = {{{', '.join(map(str, vals)) or '0'}}};")  # noqa: E731
        hdr = " ".join(f"case {i}: return {int(v)};" for i, v in enumerate(self.hdr[:D["OKIN_H_SEC0"]]) if v)
        col = lambda k: [r[k] for r in rounds]   # noqa: E731
        return "\n".join([
            "// Generated by core/topology.py (TopologyProgram.spec_source) for one topology.",
            "#pragma once",
            f"OKIN_HD constexpr int okin_spec_hdr(int f) {{ switch (f) {{ {hdr} default: return 0; }} }}",
            "namespace okin_spec {",
            arr("PHASE_ROUND", phase_round), arr("R_BASE", col(0)), arr("R_WIDTH", col(1)),
            arr("R_SLOTS", col(2)), arr("R_SLOT0", col(3)), arr("SLOT_LANES", slot_lanes),
            "OKIN_HD constexpr int phase_round(int p) { return PHASE_ROUND[p]; }",
            "OKIN_HD constexpr int r_base(int r) { return R_BASE[r]; }",
            "OKIN_HD constexpr int r_width(int r) { return R_WIDTH[r]; }",
            "OKIN_HD constexpr int r_slots(int r) { return R_SLOTS[r]; }",
            "OKIN_HD constexpr int r_slot0(int r) { return R_SLOT0[r]; }",
            "OKIN_HD constexpr int slot_lanes(int i) { return SLOT_LANES[i]; }",
            f"constexpr int DOP_NLEV = {len(self.section('OKIN_S_DOP_LEV')) - 1};",
            "}  // namespace okin_spec",
            f"#define OKIN_SPEC_WORDS {max(len(words), 1)}",
            "#ifdef __CUDACC__",
            "__device__",
            "#endif",
            f"const int32_t okin_spec_words[OKIN_SPEC_WORDS] = {{{', '.join(map(as_i32, words)) or '0'}}};",
            "",
        ])


# ---------------------------------------------------------------------------
def _constraint_rows(index: int, c: Constraint, pidx: dict, design_rules: bool) -> list:
    """Lower one constraint declaration to least-squares / report rows."""
    RULE_X, RULE_V, RULE_P = D["OKIN_RULE_EXPLICIT"], D["OKIN_RULE_DESIGN_VALUE"], D["OKIN_RULE_DESIGN_POINT"]
    pts = [pidx[k] for k in c.point_keys]
    src = ("constraint", index)
    rule_v = RULE_V if design_rules else RULE_X
    if isinstance(c, DistanceConstraint):
        return [_Row(FAMILY_CODE["distance"], pts, [c.target_distance], rule_v, src)]
    if isinstance(c, SphericalJointConstraint):
        return [_Row(FAMILY_CODE["spherical"], pts, [], RULE_X, src)]
    if isinstance(c, AngleConstraint):
        return [_Row(FAMILY_CODE["angle"], pts, [c.target_angle], rule_v, src)]
    if isinstance(c, ThreePointAngleConstraint):
        return [_Row(FAMILY_CODE["three_point_angle"], pts, [c.target_angle], RULE_X, src)]
    if isinstance(c, VectorsParallelConstraint):
        return [_Row(FAMILY_CODE["vectors_parallel"], pts, [], RULE_X, src)]
    if isinstance(c, VectorsPerpendicularConstraint):
        return [_Row(FAMILY_CODE["vectors_perpendicular"], pts, [], RULE_X, src)]
    if isinstance(c, EqualDistanceConstraint):
        return [_Row(FAMILY_CODE["equal_distance"], pts, [], RULE_X, src)]
    if isinstance(c, ScalarTripleProductConstraint):
        return [_Row(FAMILY_CODE["scalar_triple"], pts, [c.target_volume, 1.0 / c.scale], rule_v, src)]
    if isinstance(c, CoplanarPointsConstraint):
        return [_Row(FAMILY_CODE["coplanar"], pts, [], RULE_X, src)]
    if isinstance(c, FixedAxisConstraint):
        n = np.zeros(3)
        n[int(c.axis)] = 1.0
        return [_Row(FAMILY_CODE["linear_point"], pts, [*(n * c.value), *n], RULE_X, src)]
    if isinstance(c, PointOnPlaneConstraint):
        return [_Row(FAMILY_CODE["linear_point"], pts, [*c.plane_point.data, *c.plane_normal.data], RULE_X, src)]
    if isinstance(c, MidpointOnPlaneConstraint):
        return [_Row(FAMILY_CODE["midpoint_on_plane"], pts, [*c.plane_point.data, *c.plane_normal.data], RULE_X, src)]
    if isinstance(c, PointOnLineConstraint):
        # One scalar row cannot express a 2-DOF restriction and its gradient vanishes on
        # the line; the solve uses two linear pins, the original residual is kept as a
        # report row for max|r| (reference solver.py:735-747).
        d = c.line_direction.data
        n1, n2 = pin_normals(d)
        rule_p = RULE_P if design_rules else RULE_X
        p0 = list(c.line_point.data)
        return [
            _Row(FAMILY_CODE["linear_point"], pts, [*p0, *n1], rule_p, ("pin", index, 0)),
            _Row(FAMILY_CODE["linear_point"], pts, [*p0, *n2], rule_p, ("pin", index, 1)),
            _Row(FAMILY_CODE["point_on_line"], pts, [*p0, *d], rule_p, ("report", index)),
        ]
    raise TypeError(f"No device lowering for {type(c).__name__}")


def _min_degree(nodes, adjacency: list) -> tuple:
    """Greedy minimum-degree ordering of ``nodes`` with symbolic elimination on a copy of the
    graph.  Returns (order, adjacency after eliminating ``nodes``)."""
    adj = [set(a) for a in adjacency]
    alive = set(nodes)
    order = []
    while alive:
        v = min(alive, key=lambda u: (len(adj[u]), u))
        nbrs = set(adj[v])
        order.append(v)
        alive.discard(v)
        for u in nbrs:
            adj[u] |= nbrs - {u}
            adj[u].discard(v)
        adj[v] = set()
    return order, adj


def _components(nodes: set, adjacency: list) -> list:
    comps, seen = [], set()
    for start in sorted(nodes):
        if start in seen:
            continue
        comp, stack = set(), [start]
        while stack:
            v = stack.pop()
            if v in comp:
                continue
            comp.add(v)
            stack.extend(u for u in adjacency[v] if u in nodes and u not in comp)
        seen |= comp
        comps.append(comp)
    return comps


def _symbolic(nf: int, adjacency: list, order: list) -> dict:
    """Symbolic block Cholesky for a given elimination order: structure, levels, cost."""
    adj = [set(a) for a in adjacency]
    pos_of = {v: i for i, v in enumerate(order)}
    struct = []
    for v in order:
        nbrs = {u for u in adj[v] if pos_of[u] > pos_of[v]}
        struct.append(sorted(pos_of[u] for u in nbrs))
        for u in nbrs:
            adj[u] |= nbrs - {u}
            adj[u].discard(v)
    parent = [s[0] if s else -1 for s in struct]
    level = [0] * nf
    for j in range(nf):
        if parent[j] >= 0:
            level[parent[j]] = max(level[parent[j]], level[j] + 1)
    nlev = max(level) + 1 if nf else 0
    return {"order": order, "struct": struct, "level": level, "nlev": nlev,
            "blocks": nf + sum(len(s) for s in struct)}


def _best_order(nf: int, adjacency: list) -> dict:
    """Choose between plain minimum degree and a one-level nested dissection (separator of at
    most two block vertices eliminated last).  The kernel pays one warp synchronisation per
    elimination-tree level in every factor/solve phase, so fewer levels wins; ties go to the
    smaller factor."""
    nodes = set(range(nf))
    candidates = [_symbolic(nf, adjacency, _min_degree(nodes, adjacency)[0])]
    seps = [(v,) for v in range(nf)] + [(u, v) for u in range(nf) for v in range(u + 1, nf)]
    for sep in seps:
        rest = nodes - set(sep)
        comps = _components(rest, adjacency)
        if len(comps) < 2 or max(map(len, comps)) > 0.7 * nf:
            continue
        order, adj = [], adjacency
        for comp in comps:
            part, adj = _min_degree(comp, adj)
            order += part
        tail, _ = _min_degree(set(sep), adj)
        candidates.append(_symbolic(nf, adjacency, order + tail))
    return min(candidates, key=lambda c: (c["nlev"], c["blocks"]))


def compile_topology(
    initial_state,
    constraints: list,
    derived_spec: DerivedPointsSpec,
    targets: list,
    output_points=None,
    design_rules: bool = True,
    metrics=None,
    shims=None,
    diagnostics=None,
    tune_layout: bool = False,
    sensitivity_inputs=None,
) -> TopologyProgram:
    """Compile one topology.

    ``targets``: one ``PointTarget`` per sweep dimension (value ignored; point,
    direction and mode define the row).  ``design_rules=True`` makes the device
    recompute every design constant from each instance's own hardpoints (batch
    use); ``False`` bakes the explicit constants of the given constraint objects
    (the single-instance ``solve_suspension_sweep`` boundary).
    ``sensitivity_inputs``: the ``(input point key, axis)`` hardpoint coordinates whose sensitivities
    the device reports, in row order (default: every coordinate of every input point, slot order).
    """
    positions = initial_state.positions
    manager = DerivedPointsManager(derived_spec)
    derived_keys = list(manager.update_order)
    free_order = list(initial_state.free_points_order)
    if set(free_order) & set(derived_keys):
        raise ValueError("A point cannot be both free and derived")

    point_keys = sorted(positions.keys())
    pidx = {k: i for i, k in enumerate(point_keys)}
    P, NF = len(point_keys), len(free_order)
    col_of = {k: i for i, k in enumerate(free_order)}      # reference column block
    kind = np.zeros(P, np.int32)
    for k in free_order:
        kind[pidx[k]] = D["OKIN_PT_FREE"]
    for k in derived_keys:
        kind[pidx[k]] = D["OKIN_PT_DERIVED"]

    n_res = len(constraints) + len(targets)
    if 3 * NF > n_res:
        raise ValueError(
            f"System is underdetermined (n_vars={3 * NF} > m_res={n_res}). The solve method "
            "(Levenberg-Marquardt) requires at least as many residuals as variables."
        )

    # ---- derived ops -----------------------------------------------------
    in_keys = [k for k in point_keys if k not in derived_spec.functions]
    dops, par_mode, par_val = [], [], []
    dop_of = {}
    # derived points ordered by dependency level so that one level is one parallel phase
    dlevel: dict = {}
    for key in derived_keys:
        deps = [d for d in derived_spec.dependencies[key] if d in derived_spec.functions]
        dlevel[key] = 1 + max((dlevel[d] for d in deps), default=-1)
    derived_keys = sorted(derived_keys, key=lambda k: dlevel[k])   # stable: keeps topological order
    dop_lev = [0]
    for key in derived_keys:
        fn = derived_spec.functions[key]
        if fn.OP not in _DOP_CODE:
            raise TypeError(f"Derived point {key!r}: op {fn.OP!r} cannot be compiled for the device")
        ins = [pidx[k] for k in fn.inputs] + [-1] * (3 - len(fn.inputs))
        authored = -1
        if fn.design_projection is not None and design_rules:
            if fn.design_projection not in in_keys:
                in_keys.append(fn.design_projection)
            par_mode.append(D["OKIN_PAR_DESIGN_PROJECTION"])
        else:
            par_mode.append(D["OKIN_PAR_SHARED"])
        par_val.append(float(fn.param))
        dop_of[key] = len(dops)
        dops.append([_DOP_CODE[fn.OP], pidx[key], ins[0], ins[1], ins[2], len(par_val) - 1, authored, 0])
        while len(dop_lev) <= dlevel[key]:
            dop_lev.append(len(dops) - 1)
    dop_lev.append(len(dops))
    in_keys = sorted(in_keys)
    in_slot = {k: i for i, k in enumerate(in_keys)}
    for key in derived_keys:
        fn = derived_spec.functions[key]
        if fn.design_projection is not None and design_rules:
            dops[dop_of[key]][6] = in_slot[fn.design_projection]

    def base_deps(key) -> list:
        """Free points a derived point depends on (transitively), in column order."""
        seen, stack, out = set(), [key], set()
        while stack:
            k = stack.pop()
            if k in seen:
                continue
            seen.add(k)
            if k in derived_spec.functions:
                stack.extend(derived_spec.dependencies[k])
            elif k in col_of:
                out.add(k)
        return sorted(out, key=lambda k: col_of[k])

    def chain_of(key) -> list:
        """Derived ops needed to evaluate ``key``, in evaluation order."""
        need, stack = set(), [key]
        while stack:
            k = stack.pop()
            if k in derived_spec.functions and k not in need:
                need.add(k)
                stack.extend(derived_spec.dependencies[k])
        return [dop_of[k] for k in derived_keys if k in need]

    # ---- rows --------------------------------------------------------------
    ls_rows, report_rows = [], []
    for ci, c in enumerate(constraints):
        for row in _constraint_rows(ci, c, pidx, design_rules):
            (report_rows if row.source[0] == "report" else ls_rows).append(row)
    trow0 = len(ls_rows)
    if len(targets) > D["OKIN_MAX_TARGETS"]:
        raise ValueError(f"At most {D['OKIN_MAX_TARGETS']} simultaneous sweep targets are supported")
    for ti, t in enumerate(targets):
        if t.point_id not in pidx:
            raise ValueError(f"Sweep target point {t.point_id!r} is not part of the model")
        direction = resolve_target(t.direction).data
        relative = TargetPositionMode(t.mode) == TargetPositionMode.RELATIVE
        base = float(np.dot(positions[t.point_id].data, direction)) if relative else 0.0
        rule = D["OKIN_RULE_TARGET_BASE"] if (relative and design_rules) else D["OKIN_RULE_EXPLICIT"]
        ls_rows.append(_Row(FAMILY_CODE["target"], [pidx[t.point_id]], [*direction, base], rule, ("target", ti), aux=ti))
    rows = ls_rows + report_rows
    NROW, NREP = len(ls_rows), len(report_rows)

    # effective free blocks + slot maps + derived Jacobian storage
    der_desc, der_index = [], {}
    dblk_off, adj_tasks, adj_chain = {}, [], []
    ndb = 0
    ncst = nrg = 0
    for row in rows:
        eff: list = []
        per_slot = []
        for p in row.points:
            key = point_keys[p]
            if key in col_of:
                per_slot.append(("free", [key]))
            elif key in derived_spec.functions:
                per_slot.append(("derived", base_deps(key)))
            else:
                per_slot.append(("fixed", []))
            for dep in per_slot[-1][1]:
                if col_of[dep] not in eff:
                    eff.append(col_of[dep])
        row.eff = eff
        is_ls = row.source[0] != "report"
        for (what, deps), p in zip(per_slot, row.points):
            if what == "fixed" or (what == "derived" and not deps) or not is_ls:
                row.slotmap.append(-1)
            elif what == "free":
                row.slotmap.append(eff.index(col_of[deps[0]]))
            else:
                key = point_keys[p]
                if len(deps) > 3:
                    raise ValueError(f"Derived point {key!r} depends on more than 3 free points")
                desc = [len(deps)]
                for dep in deps:
                    if (key, dep) not in dblk_off:
                        dblk_off[(key, dep)] = ndb
                        chain = chain_of(key)
                        if len(chain) > D["OKIN_MAX_CHAIN"]:
                            raise ValueError(f"Derived chain of {key!r} is longer than {D['OKIN_MAX_CHAIN']}")
                        begin = len(adj_chain)
                        adj_chain.extend(chain)
                        for op_index in chain:
                            dops[op_index][7] = 1      # evaluated inside the solve iterations
                        for comp in range(3):
                            adj_tasks.append([pidx[key], pidx[dep], comp, ndb, begin, len(adj_chain), 0, 0])
                        ndb += 9
                    desc += [dblk_off[(key, dep)], eff.index(col_of[dep])]
                desc += [0] * (D["OKIN_DER_STRIDE"] - len(desc))
                tdesc = tuple(desc)
                if tdesc not in der_index:
                    der_index[tdesc] = len(der_desc)
                    der_desc.append(desc)
                row.slotmap.append(D["OKIN_SLOT_DER"] + der_index[tdesc])
        row.slotmap += [-1] * (4 - len(row.slotmap))
        row.cst_off = ncst
        ncst += len(row.consts)
        row.rg_off = nrg
        row.fast = (is_ls and row.fam == FAMILY_CODE["distance"]
                    and all(what != "derived" for what, _ in per_slot) and len(eff) >= 1)
        if row.fast:
            # sign of dR/d(block e) relative to the stored u = (p2 - p1)/|p2 - p1|
            row.eff_sign = [(-1 if col_of.get(point_keys[row.points[0]]) == c else +1) for c in eff]
            nrg += 3
        elif is_ls:
            nrg += 3 * len(eff)
    rg_zero = nrg           # a 3-vector that stays zero (padding target for fixed-length gathers)
    nrg += 3
    if nrg >= 32768:
        raise ValueError("Row-gradient storage exceeds the 15-bit index range")

    # ---- elimination order and symbolic block Cholesky ----------------------
    adjacency = [set() for _ in range(NF)]
    for row in ls_rows:
        for a in row.eff:
            for b in row.eff:
                if a != b:
                    adjacency[a].add(b)
    sym = _best_order(NF, adjacency)
    order, struct, level, NLEV = sym["order"], sym["struct"], sym["level"], sym["nlev"]
    pos_of = {v: i for i, v in enumerate(order)}             # column block -> elimination position

    block_id = {}
    for j in range(NF):
        block_id[(j, j)] = len(block_id)
        for i in struct[j]:
            block_id[(i, j)] = len(block_id)
    NB = len(block_id)
    if 9 * NB >= 32768:
        raise ValueError("Factor storage exceeds the 15-bit offset range")

    def boff(i, j) -> int:
        return 9 * block_id[(i, j)]

    # ---- optional: conflict-aware order of the row-gradient vectors (core/layout_tuning.py) --------
    rg_tuning = None
    if tune_layout:
        from .layout_tuning import UnitTrace, tune_unit_order
        units = [r for r in rows if r in ls_rows]               # rows that own gradient storage
        unit_of = {id(r): u for u, r in enumerate(units)}
        sizes = [3 if r.fast else 3 * len(r.eff) for r in units]

        def gref(r, e):                                          # (unit, offset) of d row / d block e
            return unit_of[id(r)], 0 if r.fast else 3 * e

        pattern: dict = {}
        for r in ls_rows:
            for ea, ca in enumerate(r.eff):
                for eb, cb in enumerate(r.eff):
                    pa, pb = pos_of[ca], pos_of[cb]
                    if pa < pb or (pa == pb and ea != eb):
                        continue
                    pattern.setdefault((pa, pb), []).append((gref(r, ea), gref(r, eb)))
        order_tasks = sorted(block_id.items(), key=lambda kv: (-len(pattern.get(kv[0], [])), kv[1]))
        rg_base = 3 * P + max(ncst, 1) + len(rows)
        trace = UnitTrace(rg_base, sizes)
        for r0 in range(0, len(order_tasks), 32):               # assembly: gradient pairs of every block
            ts = [pattern.get(k, []) for k, _ in order_tasks[r0:r0 + 32]]
            for q in range(max(len(c) for c in ts)):
                act = [(n, c[q]) for n, c in enumerate(ts) if len(c) > q]
                trace.access([n for n, _ in act], [c[0] for _, c in act], (0, 1, 2))
                trace.access([n for n, _ in act], [c[1] for _, c in act], (0, 1, 2))
        per_col: dict = {}
        for r in ls_rows:
            for e, cblk in enumerate(r.eff):
                per_col.setdefault(pos_of[cblk], []).append(gref(r, e))
        cols = [per_col.get(j, []) for j in range(NF)]
        for r0 in range(0, NF, 32):                              # g = J^T r, one lane per block column
            ts = cols[r0:r0 + 32]
            for q in range(max(len(c) for c in ts)):
                act = [(n, c[q]) for n, c in enumerate(ts) if len(c) > q]
                trace.access([n for n, _ in act], [c for _, c in act], (0, 1, 2))
        fast = [r for r in rows if r.fast]
        for r0 in range(0, len(fast), 32):                       # fast distance rows store u
            trace.access(list(range(len(fast[r0:r0 + 32]))), [gref(r, 0) for r in fast[r0:r0 + 32]], (0, 1, 2))
        rg_order, before, after, ideal = tune_unit_order(trace)
        start = trace.offsets(rg_order)
        first = min(r.rg_off for r in units)
        for u, r in enumerate(units):
            r.rg_off = first + int(start[u])
        rg_tuning = {"wavefronts_before": before, "wavefronts_after": after, "wavefronts_ideal": ideal}

    # ---- assembly gather lists (A = J^T J), one task per 3x3 block ----------------
    # contribution = (rg offset of the row's gradient w.r.t. the block-row point) << 16 |
    #                (rg offset of its gradient w.r.t. the block-column point)
    contrib: dict = {}
    for row in ls_rows:
        for ea, ca in enumerate(row.eff):
            for eb, cb in enumerate(row.eff):
                pa, pb = pos_of[ca], pos_of[cb]
                if pa < pb or (pa == pb and ea != eb):
                    continue
                (oa, na), (ob, nb) = row.grad_ref(ea), row.grad_ref(eb)
                word = (oa << 16) | ob | (D["OKIN_CON_NEG"] if na != nb else 0)
                contrib.setdefault((pa, pb), []).append(word)
    tasks = sorted(block_id.items(), key=lambda kv: (-len(contrib.get(kv[0], [])), kv[1]))
    asm_ptr, asm_task, asm_con = [0], [], []
    for (i, j), b in tasks:       # heaviest first: lanes take tasks round-robin
        asm_task.append(b | (D["OKIN_ASM_DIAG"] if i == j else 0))
        asm_con.extend(contrib.get((i, j), []))
        asm_ptr.append(len(asm_con))
    NAT = len(asm_task)

    g_ptr, g_con = [0], []
    row_index = {id(row): i for i, row in enumerate(rows)}
    per_block: dict = {}
    for row in ls_rows:
        for e, cblk in enumerate(row.eff):
            off_e, neg = row.grad_ref(e)
            per_block.setdefault(pos_of[cblk], []).append(
                (off_e << 16) | row_index[id(row)] | (D["OKIN_CON_NEG"] if neg else 0))
    for j in range(NF):
        g_con.extend(per_block.get(j, []))
        g_ptr.append(len(g_con))

    # ---- row-wise Jacobian lists (r + J h of the linear model, okin_linear_residuals) ------------
    # per least-squares row: (rg offset of its gradient w.r.t. one effective block) << 16 | 3 * that
    # block's elimination position, same sign convention as the assembly words
    jh_ptr, jh_con = [0], []
    for row in ls_rows:
        for e, cblk in enumerate(row.eff):
            off_e, neg = row.grad_ref(e)
            jh_con.append((off_e << 16) | (3 * pos_of[cblk]) | (D["OKIN_CON_NEG"] if neg else 0))
        jh_ptr.append(len(jh_con))
    # report rows (original point-on-line residuals) as softnorm of their two pin rows
    pin_row = {}
    for i, row in enumerate(ls_rows):
        if row.source[0] == "pin":
            pin_row[(row.source[1], row.source[2])] = i
    rep_pins = []
    for row in report_rows:
        rep_pins += [pin_row[(row.source[1], 0)], pin_row[(row.source[1], 1)]]

    # ---- left-looking update lists, scale tasks -------------------------------
    # One task per block *row* (3 entries): acc[c] -= a . B[c][:] for earlier columns K,
    # a = row r of L_iK, B = L_jK.  The right-hand side of the step equation is carried as one
    # extra block-row of the factor (a = y_K), which makes the forward substitution part of the
    # factorisation; the tangent right-hand sides ride along the same way.  Offsets are relative
    # to the instance's shared-memory base.  The contribution of column K runs in the update phase
    # of some level in [level(K) + 1, level(j)] (core/schedule.py), so a destination may be visited
    # by one task in each of several levels.
    cols_with = [[] for _ in range(NF)]        # cols_with[j] = K < j with L_jK != 0
    for k in range(NF):
        for i in struct[k]:
            cols_with[i].append(k)
    lev_cols = [[j for j in range(NF) if level[j] == lv] for lv in range(NLEV)]
    LB, VEC = "LB", "VEC"      # symbolic bases, resolved once the layout is known

    # destinations: (block row i of column j, or i = None for the carried right-hand sides, its sources)
    upd_dests = []
    for lv in range(NLEV):
        for j in lev_cols[lv]:
            for i in [j] + struct[j]:
                ks = [k for k in cols_with[j] if i == j or i in struct[k]]
                if ks:
                    upd_dests.append((i, j, ks))
            if cols_with[j]:
                upd_dests.append((None, j, cols_with[j]))
    upd_phase, upd_before, upd_after = schedule(
        [Dest(1 if i is None else 3, level[j], [level[k] + 1 for k in ks]) for i, j, ks in upd_dests], NLEV)

    lev_upd, upd_dst, upd_ptr, upd_con = [0], [], [0], []
    lev_scl, scl = [0], []
    lev_upd_mid, lev_scl_mid = [], []   # end of the tasks a solve without tangents needs, per level

    def add_update(dst, cons):
        upd_dst.append(dst)
        upd_con.extend(cons)
        upd_ptr.append(len(upd_con))

    for lv in range(NLEV):
        # heaviest first; block rows and the step right-hand side before the tangent right-hand sides: a
        # solve that does not carry tangents (lean kernel) stops at the "mid" pointer of the level
        here = [(d, [k for k, p in zip(ks, upd_phase[d]) if p == lv]) for d, (_, _, ks) in enumerate(upd_dests)]
        here = sorted((t for t in here if t[1]), key=lambda t: -len(t[1]))
        for tangent_pass in (False, True):
            for d, ks in here:
                i, j, _ = upd_dests[d]
                if i is not None and not tangent_pass:
                    for r in range(3):
                        add_update((LB, boff(i, j) + 3 * r),
                                   [((LB, boff(i, k) + 3 * r), (LB, boff(j, k))) for k in ks])
                elif i is None:
                    for rhs in (range(1, 1 + len(targets)) if tangent_pass else (0,)):
                        # carried right-hand sides: step (0) and tangents (1..NT)
                        add_update((VEC, rhs * 3 * NF + 3 * j),
                                   [((VEC, rhs * 3 * NF + 3 * k), (LB, boff(j, k))) for k in ks])
            for j in lev_cols[lv]:
                if not tangent_pass:
                    for i in struct[j]:
                        for r in range(3):
                            scl.append(((LB, boff(j, j)), (LB, boff(i, j) + 3 * r)))
                for rhs in (range(1, 1 + len(targets)) if tangent_pass else (0,)):
                    scl.append(((LB, boff(j, j)), (VEC, rhs * 3 * NF + 3 * j)))
            if not tangent_pass:
                lev_upd_mid.append(len(upd_dst))
                lev_scl_mid.append(len(scl))
        lev_upd.append(len(upd_dst))
        lev_scl.append(len(scl))

    # per-column lists of the factor products L z / L^T z (okin_factor_multiply)
    fw_ptr, fw_con, bw_ptr, bw_con = [0], [], [0], []
    for j in range(NF):
        for k in cols_with[j]:
            fw_con.append(((LB, boff(j, k)), 3 * k))
        fw_ptr.append(len(fw_con))
        for i in struct[j]:
            bw_con.append(((LB, boff(i, j)), 3 * i))
        bw_ptr.append(len(bw_con))
    lev_col_ptr, lev_col = [0], []
    for lv in range(NLEV):
        lev_col.extend(lev_cols[lv])
        lev_col_ptr.append(len(lev_col))

    # triangular solves: per phase, tasks {destination column j, finalise flag, its contributions}.  The
    # forward phases run the levels upwards (y_K is final after level(K)), the backward ones from the
    # root down (x_I is final after level(I)); a column is finalised (3x3 diagonal solve) in its own level.
    fw_phase, fw_before, fw_after = schedule(
        [Dest(1, level[j], [level[k] + 1 for k in cols_with[j]], True) for j in range(NF)], NLEV)
    bw_phase, bw_before, bw_after = schedule(
        [Dest(1, NLEV - 1 - level[j], [NLEV - level[i] for i in struct[j]], True) for j in range(NF)], NLEV)
    sol_lev, sol_task = [], []        # task = (column, finalise, [(block ref, 3 * source column)])
    for srcs, phase, of in ((cols_with, fw_phase, lambda j, k: boff(j, k)), (struct, bw_phase, lambda j, i: boff(i, j))):
        for ph in range(NLEV):
            sol_lev.append(len(sol_task))
            here = []
            for j in range(NF):
                cons = [((LB, of(j, s)), 3 * s) for s, p in zip(srcs[j], phase[j]) if p == ph]
                fin = ph == (level[j] if srcs is cols_with else NLEV - 1 - level[j])
                if cons or fin:
                    here.append((j, fin, cons))
            sol_task += sorted(here, key=lambda t: -len(t[2]))
        sol_lev.append(len(sol_task))
    sched_stats = {"factor_update": {"before": upd_before, "after": upd_after},
                   "forward_solve": {"before": fw_before, "after": fw_after},
                   "backward_solve": {"before": bw_before, "after": bw_after}}

    elim_point = [pidx[free_order[order[j]]] for j in range(NF)]
    elim_col = [order[j] for j in range(NF)]

    # tangent right-hand sides: gradient of each target row scattered to unknowns
    tgt_sc_ptr, tgt_sc = [0], []
    for row in ls_rows[trow0:]:
        for e, cblk in enumerate(row.eff):
            for r in range(3):
                tgt_sc.append(((row.rg_off + 3 * e + r) << 16) | (3 * pos_of[cblk] + r))
        tgt_sc_ptr.append(len(tgt_sc))

    out_keys = list(output_points) if output_points is not None else list(point_keys)
    for k in out_keys:
        if k not in pidx:
            raise ValueError(f"Output point {k!r} is not part of the model")

    # ---- fast distance rows: {p0 | p1 << 16, cst_off | rg_off << 16, row index}
    fast_rows = [(i, row) for i, row in enumerate(rows) if row.fast]
    drows = ([row.points[0] | (row.points[1] << 16) for _, row in fast_rows]
             + [row.cst_off | (row.rg_off << 16) for _, row in fast_rows] + [i for i, _ in fast_rows])

    # ---- evaluation order: rows of one family are adjacent so that a 32-row round of the
    # evaluation phase runs (mostly) one code path
    row_order = sorted((i for i in range(len(rows)) if not rows[i].fast), key=lambda i: (rows[i].fam, i))

    # ---- shared-memory layout (doubles) -----------------------------------------------
    NT = len(targets)
    N = 3 * NF
    off = 0

    def take(n: int) -> int:
        nonlocal off
        start = off
        off += n
        return start

    # What a solve without tangents / metrics needs comes first: the lean kernel instantiation only
    # reserves the slice up to the end of vec[0] (OKIN_H_SMEM_DOUBLES_LEAN).
    layout = {
        "OKIN_H_OFF_POS": take(3 * P), "OKIN_H_OFF_CST": take(max(ncst, 1)), "OKIN_H_OFF_R": take(NROW + NREP),
        "OKIN_H_OFF_RG": take(max(nrg, 1)), "OKIN_H_OFF_DBLK": take(max(ndb, 1)),
        "OKIN_H_OFF_LB": take(9 * NB),
        "OKIN_H_OFF_RED": take(32), "OKIN_H_OFF_PAR": take(max(len(par_val), 1)),
        "OKIN_H_OFF_TGT": take(2 * D["OKIN_MAX_TARGETS"]),
        # extrapolation predictor: previous solution (doubles) + three older increments (float32 pairs)
        "OKIN_H_OFF_XPREV": take(N), "OKIN_H_OFF_DHIST": take(3 * ((N + 1) // 2)),
        "OKIN_H_OFF_VEC": take(N),
    }
    layout["OKIN_H_SMEM_DOUBLES_LEAN"] = off
    take(NT * N)                         # vec[1..NT]: tangents (contiguous with vec[0])
    if off >= 65536:
        raise ValueError("Per-instance state exceeds the 16-bit shared-memory offset range")
    base = {LB: layout["OKIN_H_OFF_LB"], VEC: layout["OKIN_H_OFF_VEC"]}

    # ---- optional: bank-conflict-aware placement of the factor blocks (core/layout_tuning.py) ------
    slot = list(range(NB))
    tuning = None
    if tune_layout and NB > 1:
        from .layout_tuning import AccessTrace, tune_block_slots
        trace = AccessTrace(base[LB])

        def ref(r):
            return ("LB", r[1]) if r[0] == LB else ("ABS", base[r[0]] + r[1])

        for lv in range(NLEV):
            for r0 in range(lev_upd[lv], lev_upd[lv + 1], 32):          # update rounds
                ts = range(r0, min(r0 + 32, lev_upd[lv + 1]))
                lanes = [t - r0 for t in ts]
                trace.access(lanes, [ref(upd_dst[t]) for t in ts], (0, 1, 2))          # load c0..c2
                for q in range(max(upd_ptr[t + 1] - upd_ptr[t] for t in ts)):
                    act = [t for t in ts if upd_ptr[t + 1] - upd_ptr[t] > q]
                    la = [t - r0 for t in act]
                    trace.access(la, [ref(upd_con[upd_ptr[t] + q][0]) for t in act], (0, 1, 2))
                    trace.access(la, [ref(upd_con[upd_ptr[t] + q][1]) for t in act], range(9))
                trace.access(lanes, [ref(upd_dst[t]) for t in ts], (0, 1, 2))          # store
            for r0 in range(lev_scl[lv], lev_scl[lv + 1], 32):          # scale rounds
                ts = range(r0, min(r0 + 32, lev_scl[lv + 1]))
                lanes = [t - r0 for t in ts]
                trace.access(lanes, [ref(scl[t][0]) for t in ts], (1, 3, 4, 6, 7, 8))
                trace.access(lanes, [ref(scl[t][1]) for t in ts], (0, 1, 2, 0, 1, 2))   # load + store
        nrhs = 1 + len(targets)
        for ph in range(NLEV):                                        # backward solve, all right-hand sides
            tasks = [t for t in sol_task[sol_lev[NLEV + 1 + ph]:sol_lev[NLEV + 2 + ph]] for _ in range(nrhs)]
            for r0 in range(0, len(tasks), 32):
                ts = tasks[r0:r0 + 32]
                for q in range(max(len(t[2]) for t in ts)):
                    act = [(n, t) for n, t in enumerate(ts) if len(t[2]) > q]
                    trace.access([n for n, _ in act], [ref(t[2][q][0]) for _, t in act], range(9))
                fin = [(n, t[0]) for n, t in enumerate(ts) if t[1]]
                trace.access([n for n, _ in fin], [("LB", boff(j, j)) for _, j in fin], (1, 3, 4, 6, 7, 8))
        for r0 in range(0, NAT, 32):                                  # assembly: block stores
            ts = range(r0, min(r0 + 32, NAT))
            trace.access([t - r0 for t in ts], [("LB", 9 * (asm_task[t] & 0xFFFF)) for t in ts], range(9))
        tuned, before, after, ideal = tune_block_slots(trace, NB)
        slot = [int(v) for v in tuned]
        tuning = {"wavefronts_before": before, "wavefronts_after": after, "wavefronts_ideal": ideal,
                  "row_gradients": rg_tuning}

    def sm(ref) -> int:
        if ref[0] == LB:
            return base[LB] + 9 * slot[ref[1] // 9] + ref[1] % 9
        return base[ref[0]] + ref[1]

    asm_task = [(t & ~0xFFFF) | slot[t & 0xFFFF] for t in asm_task]
    diag_off = [sm((LB, boff(j, j))) for j in range(NF)]
    upd_dst = [sm(d) for d in upd_dst]
    upd_con = [(sm(a) << 16) | sm(b) for a, b in upd_con]
    scl = [sm(d) | (sm(r) << 16) for d, r in scl]
    fw_con = [(sm(b) << 16) | v for b, v in fw_con]
    bw_con = [(sm(b) << 16) | v for b, v in bw_con]
    sol_con, sol_words = [], []
    for j, fin, cons in sol_task:
        sol_words.append((len(sol_con) << 16) | (D["OKIN_SOLVE_FIN"] if fin else 0) | j)
        sol_con += [(sm(b) << 16) | v for b, v in cons]
    sol_words.append(len(sol_con) << 16)          # end of the last task's contributions
    if len(sol_con) >= 65536:
        raise ValueError("Triangular-solve lists exceed the 16-bit index range")

    # ---- blobs ------------------------------------------------------------------
    row_tab = []
    for row in rows:
        pts = row.points + [-1] * (4 - len(row.points))
        rec = [row.fam, *pts, row.cst_off, row.rg_off, len(row.eff), row.rule, *row.slotmap, row.aux]
        row_tab.append(rec + [0] * (D["OKIN_ROW_STRIDE"] - len(rec)))
    row_hot = []
    for i in row_order:
        rec = list(row_tab[i])
        rec[D["OKIN_R_ROWID"]] = i
        row_hot.append(rec)
    cst_init = [v for row in rows for v in row.consts]

    point_elim = [-1] * P
    for j in range(NF):
        point_elim[elim_point[j]] = j
    point_dop = [-1] * P
    for key, d in dop_of.items():
        point_dop[pidx[key]] = d
    shim_recs, shim_pts, param_default, param_names = [], [], [], []
    for sh in (shims or []):
        ix = lambda k: -1 if k is None else pidx[k]   # noqa: E731
        up_begin = len(shim_pts)
        shim_pts += [pidx[k] for k in sh["upright_points"]]
        rk_begin = len(shim_pts)
        shim_pts += [pidx[k] for k in sh["rocker_points"]]
        rocker = sh.get("rocker")
        rec = [ix(sh["ubj"]), ix(sh["lbj"]), ix(sh["uw_front"]), ix(sh["uw_rear"]), ix(sh["heading_in"]),
               ix(sh["heading_out"]), 1 if rocker else 0,
               *([ix(k) for k in rocker] if rocker else [-1, -1, -1, -1]),
               len(param_default), up_begin, rk_begin, rk_begin, len(shim_pts)]
        shim_recs.append(rec + [0] * (D["OKIN_SHIM_STRIDE"] - len(rec)))
        param_default += [float(v) for v in sh["params"]]
        param_names += [f"{sh['label']}.{n}" for n in (
            "face_a.x", "face_a.y", "face_a.z", "face_b.x", "face_b.y", "face_b.z", "normal.x", "normal.y",
            "normal.z", "design_thickness", "setup_thickness")]
    if len(shim_recs) > 32:
        raise ValueError("At most 32 shimmed corners per topology")
    mprog = metrics(pidx) if metrics is not None else None
    mcorners = mprog.corners if mprog else []
    mops = mprog.mops if mprog else []
    maxle = [mprog.axle] if (mprog and mprog.axle) else []
    design_pts = mprog.design_pts if mprog else []
    mconst = mprog.fconst if mprog else []
    metric_names = list(mprog.names) if mprog else []
    design_pts = list(design_pts)
    dprog = diagnostics(pidx, design_pts) if diagnostics is not None else None
    free_out = [out_keys.index(k) if k in out_keys else -1 for k in free_order]
    if sensitivity_inputs is None:
        sensitivity_inputs = [(k, axis) for k in in_keys for axis in range(3)]
    sensitivity_inputs = [(k, int(axis)) for k, axis in sensitivity_inputs]
    for k, axis in sensitivity_inputs:
        if k not in in_slot or axis not in (0, 1, 2):
            raise ValueError(f"Sensitivity input {(k, axis)!r} is not a hardpoint coordinate of this topology")
    ndsn = len(design_pts)
    layout["OKIN_H_OFF_DSN"] = take(max(3 * ndsn, 1))
    layout["OKIN_H_OFF_MCTX"] = take(4 * max(len(mcorners), 2))

    isecs = {
        "OKIN_S_POINT_KIND": kind, "OKIN_S_IN_POINT": [pidx[k] for k in in_keys],
        "OKIN_S_DOP": dops, "OKIN_S_PAR_MODE": par_mode, "OKIN_S_ADJ": adj_tasks, "OKIN_S_ADJ_CHAIN": adj_chain,
        "OKIN_S_ROW": row_tab, "OKIN_S_DER": der_desc,
        "OKIN_S_ASM_PTR": asm_ptr, "OKIN_S_ASM_TASK": asm_task, "OKIN_S_ASM_CON": asm_con,
        "OKIN_S_G_PTR": g_ptr, "OKIN_S_G_CON": g_con,
        "OKIN_S_LEV_UPD_MID": lev_upd_mid, "OKIN_S_LEV_SCL_MID": lev_scl_mid,
        "OKIN_S_JH_PTR": jh_ptr, "OKIN_S_JH_CON": jh_con, "OKIN_S_REP_PINS": rep_pins,
        "OKIN_S_LEV_UPD": lev_upd, "OKIN_S_UPD_DST": upd_dst, "OKIN_S_UPD_PTR": upd_ptr, "OKIN_S_UPD_CON": upd_con,
        "OKIN_S_LEV_SCL": lev_scl, "OKIN_S_SCL": scl,
        "OKIN_S_LEV_COL_PTR": lev_col_ptr, "OKIN_S_LEV_COL": lev_col,
        "OKIN_S_SOLVE_LEV": sol_lev, "OKIN_S_SOLVE_TASK": sol_words, "OKIN_S_SOLVE_CON": sol_con,
        "OKIN_S_FW_PTR": fw_ptr, "OKIN_S_FW_CON": fw_con, "OKIN_S_BW_PTR": bw_ptr, "OKIN_S_BW_CON": bw_con,
        "OKIN_S_ELIM_POINT": elim_point, "OKIN_S_ELIM_COL": elim_col,
        "OKIN_S_TGT_SC_PTR": tgt_sc_ptr, "OKIN_S_TGT_SC": tgt_sc,
        "OKIN_S_OUT_POINT": [pidx[k] for k in out_keys], "OKIN_S_ROW_ORDER": row_order, "OKIN_S_DROW": drows, "OKIN_S_DIAG_OFF": diag_off,
        "OKIN_S_DOP_LEV": dop_lev, "OKIN_S_POINT_ELIM": point_elim, "OKIN_S_POINT_DOP": point_dop,
        "OKIN_S_DESIGN_PT": design_pts, "OKIN_S_MCORNER": mcorners, "OKIN_S_MOP": mops, "OKIN_S_MAXLE": maxle,
        "OKIN_S_SHIM": shim_recs, "OKIN_S_SHIM_PTS": shim_pts,
        "OKIN_S_FREE_OUT": free_out, "OKIN_S_DGOP": dprog.ops if dprog else [],
        "OKIN_S_ELIM_OUT": [free_out[c] for c in elim_col],
        "OKIN_S_SENS_IN": [3 * in_slot[k] + axis for k, axis in sensitivity_inputs],
    }
    isecs["OKIN_S_ROW_HOT"] = row_hot
    # Cold sections (setup, outputs requested per state, metrics, diagnostics) go last: the kernel
    # copies only the hot prefix of the blob to shared memory.
    cold = [k for k in isecs if D[k] >= D["OKIN_S_COLD0"]]
    isecs = {**{k: v for k, v in isecs.items() if k not in cold}, **{k: isecs[k] for k in cold}}
    hdr = np.zeros(D["OKIN_HDR_SIZE"], np.int32)
    chunks, cursor, n_hot = [], 0, None
    for name, data in isecs.items():
        if name == cold[0]:
            n_hot = cursor
        arr = np.asarray(data, dtype=np.int64).reshape(-1)
        if arr.size and (arr.max() > 2**32 - 1 or arr.min() < -(2**31)):
            raise ValueError(f"section {name} overflows 32 bits")
        s = D[name]
        hdr[D["OKIN_H_SEC0"] + 2 * s] = cursor
        hdr[D["OKIN_H_SEC0"] + 2 * s + 1] = arr.size
        chunks.append((arr & 0xFFFFFFFF).astype(np.uint32).view(np.int32))   # flag bit 31 wraps to sign
        cursor += arr.size
    iblob = np.concatenate(chunks) if chunks else np.zeros(0, np.int32)
    fsecs = {"OKIN_F_PAR_VAL": par_val, "OKIN_F_CST_INIT": cst_init, "OKIN_F_MCONST": mconst,
             "OKIN_F_PARAM_DEFAULT": param_default}
    fchunks, cursor = [], 0
    for name, data in fsecs.items():
        arr = np.asarray(data, dtype=np.float64).reshape(-1)
        s = D[name]
        hdr[D["OKIN_H_FSEC0"] + 2 * s] = cursor
        hdr[D["OKIN_H_FSEC0"] + 2 * s + 1] = arr.size
        fchunks.append(arr)
        cursor += arr.size
    fblob = np.concatenate(fchunks) if fchunks else np.zeros(0, np.float64)
    if fblob.size == 0:
        fblob = np.zeros(1, np.float64)

    counts = {
        "OKIN_H_MAGIC": D["OKIN_MAGIC"], "OKIN_H_P": P, "OKIN_H_NF": NF, "OKIN_H_NIN": len(in_keys),
        "OKIN_H_NDOP": len(dops), "OKIN_H_NPAR": len(par_val), "OKIN_H_NROW": NROW, "OKIN_H_NREP": NREP,
        "OKIN_H_NT": NT, "OKIN_H_NCST": ncst, "OKIN_H_NRG": nrg, "OKIN_H_NAD": len(adj_tasks), "OKIN_H_NDB": ndb,
        "OKIN_H_NB": NB, "OKIN_H_NLEV": NLEV, "OKIN_H_NAT": NAT, "OKIN_H_NOUT": len(out_keys),
        "OKIN_H_TROW0": trow0, "OKIN_H_SMEM_DOUBLES": off, "OKIN_H_NM": len(metric_names),
        "OKIN_H_NMC": len(mcorners), "OKIN_H_NMOP": len(mops), "OKIN_H_NMAXLE": len(maxle), "OKIN_H_NDSN": ndsn,
        "OKIN_H_NSHIM": len(shim_recs), "OKIN_H_NPARAM": len(param_default),
        "OKIN_H_NDROW": len(fast_rows), "OKIN_H_NGROW": len(row_order),
        "OKIN_H_FREE_ALL_OUT": int(all(v >= 0 for v in free_out)),
        "OKIN_H_NHOT": n_hot, "OKIN_H_NSENS": len(sensitivity_inputs), "OKIN_H_NDIAG": len(dprog.names) if dprog else 0, "OKIN_H_NDGOP": len(dprog.ops) if dprog else 0,
        **layout,
    }
    for name, value in counts.items():
        hdr[D[name]] = value

    dense_flops = 2 * N**3 // 3
    stats = {
        "n_points": P, "n_free": NF, "n_unknowns": N, "n_rows": NROW, "n_report_rows": NREP, "n_targets": NT,
        "n_blocks": NB, "n_levels": NLEV, "fill_blocks": NB - NF - sum(len(a) for a in adjacency) // 2,
        "asm_fma": 9 * len(asm_con), "g_fma": 3 * len(g_con), "update_fma": 9 * len(upd_con),
        "scale_tasks": len(scl) + NF, "solve_fma": 9 * (len(fw_con) + len(bw_con)) + 12 * NF,
        "smem_doubles": off, "iblob_words": int(iblob.size), "dense_lu_flops": dense_flops,
        "layout_tuning": tuning, "schedule_wavefronts": sched_stats,
    }
    return TopologyProgram(
        hdr=hdr, iblob=iblob, fblob=fblob, point_keys=point_keys, free_order=free_order, in_keys=in_keys,
        out_keys=out_keys, n_constraints=len(constraints), row_source=[r.source for r in rows],
        target_points=[t.point_id for t in targets], stats=stats, metric_names=metric_names,
        metric_locations=list(mprog.locations) if mprog else [],
        diagnostic_names=list(dprog.names) if dprog else [],
        diagnostic_checks=list(dprog.checks) if dprog else [],
        param_names=param_names, param_default=np.asarray(param_default, dtype=np.float64),
        sensitivity_inputs=sensitivity_inputs,
    )


def structure_point_index(suspension) -> dict:
    """``{point key: index}`` of a suspension's points in the compiled topology (sorted keys), without
    compiling anything."""
    state, _ = suspension.structure()
    return {k: i for i, k in enumerate(sorted(state.positions.keys()))}


def compile_suspension(suspension, sweep_config, output_points=None, design_rules: bool = True,
                       with_metrics: bool = True, tune_layout: bool = False, sensitivity_inputs=None,
                       with_shims: bool = True) -> TopologyProgram:
    """Compile a built suspension + sweep (first-step targets define the target rows).
    ``with_shims=False`` leaves the camber-shim pre-solve out (hardpoint sensitivities need that; the
    caller must make sure every shim is at its design thickness)."""
    from .diagnostics_program import build_diagnostic_program
    from .metrics_program import build_metric_program
    from .shim_program import shim_records

    targets = [sweep[0] for sweep in sweep_config.target_sweeps]
    metrics = (lambda pidx: build_metric_program(suspension, targets, pidx)) if with_metrics else None
    state, constraints = suspension.structure() if design_rules else (suspension.initial_state(),
                                                                       suspension.constraints())
    return compile_topology(
        state, constraints, suspension.derived_spec(), targets,
        output_points=output_points, design_rules=design_rules, metrics=metrics,
        shims=shim_records(suspension) if (design_rules and with_shims) else None,
        diagnostics=lambda pidx, design_pts: build_diagnostic_program(suspension, pidx, design_pts),
        tune_layout=tune_layout, sensitivity_inputs=sensitivity_inputs,
    )
