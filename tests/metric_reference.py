"""Plain high-precision restatement of every metric column (mpmath, 32 digits).

Each column is computed from point positions looked up by the column's name and the suspension
type -- never from the records of ``core/metrics_program.py`` -- so a wrong index, side or constant
in the program builder, or a wrong formula in ``csrc/okin_metrics.cuh`` / ``okin_core.cuh``, shows up
as a disagreement.  The definitions are those cited in the headers of both files (reference
``metrics/catalog.py``, ``context.py``, ``angles.py``, ``steering_geometry.py``, ``swing_arms.py``,
``travel.py``, ``anti_geometry.py``, ``axle_metrics.py``, the mechanism metrics of
``corner/mechanisms.py`` / ``axle/mechanisms.py`` and ``metrics/derivatives.py``):

* instant centres: the instant axis is the line common to two planes (double wishbone: the upper
  and the lower arm planes; MacPherson: the lower-arm plane and the plane through the strut top
  normal to the steering axis, lower ball joint -> strut top).  The side-view centre is where that
  line crosses the plane y = wheel-centre y, the front-view centre where it crosses x = wheel-centre
  x; both are solved here as one 3x3 linear system;
* anti geometry (side-view swing arm from the contact patch, height of the centre of gravity above
  the contact patch): front axle, brake bias b: anti_dive = 100 b (wb / h) (svic_z - cp_z) /
  (cp_x - svic_x); rear axle: anti_lift = 100 (1 - b) (wb / h) (svic_z - cp_z) / (svic_x - cp_x);
  driven axle: anti_squat = 100 (wb / h) (svic_z - wc_z) / run with run = wc_x - svic_x at the front
  and svic_x - wc_x at the rear.  "None" (NaN) wherever a flag is unset or a guard trips;
* derivative metrics: the response's directional derivative along the velocities of the driver
  tangent (a central difference at h = 1e-12 in 32-digit arithmetic, error ~1e-20 relative), over
  the driver rate.  The driver tangent is the one whose side-local target (or shared-actuator
  equivalent) is the driver point with the strongest |rate|; None below 1e-6; +inf when two
  candidates are within 1e-6 of the strongest.

Every entry also carries the guard quantities it was decided on (``(name, value, threshold)``) and
``scale``: the magnitude of the absolute rounding error per unit of relative input rounding (for an
instant centre ~ P (P / L) / (|n1 x n2| |dir_y|), P the coordinate magnitude, L the shortest arm
edge); ``kappa = max(1, scale / max(1, |value|))`` is the entry's condition factor.
"""

from __future__ import annotations

from dataclasses import dataclass, field

import mpmath as mp
import numpy as np

mp.mp.dps = 32
EPS = 1e-6                  # the reference's degenerate-geometry guard (OKIN_GEOM_EPS)
H = mp.mpf("1e-12")         # central-difference step along the velocities
RAD2DEG = 180 / mp.pi
NAN = float("nan")

IC_FAMILY = ("svic_x", "svic_z", "svsa_length", "fvic_y", "fvic_z", "fvsa_length", "svsa_angle", "anti_dive",
             "anti_lift", "anti_squat", "roll_center_y", "roll_center_z")


@dataclass
class Entry:
    value: float
    scale: float = 0.0
    guards: list = field(default_factory=list)     # (name, value, threshold)

    @property
    def kappa(self) -> float:
        if not np.isfinite(self.value):
            return 1.0
        return max(1.0, self.scale / max(1.0, abs(self.value)))

    def guard_margin(self) -> float:
        """Smallest relative distance of a guard quantity to its threshold (inf without guards)."""
        return min((abs(abs(v) - t) / t for _, v, t in self.guards), default=float("inf"))


@dataclass
class Model:
    """What the restatement needs to know about a suspension, read from the built product model
    and its geometry mapping (no metric-program records)."""
    axle: bool
    kind: dict                  # side prefix ("" or "left_"/"right_") -> "dw" | "mac"
    spring: str                 # "none" | "coilover" | "torsion_bar"
    rocker: bool
    steered: bool
    arb: str                    # "none" | "u_bar" | "t_bar"
    heave_link: bool
    cg_z: float
    wheelbase: float
    bias: float | None
    axle_position: str | None   # "front" | "rear" | None
    driven: str | None


def model_of(sus) -> Model:
    from open_kinematics_b200.core.suspensions.axle import ArbTBar, ArbUBar, AxleSuspension
    from open_kinematics_b200.core.suspensions.corner import ActuationPushrodRocker, MacPhersonSuspension
    axle = isinstance(sus, AxleSuspension)
    corners = dict(sus.corners) if axle else {None: sus}
    c0 = next(iter(corners.values()))
    cfg = c0.config
    pos = lambda a: None if a is None else a.name.lower()   # noqa: E731
    kind = {("" if s is None else s.name.lower() + "_"): ("mac" if isinstance(c, MacPhersonSuspension) else "dw")
            for s, c in corners.items()}
    return Model(
        axle=axle, kind=kind, spring=getattr(getattr(c0, "spring", None), "kind", "none"),
        rocker=isinstance(getattr(c0, "actuation", None), ActuationPushrodRocker),
        steered=c0.rack_attachment_point() is not None,
        arb=("u_bar" if isinstance(sus.anti_roll, ArbUBar) else "t_bar" if isinstance(sus.anti_roll, ArbTBar)
             else "none") if axle else "none",
        heave_link=axle and sus.heave_link.kind == "rocker_to_rocker",
        cg_z=float(cfg.cg_position.data[2]), wheelbase=float(cfg.wheelbase), bias=cfg.front_brake_bias,
        axle_position=pos(cfg.axle_position), driven=pos(cfg.driven_axle))


def key_str(key) -> str:
    side = getattr(key, "side", None)
    if side is not None:
        return f"{side.name.lower()}_{key.point.name.lower()}"
    return key.name.lower()


# ---- small mp vector algebra ----------------------------------------------------------------------
def _v(p):
    return [mp.mpf(float(c)) for c in p]


def sub(a, b):
    return [a[0] - b[0], a[1] - b[1], a[2] - b[2]]


def add(a, b):
    return [a[0] + b[0], a[1] + b[1], a[2] + b[2]]


def mul(a, s):
    return [a[0] * s, a[1] * s, a[2] * s]


def dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def norm(a):
    return mp.sqrt(dot(a, a))


def det3(a, b, c):
    return dot(a, cross(b, c))


def _f(x) -> float:
    return float(x)


# ---- responses (values of the metric functions; used for state columns and for derivatives) -------
def camber(ai, ao, side):
    """Wheel-plane inclination from vertical, positive with the wheel top leaning outboard."""
    a = sub(ao, ai)
    return side * RAD2DEG * mp.atan2(-side * a[2], side * a[1])


def toe(ai, ao, side):
    a = sub(ao, ai)
    return RAD2DEG * mp.atan2(a[0], side * a[1])


def caster(lo, up):
    s = sub(up, lo)
    return RAD2DEG * mp.atan2(-s[0], s[2])


def kpi(lo, up, side):
    s = sub(up, lo)
    return RAD2DEG * mp.atan2(-side * s[1], s[2])


def rotation(p, design, a, b):
    """Signed angle (deg) of ``p`` about the axis a -> b, from the design position."""
    u = sub(b, a)
    u = mul(u, 1 / norm(u))
    r0, r1 = sub(design, a), sub(p, a)
    r0, r1 = sub(r0, mul(u, dot(r0, u))), sub(r1, mul(u, dot(r1, u)))
    return RAD2DEG * mp.atan2(dot(u, cross(r0, r1)), dot(r0, r1))


def tbar_twist(left, right, pivot):
    """Twist (rad) of the T-bar crossbar about its stem, measured from the lateral axis."""
    stem = sub(mul(add(left, right), mp.mpf(1) / 2), pivot)
    stem = mul(stem, 1 / norm(stem))
    cb = sub(left, right)
    cb = sub(cb, mul(stem, dot(stem, cb)))
    return mp.atan2(dot(stem, cross([0, 1, 0], cb)), cb[1])


def dist(a, b):
    return norm(sub(a, b))


# ---- the instant axis and the corner state metrics --------------------------------------------------
def _plane(a, b, c):
    n = cross(sub(b, a), sub(c, a))
    return n, norm(n)


def corner_state(m: Model, pre: str, side: float, at, design) -> dict:
    P = lambda n: at[pre + n]   # noqa: E731
    scale_p = max(abs(x) for k, p in at.items() if k.startswith(pre) for x in p)
    ai, ao, wc, cp = P("axle_inboard"), P("axle_outboard"), P("wheel_center"), P("contact_patch_center")
    lo = P("lower_wishbone_outboard")
    up = P("strut_top") if m.kind[pre] == "mac" else P("upper_wishbone_outboard")
    e = {}
    a, s = sub(ao, ai), sub(up, lo)
    ang_scale = float(RAD2DEG) * scale_p
    e["camber"] = Entry(_f(camber(ai, ao, side)), ang_scale / _f(norm(a)))
    e["roadwheel_angle"] = Entry(_f(toe(ai, ao, side)), ang_scale / _f(norm(a)))
    e["caster"] = Entry(_f(caster(lo, up)), ang_scale / _f(norm(s)))
    e["kpi"] = Entry(_f(kpi(lo, up, side)), ang_scale / _f(norm(s)))
    g = [("steer_axis_z", _f(s[2]), EPS)]
    if abs(s[2]) < EPS:
        e["scrub_radius"] = Entry(NAN, 0.0, g)
        e["mechanical_trail"] = Entry(NAN, 0.0, g)
    else:
        gp = add(lo, mul(s, (cp[2] - lo[2]) / s[2]))      # steering axis at the ground (contact-patch) height
        h = [a[0], a[1], 0]
        h = mul(h, 1 / norm(h))
        sc = scale_p * _f(norm(s) / abs(s[2]))
        e["scrub_radius"] = Entry(_f(-dot(sub(gp, cp), h)), sc, g)
        e["mechanical_trail"] = Entry(_f(gp[0] - cp[0]), sc, g)

    # the two planes of the instant axis, n . x = c
    guards, ok = [], True
    if m.kind[pre] == "dw":
        pl = [P(f"{arm}_wishbone_inboard_front") for arm in ("upper", "lower")]
        tri1 = (P("upper_wishbone_inboard_front"), P("upper_wishbone_inboard_rear"), P("upper_wishbone_outboard"))
        tri2 = (P("lower_wishbone_inboard_front"), P("lower_wishbone_inboard_rear"), P("lower_wishbone_outboard"))
        n1, m1 = _plane(*tri1)
        n2, m2 = _plane(*tri2)
        guards += [("plane1", _f(m1), EPS), ("plane2", _f(m2), EPS)]
        ok = m1 >= EPS and m2 >= EPS
        edges = [norm(sub(t[i], t[j])) for t in (tri1, tri2) for i, j in ((0, 1), (0, 2), (1, 2))]
        c1, c2 = dot(n1, pl[0]), dot(n2, pl[1])
    else:
        tri1 = (P("lower_wishbone_inboard_front"), P("lower_wishbone_inboard_rear"), P("lower_wishbone_outboard"))
        n1, m1 = _plane(*tri1)
        guards.append(("plane1", _f(m1), EPS))
        ok = m1 >= EPS
        top = P("strut_top")
        n2 = sub(top, P("lower_wishbone_outboard"))
        m2 = norm(n2)
        edges = [norm(sub(tri1[i], tri1[j])) for i, j in ((0, 1), (0, 2), (1, 2))] + [m2]
        c1, c2 = dot(n1, tri1[0]), dot(n2, top)
    if m1 > 0 and m2 > 0:
        n1, c1, n2, c2 = mul(n1, 1 / m1), c1 / m1, mul(n2, 1 / m2), c2 / m2
    d = cross(n1, n2)
    dn = norm(d)
    guards.append(("axis", _f(dn), EPS))
    ok = ok and dn >= EPS
    u = mul(d, 1 / dn) if dn > 0 else [mp.mpf(0)] * 3
    amp = scale_p * scale_p / _f(min(edges)) / max(_f(dn), 1e-300)
    sv_g = guards + [("dir_y", _f(u[1]), EPS)]
    fv_g = guards + [("dir_x", _f(u[0]), EPS)]
    sv_ok, fv_ok = ok and abs(u[1]) >= EPS, ok and abs(u[0]) >= EPS
    nan3 = [mp.nan] * 3

    def ic(row, val):    # n1 . x = c1, n2 . x = c2, row . x = val (Cramer)
        D = det3(n1, n2, row)
        b = [c1, c2, val]
        cols = [[n1[k], n2[k], row[k]] for k in range(3)]
        out = []
        for k in range(3):
            ck = [list(cols[0]), list(cols[1]), list(cols[2])]
            ck[k] = b
            out.append(det3(*[[ck[0][r], ck[1][r], ck[2][r]] for r in range(3)]) / D)
        return out
    svic = ic([0, 1, 0], wc[1]) if sv_ok else nan3
    fvic = ic([1, 0, 0], wc[0]) if fv_ok else nan3
    sv_scale = amp / max(abs(_f(u[1])), 1e-300) * max(1.0, _f(norm(sub(svic, wc))) / scale_p if sv_ok else 1.0)
    fv_scale = amp / max(abs(_f(u[0])), 1e-300) * max(1.0, _f(norm(sub(fvic, wc))) / scale_p if fv_ok else 1.0)
    e["svic_x"] = Entry(_f(svic[0]), sv_scale, sv_g)
    e["svic_z"] = Entry(_f(svic[2]), sv_scale, sv_g)
    e["svsa_length"] = Entry(_f(svic[0] - cp[0]) if sv_ok else NAN, sv_scale, sv_g)
    e["fvic_y"] = Entry(_f(fvic[1]), fv_scale, fv_g)
    e["fvic_z"] = Entry(_f(fvic[2]), fv_scale, fv_g)
    if fv_ok:
        dy, dz = fvic[1] - cp[1], fvic[2] - cp[2]
        e["fvsa_length"] = Entry(_f(mp.sqrt(dy * dy + dz * dz) * (-side * mp.sign(dy))), fv_scale, fv_g)
    else:
        e["fvsa_length"] = Entry(NAN, 0.0, fv_g)
    e["wheel_travel"] = Entry(_f(wc[2] - design[pre + "wheel_center"][2]), scale_p)
    e["half_track"] = Entry(_f(abs(cp[1])), scale_p)
    if m.spring == "coilover" or m.kind[pre] == "mac":
        e["damper_length"] = Entry(_f(dist(P("strut_top"), P("strut_bottom"))), scale_p)
    else:
        e["damper_length"] = Entry(NAN)

    # anti geometry
    run_cp = svic[0] - cp[0]
    rise_cp = svic[2] - cp[2]
    run_g = sv_g + ([("run_cp", _f(run_cp), EPS)] if sv_ok else [])
    ratio_scale = sv_scale * (1 + abs(_f(rise_cp / run_cp))) / abs(_f(run_cp)) if sv_ok and run_cp != 0 else 0.0
    svsa_ok = sv_ok and abs(run_cp) >= EPS
    e["svsa_angle"] = Entry(_f(RAD2DEG * mp.atan(rise_cp / run_cp)) if svsa_ok else NAN,
                            float(RAD2DEG) * ratio_scale, run_g)
    height = mp.mpf(m.cg_z) - cp[2]
    h_g = [("height", _f(height), EPS)]
    h_ok = height > EPS
    wb_h = m.wheelbase / height
    h_scale = scale_p / max(abs(_f(height)), 1e-300)
    front, rear = m.axle_position == "front", m.axle_position == "rear"
    b = m.bias
    e["anti_dive"] = Entry(NAN, 0.0, run_g + h_g)
    e["anti_lift"] = Entry(NAN, 0.0, run_g + h_g)
    e["anti_squat"] = Entry(NAN, 0.0, sv_g + h_g)
    if b is not None and svsa_ok and h_ok:
        if front:
            v = 100 * b * wb_h * rise_cp / (cp[0] - svic[0])
            e["anti_dive"] = Entry(_f(v), 100 * b * _f(wb_h) * ratio_scale + abs(_f(v)) * h_scale, run_g + h_g)
        if rear:
            v = 100 * (1 - b) * wb_h * rise_cp / run_cp
            e["anti_lift"] = Entry(_f(v), 100 * (1 - b) * _f(wb_h) * ratio_scale + abs(_f(v)) * h_scale, run_g + h_g)
    if m.driven is not None and m.driven == m.axle_position and sv_ok and h_ok:
        run = wc[0] - svic[0] if front else svic[0] - wc[0]
        g = sv_g + h_g + [("run_wc", _f(run), EPS)]
        if abs(run) >= EPS:
            v = 100 * wb_h * (svic[2] - wc[2]) / run
            sc = 100 * _f(wb_h) * sv_scale * (1 + abs(_f((svic[2] - wc[2]) / run))) / abs(_f(run))
            e["anti_squat"] = Entry(_f(v), sc + abs(_f(v)) * h_scale, g)
        else:
            e["anti_squat"] = Entry(NAN, 0.0, g)
    return {"entries": e, "fvic": fvic, "fv_ok": fv_ok}


# ---- derivative metrics -------------------------------------------------------------------------------
def _responses(m: Model, pre: str, side: float, design) -> dict:
    """name (without side suffix) -> (response(at), driver point, driver axis)."""
    R = {}
    P = lambda n: pre + n   # noqa: E731
    ai, ao, lo = P("axle_inboard"), P("axle_outboard"), P("lower_wishbone_outboard")
    up = P("strut_top") if m.kind[pre] == "mac" else P("upper_wishbone_outboard")
    hub = (P("wheel_center"), 2)
    R["deriv_camber_wrt_hub_z"] = (lambda x: camber(x[ai], x[ao], side), *hub)
    R["deriv_roadwheel_angle_wrt_hub_z"] = (lambda x: toe(x[ai], x[ao], side), *hub)
    R["deriv_caster_wrt_hub_z"] = (lambda x: caster(x[lo], x[up]), *hub)
    R["deriv_kpi_wrt_hub_z"] = (lambda x: kpi(x[lo], x[up], side), *hub)
    R["deriv_half_track_wrt_hub_z"] = (lambda x: side * x[P("contact_patch_center")][1], *hub)
    R["deriv_wheel_center_x_wrt_hub_z"] = (lambda x: x[P("wheel_center")][0], *hub)
    if m.steered:
        rack = (P("trackrod_inboard"), 1)
        R["deriv_roadwheel_angle_wrt_rack_displacement"] = (lambda x: toe(x[ai], x[ao], side), *rack)
        R["deriv_camber_wrt_rack_displacement"] = (lambda x: camber(x[ai], x[ao], side), *rack)
    pin, ra, rb = P("pushrod_inboard"), P("rocker_axis_a"), P("rocker_axis_b")
    if m.rocker:
        R["deriv_rocker_angle_wrt_hub_z"] = (lambda x: side * rotation(x[pin], design[pin], x[ra], x[rb]), *hub)
    if m.spring == "coilover" or m.kind[pre] == "mac":
        R["deriv_damper_length_wrt_hub_z"] = (lambda x: dist(x[P("strut_top")], x[P("strut_bottom")]), *hub)
    if m.spring == "torsion_bar":
        R["deriv_torsion_bar_twist_wrt_hub_z"] = (lambda x: side * rotation(x[pin], design[pin], x[ra], x[rb]), *hub)
    return R


def _axle_responses(m: Model, design) -> dict:
    R = {}
    if m.arb == "u_bar":
        a, b = "center_arb_u_bar_axis_a", "center_arb_u_bar_axis_b"
        L, Rr = "left_droplink_u_bar", "right_droplink_u_bar"
        f = lambda x: rotation(x[L], design[L], x[a], x[b]) - rotation(x[Rr], design[Rr], x[a], x[b])  # noqa: E731
        for s in ("left", "right"):
            R[f"deriv_arb_twist_wrt_hub_z_{s}"] = (f, f"{s}_wheel_center", 2)
    elif m.arb == "t_bar":
        L, Rr, pv = "left_droplink_t_bar", "right_droplink_t_bar", "center_arb_t_bar_pivot"
        for s in ("left", "right"):
            R[f"deriv_t_bar_center_x_wrt_hub_z_{s}"] = (lambda x: (x[L][0] + x[Rr][0]) / 2, f"{s}_wheel_center", 2)
            R[f"deriv_arb_twist_wrt_hub_z_{s}"] = (lambda x: RAD2DEG * tbar_twist(x[L], x[Rr], x[pv]),
                                                    f"{s}_wheel_center", 2)
    if m.heave_link:
        for s in ("left", "right"):
            R[f"deriv_heave_link_length_wrt_hub_z_{s}"] = (
                lambda x: dist(x["left_heave_link_rocker"], x["right_heave_link_rocker"]), f"{s}_wheel_center", 2)
    return R


def local_target(head: str, pre: str, steered: bool):
    """Side-local name of a target point seen from corner ``pre``, or its shared-actuator
    equivalent (the steering rack links left and right track-rod inboard points)."""
    if pre == "" or head.startswith(pre):
        return head[len(pre):]
    if steered and head.endswith("_trackrod_inboard"):
        return "trackrod_inboard"
    return None


def select_driver(vel, heads, driver, axis, pre, steered, exact=False):
    """(tangent index | None, rate, guards, tied)."""
    point = driver[len(pre):]
    cand = [j for j, h in enumerate(heads) if (h == driver if exact else local_target(h, pre, steered) == point)]
    rates = [(abs(float(vel[j][driver][axis])), j) for j in cand]
    if not rates:
        return None, 0.0, [], False
    strongest, best = max(rates)
    guards = [("rate", strongest, EPS)]
    others = [r for r, j in rates if j != best]
    tied = any(strongest - r <= EPS for r in others)
    guards += [("tie", strongest - r + EPS, EPS) for r in others]    # |gap - eps| / eps is the tie margin
    if strongest < EPS:
        return None, strongest, guards, False
    return best, float(vel[best][driver][axis]), guards, tied


def _deriv(f, at, v):
    plus = {k: add(p, mul(v[k], H)) for k, p in at.items()}
    minus = {k: sub(p, mul(v[k], H)) for k, p in at.items()}
    return (f(plus) - f(minus)) / (2 * H)


def _deriv_entry(f, at, vel, heads, driver, axis, pre, steered, exact, resp_gain) -> Entry:
    j, rate, guards, tied = select_driver(vel, heads, driver, axis, pre, steered, exact)
    if j is None:
        return Entry(NAN, 0.0, guards)
    if tied:
        return Entry(float("inf"), 0.0, guards)
    v = {k: _v(x) for k, x in vel[j].items()}
    d = _deriv(f, at, v) / rate
    vmax = max(abs(float(c)) for x in vel[j].values() for c in x)
    return Entry(_f(d), resp_gain * vmax / abs(rate) * 8, guards)


def metric_row(m: Model, names, at: dict, design: dict, vel=None, heads=None) -> dict:
    """{column: Entry} for ``names``; ``at`` / ``design``: point name -> xyz of the state / the
    design pose; ``vel``: per tangent j, point name -> velocity; ``heads``: per tangent j, the name of
    its target point."""
    at = {k: _v(p) for k, p in at.items()}
    design = {k: _v(p) for k, p in design.items()}
    out = {}
    sides = [("left_", 1.0, "_left"), ("right_", -1.0, "_right")] if m.axle else [("", 1.0, "")]
    corner = {}
    for pre, side, suf in sides:
        scale_p = max(abs(float(x)) for k, p in at.items() if k.startswith(pre) for x in p)
        cs = corner_state(m, pre, side, at, design)
        corner[pre] = cs
        for name, entry in cs["entries"].items():
            out[name + suf] = entry
        pin = pre + "pushrod_inboard"
        for col in ("rocker_angle", "torsion_bar_twist"):
            if (col == "rocker_angle" and m.rocker) or (col == "torsion_bar_twist" and m.spring == "torsion_bar"):
                ax = sub(at[pre + "rocker_axis_b"], at[pre + "rocker_axis_a"])
                r = rotation(at[pin], design[pin], at[pre + "rocker_axis_a"], at[pre + "rocker_axis_b"])
                out[col + suf] = Entry(_f(side * r), float(RAD2DEG) * scale_p / _f(dist(at[pin], at[pre + "rocker_axis_a"]))
                                       * (1 + scale_p / _f(norm(ax))))
        if m.arb == "u_bar":
            arm = pre + "droplink_u_bar"
            a, b = at["center_arb_u_bar_axis_a"], at["center_arb_u_bar_axis_b"]
            out["arb_arm_angle" + suf] = Entry(_f(rotation(at[arm], design[arm], a, b)),
                                               float(RAD2DEG) * scale_p / _f(dist(at[arm], a)) * (1 + scale_p / _f(dist(a, b))))
        if vel is not None:
            for name, (f, driver, axis) in _responses(m, pre, side, design).items():
                gain = float(RAD2DEG) * 4 if "angle" in name or "camber" in name or "caster" in name or "kpi" in name \
                    or "twist" in name else 1.0
                out[name + suf] = _deriv_entry(f, at, vel, heads, driver, axis, pre, m.steered, False,
                                               gain * max(1.0, scale_p / 100.0))
    if m.axle:
        scale_p = max(abs(float(x)) for p in at.values() for x in p)
        wcL, wcR, cpL, cpR = at["left_wheel_center"], at["right_wheel_center"], at["left_contact_patch_center"], \
            at["right_contact_patch_center"]
        lz = wcL[2] - design["left_wheel_center"][2]
        rz = wcR[2] - design["right_wheel_center"][2]
        clz = cpL[2] - design["left_contact_patch_center"][2]
        crz = cpR[2] - design["right_contact_patch_center"][2]
        track = abs(cpL[1] - cpR[1])
        out["heave"] = Entry(_f((lz + rz) / 2), scale_p)
        out["roll"] = Entry(_f(RAD2DEG * mp.atan2(lz - rz, track)), float(RAD2DEG) * scale_p / _f(track))
        out["ride_height_change"] = Entry(_f(-(clz + crz) / 2), scale_p)
        out["track"] = Entry(_f(track), scale_p)
        # roll centre: the lines contact patch -> front-view centre of both sides, in the YZ plane
        cl, cr = corner["left_"], corner["right_"]
        guards = [("fv_left", 1.0 if cl["fv_ok"] else 0.0, 0.5), ("fv_right", 1.0 if cr["fv_ok"] else 0.0, 0.5)]
        rc = (NAN, NAN)
        rc_scale = 0.0
        if cl["fv_ok"] and cr["fv_ok"]:
            l = (cl["fvic"][1] - cpL[1], cl["fvic"][2] - cpL[2])
            r = (cr["fvic"][1] - cpR[1], cr["fvic"][2] - cpR[2])
            den = l[0] * r[1] - l[1] * r[0]
            guards.append(("den", _f(den), EPS))
            if abs(den) >= EPS:
                # cpL + a l = cpR + b r  ->  a = ((cpR - cpL) x r) / (l x r)
                a = ((cpR[1] - cpL[1]) * r[1] - (cpR[2] - cpL[2]) * r[0]) / den
                rc = (_f(cpL[1] + a * l[0]), _f(cpL[2] + a * l[1]))
                ln, rn = _f(mp.sqrt(l[0] ** 2 + l[1] ** 2)), _f(mp.sqrt(r[0] ** 2 + r[1] ** 2))
                # each line turns by the relative rounding of its end points (an error of a far
                # front-view centre lies along its line and does not turn it); the roll centre then moves
                # by its lever arm from the contact patches over the sine of the angle between the lines
                lever = _f(mp.sqrt((rc[0] - cpL[1]) ** 2 + (rc[1] - cpL[2]) ** 2)) + \
                    _f(mp.sqrt((rc[0] - cpR[1]) ** 2 + (rc[1] - cpR[2]) ** 2))
                rc_scale = (lever + scale_p) * ln * rn / abs(_f(den))
        out["roll_center_y"] = Entry(rc[0], rc_scale, guards)
        out["roll_center_z"] = Entry(rc[1], rc_scale, guards)
        if m.steered:
            out["rack_displacement"] = Entry(_f(at["left_trackrod_inboard"][1] - design["left_trackrod_inboard"][1]),
                                             scale_p)
        else:
            out["rack_displacement"] = Entry(NAN)
        if m.arb == "u_bar":
            a, b = at["center_arb_u_bar_axis_a"], at["center_arb_u_bar_axis_b"]
            L, R = "left_droplink_u_bar", "right_droplink_u_bar"
            out["arb_twist"] = Entry(_f(rotation(at[L], design[L], a, b) - rotation(at[R], design[R], a, b)),
                                     float(RAD2DEG) * scale_p / _f(dist(at[L], a)) * (1 + scale_p / _f(dist(a, b))) * 2)
        elif m.arb == "t_bar":
            L, R, pv = "left_droplink_t_bar", "right_droplink_t_bar", "center_arb_t_bar_pivot"
            span = _f(dist(at[L], at[R]))
            tw = tbar_twist(at[L], at[R], at[pv]) - tbar_twist(design[L], design[R], at[pv])
            out["arb_twist"] = Entry(_f(RAD2DEG * tw), float(RAD2DEG) * scale_p / span * 8)
            c = mul(add(at[L], at[R]), mp.mpf(1) / 2)
            dc = mul(add(design[L], design[R]), mp.mpf(1) / 2)
            out["t_bar_heave_angle"] = Entry(_f(rotation(c, dc, at[pv], add(at[pv], [0, 1, 0]))),
                                             float(RAD2DEG) * scale_p / _f(dist(c, at[pv])) * 4)
        if m.heave_link:
            out["heave_link_length"] = Entry(_f(dist(at["left_heave_link_rocker"], at["right_heave_link_rocker"])),
                                             scale_p)
        if vel is not None:
            for name, (f, driver, axis) in _axle_responses(m, design).items():
                gain = float(RAD2DEG) * 8 if "twist" in name else 1.0
                out[name] = _deriv_entry(f, at, vel, heads, driver, axis, "", m.steered, True,
                                         gain * max(1.0, scale_p / 100.0))
    missing = [n for n in names if n not in out]
    assert not missing, missing
    return {n: out[n] for n in names}
