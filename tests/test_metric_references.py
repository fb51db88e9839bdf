"""Every metric column against a plain high-precision restatement (tests/metric_reference.py).

The restatement is first pinned to the reference's own metric rows: evaluated at the reference's
tight-tolerance states, design pose and velocities of every golden sweep and of batch256_c3, it
reproduces them (state columns within 1e-12 max(1, |ref|), derivative columns within 1e-10
relative, identical NaN pattern).  It is then evaluated at the device's own returned positions,
design pose and velocities, so that solve error drops out and what is left is the metric code:

* state columns: |dev - ref| <= C_STATE eps kappa max(1, |ref|) per entry, kappa the entry's
  condition factor (for an instant centre ~ (P / L) / (|n1 x n2| |dir_y|));
* derivative columns along the device's own velocities: the same form with C_DERIV; along the
  oracle's velocities (SVD tangents at the device state) with a bar from TANGENT_TOL;
* NaN / +inf pattern identical, except entries whose guard quantity lies within 1e-9 relative of its
  threshold (counted; none on the golden inputs).

Cases: the golden sweeps at authored hardpoints; perturbed instances of the C1, C2, C3 and shimmed
C4 batches; anti-geometry variants of the C1 corner and the C3 axle (axle position, brake bias,
driven axle, centre of gravity at the contact patch); near-parallel arm planes; driver selection
with no hub candidate (None), with two hub candidates, the weaker listed first (the strongest wins),
and with two equal ones (+inf).

The anti-geometry columns are NaN in every golden file (no golden sets front_brake_bias or
driven_axle), so their signs follow the textbook definitions and the reference lines cited in
csrc/okin_core.cuh (anti_geometry.py:33-206), as restated in metric_reference.py; a golden generated
by the reference with these flags set is still to be added.

Worst measured errors on the lane emulation, in units of eps kappa max(1, |ref|): state columns
0.47, instant-centre family 0.33, derivative columns along the device's velocities 0.012; along
the oracle's velocities 2.1e-5 of the TANGENT_TOL bar.  Through the C ABI on a B200 (1000 W power
limit): 0.94, 0.33, 0.012 and 1.5e-5.  No entry fell in the guard band on either.  Pinning:
derivative columns 9e-14; state columns 1.4e-14 of a bar of 1e-12 max(1, |ref|) widened, per entry,
to C_STATE eps kappa max(1, |ref|) where the reference's own float64 rounding is larger than that.
The widest widening applied was 3.8e5 on the sweeps (c3_rocker_ubar_coilover_roll) and 2.8e6
on batch256_c3.  The roll-centre |den| guard is never approached: its smallest |den| is 9e9
times the guard (den is the cross product of the two contact-patch lines, whose lengths grow with
the front-view centres, so near-parallel arm planes make it larger, not smaller).
"""

import copy

import numpy as np
import pytest

import metric_reference as MR
from helpers import SHIM_CASES, SWEEP_CASES, authored_positions, build_case, emu_solve, key_from_name, load_golden
from open_kinematics_b200.core.input import build_suspension, build_sweep
from open_kinematics_b200.core.solver import sweep_target_values
from test_batches import batch_geometry, batch_inputs, compile_batch
from test_output_references import TANGENT_TOL, golden_oracle, sample_steps

EPS = np.finfo(float).eps
C_STATE = 8.0           # state columns, units of eps kappa max(1, |ref|)
C_DERIV = 1.0           # derivative columns along the device's own velocities
C_ORACLE = 1.0          # derivative columns along the oracle's velocities, units of TANGENT_TOL max(1, |v|) max(1, |ref|)
GUARD_BAND = 1e-9       # guard quantities this close (relative) to their threshold may flip NaN
PIN_STATE, PIN_DERIV = 1e-12, 1e-10
DERIV_FLOOR = 1e-6    # derivative columns: relative to max(|ref|, 1e-6) (a near-zero derivative keeps the reference's rounding)
METRIC_SWEEPS = SWEEP_CASES + SHIM_CASES
METRIC_BATCHES = ["batch256_c1", "batch256_c2", "batch256_c3", "batch64_c4_roll", "batch64_c4_bump"]


def _family(name: str) -> str:
    base = name.replace("_left", "").replace("_right", "")
    if base.startswith("deriv_"):
        return "deriv"
    return "ic" if base in MR.IC_FAMILY else "state"


def head_names(sweep) -> list:
    heads, _ = sweep_target_values(sweep)
    return [MR.key_str(h.point_id) for h in heads]


class Points:
    """Point name <-> slot of a position row."""

    def __init__(self, keys):
        self.names = [MR.key_str(k) for k in keys]

    def at(self, row) -> dict:
        return {n: row[i] for i, n in enumerate(self.names) if np.all(np.isfinite(row[i]))}

    def vel(self, rows) -> list:
        return [{n: v[i] for i, n in enumerate(self.names)} for v in rows]


def compare(names, got, ref: dict, stats: dict, label, boundary: list, deriv_bar=None, checked=None) -> None:
    """One row: device ``got`` [n_cols] against the restatement's entries; ``checked`` collects the
    names of the columns compared."""
    for c, name in enumerate(names):
        e = ref[name]
        g, r = got[c], e.value
        fam = _family(name)
        if checked is not None:
            checked.add(name)
        den = [abs(v) / t for gname, v, t in e.guards if gname == "den"]
        if den:    # how close the roll-centre construction came to its |den| guard
            stats["den_over_guard"] = min(stats.get("den_over_guard", np.inf), den[0])
        if np.isnan(r) or np.isnan(g) or np.isinf(r) or np.isinf(g):
            same = (np.isnan(r) and np.isnan(g)) or (g == r)
            if not same:
                assert e.guard_margin() <= GUARD_BAND, (label, name, g, r, e.guards)
                boundary.append((label, name))
            continue
        if fam == "deriv" and deriv_bar is not None:
            bar = deriv_bar(name, e)
            err = abs(g - r)
            stats[fam + "_oracle"] = max(stats.get(fam + "_oracle", 0.0), err / bar)
            assert err <= bar, (label, name, g, r, bar)
            continue
        c_ = C_DERIV if fam == "deriv" else C_STATE
        unit = EPS * e.kappa * max(1.0, abs(r))
        err = abs(g - r) / unit
        stats[fam] = max(stats.get(fam, 0.0), err)
        assert err <= c_, (label, name, g, r, err, e.kappa)


# ---------------------------------------------------------------------------------------------
# 1. pin the restatement to the reference's own metric rows
# ---------------------------------------------------------------------------------------------
def _pin_rows(model, names, pts, positions, design, velocities, heads, ref_rows, label):
    worst = {"state": 0.0, "deriv": 0.0}
    for s in range(positions.shape[0]):
        vel = None if velocities is None else pts.vel(velocities[s])
        row = MR.metric_row(model, names, pts.at(positions[s]), pts.at(design), vel, heads)
        for c, name in enumerate(names):
            r, got = ref_rows[s, c], row[name].value
            assert np.isnan(r) == np.isnan(got), (label, s, name, got, r)
            if np.isnan(r):
                continue
            if name.startswith("deriv_"):
                err = abs(got - r) / max(abs(r), DERIV_FLOOR)
                worst["deriv"] = max(worst["deriv"], err)
                assert err <= PIN_DERIV, (label, s, name, got, r)
            else:
                # the reference's own float64 rounding, amplified by the entry's condition factor
                relax = max(1.0, C_STATE * EPS * row[name].kappa / PIN_STATE)
                err = abs(got - r) / max(1.0, abs(r)) / relax
                worst["state"] = max(worst["state"], err)
                worst["relax"] = max(worst.get("relax", 1.0), relax)
                assert err <= PIN_STATE, (label, s, name, got, r, row[name].kappa)
    return worst


@pytest.mark.parametrize("case", METRIC_SWEEPS)
def test_restatement_reproduces_reference_rows(case):
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    pts = Points([key_from_name(n) for n in meta["point_keys"]])
    worst = _pin_rows(MR.model_of(sus), meta["metric_names"], pts, arr["positions_tight"], arr["design_positions"],
                      arr["velocities"], head_names(sweep), arr["metrics"], case)
    print(case, "pinning worst", worst)


def test_restatement_reproduces_reference_batch_c3():
    """The state columns of batch256_c3's 768 rows (perturbed instances; the golden keeps no
    velocities, so derivative columns are pinned on the sweeps above)."""
    meta, arr = load_golden("batch256_c3")
    sus, sweep, prog = compile_batch(meta)
    names = meta["metric_names"]
    state = [c for c, n in enumerate(names) if not n.startswith("deriv_")]
    pts = Points([key_from_name(n) for n in meta["point_keys"]])
    worst = {"state": 0.0}
    for i in range(arr["hardpoints"].shape[0]):
        sus_i = build_suspension(batch_geometry(meta, arr["hardpoints"][i]))
        pose = sus_i.initial_state().positions
        design = np.array([pose[key_from_name(n)].data for n in meta["point_keys"]])
        w = _pin_rows(MR.model_of(sus_i), [names[c] for c in state], pts, arr["positions_tight"][i], design, None,
                      None, arr["metrics"][i][:, state], f"batch256_c3[{i}]")
        worst["state"] = max(worst["state"], w["state"])
        worst["relax"] = max(worst.get("relax", 1.0), w.get("relax", 1.0))
    print("batch256_c3 pinning worst", worst)


# ---------------------------------------------------------------------------------------------
# 2. the device at its own states
# ---------------------------------------------------------------------------------------------
def emu_backend(prog, hp, values, params=None):
    return emu_solve(prog, hp, values, params=params)


def gpu_backend(prog, hp, values, params=None):
    from open_kinematics_b200 import _lib
    topo = _lib.DeviceTopology(prog)
    try:
        return topo.solve_batch(hp, values, params=params, want_positions=True, want_metrics=True, want_design=True,
                                want_velocities=True, want_tangents=True)
    finally:
        topo.close()


def oracle_velocities(oracle, row, column) -> np.ndarray:
    from oracle.solve import state_tangents
    x = row[oracle.cols].reshape(-1)
    ref = state_tangents(oracle.problem, oracle.rc, x, oracle.bases + column)
    return oracle.velocities(x, ref["tangents"])


def check_device_rows(sus, sweep, prog, out, values, rows, steps, label, stats, boundary, oracle_of=None,
                      checked=None) -> None:
    """Device metric rows of instances ``rows`` (indices into ``out``) at ``steps`` against the
    restatement at the device's own positions / design / velocities; with ``oracle_of(k)`` also
    the derivative columns along the oracle's velocities."""
    model = MR.model_of(sus)
    names = prog.metric_names
    pts = Points(prog.out_keys)
    heads = head_names(sweep)
    deriv_cols = [c for c, n in enumerate(names) if n.startswith("deriv_")]
    for k in rows:
        assert out["status"][k] == 0, (label, k)
        oracle = None if oracle_of is None else oracle_of(k)
        design = pts.at(out["design"][k])
        for s in steps:
            at = pts.at(out["positions"][k, s])
            ref = MR.metric_row(model, names, at, design, pts.vel(out["velocities"][k, s]), heads)
            compare(names, out["metrics"][k, s], ref, stats, f"{label}[{k}]@{s}", boundary, checked=checked)
            if oracle is not None:
                v_ref = oracle_velocities(oracle, out["positions"][k, s], values[:, s])
                vs = max(1.0, np.abs(v_ref).max())
                ref_o = MR.metric_row(model, [names[c] for c in deriv_cols], at, design, pts.vel(v_ref), heads)

                def bar(name, e, vs=vs):
                    return C_ORACLE * TANGENT_TOL * vs * max(1.0, abs(e.value))
                compare([names[c] for c in deriv_cols], out["metrics"][k, s][deriv_cols], ref_o, stats,
                        f"{label}[{k}]@{s}/oracle", boundary, deriv_bar=bar)


def _sweep_case(case, backend, stats, boundary, n_steps=None, checked=None):
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    from open_kinematics_b200.core.topology import compile_suspension
    prog = compile_suspension(sus, sweep)
    _, values = sweep_target_values(sweep)
    values = values[:, :n_steps]
    auth = authored_positions(sus)
    hp = np.concatenate([auth[k] for k in prog.in_keys])[None, :]
    out = backend(prog, hp, values)

    def oracle_of(k):
        from test_output_references import StateOracle
        if prog.param_names:
            setup = {key: out["design"][k][prog.out_keys.index(key)] for key in prog.in_keys}
            return StateOracle(sus, sweep, prog, setup, shimmed=True)
        return StateOracle(sus, sweep, prog, authored_positions(sus), shimmed=False)
    check_device_rows(sus, sweep, prog, out, values, [0], range(values.shape[1]), case, stats, boundary,
                      None if n_steps else oracle_of, checked)
    return prog


def _batch_case(name, backend, stats, boundary, n_inst=64, n_steps=None, checked=None):
    meta, arr = load_golden(name)
    sus, sweep, prog = compile_batch(meta)
    n = arr["hardpoints"].shape[0]
    rows = sorted(set(np.linspace(0, n - 1, n_inst).astype(int).tolist()))
    hp, par = batch_inputs(meta, arr, prog, rows)
    _, values = sweep_target_values(sweep)
    values = values[:, :n_steps]
    out = backend(prog, hp, values, par)
    steps = sample_steps(values.shape[1])
    oracle_rows = set(rows[::16])

    def oracle_of(k):
        return golden_oracle(meta, arr, rows[k], sweep, prog, out["design"][k]) if rows[k] in oracle_rows else None
    check_device_rows(sus, sweep, prog, out, values, range(len(rows)), steps, name, stats, boundary,
                      None if n_steps else oracle_of, checked)
    return prog


def _variant_case(meta, geometry, sweep_spec, backend, stats, boundary, steps=None, oracle=False):
    from open_kinematics_b200.core.topology import compile_suspension
    sus = build_suspension(geometry)
    sweep = build_sweep(sweep_spec, sus)
    prog = compile_suspension(sus, sweep)
    _, values = sweep_target_values(sweep)
    auth = authored_positions(sus)
    out = backend(prog, np.concatenate([auth[k] for k in prog.in_keys])[None, :], values)
    steps = range(values.shape[1]) if steps is None else steps

    def oracle_of(k):
        from test_output_references import StateOracle
        return StateOracle(sus, sweep, prog, authored_positions(sus), shimmed=False)
    check_device_rows(sus, sweep, prog, out, values, [0], steps, meta.get("name", "variant"), stats, boundary,
                      oracle_of if oracle else None)
    return sus, prog, out, values


# ---- anti-geometry variants ------------------------------------------------------------------------
ANTI_BASES = {"c1": "c1_dw_corner_bump", "c3": "c3_rocker_ubar_coilover_roll"}
BIASES = [None, 0.0, 0.65, 1.0]
AXLES = ["front", "rear"]
DRIVEN = [None, "front", "rear"]


def anti_geometry(base: str, axle_position, bias, driven, cg_z=None) -> tuple:
    meta, _ = load_golden(ANTI_BASES[base])
    geom = copy.deepcopy(meta["geometry"])
    vehicle = geom["config"] if base == "c1" else geom["vehicle_config"]
    (geom["config"] if base == "c1" else geom["axle_config"])["axle_position"] = axle_position
    for key, value in (("front_brake_bias", bias), ("driven_axle", driven)):
        vehicle.pop(key, None)
        if value is not None:
            vehicle[key] = value
    if cg_z is not None:
        vehicle["cg_position"]["z"] = cg_z
    return meta, geom


def run_anti_variants(base, backend) -> dict:
    """Every (axle position, brake bias, driven axle) variant plus the centre of gravity below the
    contact patch; returns {variant: (prog, out)} after the restatement checks."""
    stats, boundary, results = {}, [], {}
    variants = [(a, b, d, None) for a in AXLES for b in BIASES for d in DRIVEN] + [("front", 0.65, "front", -400.0)]
    for a, b, d, cg in variants:
        meta, geom = anti_geometry(base, a, b, d, cg)
        steps = sample_steps(load_golden(ANTI_BASES[base])[1]["sweep_values"].shape[1])
        sus, prog, out, _ = _variant_case(meta, geom, meta["sweep"], backend, stats, boundary, steps)
        results[(a, b, d, cg)] = (prog, out, steps, MR.model_of(sus))
    assert not boundary, boundary
    print(base, "anti variants worst", stats)
    return results


def check_anti_flags(results) -> None:
    """NaN exactly where the flags say; device-only identities between the anti columns and
    svsa_angle; linearity in the brake bias."""
    seen = {"anti_dive": set(), "anti_lift": set(), "anti_squat": set()}
    for (a, b, d, cg), (prog, out, steps, model) in results.items():
        names = prog.metric_names
        pts = Points(prog.out_keys)
        m = out["metrics"][0][steps]
        sides = ["_left", "_right"] if "camber_left" in names else [""]
        for suf in sides:
            col = {n: names.index(n + suf) for n in ("anti_dive", "anti_lift", "anti_squat", "svsa_angle")}
            cp = pts.names.index(("left_" if suf == "_left" else "right_" if suf == "_right" else "")
                                 + "contact_patch_center")
            h = model.cg_z - out["positions"][0][steps][:, cp, 2]
            wb = model.wheelbase
            tan_sv = np.tan(np.radians(m[:, col["svsa_angle"]]))
            sv_fin = np.isfinite(tan_sv)
            dive, lift, squat = m[:, col["anti_dive"]], m[:, col["anti_lift"]], m[:, col["anti_squat"]]
            want_dive = (a == "front") & (b is not None) & (cg is None) & sv_fin
            want_lift = (a == "rear") & (b is not None) & (cg is None) & sv_fin
            assert np.array_equal(np.isfinite(dive), want_dive), (a, b, d, cg, suf)
            assert np.array_equal(np.isfinite(lift), want_lift), (a, b, d, cg, suf)
            if d != a or cg is not None:
                assert np.isnan(squat).all(), (a, b, d, cg, suf)
            else:
                assert np.isfinite(squat).any()
            for name, v in (("anti_dive", dive), ("anti_lift", lift), ("anti_squat", squat)):
                seen[name] |= {bool(x) for x in np.isfinite(v)}
            bb = 0.0 if b is None else b
            if want_dive.any():
                ref = -100.0 * bb * (wb / h) * tan_sv
                assert np.allclose(dive[want_dive], ref[want_dive], rtol=1e-12, atol=1e-12), (a, b, d, suf)
            if want_lift.any():
                ref = 100.0 * (1.0 - bb) * (wb / h) * tan_sv
                assert np.allclose(lift[want_lift], ref[want_lift], rtol=1e-12, atol=1e-12), (a, b, d, suf)
    # anti-dive / anti-lift are linear in the brake bias
    for a, name in (("front", "anti_dive"), ("rear", "anti_lift")):
        full = results[(a, 1.0 if a == "front" else 0.0, None, None)]
        part = results[(a, 0.65, None, None)]
        c = full[0].metric_names.index(name if name in full[0].metric_names else name + "_left")
        f = 0.65 if a == "front" else 0.35
        assert np.allclose(part[1]["metrics"][0][:, c], f * full[1]["metrics"][0][:, c], rtol=1e-13, atol=1e-12,
                           equal_nan=True)
    assert all(v == {True, False} for v in seen.values()), seen


def _check_anti_symmetry(results) -> None:
    """Left equals right on the symmetric C3 axle at its design state (the middle of the roll sweep)."""
    prog, out, _, _ = results[("front", 0.65, "front", None)]
    names = prog.metric_names
    mid = out["metrics"].shape[1] // 2
    for n in ("anti_dive", "anti_squat", "svsa_angle"):
        l, r = out["metrics"][0, mid, names.index(n + "_left")], out["metrics"][0, mid, names.index(n + "_right")]
        assert (np.isnan(l) and np.isnan(r)) or abs(l - r) <= 1e-9 * max(1.0, abs(l)), (n, l, r)


# ---- near-degenerate instant centres -----------------------------------------------------------------
def near_parallel_geometry(base: str, delta: float) -> tuple:
    """Both arm planes of the C1 corner and of the C3 axle are horizontal at the authored pose (their
    instant centres are None there).  Raising the upper-arm rear inboard pivot (left side on the axle)
    by ``delta`` mm tilts the upper plane by ~delta / 500 rad: near the design state the instant axis
    is then ~1e5 / delta mm away, and the sweep carries it back to ordinary distances."""
    meta, _ = load_golden(ANTI_BASES[base])
    geom = copy.deepcopy(meta["geometry"])
    hp = geom["hardpoints"] if base == "c1" else geom["hardpoints"]["left"]
    hp["upper_wishbone_inboard_rear"]["z"] = float(hp["upper_wishbone_inboard_rear"]["z"]) + delta
    return meta, geom


DELTAS = [1e-4, 1e-2, 1.0]


def run_near_parallel(base, backend) -> dict:
    stats, boundary = {}, []
    span = {}
    for delta in DELTAS:
        meta, geom = near_parallel_geometry(base, delta)
        _, prog, out, _ = _variant_case(meta, geom, meta["sweep"], backend, stats, boundary)
        suf = "_left" if base == "c3" else ""
        for col in ("svic_x", "fvic_y"):
            v = np.abs(out["metrics"][0][:, prog.metric_names.index(col + suf)])
            span[(col, delta)] = (float(np.nanmin(v)), float(np.nanmax(v)))
    print(base, "near-parallel worst", stats, "IC magnitude span", span, "boundary entries", len(boundary))
    assert max(hi for _, hi in span.values()) > 1e7 and min(lo for lo, _ in span.values()) < 1e5
    return stats


# ---- driver selection ----------------------------------------------------------------------------------
def run_driver_nan(backend) -> None:
    """Bump target on the lower ball joint instead of the wheel centre: no tangent drives the hub, so
    every *_wrt_hub_z column is None (NaN); the rack columns keep their driver."""
    meta, _ = load_golden("c1_dw_corner_bump_steer")
    spec = copy.deepcopy(meta["sweep"])
    spec["targets"][1]["point"] = "lower_wishbone_outboard"
    spec["targets"][1]["mode"] = "relative"
    spec["targets"][1]["start"], spec["targets"][1]["stop"] = -30, 40
    stats, boundary = {}, []
    _, prog, out, _ = _variant_case(meta, meta["geometry"], spec, backend, stats, boundary, oracle=True)
    names = prog.metric_names
    m = out["metrics"][0]
    for c, n in enumerate(names):
        if n.endswith("_wrt_hub_z"):
            assert np.isnan(m[:, c]).all(), n
        elif n.endswith("_wrt_rack_displacement"):
            assert np.isfinite(m[:, c]).all(), n
    assert not boundary


def _steer_sweep_values(spec: dict, n: int) -> dict:
    """The steered C1 sweep with explicit value lists (so that targets can be added)."""
    spec = copy.deepcopy(spec)
    for t in spec["targets"]:
        t["values"] = np.linspace(t.pop("start"), t.pop("stop"), n).tolist()
    spec.pop("steps")
    return spec


def run_driver_two_candidates(backend) -> None:
    """Two tangents drive the hub: a wheel-centre x target, listed first, and the wheel-centre z
    target.  The x target takes the wheel-centre x the device solved on the plain sweep, so the
    three targets (rack, x, z) stay consistent on the two-degree-of-freedom corner and the solve is
    the plain sweep's.  The x tangent moves the hub by ~3e-3 in z, the z tangent by ~1: the strongest
    |rate| must win, not the first candidate."""
    from open_kinematics_b200.core.topology import compile_suspension
    meta, _ = load_golden("c1_dw_corner_bump_steer")
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    _, values = sweep_target_values(sweep)
    auth = authored_positions(sus)
    plain = backend(prog, np.concatenate([auth[k] for k in prog.in_keys])[None, :], values)
    wc = Points(prog.out_keys).names.index("wheel_center")
    spec = _steer_sweep_values(meta["sweep"], values.shape[1])
    spec["targets"].insert(1, {"point": "wheel_center", "direction": {"axis": "x"}, "mode": "absolute",
                               "values": plain["positions"][0, :, wc, 0].tolist()})
    stats, boundary = {}, []
    _, prog2, out, _ = _variant_case(meta, meta["geometry"], spec, backend, stats, boundary)
    assert not boundary, boundary
    rates = np.abs(out["velocities"][0, :, 1:, Points(prog2.out_keys).names.index("wheel_center"), 2])
    assert (rates[:, 0] < 1e-2).all() and (rates[:, 1] > 0.99).all(), rates
    names = prog2.metric_names
    for c, n in enumerate(names):
        if n.endswith("_wrt_hub_z"):
            assert np.isfinite(out["metrics"][0, :, c]).all(), n
    print("two hub candidates worst", stats)


def run_driver_tie(backend) -> None:
    """The wheel-centre z target given twice: the pinned tangent system is still of full column
    rank, its least-squares tangents split the hub motion 0.5 / 0.5 between the two, and the
    equal-strength drivers give +inf (the reference raises) in every *_wrt_hub_z column."""
    meta, _ = load_golden("c1_dw_corner_bump_steer")
    spec = copy.deepcopy(meta["sweep"])
    spec["targets"].append(copy.deepcopy(spec["targets"][1]))
    stats, boundary = {}, []
    _, prog, out, _ = _variant_case(meta, meta["geometry"], spec, backend, stats, boundary, oracle=True)
    assert not boundary, boundary
    for c, n in enumerate(prog.metric_names):
        if n.endswith("_wrt_hub_z"):
            assert np.isposinf(out["metrics"][0, :, c]).all(), n
        elif n.endswith("_wrt_rack_displacement"):
            assert np.isfinite(out["metrics"][0, :, c]).all(), n


# ---------------------------------------------------------------------------------------------
# tests
# ---------------------------------------------------------------------------------------------
BACKENDS = [pytest.param(emu_backend, id="emu"), pytest.param(gpu_backend, id="gpu", marks=pytest.mark.gpu)]


@pytest.mark.parametrize("backend", BACKENDS)
def test_golden_sweeps_at_device_states(backend):
    stats, boundary = {}, []
    for case in METRIC_SWEEPS:
        _sweep_case(case, backend, stats, boundary)
    assert not boundary, boundary
    print("golden sweeps worst", stats)


@pytest.mark.parametrize("name", METRIC_BATCHES)
@pytest.mark.parametrize("backend", BACKENDS)
def test_perturbed_batches_at_device_states(backend, name):
    stats, boundary = {}, []
    _batch_case(name, backend, stats, boundary)
    print(name, "worst", stats)
    assert not boundary, boundary


@pytest.mark.parametrize("base", ["c1", "c3"])
@pytest.mark.parametrize("backend", BACKENDS)
def test_anti_geometry_variants(backend, base):
    results = run_anti_variants(base, backend)
    check_anti_flags(results)
    if base == "c3":
        _check_anti_symmetry(results)


@pytest.mark.parametrize("base", ["c1", "c3"])
@pytest.mark.parametrize("backend", BACKENDS)
def test_near_parallel_arm_planes(backend, base):
    run_near_parallel(base, backend)


@pytest.mark.parametrize("backend", BACKENDS)
def test_driver_selection_without_hub_target(backend):
    run_driver_nan(backend)


@pytest.mark.parametrize("backend", BACKENDS)
def test_driver_selection_strongest_of_two_candidates(backend):
    run_driver_two_candidates(backend)


@pytest.mark.parametrize("backend", BACKENDS)
def test_driver_selection_tie(backend):
    run_driver_tie(backend)


def test_every_metric_column_is_checked():
    """The device-at-own-state cases above compare every metric column of C1, C2, C3 and C4: the
    golden sweeps and the perturbed batches, run here on two steps / two instances, record in
    compare() which device columns they compared, and that set equals the union of the programs'
    metric names."""
    progs, checked = set(), set()
    for case in METRIC_SWEEPS:
        progs |= set(_sweep_case(case, emu_backend, {}, [], n_steps=2, checked=checked).metric_names)
    for name in METRIC_BATCHES:
        progs |= set(_batch_case(name, emu_backend, {}, [], n_inst=2, n_steps=2, checked=checked).metric_names)
    assert checked == progs, sorted(progs ^ checked)
