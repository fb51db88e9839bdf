"""On-device metric program (csrc/okin_metrics.cuh) vs the reference's metric rows
(compute_sweep_metrics on the reference's tight-tolerance states, tests/golden)."""

import numpy as np
import pytest

from helpers import SWEEP_CASES, authored_positions, build_case, emu_solve, load_golden
from open_kinematics_b200.core.topology import compile_suspension

ANGLE_TOL_DEG = np.degrees(1e-9)      # north star: angles within 1e-9 rad


def metric_tolerances(names):
    """Per-column absolute tolerance.  Angles (deg): 1e-9 rad.  Lengths (mm): 1e-6 mm, except
    instant-centre constructions (and the roll centre built from two of them), which amplify
    the 3e-8 mm position agreement by the lever arm of two nearly parallel planes/lines: 1e-6
    relative to each entry's own magnitude (values reach 1e7 mm).  A roll centre moves with the
    turn of its two contact-patch lines times its lever arm from the contact patches, so its entries
    are scaled by that lever arm (|rc_y| + track / 2 and |rc_z|, the patches on the ground plane), but
    never by more than the column's largest entry: a roll centre at y = 0.007 mm, 800 mm from the
    patches, moves by ~1e-5 mm with 3e-8 mm of position when its front-view centres are 3e7 mm away.
    Derivative columns: the reference takes its tangents from an SVD least-squares solve at slightly
    different states; 1e-9 relative to the column's scale (measured: below 3e-11)."""
    angle = ("camber", "caster", "kpi", "roadwheel_angle", "roll", "rocker_angle", "torsion_bar_twist",
             "arb_arm_angle", "arb_twist", "t_bar_heave_angle", "svsa_angle")
    ic = ("svic", "fvic", "svsa_length", "fvsa_length", "roll_center", "anti_")
    tol = []
    for n in names:
        base = n.replace("_left", "").replace("_right", "")
        if base.startswith("deriv_"):
            tol.append(("rel", 1e-9))
        elif base in angle:
            tol.append(("abs", ANGLE_TOL_DEG))          # every angle column, svsa_angle included (measured ~1e-13 rad)
        elif base.startswith(ic):
            tol.append(("rel", 1e-6))     # never tighter than the 1e-6 mm position bar it is built from
        else:
            tol.append(("abs", 1e-6))
    return tol


def check_metrics(names, got, ref):
    assert got.shape == ref.shape
    if "roll_center_y" in names:
        rc_y, rc_z = np.abs(ref[:, names.index("roll_center_y")]), np.abs(ref[:, names.index("roll_center_z")])
        lever = np.maximum(rc_y + 0.5 * ref[:, names.index("track")], rc_z)
    for c, (name, (kind, t)) in enumerate(zip(names, metric_tolerances(names))):
        g, r = got[:, c], ref[:, c]
        assert np.array_equal(np.isnan(g), np.isnan(r)), name
        ok = ~np.isnan(r)
        if not ok.any():
            continue
        if name.startswith("deriv_"):
            scale = max(1.0, np.abs(r[ok]).max())
        elif name.startswith("roll_center"):    # lever arm, never looser than the column scale
            scale = np.minimum(np.maximum(1.0, lever[ok]), max(1.0, np.abs(r[ok]).max()))
        elif kind == "rel":     # each entry's own magnitude
            scale = np.maximum(1.0, np.abs(r[ok]))
        else:
            scale = 1.0
        err = np.abs(g[ok] - r[ok]) / scale
        assert err.max() <= t, (name, err.max(), t)


@pytest.mark.parametrize("case", SWEEP_CASES)
def test_metric_rows_match_reference(case):
    meta, arr = load_golden(case)
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    assert prog.metric_names == meta["metric_names"]
    auth = authored_positions(sus)
    hp = np.concatenate([auth[k] for k in prog.in_keys])[None, :]
    out = emu_solve(prog, hp, arr["sweep_values"])
    assert out["status"][0] == 0
    check_metrics(prog.metric_names, out["metrics"][0], arr["metrics"])
