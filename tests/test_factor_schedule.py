"""Phase schedule of the block factorisation and the triangular solves (core/schedule.py), read back from
the compiled tables: every left-looking contribution runs exactly once, after its source column is final
and no later than its destination's own level; a phase never updates one destination twice nor reads a
destination it writes; every solve column is finalised once, in its own level; tangent update tasks
stay behind the "mid" pointers; and the modelled wavefront count is no worse than the schedule that runs
every contribution in its destination's level.
"""

from collections import Counter

import numpy as np
import pytest

import open_kinematics_b200.core.topology as T
from helpers import SHIM_CASES, SWEEP_CASES, build_case, load_golden
from linkage_corpus import CASES, build

D = T.D
FIN = D["OKIN_SOLVE_FIN"]


def _golden(case, design_rules):
    meta, _ = load_golden(case)
    sus, sweep = build_case(meta)
    return T.compile_suspension(sus, sweep, design_rules=design_rules)


def _corpus(name, design_rules):
    lk = build(next(c for c in CASES if c.name == name))
    return T.compile_topology(lk.state, lk.constraints, lk.spec, lk.heads, design_rules=design_rules)


def _home_schedule(dests, n_phases):
    home = [[d.home] * len(d.lo) for d in dests]
    return home, 0, 0


def _update_tasks(prog):
    """[(level, tangent, destination offset, [contribution words])] of the factor update lists."""
    lev, mid = prog.section("OKIN_S_LEV_UPD"), prog.section("OKIN_S_LEV_UPD_MID")
    dst, ptr, con = prog.section("OKIN_S_UPD_DST"), prog.section("OKIN_S_UPD_PTR"), prog.section("OKIN_S_UPD_CON")
    out = []
    for lv in range(len(lev) - 1):
        for t in range(lev[lv], lev[lv + 1]):
            out.append((lv, t >= mid[lv], int(dst[t]), [int(w) & 0xFFFFFFFF for w in con[ptr[t]:ptr[t + 1]]]))
    return out


def _solve_tasks(prog):
    """[(backward, phase, column, finalise, [contribution words])] of the triangular solves."""
    nlev = prog.stats["n_levels"]
    lev, task, con = prog.section("OKIN_S_SOLVE_LEV"), prog.section("OKIN_S_SOLVE_TASK"), prog.section("OKIN_S_SOLVE_CON")
    out = []
    for bw in (0, 1):
        for ph in range(nlev):
            for t in range(lev[bw * (nlev + 1) + ph], lev[bw * (nlev + 1) + ph + 1]):
                w, nxt = int(task[t]) & 0xFFFFFFFF, int(task[t + 1]) & 0xFFFFFFFF
                out.append((bw, ph, w & 0x7FFF, bool(w & FIN), [int(c) for c in con[w >> 16:nxt >> 16]]))
    return out


def check_schedule(prog, home):
    nf, nlev = prog.stats["n_free"], prog.stats["n_levels"]
    hdr = prog.hdr
    vec0, n = int(hdr[D["OKIN_H_OFF_VEC"]]), 3 * nf
    level = np.zeros(nf, int)
    lcp, lcol = prog.section("OKIN_S_LEV_COL_PTR"), prog.section("OKIN_S_LEV_COL")
    for lv in range(nlev):
        level[lcol[lcp[lv]:lcp[lv + 1]]] = lv

    # column of every factor row (scale tasks name each off-diagonal row with its column's diagonal block)
    col_of = {}
    diag = prog.section("OKIN_S_DIAG_OFF")
    for j, off in enumerate(diag):
        for r in range(3):
            col_of[int(off) + 3 * r] = j
    for w in prog.section("OKIN_S_SCL"):
        w = int(w) & 0xFFFFFFFF
        row, d = w >> 16, w & 0xFFFF
        if row < vec0:
            col_of[row] = col_of[d]

    def column(off):
        return (off - vec0) % n // 3 if off >= vec0 else col_of[off]

    # factor: same contributions as the home schedule, each in a phase it may run in
    tasks, ref = _update_tasks(prog), _update_tasks(home)
    assert Counter((d, w) for _, _, d, ws in tasks for w in ws) == Counter((d, w) for _, _, d, ws in ref for w in ws)
    for lv in range(nlev):
        here = [t for t in tasks if t[0] == lv]
        assert len({d for _, _, d, _ in here}) == len(here)
        written = {d + c for _, _, d, _ in here for c in range(3)}
        for _, tangent, d, ws in here:
            assert tangent == (d >= vec0 + n)
            assert lv <= level[column(d)]
            for w in ws:
                a, b = w >> 16, w & 0xFFFF
                assert level[column(a)] + 1 <= lv and column(b) == column(a)
                assert not written & ({a + c for c in range(3)} | {b + c for c in range(9)})
        flags = [tangent for _, tangent, _, _ in here]
        assert flags == sorted(flags)

    # solves: each column's contributions are the per-column lists of L z / L^T z, finalised once
    solve = _solve_tasks(prog)
    for bw, name in ((0, "FW"), (1, "BW")):
        ptr, con = prog.section(f"OKIN_S_{name}_PTR"), prog.section(f"OKIN_S_{name}_CON")
        want = Counter((j, int(w)) for j in range(nf) for w in con[ptr[j]:ptr[j + 1]])
        mine = [t for t in solve if t[0] == bw]
        assert Counter((j, w) for _, _, j, _, ws in mine for w in ws) == want
        assert sorted(j for _, _, j, fin, _ in mine if fin) == list(range(nf))
        for _, ph, j, fin, ws in mine:
            own = nlev - 1 - level[j] if bw else level[j]
            assert ph <= own and fin == (ph == own)
            for w in ws:
                s = (w & 0xFFFF) // 3
                assert ph >= (nlev - level[s] if bw else level[s] + 1)
        for ph in range(nlev):
            cols = [j for _, p, j, _, _ in mine if p == ph]
            assert len(set(cols)) == len(cols)

    for name, cost in prog.stats["schedule_wavefronts"].items():
        assert cost["after"] <= cost["before"], name


def _pair(make, monkeypatch):
    prog = make()
    with monkeypatch.context() as m:
        m.setattr(T, "schedule", _home_schedule)
        home = make()
    return prog, home


# a shimmed corner's explicit-constant model needs the device pre-solve: design-rule compile only
@pytest.mark.parametrize("case,design_rules", [(c, d) for c in SWEEP_CASES for d in (True, False)]
                         + [(c, True) for c in SHIM_CASES])
def test_golden_topology_schedule(case, design_rules, monkeypatch):
    check_schedule(*_pair(lambda: _golden(case, design_rules), monkeypatch))


@pytest.mark.parametrize("design_rules", [True, False])
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_generated_linkage_schedule(name, design_rules, monkeypatch):
    check_schedule(*_pair(lambda: _corpus(name, design_rules), monkeypatch))


def test_flagship_schedule_saves_wavefronts():
    """The C3 axle: the trunk of its elimination tree (one column per level over the last four levels)
    leaves most lanes idle when every contribution waits for its destination's level."""
    prog = _golden("c3_rocker_ubar_coilover_roll", True)
    cost = prog.stats["schedule_wavefronts"]
    before = sum(c["before"] for c in cost.values())
    after = sum(c["after"] for c in cost.values())
    assert after <= 0.75 * before
