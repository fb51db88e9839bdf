"""Packing of the row-evaluation, linear-model and derived-point phases of a topology spec
(``TopologyProgram.spec_source``): every distance row, least-squares row and derived op of the program
appears exactly once in the packed words, with its words as the generic build reads them from the tables.

The distance rows must also keep their lane and order: their squared residuals go into per-lane partial
sums that are reduced across lanes, so slot s has to run in lane s % 32 of round s // 32, as the generic
lane loop runs it, or the sum of squares (and with it accept / reject decisions) would change by rounding.
A linear-model row and a derived op write only their own residual or point, so their lane is free; a
row's contributions keep their order, which fixes the row's own sum.
"""

import numpy as np
import pytest

import open_kinematics_b200.core.topology as T
from helpers import SWEEP_CASES
from linkage_corpus import CASES, build
from test_specialised_kernel import golden_program

D = T.D


def spec_arrays(prog):
    arrays = {}
    for line in prog.spec_source().splitlines():
        if line.startswith(("constexpr int32_t", "const int32_t okin_spec_words")):
            name = line.split("[")[0].split()[-1]
            arrays[name] = [int(v) & 0xFFFFFFFF for v in line.split("{")[1].split("}")[0].split(",")]
        elif line.startswith("constexpr int DOP_NLEV"):
            arrays["DOP_NLEV"] = int(line.split("=")[1].strip(" ;"))
    return arrays


def packed(a, p):
    """``[(round within the phase, lane, task word, [contribution words])]`` of phase p."""
    out = []
    for k, r in enumerate(range(a["PHASE_ROUND"][p], a["PHASE_ROUND"][p + 1])):
        base, width, slots, s0 = (a[n][r] for n in ("R_BASE", "R_WIDTH", "R_SLOTS", "R_SLOT0"))
        for lane in range(width):
            cons = [a["okin_spec_words"][base + (s + 1) * width + lane] for s in range(slots)
                    if lane < a["SLOT_LANES"][s0 + s]]
            out.append((k, lane, a["okin_spec_words"][base + lane], cons))
    return out


def check_program(prog):
    a = spec_arrays(prog)
    u32 = lambda name: [int(w) & 0xFFFFFFFF for w in prog.section(name)]   # noqa: E731
    h = prog.hdr
    nlev, nls, ndrow = int(h[D["OKIN_H_NLEV"]]), int(h[D["OKIN_H_NROW"]]), int(h[D["OKIN_H_NDROW"]])
    first = 2 + 5 * nlev                     # OKIN_PH_DROW(nlev)
    assert len(a["PHASE_ROUND"]) - 1 == first + 2 + 2 * a["DOP_NLEV"]

    drow = u32("OKIN_S_DROW")
    assert packed(a, first) == [(s // 32, s % 32, drow[s], [drow[ndrow + s], drow[2 * ndrow + s]])
                                for s in range(ndrow)]

    jptr, jcon = u32("OKIN_S_JH_PTR"), u32("OKIN_S_JH_CON")
    got = sorted((t, c) for _, _, t, c in packed(a, first + 1))
    assert got == [(t, jcon[jptr[t]:jptr[t + 1]]) for t in range(nls)]

    dop = np.asarray(prog.section("OKIN_S_DOP")).reshape(-1, D["OKIN_DOP_STRIDE"])
    dlev = u32("OKIN_S_DOP_LEV")
    assert a["DOP_NLEV"] == len(dlev) - 1
    for active in (0, 1):
        for lv in range(a["DOP_NLEV"]):
            want = []
            for d in range(dlev[lv], dlev[lv + 1]):
                op, o, ia, ib, ic, p = (int(v) for v in dop[d, :6])
                if active and not dop[d, 7]:
                    continue
                ib, ic = ia if ib < 0 else ib, ia if ic < 0 else ic
                want.append((o | op << 16, [ia | ib << 16, ic | p << 16]))
            got = [(t, c) for _, _, t, c in packed(a, first + 2 + active * a["DOP_NLEV"] + lv)]
            assert sorted(got) == sorted(want), (active, lv)


@pytest.mark.parametrize("design_rules", [True, False])
@pytest.mark.parametrize("case", SWEEP_CASES)
def test_row_phases_packed_golden(case, design_rules):
    check_program(golden_program(case, design_rules)[0])


@pytest.mark.parametrize("design_rules", [True, False])
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_row_phases_packed_linkages(name, design_rules):
    lk = build(next(c for c in CASES if c.name == name))
    check_program(T.compile_topology(lk.state, lk.constraints, lk.spec, lk.heads, design_rules=design_rules))
