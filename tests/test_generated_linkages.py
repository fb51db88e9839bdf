"""Generated linkages (tests/linkage_corpus.py) through the generic solver API: the lane emulation of
the device core against the oracle's tight SciPy run, and the device against the emulation.

The corpus reaches plans the shipped topologies never produce: a level of 65 blocks (lane loops take
three trips), 33 elimination levels, four targets, 285 unknowns, 500+ fill blocks and derived chains of
``OKIN_MAX_CHAIN`` ops.  Bars:

* positions within ``POS_TOL_MM`` of the oracle's root where the pinned Jacobian at that root is well
  conditioned (``cond <= COND_POSITIONS``): the error of a state within ``step_tol`` of the root, pushed
  through ``1/sigma_min``, stays far below the bar there;
* the flag contract (``test_emu_core.check_flag_contract``) on every sweep;
* the reported ``max_residual`` against the oracle's max|r| at the device's own state: the lean kernel
  reports the residual of the linear model of its last step (error second order in a step below
  ``fine_tol`` = 1e-4 mm: ~1e-8 on unit-curvature rows), so the bar is ``RES_TOL``;
* tangents, velocities and tangent health against the SVD solve of ``[J; pins]`` at the device's state.

The flag contract holds in full on linkages whose pinned Jacobian at the design pose has
``cond <= COND_CONTRACT``.  Above it the device may stop on a different flag than the reference (a
damped iteration that used its budget reports its current point to the residual test), but every
state it accepts is a verified root: the oracle's own max|r| there is within the acceptance tolerance.
The damping cycle these linkages exposed (rejected undamped step -> ``mu_init`` -> damped step below
``step_tol`` -> undamped again, until ``max_iter``) broke the contract on ``well_reach_12`` and
``random_60_4``.
"""

import numpy as np
import pytest

from helpers import emu_solve, oracle_problem_of
from linkage_corpus import CASES, SWAPS, build
from open_kinematics_b200.core.topology import compile_topology
from oracle.solve import ResidualComputer, design_setup, solve_sweep, state_tangents, target_bases
from test_emu_core import POS_TOL_MM, check_flag_contract

COND_POSITIONS = 1e5
COND_CONTRACT = 1e5
RES_TOL = 1e-7
ACCEPT_TOL = 1e-3     # the reference's acceptance tolerance (SolverConfig.residual_tolerance)
BY_NAME = {c.name: c for c in CASES}

_cache: dict = {}


def linkage(name: str):
    if name not in _cache:
        _cache[name] = build(BY_NAME[name])
    return _cache[name]


def program(lk, design_rules=True, tune_layout=False):
    return compile_topology(lk.state, lk.constraints, lk.spec, lk.heads, design_rules=design_rules,
                            tune_layout=tune_layout)


def instances(lk, prog):
    """Nominal instance and one perturbed by 0.5 mm per coordinate (``{key: xyz}``, hardpoint rows)."""
    rows = np.array([lk.hardpoints(prog.in_keys), lk.hardpoints(prog.in_keys, sigma=0.5, seed=BY_NAME[
        lk.case.name].seed)])
    dicts = []
    for row in rows:
        d = {k: v.copy() for k, v in lk.design.items()}
        d.update({k: row[3 * i: 3 * i + 3].copy() for i, k in enumerate(prog.in_keys)})
        dicts.append(d)
    return rows, dicts


class Oracle:
    """The oracle's view of one instance: tight sweep, residuals and tangents at any state."""

    def __init__(self, lk, authored):
        self.pb = oracle_problem_of(lk.state, lk.constraints, lk.spec, lk.heads)
        self.ref = solve_sweep(self.pb, authored, lk.values, ftol=1e-15, xtol=1e-15, gtol=1e-15)
        pos0, consts = design_setup(self.pb, authored)
        self.rc = ResidualComputer(self.pb, pos0, consts)
        self.bases = target_bases(self.pb, pos0)
        self.values = lk.values

    def x_of(self, prog, row):
        return np.concatenate([row[prog.out_keys.index(k)] for k in self.pb.free_order])

    def max_residual(self, prog):
        return lambda row, column: float(np.abs(self.rc.compute(self.x_of(prog, row), self.bases + column)).max())

    def tangents(self, prog, row, s):
        return state_tangents(self.pb, self.rc, self.x_of(prog, row), self.bases + self.values[:, s])


def design_cond(lk, prog) -> float:
    """cond([J; pins]) of the oracle at the nominal design pose."""
    o = Oracle.__new__(Oracle)
    o.pb = oracle_problem_of(lk.state, lk.constraints, lk.spec, lk.heads)
    pos0, consts = design_setup(o.pb, lk.design)
    o.rc, o.bases, o.values = ResidualComputer(o.pb, pos0, consts), target_bases(o.pb, pos0), lk.values
    return o.tangents(prog, np.array([pos0[k] for k in prog.out_keys]), 0)["condition_number"]


def check_against_oracle(name, design_rules=True):
    lk = linkage(name)
    prog = program(lk, design_rules)
    hp, authored = instances(lk, prog)
    if not design_rules:      # explicit constants: the declared (nominal) ones for every instance
        hp, authored = hp[:1], authored[:1]
    full = emu_solve(prog, hp, lk.values, want_health=True)
    lean = emu_solve(prog, hp, lk.values, lean=True)
    cond0 = design_cond(lk, prog)
    for i, auth in enumerate(authored):
        o = Oracle(lk, auth)
        ref = o.ref
        label = f"{name}[{i}]"
        for out in (full, lean):
            st, fs = int(out["status"][i]), int(out["failed_step"][i])
            if cond0 <= COND_CONTRACT:
                check_flag_contract(label, ref["status"], ref["failed_step"], st, fs, out["positions"][i], lk.values,
                                    o.max_residual(prog))
            else:     # every accepted state is a verified root of the reference's residual function
                accepted_to = lk.values.shape[1] if st == 0 else fs
                assert np.isfinite(out["positions"][i, :accepted_to]).all(), label
                for s in range(accepted_to):
                    assert o.max_residual(prog)(out["positions"][i, s], lk.values[:, s]) <= ACCEPT_TOL, (label, s)
        assert np.array_equal(np.isnan(full["positions"][i]), np.isnan(lean["positions"][i]))
        ok = ~np.isnan(full["positions"][i, :, 0, 0])
        assert np.nanmax(np.abs(full["positions"][i] - lean["positions"][i]), initial=0.0) <= 1e-8, label
        order = [prog.out_keys.index(k) for k in ref["keys"]]
        ref_ok = ~np.isnan(ref["positions"][:, 0, 0])
        for s in np.flatnonzero(ok):
            # reported max|r| against the oracle's residuals at the device's own state
            for out in (full, lean):
                r = o.max_residual(prog)(out["positions"][i, s], lk.values[:, s])
                assert abs(out["max_residual"][i, s] - r) <= RES_TOL, (label, s, out["max_residual"][i, s], r)
            if not ref_ok[s]:
                continue
            cond = o.tangents(prog, ref["positions"][s][np.argsort(order)], s)["condition_number"]
            if cond <= COND_POSITIONS:
                diff = np.abs(full["positions"][i, s][order] - ref["positions"][s]).max()
                assert diff <= POS_TOL_MM, (label, s, diff, cond)
    return lk, prog, hp, full


@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_emulation_matches_oracle(name):
    check_against_oracle(name)


@pytest.mark.parametrize("name", ["well_chain_33", "well_random_63", "well_families_30", "random_29_2"])
def test_emulation_matches_oracle_explicit_constants(name):
    """``design_rules=False``: the declared constants baked into the program, as solve_suspension_sweep
    compiles a linkage."""
    check_against_oracle(name, design_rules=False)


@pytest.mark.parametrize("name", ["well_star_40", "well_chain_31", "well_random_63", "well_families_30"])
def test_tangents_velocities_and_health_match_svd(name):
    lk = linkage(name)
    prog = program(lk)
    hp, authored = instances(lk, prog)
    out = emu_solve(prog, hp[:1], lk.values, want_health=True)
    assert out["status"][0] == 0
    o = Oracle(lk, authored[0])
    for s in range(lk.values.shape[1]):
        t = o.tangents(prog, out["positions"][0, s], s)
        assert t["rank"] == prog.n_unknowns
        ref_t = t["tangents"]
        scale = max(1.0, np.abs(ref_t).max())
        assert np.abs(out["tangents"][0, s] - ref_t).max() <= 1e-7 * scale, (name, s)
        # velocities of every output point: free from the tangent, fixed at rest, derived through the ops
        for j in range(len(lk.heads)):
            o.rc._refresh(o.x_of(prog, out["positions"][0, s]))
            eps = 1e-6
            xp = o.x_of(prog, out["positions"][0, s]) + eps * ref_t[j]
            xm = o.x_of(prog, out["positions"][0, s]) - eps * ref_t[j]
            o.rc._refresh(xp)
            pp = {k: v.copy() for k, v in o.rc.pos.items()}
            o.rc._refresh(xm)
            vel = np.array([(pp[k] - o.rc.pos[k]) / (2 * eps) for k in prog.out_keys])
            assert np.abs(out["velocities"][0, s, j] - vel).max() <= 1e-6 * scale, (name, s, j)
        smin, cond = out["tangent_health"][0, s]
        assert abs(smin / t["smallest_singular_value"] - 1) <= 1e-5, (name, s)
        assert abs(cond / t["condition_number"] - 1) <= 1e-5, (name, s)


@pytest.mark.parametrize("name", ["well_random_95", "well_families_30", "random_29_2"])
def test_tuned_layout_keeps_the_answer(name):
    lk = linkage(name)
    plain, tuned = program(lk), program(lk, tune_layout=True)
    hp, _ = instances(lk, plain)
    a = emu_solve(plain, hp, lk.values)
    b = emu_solve(tuned, hp, lk.values)
    assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["failed_step"], b["failed_step"])
    assert np.nanmax(np.abs(a["positions"] - b["positions"])) <= 1e-9


def test_corpus_reaches_the_edges():
    """The plans the corpus exists for: checked on the compiled programs, not assumed."""
    stats = {c.name: program(linkage(c.name)).stats for c in CASES}
    assert max(s["n_levels"] for s in stats.values()) >= 30
    # one level wider than a warp: the star linkages eliminate every free block in level 0
    assert any(s["n_levels"] == 1 and s["n_free"] > 32 for s in stats.values())
    assert max(s["n_targets"] for s in stats.values()) == 4
    assert max(s["n_unknowns"] for s in stats.values()) >= 285
    assert max(s["fill_blocks"] for s in stats.values()) >= 500
    # free blocks on both sides of one and two warps; 95 is as close to three as four fixed points
    # and the 102 keys allow with room for targets
    assert {31, 33, 63, 65, 95} <= {s["n_free"] for s in stats.values()}
    families, ops, modes, reach = set(), set(), set(), False
    longest = 0
    for c in CASES:
        lk = linkage(c.name)
        families |= {type(x).__name__ for x in lk.constraints}
        ops |= {fn.OP for fn in lk.spec.functions.values()}
        modes |= {h.mode for h in lk.heads}
        reach |= c.reach
        for key in lk.spec.functions:
            depth, k = 0, key
            while k in lk.spec.functions:
                depth += 1
                k = lk.spec.functions[k].inputs[0]
            longest = max(longest, depth)
    assert len(families) == 13, families      # every generic family the API exposes
    assert ops == {"midpoint", "along_line", "contact_patch"}
    assert len(modes) == 2 and reach
    assert longest >= 4
    assert set(SWAPS) <= {k for c in CASES for k in c.families} | {"distance"}


# ---------------------------------------------------------------------------------------------
# On the device
# ---------------------------------------------------------------------------------------------
# Its tables (the hot int sections live in shared memory, 146 kB) and one slice need more shared
# memory than one CTA of a B200 may have (227 kB): the device refuses it.
OVERSIZED = "well_random_95"


def cta_bytes(prog, lean=False) -> int:
    """Shared memory of a one-warp CTA: tables plus one slice (okin_abi.cu, CTA shape rule)."""
    from open_kinematics_b200.csrc_defs import D
    hdr = prog.hdr
    tables = D["OKIN_S_COUNT"] + ((int(hdr[D["OKIN_H_NHOT"]]) + D["OKIN_HDR_SIZE"]) * 4 + 7) // 8
    return 8 * (tables + int(hdr[D["OKIN_H_SMEM_DOUBLES_LEAN" if lean else "OKIN_H_SMEM_DOUBLES"]]))


@pytest.mark.gpu
def test_oversized_linkage_is_refused():
    from open_kinematics_b200 import _lib
    lk = linkage(OVERSIZED)
    prog = program(lk)
    assert cta_bytes(prog, lean=True) > 227 * 1024      # sm_100's opt-in limit per block
    topo = _lib.DeviceTopology(prog)
    try:
        with pytest.raises(RuntimeError, match=r"\(code -1\): topology needs more shared memory per CTA"):
            topo.solve_batch(instances(lk, prog)[0], lk.values)
    finally:
        topo.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c.name for c in CASES if c.name != OVERSIZED])
def test_device_matches_emulation(name):
    from open_kinematics_b200 import _lib
    lk = linkage(name)
    prog = program(lk, tune_layout=True)
    hp, _ = instances(lk, prog)
    emu = emu_solve(prog, hp, lk.values)
    topo = _lib.DeviceTopology(prog)
    try:
        dev = topo.solve_batch(hp, lk.values, want_tangents=True)
        lean = topo.solve_batch(hp, lk.values)
    finally:
        topo.close()
    if design_cond(lk, prog) > COND_CONTRACT:
        # Past the contract's envelope a damped iteration creeps along a direction as weak as 1/cond: the
        # rounding differences between the device and the emulation (reduction order, FMA contraction)
        # are amplified to where flags and states may differ.  Both must still accept verified roots only.
        o = Oracle(lk, lk.design)
        for out in (dev, lean):
            accepted_to = lk.values.shape[1] if out["status"][0] == 0 else out["failed_step"][0]
            for s in range(accepted_to):
                assert o.max_residual(prog)(out["positions"][0, s], lk.values[:, s]) <= ACCEPT_TOL, (name, s)
        return
    for out in (dev, lean):
        assert np.array_equal(out["status"], emu["status"]), (out["status"], emu["status"])
        assert np.array_equal(out["failed_step"], emu["failed_step"])
        assert np.array_equal(np.isnan(out["positions"]), np.isnan(emu["positions"]))
        assert np.nanmax(np.abs(out["positions"] - emu["positions"]), initial=0.0) <= 1e-9


@pytest.mark.gpu
def test_lean_families_bit_identical_on_the_largest_linkages(monkeypatch):
    """The 128- and 168-register lean families on the largest linkage the device runs and the widest level."""
    from open_kinematics_b200 import _lib
    runs = [c.name for c in CASES if c.name != OVERSIZED]
    largest = max(runs, key=lambda n: cta_bytes(program(linkage(n))))
    assert largest == "random_60_4"
    for name in (largest, "well_star_65"):
        lk = linkage(name)
        prog = program(lk)
        hp = np.repeat(instances(lk, prog)[0], 200, axis=0)
        hp[2:] += np.random.default_rng(5).normal(0.0, 0.5, hp[2:].shape)
        results = {}
        for regs in ("128", "168"):
            monkeypatch.setenv("OKIN_LEAN_REGS", regs)
            topo = _lib.DeviceTopology(prog)
            try:
                results[regs] = topo.solve_batch(hp, lk.values)
            finally:
                topo.close()
        a, b = results["128"], results["168"]
        assert np.array_equal(a["positions"], b["positions"], equal_nan=True)
        assert np.array_equal(a["iters"], b["iters"]) and np.array_equal(a["status"], b["status"])
