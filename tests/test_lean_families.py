"""Every lean kernel family on the device.

Positions-only solves run one of four lean kernels: the generic one or the one specialised to the topology
(compiled at run time by NVRTC, OKIN_SPEC), each at 168 and at 128 registers.  The first launch of a
topology on a device that is large enough times the four and keeps the fastest (``launch`` in
``csrc/okin_abi.cu``); smaller launches take the generic 168-register kernel.  So which kernel produced a
user's numbers depends on the topology, the device and the timing of that moment, and all four must
compute the same thing.  The families are pinned here with OKIN_LEAN_REGS, and each test checks that:

* every family meets the reference batches of tests/test_batches.py (positions of the reference's tight
  run, plain and tuned layout) and the flag contract on its failing batches;
* the four agree bit for bit (positions, status, failed step, iterations, reported residuals and worst
  row) at 40 000 instances on every golden and camber-shimmed topology with the tuned layout the benchmark
  uses, with per-instance setup thicknesses, on every generated linkage the device runs, and on the
  flagship with the benchmark's moving-point output subset and with per-instance target tables;
* the calibrated choice computes what the pinned generic 128-register family computes, including the
  leading instances the calibration launches solved first;
* a tolerance study is identical whichever family solves it: each device of a study calibrates on its
  own, and a study must not depend on the device list (DESIGN section 10).
"""

from __future__ import annotations

import hashlib
from types import SimpleNamespace

import numpy as np
import pytest

import open_kinematics_b200.core.topology as T
from helpers import SHIM_CASES, SWEEP_CASES
from linkage_corpus import CASES
from test_batches import BATCHES, FAIL_BATCHES, _check_failure_report, check_batch, failure_batch_report
from test_generated_linkages import OVERSIZED, instances, linkage, program
from test_specialised_kernel import golden_program, instance_inputs, perturbed
from test_study import solver_of
from test_study_gpu import c1_lean_study, tbar_shim_study

pytestmark = pytest.mark.gpu

FAMILIES = ("128", "168", "spec128", "spec168")   # OKIN_LEAN_REGS values; "128" is the reference
# Above the calibration threshold (2 x 4 x SMs x resident lean warps: 18 944 on a 148-SM B200) and past
# one pipelined chunk (32 768 instances), so the second chunk solves where the first one left off.
N = 40000
STUDY_FIELDS = ("count", "nonfinite", "mean", "std", "min", "max", "argmin", "argmax", "histogram",
                "status_counts", "failed_at_step")


def check_family(topology, family: str) -> None:
    """The family the library reports for ``topology`` on device 0 is ``family``: a specialised pin that
    silently fell back to the generic kernel fails here."""
    cal = topology.lean_calibration()
    want = (int(family.removeprefix("spec")), family.startswith("spec"))
    assert (cal["registers"], cal["specialised"]) == want, (family, cal)


def differing_instances(a: np.ndarray, b: np.ndarray) -> int:
    same = a == b
    if a.dtype.kind == "f":
        same |= np.isnan(a) & np.isnan(b)
    return int((~same.reshape(len(a), -1)).any(axis=1).sum())


def assert_identical(a: dict, b: dict, what) -> None:
    """Every output both solves returned (``worst_row`` always, ``design`` where asked), bit for bit."""
    assert a.keys() == b.keys()
    for k in a:
        assert (a[k] is None) == (b[k] is None), (what, k)
        if a[k] is not None:
            assert np.array_equal(a[k], b[k], equal_nan=True), (what, k, differing_instances(a[k], b[k]))


class Pinned:
    """A device topology whose lean family is pinned to ``family``."""

    def __init__(self, mp, topology, family: str):
        self.mp, self.topology, self.family = mp, topology, family

    def solve(self, hardpoints, values, **kw) -> dict:
        # The library reads OKIN_LEAN_REGS when the topology becomes resident on a device (its first
        # solve); other pinned topologies of this module may have set it since this one was made.
        self.mp.setenv("OKIN_LEAN_REGS", self.family)
        out = self.topology.solve_batch(hardpoints, values, want_worst_row=True, **kw)
        check_family(self.topology, self.family)
        return out


class Pins:
    """Pinned topologies and solvers of this module.  A topology is made once per program and family (an
    NVRTC compile of a specialised family takes seconds), so the reference batches and the 40 000-instance
    runs of one program share it."""

    def __init__(self, mp):
        self.mp = mp
        self.topologies: dict = {}

    def topology(self, prog, family: str) -> Pinned:
        key = hashlib.sha1(b"".join([prog.spec_source().encode(), np.ascontiguousarray(prog.hdr).tobytes(),
                                     np.ascontiguousarray(prog.iblob).tobytes(),
                                     np.ascontiguousarray(prog.fblob).tobytes()])).hexdigest()
        if (key, family) not in self.topologies:
            from open_kinematics_b200 import _lib
            self.topologies[key, family] = Pinned(self.mp, _lib.DeviceTopology(prog), family)
        return self.topologies[key, family]

    def solver(self, family: str, make):
        """A fresh ``BatchSolver`` from ``make()`` with ``family`` pinned; use it before pinning another."""
        self.mp.setenv("OKIN_LEAN_REGS", family)
        return make()

    def close(self) -> None:
        for p in self.topologies.values():
            p.topology.close()
        self.topologies.clear()


@pytest.fixture(scope="module")
def pins():
    with pytest.MonkeyPatch.context() as mp:
        p = Pins(mp)
        try:
            yield p
        finally:
            p.close()


def check_families(pins, prog, values, batches) -> None:
    """``batches``: ``(label, hardpoints, solve keywords)``; every family against the generic 128."""
    for what, hp, kw in batches:
        ref = pins.topology(prog, "128").solve(hp, values, **kw)
        for family in FAMILIES[1:]:
            assert_identical(pins.topology(prog, family).solve(hp, values, **kw), ref, (what, family))


# ---------------------------------------------------------------------------------------------
# Reference batches through every family
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tune_layout", [False, True])
@pytest.mark.parametrize("name", BATCHES)
def test_reference_batch_every_family(name, tune_layout, pins):
    outs = {}
    for family in FAMILIES:
        def solve(prog, hp, values, par, family=family):
            outs[family] = pins.topology(prog, family).solve(hp, values, params=par)
            return outs[family]
        check_batch(name, solve, tune_layout=tune_layout)
    for family in FAMILIES[1:]:
        assert_identical(outs[family], outs["128"], family)


@pytest.mark.parametrize("name", FAIL_BATCHES)
def test_failure_batch_every_family(name, pins):
    outs = {}
    for family in FAMILIES:
        def solve(prog, hp, values, par, family=family):
            outs[family] = pins.topology(prog, family).solve(hp, values, params=par, want_design=True)
            return outs[family]
        _check_failure_report(name, failure_batch_report(name, solve))
    for family in FAMILIES[1:]:
        assert_identical(outs[family], outs["128"], family)


# ---------------------------------------------------------------------------------------------
# The four families bit-identical at scale
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", SWEEP_CASES + SHIM_CASES)
def test_families_bit_identical_golden(case, pins):
    prog, nominal, values = golden_program(case, True, tune_layout=True)
    hp = perturbed(nominal, N, 0.5, 1)
    batches = [("sigma 0.5", hp, {}), ("sigma 10", perturbed(nominal, N, 10.0, 2), {})]
    if prog.param_names:     # every camber-shimmed model: C1 at design thickness, the SHIM_CASES away from it
        batches.append(("setup thickness", hp, {"params": instance_inputs(prog, values, N, 3)["params"]}))
    check_families(pins, prog, values, batches)


@pytest.mark.parametrize("name", [c.name for c in CASES if c.name != OVERSIZED])
def test_families_bit_identical_linkages(name, pins):
    lk = linkage(name)
    prog = program(lk)
    check_families(pins, prog, lk.values, [("sigma 0.5", perturbed(instances(lk, prog)[0][0], N, 0.5, 4), {})])


def test_families_bit_identical_flagship_outputs_and_targets(pins):
    """The benchmark's packed result (moving points per state, the design pose per instance) and
    per-instance target tables, on the flagship with the tuned layout."""
    import bench
    sus, sweep = bench.workload_case()
    prog, nominal, values = golden_program("c3_rocker_ubar_coilover_roll", True, tune_layout=True)
    moving = bench.moving_point_keys(SimpleNamespace(program=prog, suspension=sus))
    sub = T.compile_suspension(sus, sweep, output_points=moving, tune_layout=True)
    assert 0 < sub.n_out < prog.n_out and sub.in_keys == prog.in_keys
    hp = bench.make_hardpoints_numpy(nominal, prog, N, 5)
    check_families(pins, sub, values, [("moving points", hp, {"want_design": True})])
    targets = instance_inputs(prog, values, N, 6)["instance_targets"]
    check_families(pins, prog, values, [("instance targets", hp, {"instance_targets": targets})])


# ---------------------------------------------------------------------------------------------
# The calibrated path
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["c1_dw_corner_bump", "c4_tbar_heave_shim_bump"])
def test_calibrated_family_matches_generic_128(case, pins, monkeypatch):
    from open_kinematics_b200 import _lib
    prog, nominal, values = golden_program(case, True)
    hp = perturbed(nominal, N, 0.5, 7)
    want = pins.topology(prog, "128").solve(hp, values)
    monkeypatch.delenv("OKIN_LEAN_REGS", raising=False)
    topo = _lib.DeviceTopology(prog)
    try:
        got = topo.solve_batch(hp, values, want_worst_row=True)
        cal = topo.lean_calibration()
    finally:
        topo.close()
    ms = [cal["ms_168"], cal["ms_128"], cal["ms_spec_168"], cal["ms_spec_128"]]
    if cal["spec_error"]:     # only the generic families were timed, and the library says why
        assert min(ms[:2]) > 0 and ms[2:] == [0.0, 0.0], cal
    else:
        assert min(ms) > 0, cal
    timed = [m for m in ms if m > 0]
    best = [(168, False), (128, False), (168, True), (128, True)][int(np.argmin(timed))]
    assert (cal["registers"], cal["specialised"]) == best, cal
    assert_identical(got, want, cal)


# ---------------------------------------------------------------------------------------------
# Studies
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,study", [("c1_dw_corner_bump", c1_lean_study),
                                        ("c4_tbar_heave_shim_bump", tbar_shim_study)])
def test_study_identical_across_families(case, study, pins):
    results = {}
    for family in FAMILIES:
        solver = pins.solver(family, lambda: solver_of(case))
        try:
            smp, n, seed, kw = study(solver)
            results[family] = solver.study(smp, n, seed=seed, **kw)
            check_family(solver.topology, family)
        finally:
            solver.close()
    for family in FAMILIES[1:]:
        for f in STUDY_FIELDS:
            a, b = getattr(results[family], f), getattr(results["128"], f)
            assert (a is None) == (b is None), (family, f)
            assert a is None or a.tobytes() == b.tobytes(), (family, f)
