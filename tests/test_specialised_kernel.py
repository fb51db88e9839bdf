"""Topology-specialised lean kernel: ``csrc/okin_core.cuh`` built with a program's generated spec
(``TopologyProgram.spec_source``, OKIN_SPEC) must compute exactly what the generic build computes.

On the CPU the lane emulation is built with the spec and compared bit for bit with the generic emulation
for every golden topology (camber-shimmed and failing-batch ones included) and every generated linkage, in
both compile modes and with the tuned layout, at nominal hardpoints, at sigma = 10 mm, and at sigma = 10 mm
with per-instance target tables and setup thicknesses.  NVRTC compiles one spec of each kind for sm_100a
when the toolkit's libnvrtc is present.  On the device the specialised lean kernel (pinned with
OKIN_LEAN_REGS) is compared bit for bit with the generic lean kernel (tests/test_lean_families.py covers
every topology).
"""

import contextlib
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

import helpers
import open_kinematics_b200.core.topology as T
from helpers import SHIM_CASES, SWEEP_CASES, build_case, emu_solve, load_golden
from linkage_corpus import CASES, build
from test_batches import FAIL_BATCHES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "open-kinematics_b200", "csrc")
_SPEC_LIBS: dict = {}


def spec_emu_lib(prog):
    """Lane emulation of ``prog``'s specialised lean kernel (``tests/emu/okin_emu_spec.cpp``, one build per
    distinct spec, in a temporary directory)."""
    src = prog.spec_source()
    key = hashlib.sha1(src.encode()).hexdigest()
    if key not in _SPEC_LIBS:
        d = tempfile.mkdtemp(prefix="okin_spec_emu_")
        with open(os.path.join(d, "okin_spec.h"), "w") as f:
            f.write(src)
        out = os.path.join(d, "libokin_emu_spec.so")
        subprocess.run(["g++", "-O1", "-shared", "-fPIC", "-std=c++17", "-DOKIN_SPEC", f"-I{d}", f"-I{CSRC}", "-o", out,
                        os.path.join(ROOT, "tests", "emu", "okin_emu_spec.cpp")], check=True)
        lib = ctypes.CDLL(out)
        lib.okin_emu_sweep.restype = ctypes.c_int
        lib.okin_emu_sweep.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_long, ctypes.c_int] + [ctypes.c_void_p] * 2
        _SPEC_LIBS[key] = lib
    return _SPEC_LIBS[key]


@contextlib.contextmanager
def emulation(lib):
    saved = helpers.emu_lib()
    helpers._EMU = lib
    try:
        yield
    finally:
        helpers._EMU = saved


FIELDS = ("positions", "status", "failed_step", "iters", "max_residual", "worst_row")


def assert_bit_identical(a, b, what):
    for k in FIELDS:
        assert np.array_equal(a[k], b[k], equal_nan=True), (what, k)


def perturbed(nominal, n, sigma, seed=0):
    hp = np.repeat(nominal.reshape(1, -1), n, axis=0)
    hp[1:] += np.random.default_rng(seed).normal(0.0, sigma, hp[1:].shape)
    return hp


def instance_inputs(prog, values, n, seed=0) -> dict:
    """Per-instance inputs of ``n`` instances: target tables shifted by up to 2 mm per target, and
    camber-shim setup thicknesses uniform within 0.5 mm of the model's (None without shims)."""
    rng = np.random.default_rng(seed)
    targets = values[None] + rng.uniform(-2.0, 2.0, (n, values.shape[0], 1))
    params = None
    if prog.param_names:
        params = np.repeat(prog.param_default[None].astype(np.float64), n, axis=0)
        for j, name in enumerate(prog.param_names):
            if name.endswith("setup_thickness"):
                params[:, j] += rng.uniform(-0.5, 0.5, n)
    return {"instance_targets": targets, "params": params}


def golden_program(case, design_rules, tune_layout=False):
    meta, _ = load_golden(case)
    sus, sweep = build_case(meta)
    prog = T.compile_suspension(sus, sweep, design_rules=design_rules, tune_layout=tune_layout)
    auth = helpers.authored_positions(sus)
    nominal = np.concatenate([auth[k] for k in prog.in_keys])
    from open_kinematics_b200.core.solver import sweep_target_values
    return prog, nominal, sweep_target_values(sweep)[1]


def check_spec_matches_generic(prog, nominal, values, n=6, rows=None):
    """Nominal instance; ``n`` instances at sigma = 10 mm (or the hardpoint ``rows`` given); the same
    again with per-instance target tables and setup thicknesses (``instance_inputs``)."""
    hp = perturbed(nominal, n, 10.0) if rows is None else rows
    runs = [("nominal", perturbed(nominal, 1, 0.0), {}), ("sigma 10", hp, {}),
            ("per-instance inputs", hp, instance_inputs(prog, values, len(hp)))]
    for what, hp, kw in runs:
        generic = emu_solve(prog, hp, values, lean=True, **kw)
        with emulation(spec_emu_lib(prog)):
            spec = emu_solve(prog, hp, values, lean=True, **kw)
        assert_bit_identical(spec, generic, what)


def failing_rows(name, prog, n=6):
    """Hardpoint rows of a failing batch (tests/test_batches.py FAIL_BATCHES): the reference's failing
    instances first."""
    from test_batches import batch_inputs
    meta, arr = load_golden(name)
    order = np.argsort(arr["status"] == 0, kind="stable")
    return batch_inputs(meta, arr, prog, order[:n])[0]


# Explicit design constants take the model's initial_state(), whose camber-shim pre-solve needs the device
# when a shim's setup thickness differs from design: the shimmed and failing-batch topologies run with
# design rules only.
GOLDEN_SPEC_CASES = (
    [pytest.param(c, dr, False, id=f"{c}-{dr}") for c in SWEEP_CASES for dr in (True, False)]
    + [pytest.param(c, True, False, id=f"{c}-True") for c in SHIM_CASES + FAIL_BATCHES]
    + [pytest.param(c, True, True, id=f"{c}-tuned") for c in SWEEP_CASES + SHIM_CASES + FAIL_BATCHES])


@pytest.mark.parametrize("case,design_rules,tune_layout", GOLDEN_SPEC_CASES)
def test_spec_emulation_matches_generic_golden(case, design_rules, tune_layout):
    prog, nominal, values = golden_program(case, design_rules, tune_layout)
    rows = failing_rows(case, prog) if case in FAIL_BATCHES else None
    check_spec_matches_generic(prog, nominal, values, rows=rows)


@pytest.mark.parametrize("design_rules,tune_layout", [pytest.param(True, False, id="True"),
                                                      pytest.param(False, False, id="False"),
                                                      pytest.param(True, True, id="tuned")])
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_spec_emulation_matches_generic_linkages(name, design_rules, tune_layout):
    lk = build(next(c for c in CASES if c.name == name))
    prog = T.compile_topology(lk.state, lk.constraints, lk.spec, lk.heads, design_rules=design_rules,
                              tune_layout=tune_layout)
    nominal = np.concatenate([lk.design[k] for k in prog.in_keys])
    check_spec_matches_generic(prog, nominal, lk.values, n=3)


def test_spec_rounds_pack_every_task_once():
    """Every task of every phase appears once in the packed words, with its contributions in order."""
    prog, _, _ = golden_program(SWEEP_CASES[0], True)
    src = prog.spec_source()
    arrays = {}
    for line in src.splitlines():
        if line.startswith(("constexpr int32_t", "const int32_t okin_spec_words")):
            name = line.split("[")[0].split()[-1]
            arrays[name] = [int(v) for v in line.split("{")[1].split("}")[0].split(",")]
    words = arrays["okin_spec_words"]
    for p, tasks in enumerate(prog.spec_phases()):
        got = []
        for r in range(arrays["PHASE_ROUND"][p], arrays["PHASE_ROUND"][p + 1]):
            base, width, slots, s0 = (arrays[k][r] for k in ("R_BASE", "R_WIDTH", "R_SLOTS", "R_SLOT0"))
            for lane in range(width):
                cons = [words[base + (s + 1) * width + lane] & 0xFFFFFFFF for s in range(slots)
                        if lane < arrays["SLOT_LANES"][s0 + s]]
                got.append((words[base + lane] & 0xFFFFFFFF, cons))
        assert sorted(got) == sorted(tasks), p


def check_nvrtc_compile(prog):
    """NVRTC builds both specialised lean kernels of ``prog`` for sm_100a: the instantiation with the
    camber-shim pre-solve when the program has shim records, at 512 threads within 128 registers and at
    384 threads within 168."""
    from open_kinematics_b200 import _lib
    if not _lib.nvrtc_available():
        pytest.skip("libnvrtc not found")
    cubin, log = _lib.spec_compile(prog)
    assert len(cubin) > 0, log
    used, entry = {}, None
    for line in log.splitlines():
        if "Compiling entry function" in line:
            entry = line.split("'")[1]
        elif "Used " in line and "registers" in line:
            used[entry] = int(line.split("Used ")[1].split()[0])
    shim = int(prog.hdr[T.D["OKIN_H_NSHIM"]] > 0)
    want = {f"_Z17okin_sweep_kernelILb0ELb{shim}ELi{threads}ELb0EE": cap for threads, cap in ((512, 128), (384, 168))}
    got = {name.split("EEvPKi")[0] + "EE": regs for name, regs in used.items()}
    assert set(got) == set(want), log
    for name, cap in want.items():
        assert got[name] <= cap, (name, got[name], log)


def test_nvrtc_compiles_flagship_spec():
    import bench
    sus, sweep = bench.workload_case()
    check_nvrtc_compile(T.compile_suspension(sus, sweep))


# One spec of each kind (a CPU-only NVRTC compile takes 15-20 s): C1 is the shim instantiation (one record
# at design thickness), C2 a MacPherson strut, the C4 T-bar axle has two shim records away from design, and
# random_60_4 is the largest generated linkage the device runs.
@pytest.mark.parametrize("case", ["c1_dw_corner_bump", "c2_macpherson_bump_steer", "c4_tbar_heave_shim_bump",
                                  "random_60_4"])
def test_nvrtc_compiles_spec(case):
    if case in SWEEP_CASES + SHIM_CASES:
        prog = golden_program(case, True)[0]
    else:
        lk = build(next(c for c in CASES if c.name == case))
        prog = T.compile_topology(lk.state, lk.constraints, lk.spec, lk.heads)
    check_nvrtc_compile(prog)


@pytest.mark.gpu
def test_specialised_lean_kernel_bit_identical(monkeypatch):
    """Flagship at sigma 0.5 and 10 mm, and the largest generated linkage the device runs: the specialised
    lean kernel against the generic lean kernel, both families, big enough to trigger the calibration."""
    import bench
    from open_kinematics_b200 import _lib
    from test_generated_linkages import OVERSIZED, cta_bytes, instances, linkage, program
    sus, sweep = bench.workload_case()
    flag = T.compile_suspension(sus, sweep)
    from open_kinematics_b200.core.solver import sweep_target_values
    flag_values = sweep_target_values(sweep)[1]
    auth = helpers.authored_positions(sus)
    flag_nominal = np.concatenate([auth[k] for k in flag.in_keys])
    runs = [c.name for c in CASES if c.name != OVERSIZED]
    largest = max(runs, key=lambda n: cta_bytes(program(linkage(n))))
    lk = linkage(largest)
    lprog = program(lk)
    cases = [(flag, perturbed(flag_nominal, 40000, 0.5, 1), flag_values),
             (flag, perturbed(flag_nominal, 40000, 10.0, 2), flag_values),
             (lprog, np.repeat(instances(lk, lprog)[0][:1], 40000, axis=0) +
              np.random.default_rng(3).normal(0.0, 0.5, (40000, 3 * lprog.n_in)), lk.values)]
    for prog, hp, values in cases:
        results = {}
        for regs in ("128", "168", "spec128", "spec168"):
            monkeypatch.setenv("OKIN_LEAN_REGS", regs)
            topo = _lib.DeviceTopology(prog)
            try:
                results[regs] = topo.solve_batch(hp, values, want_worst_row=True)
                cal = topo.lean_calibration()
            finally:
                topo.close()
            assert cal["specialised"] == regs.startswith("spec"), (regs, cal)
        for regs in ("168", "spec128", "spec168"):
            assert_bit_identical(results[regs], results["128"], regs)
