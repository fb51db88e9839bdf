"""Scrambled Sobol' variates of tolerance studies on the CPU: the committed direction-number table
against SciPy's, the numpy restatement (tests/sobol_reference.py) against SciPy's unscrambled
sequence, the lane-emulation generator and the tables uploaded for the device against the
restatement, the net properties the scramble must keep, AS241 against mpmath, emulated Sobol' studies against numpy statistics and across
emulated device counts, and the new usage errors of the C ABI."""

from __future__ import annotations

import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import sobol_reference as sref
from helpers import ROOT
from study_emu import emu_study, emu_study_inputs
from test_study import call_study, check_against_numpy, solver_of


@pytest.fixture(scope="module")
def c1():
    s = solver_of("c1_dw_corner_bump")
    yield s
    s.close()


@pytest.fixture(scope="module")
def axle():
    s = solver_of("c4_tbar_heave_shim_bump")
    yield s
    s.close()


def test_table_matches_scipy():
    text = open(os.path.join(ROOT, "open-kinematics_b200", "csrc", "okin_sobol.h")).read()
    body = lambda name: text[text.index(name):].split("};")[0].split("= {", 1)[1]
    poly = np.array([int(x) for x in re.findall(r"\d+", body("okin_sobol_poly["))])
    vinit = np.array([int(x) for x in re.findall(r"\d+", body("okin_sobol_vinit["))]).reshape(1024, -1)
    want_poly, want_vinit = sref.scipy_table()
    assert np.array_equal(poly, want_poly[:1024])
    cols = vinit.shape[1]
    assert np.array_equal(vinit, want_vinit[:1024, :cols]) and not want_vinit[:1024, cols:].any()


def test_unscrambled_matches_scipy():
    """The restatement with the identity scramble is SciPy's sequence bit for bit (SciPy's
    fast_forward does not take bits > 32, so both start at point 0)."""
    from scipy.stats import qmc
    X = sref.points(sref.directions(1024), np.arange(4096))
    want = qmc.Sobol(1024, scramble=False, bits=52).random(4096)
    assert np.array_equal(X.astype(np.float64) * 2.0 ** -52, want)
    assert list(X[:8, 0].astype(np.float64) * 2.0 ** -52) == [0, 0.5, 0.75, 0.25, 0.375, 0.875, 0.625, 0.125]


def mixed_sobol_sampling(solver, mirror_right=False):
    """Philox normals, Sobol' normals and uniforms, a grid factor (crossed index) and, where the
    topology has them, the setup thicknesses as Sobol' uniforms."""
    from open_kinematics_b200.core.study import Sampling
    keys = [k for k in solver.program.in_keys]
    smp = Sampling(solver, mirror_right=mirror_right)
    own = [k for i, k in enumerate(keys) if i not in smp._followers]
    smp.normal(own[0], 0.4).normal(own[1], 0.3, sequence="sobol").uniform([(own[2], "x"), own[3]], 0.25,
                                                                       sequence="sobol")
    smp.grid((own[4], 2), 1.0, 3).normal(own[5], [0.1, 0.2, 0.3], sequence="sobol")
    smp.uniform((own[2], "z"), 0.2)
    thick = [n for n in solver.program.param_names if n.endswith("setup_thickness")]
    if thick:
        smp.uniform(thick, 0.5, sequence="sobol")
    return smp


def compare_inputs(solver, smp, seed, ids):
    hp, par = emu_study_inputs(solver, smp, seed, ids)
    got = np.concatenate([hp, par], axis=1)
    tables = smp.tables()
    want = sref.inputs(tables, seed, ids)
    kind = np.asarray(smp.variate_kind)
    src = smp.source
    normal = (src >= 0) & np.isin(kind[np.maximum(src, 0)], (0, 4))
    assert np.array_equal(got[:, ~normal], want[:, ~normal])
    z = (want[:, normal] - smp.nominal[normal]) / smp.scale[normal]
    tol = 4 * np.spacing(np.abs(z)) * np.abs(smp.scale[normal]) + np.spacing(np.abs(want[:, normal]))
    assert (np.abs(got[:, normal] - want[:, normal]) <= tol).all()
    return got, want


@pytest.mark.parametrize("case", ["c1", "axle"])
def test_emulation_matches_restatement(case, request):
    solver = request.getfixturevalue(case)
    smp = mixed_sobol_sampling(solver, mirror_right=case == "axle")
    kinds = set(smp.variate_kind)
    assert {0, 1, 2, 3, 4} <= kinds
    ids = np.concatenate([np.arange(600), [2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 40 + 12345, 3 * 2 ** 51 - 1]])
    for seed in (0, 12345, 2 ** 40 + 99):
        got, _ = compare_inputs(solver, smp, seed, ids)
    # crossed design: the three grid levels of one Sobol' point share its Sobol' coordinates
    sob = np.isin(np.asarray(smp.variate_kind)[np.maximum(smp.source, 0)], (3, 4)) & (smp.source >= 0)
    assert np.array_equal(got[0:600:3][:, sob], got[1:600:3][:, sob])
    assert np.array_equal(got[0:600:3][:, sob], got[2:600:3][:, sob])
    assert len(np.unique(got[0:600:3][:, sob], axis=0)) == 200
    if case == "axle":       # mirrored right twins share the left point's Sobol' variate
        twins = [(c, r) for c in range(smp.n_hardpoint_coords) for r in range(smp.n_hardpoint_coords)
                 if c != r and smp.source[c] >= 0 and smp.source[r] == smp.source[c] and sob[c]]
        assert twins
        for c, r in twins:
            sign = -1.0 if c % 3 == 1 else 1.0
            assert np.array_equal(got[:, r] - smp.nominal[r], sign * (got[:, c] - smp.nominal[c]))


def unit_sobol_points(solver, seed, n):
    """``X [n, D]`` read back from the emulated generator: Sobol' uniforms of scale 1 about nominal 0."""
    from open_kinematics_b200.core.study import Sampling
    smp = Sampling(solver).uniform("all", 1.0, sequence="sobol")
    smp.nominal = np.zeros_like(smp.nominal)
    hp, _ = emu_study_inputs(solver, smp, seed, np.arange(n))
    z = hp[:, smp.source[:hp.shape[1]] >= 0]
    X = (z + 1.0) * 2.0 ** 51
    assert np.array_equal(X, np.round(X))
    return X.astype(np.uint64)


@pytest.mark.parametrize("m", [4, 9, 12])
def test_net_properties(c1, m):
    """First 2^m scrambled points: every dimension puts one point in each of the 2^m intervals, and
    dimensions (0, 1) form a (0, m, 2)-net (every elementary box of area 2^-m holds one point)."""
    for seed in (1, 2 ** 35 + 17):
        X = unit_sobol_points(c1, seed, 2 ** m)
        top = X >> np.uint64(52 - m)
        for d in range(X.shape[1]):
            assert np.array_equal(np.sort(top[:, d]), np.arange(2 ** m, dtype=np.uint64)), d
        for k in range(m + 1):
            a = X[:, 0] >> np.uint64(52 - k) if k else np.zeros(2 ** m, np.uint64)
            b = X[:, 1] >> np.uint64(52 - (m - k)) if m - k else np.zeros(2 ** m, np.uint64)
            assert len(np.unique(a * np.uint64(2 ** (m - k)) + b)) == 2 ** m, k
        assert X.shape[1] > 20


def test_scramble_changes_with_seed_and_variate(c1):
    X1, X2 = unit_sobol_points(c1, 1, 64), unit_sobol_points(c1, 2, 64)
    assert not np.array_equal(X1, X2)
    assert len({tuple(X1[:, d]) for d in range(X1.shape[1])}) == X1.shape[1]
    assert (X1[0] != 0).all()


@pytest.fixture(scope="module")
def sobol_lib(tmp_path_factory):
    """tests/emu/okin_emu_sobol.cpp built with g++ outside the tree: the library's Sobol' table
    builder and AS241 on the host."""
    src = os.path.join(ROOT, "tests", "emu", "okin_emu_sobol.cpp")
    out = str(tmp_path_factory.mktemp("sobol_emu") / "libokin_emu_sobol.so")
    csrc = os.path.join(ROOT, "open-kinematics_b200", "csrc")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", f"-I{csrc}", "-o", out, src], check=True)
    lib = ctypes.CDLL(out)
    lib.okin_emu_sobol_tables.restype = ctypes.c_int
    lib.okin_emu_sobol_tables.argtypes = [ctypes.c_uint64, ctypes.c_int] + [ctypes.c_void_p] * 5
    lib.okin_emu_ppnd16.restype = None
    lib.okin_emu_ppnd16.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong]
    return lib


def test_uploaded_tables_match_restatement(c1, sobol_lib):
    """The scrambled direction numbers and shifts okin_study uploads for the device are M_v V[d][k]
    and S_v of the restatement, with d counting Sobol' variates only."""
    smp = mixed_sobol_sampling(c1)
    t = smp.tables()
    kind, levels = t["variate_kind"], t["grid_levels"]
    nv = kind.size
    sob = [v for v in range(nv) if kind[v] in (3, 4)]
    V = sref.directions(len(sob))
    for seed in (0, 2 ** 40 + 99):
        rank = np.zeros(nv, np.int32)
        dirs = np.zeros((nv, sref.BITS), np.uint64)
        shift = np.zeros(nv, np.uint64)
        n = sobol_lib.okin_emu_sobol_tables(seed, nv, kind.ctypes.data, levels.ctypes.data, rank.ctypes.data,
                                            dirs.ctypes.data, shift.ctypes.data)
        assert n == len(sob) and list(rank) == [sob.index(v) if v in sob else -1 for v in range(nv)]
        for d, v in enumerate(sob):
            rows, s = sref.scramble(seed, v)
            assert np.array_equal(dirs[d], sref.apply_matrix(rows, V[d])) and int(shift[d]) == s


def ppnd16_emu(lib, p: np.ndarray) -> np.ndarray:
    p = np.ascontiguousarray(p, np.float64)
    z = np.empty_like(p)
    lib.okin_emu_ppnd16(p.ctypes.data, z.ctypes.data, p.size)
    return z


def test_ppnd16_against_mpmath(sobol_lib):
    import mpmath
    k = np.arange(0, 53, 0.25)
    tails = np.unique(np.concatenate([np.ldexp(1.0, -53) * (2 * np.arange(4) + 1), np.exp2(-k)]))
    tails = tails[(tails >= 2.0 ** -53) & (tails < 0.5)]
    rng = np.random.default_rng(3)
    central = np.concatenate([rng.random(400), 0.5 + np.ldexp(1.0, -np.arange(2, 53)),
                              np.nextafter([0.075, 0.075, 0.925, 0.925], [0, 1, 0, 1])])
    p = np.unique(np.concatenate([tails, 1.0 - tails, central, [0.5]]))
    p = p[(p >= 2.0 ** -53) & (p <= 1.0 - 2.0 ** -53)]
    mpmath.mp.dps = 50
    want = np.array([float(mpmath.sqrt(2) * mpmath.erfinv(2 * mpmath.mpf(float(x)) - 1)) for x in p])
    for got in (ppnd16_emu(sobol_lib, p), sref.ppnd16(p)):
        assert (np.abs(got - want) <= 1e-15 * np.abs(want)).all(), np.max(np.abs(got - want) / np.abs(want))
    assert ppnd16_emu(sobol_lib, np.array([2.0 ** -53]))[0] < -8.2


def test_emulated_study_matches_numpy(c1, axle):
    from open_kinematics_b200.core.study import Sampling
    smp = Sampling(c1).normal("all", 0.5, sequence="sobol")
    kw = dict(points=[c1.program.out_keys[0], c1.program.out_keys[-1]], metrics="all",
              solver_quantities=("solver_max_residual", "solver_nfev"))
    res = emu_study(c1, smp, 256, seed=7, chunk=64, **kw)
    check_against_numpy(c1, smp, 7, 256, res, want_metrics=True)
    res_lean = emu_study(c1, mixed_sobol_sampling(c1), 150, seed=8, points="all", chunk=64)
    check_against_numpy(c1, mixed_sobol_sampling(c1), 8, 150, res_lean, want_metrics=False)
    smp = mixed_sobol_sampling(axle, mirror_right=True)
    res = emu_study(axle, smp, 96, seed=5, points=axle.program.out_keys[:6], solver_quantities=("solver_nfev",),
                    chunk=40)
    check_against_numpy(axle, smp, 5, 96, res, want_metrics=False)


def test_emulated_study_device_splits_bit_identical(c1):
    from open_kinematics_b200.core.study import Sampling
    smp = Sampling(c1).normal("all", 1.0, sequence="sobol").uniform("camber_shim.setup_thickness", 0.5,
                                                                    sequence="sobol")
    runs = [emu_study(c1, smp, 170, seed=3, points="all", solver_quantities=("solver_nfev",), chunk=32, n_devices=g)
            for g in (1, 2, 3)]
    for other in runs[1:]:
        for field in ("count", "nonfinite", "mean", "std", "min", "max", "argmin", "argmax", "status_counts",
                      "failed_at_step"):
            assert getattr(runs[0], field).tobytes() == getattr(other, field).tobytes(), field


def test_usage_errors(c1):
    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.study import Sampling, study_quantities
    prog = c1.program
    _, _, kinds, idx = study_quantities(prog, points=[prog.out_keys[0]])
    quantities = dict(quantity_kind=kinds, quantity_index=idx, hist_lo=np.zeros(kinds.size),
                      hist_hi=np.ones(kinds.size))
    base = dict(Sampling(c1).normal((prog.in_keys[0], 0), 1.0, sequence="sobol").tables(), **quantities)

    def expect(arrays, match, **kw):
        rc, msg = call_study(c1, arrays, **kw)
        assert rc == -1 and match in msg, (rc, msg)

    def variates(kinds, levels=None):
        kinds = np.asarray(kinds, np.int32)
        return dict(base, variate_kind=kinds,
                    grid_levels=np.asarray(levels if levels is not None else np.zeros(kinds.size), np.int32))

    expect(variates([3] * 1025), "at most 1024 Sobol' variates")
    rc, msg = call_study(c1, variates([4] * 1024), n=-1)
    assert rc == -1 and "negative size" in msg, msg          # 1024 is accepted
    expect(variates([3] + [2] * 64, [0] + [2] * 64), "grid period below 2^63")
    expect(base, "below 2^52", n=2 ** 52 + 1)
    expect(variates([3, 2], [0, 3]), "below 2^52", n=3 * 2 ** 52 + 1)
    rc, msg = call_study(c1, variates([0, 2], [0, 3]), n=-1)
    assert rc == -1 and "negative size" in msg, msg
    vk = base["variate_kind"].copy()
    vk[0] = 5
    expect(dict(base, variate_kind=vk), "unknown variate kind")
    # okin_study_sample checks each id's point index
    desc = _lib.StudyDesc.of(base)
    hp = np.zeros((2, 3 * prog.n_in))
    par = np.zeros((2, len(prog.param_names)))
    ids = np.array([0, 2 ** 52], np.int64)
    rc = _lib.load().okin_study_sample(c1.topology.handle, ctypes.byref(desc), 2, ids.ctypes.data, hp.ctypes.data,
                                       par.ctypes.data, 0)
    assert rc == -1 and "below 2^52" in _lib.last_error()
    with pytest.raises(ValueError, match="Unknown sequence"):
        Sampling(c1).normal("all", 1.0, sequence="halton")
    t = Sampling(c1).normal("all", 1.0, sequence="sobol").uniform("camber_shim.setup_thickness", 0.5,
                                                                   sequence="sobol").tables()
    assert set(t["variate_kind"][:-1]) == {4} and t["variate_kind"][-1] == 3
    assert set(Sampling(c1).normal("all", 1.0).tables()["variate_kind"]) == {0}
