"""Hardpoint sensitivities through the C ABI on a device (``pytest -m gpu``): agreement with the lane
emulation and the oracle restatement on perturbed batches, chunked and multi-device batches against instances solved alone, the
device-buffer entry point, the camber-shim usage error and the linearised spread against Monte Carlo."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import authored_positions, build_case, load_golden
from sens_emu import emu_solve_sens
from test_batches import batch_inputs
from test_hardpoint_sensitivity import FULL_OUTPUTS

pytestmark = pytest.mark.gpu

BATCHES = ["batch256_c1", "batch256_c2", "batch256_c3"]


def compile_batch_sens(name, **kw):
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_suspension
    from helpers import build_suspension, build_sweep
    meta, arr = load_golden(name)
    sus = build_suspension(meta["geometry"])
    sweep = build_sweep(meta["sweep"], sus)
    prog = compile_suspension(sus, sweep, with_shims=False, **kw)
    _, values = sweep_target_values(sweep)
    return meta, arr, prog, np.asarray(values, dtype=np.float64)


@pytest.mark.parametrize("name", BATCHES)
def test_device_matches_emulation(name):
    from open_kinematics_b200 import _lib
    meta, arr, prog, values = compile_batch_sens(name)
    hp, _ = batch_inputs(meta, arr, prog, range(64))
    topo = _lib.DeviceTopology(prog)
    try:
        dev = topo.solve_batch(hp, values, want_tangents=True, want_velocities=True, want_health=True,
                               want_metrics=bool(prog.metric_names), want_design=True,
                               want_diagnostics=bool(prog.diagnostic_names), want_hardpoint_sensitivity=True)
        base = topo.solve_batch(hp, values, want_tangents=True, want_velocities=True, want_health=True,
                                want_metrics=bool(prog.metric_names), want_design=True,
                                want_diagnostics=bool(prog.diagnostic_names))
    finally:
        topo.close()
    for key in FULL_OUTPUTS:      # requesting sensitivities changes no other output
        if base.get(key) is not None:
            assert np.array_equal(base[key], dev[key], equal_nan=True), (name, key)
    emu = emu_solve_sens(prog, hp, values)
    assert (dev["status"] == 0).all() and (emu["status"] == 0).all()
    s_dev, s_emu = dev["hardpoint_sensitivity"], emu["hardpoint_sensitivity"]
    # same algorithm, different contraction / rounding of the fp64 arithmetic; the states themselves agree
    # to ~1e-12 mm, the sensitivities to round-off amplified by the conditioning of A
    err = np.abs(s_dev - s_emu) / np.maximum(1.0, np.abs(s_emu))
    assert err.max() <= 1e-9, (name, err.max())
    from helpers import build_suspension, build_sweep
    from test_hardpoint_sensitivity_reference import compare
    sus = build_suspension(meta["geometry"])
    S, K = values.shape[1], len(prog.sensitivity_inputs)
    compare(prog, sus, build_sweep(meta["sweep"], sus), hp[:4], {k: v[:4] for k, v in dev.items() if v is not None},
            [S - 1], list(range(0, K, max(1, K // 4))))


def test_chunked_two_device_batch_matches_instances_alone():
    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_suspension
    meta, _ = load_golden("c1_dw_corner_bump")
    sus, sweep = build_case(meta)
    first_free = compile_suspension(sus, sweep, with_shims=False).free_order[0]
    prog = compile_suspension(sus, sweep, with_shims=False, output_points=[first_free])
    _, values = sweep_target_values(sweep)
    values = np.asarray(values, dtype=np.float64)[:, :3]
    auth = authored_positions(sus)
    nominal = np.concatenate([auth[k] for k in prog.in_keys])
    n = 3 * 32768 + 123
    rng = np.random.default_rng(7)
    hp = nominal + rng.normal(0.0, 0.2, (n, nominal.size))
    devices = [0, 1] if _lib.device_count() >= 2 else [0]
    topo = _lib.DeviceTopology(prog)
    try:
        big = topo.solve_batch(hp, values, devices=devices, want_hardpoint_sensitivity=True)
        pick = [0, 32767, 32768, 65535, 65536, 98303, 98304, n - 1, n // 2]
        for i in pick:
            one = topo.solve_batch(hp[i:i + 1], values, want_hardpoint_sensitivity=True)
            assert np.array_equal(one["hardpoint_sensitivity"][0], big["hardpoint_sensitivity"][i], equal_nan=True), i
            assert np.array_equal(one["positions"][0], big["positions"][i], equal_nan=True), i
    finally:
        topo.close()
    assert big["hardpoint_sensitivity"].shape == (n, 3, len(prog.sensitivity_inputs), 1, 3)
    assert np.isfinite(big["hardpoint_sensitivity"][big["status"] == 0]).all()


def test_device_entry_point_fills_every_entry():
    import torch
    from open_kinematics_b200 import _lib
    meta, arr, prog, values = compile_batch_sens("batch256_c2")
    hp, _ = batch_inputs(meta, arr, prog, range(40))
    n, S, K = len(hp), values.shape[1], len(prog.sensitivity_inputs)
    dev = torch.device("cuda:0")
    sentinel = -7.25e33
    t_hp = torch.tensor(hp, device=dev)
    t_tv = torch.tensor(values, device=dev)
    status = torch.full((n,), -99, dtype=torch.int32, device=dev)
    failed = torch.full((n,), -99, dtype=torch.int32, device=dev)
    pos = torch.full((n, S, prog.n_out, 3), sentinel, dtype=torch.float64, device=dev)
    sens = torch.full((n, S, K, prog.n_out, 3), sentinel, dtype=torch.float64, device=dev)
    io = _lib.BatchIO.of(hardpoints=t_hp.data_ptr(), target_values=t_tv.data_ptr(), status=status.data_ptr(),
                         failed_step=failed.data_ptr(), positions=pos.data_ptr(),
                         hardpoint_sensitivity=sens.data_ptr())
    import ctypes
    cfg = _lib.default_cfg()
    stream = torch.cuda.current_stream(dev)
    topo = _lib.DeviceTopology(prog)
    try:
        _lib.check(_lib.load().okin_solve_batch_device(topo.handle, ctypes.byref(cfg), 0,
                                                       ctypes.c_void_p(stream.cuda_stream), n, S, ctypes.byref(io)),
                   "okin_solve_batch_device")
        torch.cuda.synchronize(dev)
        host = topo.solve_batch(hp, values, want_hardpoint_sensitivity=True)
    finally:
        topo.close()
    got = sens.cpu().numpy()
    assert not (got == sentinel).any()
    assert (status.cpu().numpy() == host["status"]).all()
    assert np.array_equal(got, host["hardpoint_sensitivity"], equal_nan=True)


def test_shim_topology_usage_error():
    from open_kinematics_b200 import _lib
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.sweep import BatchSolver
    from open_kinematics_b200.core.topology import compile_suspension
    meta, _ = load_golden("c4_tbar_heave_shim_roll")
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep)
    hp = np.concatenate([authored_positions(sus)[k] for k in prog.in_keys])[None]
    _, values = sweep_target_values(sweep)
    topo = _lib.DeviceTopology(prog)
    try:
        with pytest.raises(RuntimeError, match="camber-shim"):
            topo.solve_batch(hp, values, want_hardpoint_sensitivity=True)
    finally:
        topo.close()
    solver = BatchSolver(sus, sweep)
    try:
        with pytest.raises(ValueError, match="camber shims"):
            solver.solve(hp, want_hardpoint_sensitivity=True)
    finally:
        solver.close()


def test_linearised_spread_matches_monte_carlo():
    """C1, every hardpoint coordinate with sigma = 0.01 mm: the sample standard deviation of 16384
    solved instances against the helper's first-order spread at the nominal geometry.  The sample
    standard deviation has a relative sampling error of about 1/sqrt(2N) = 0.55 %; second-order terms
    are ~sigma x curvature ~ 1e-5 relative.  Bar: 5 sampling errors (2.8 %) on every output coordinate
    whose spread is at least 1e-4 mm."""
    from open_kinematics_b200.core.sensitivity import linearised_std
    from open_kinematics_b200.core.sweep import BatchSolver
    meta, _ = load_golden("c1_dw_corner_bump")
    sus, sweep = build_case(meta)
    solver = BatchSolver(sus, sweep)
    try:
        nominal = solver.nominal_hardpoints()
        lin = linearised_std(solver.solve(nominal[None], want_hardpoint_sensitivity=True).hardpoint_sensitivity,
                             0.01)[0]
        N, sigma = 16384, 0.01
        hp = nominal + np.random.default_rng(11).normal(0.0, sigma, (N, nominal.size))
        res = solver.solve(hp)
    finally:
        solver.close()
    assert (res.status == 0).all()
    sample = res.positions.std(axis=0, ddof=1)
    mask = lin >= 1e-4
    rel = np.abs(sample[mask] - lin[mask]) / lin[mask]
    assert rel.max() <= 5.0 / np.sqrt(2 * N), rel.max()
