"""Independent restatement of the hardpoint sensitivities from the oracle alone, at the device's own
solved states (lane emulation here; ``test_hardpoint_sensitivity_gpu`` runs the C ABI against it).

For a state x (the device's) and hardpoints p, the least-squares residual vector of the oracle is
    R(x, p) = [constraint rows without the point-on-line rows; their pins n.(x - p0(p)); targets]
with the design pose, constants, derived-op parameters and relative-target bases recomputed from p by
``design_setup`` / ``target_bases``.  dR/dp_k comes from Richardson-extrapolated central differences in
p with x held, dx = -lstsq(J, dR/dp_k) with J the oracle's Jacobian (plus pin rows), and every output
point's total derivative from central differences of the oracle's derived points along (dx, e_k)."""

from __future__ import annotations

import numpy as np
import pytest

from helpers import authored_positions, build_case, emu_solve, load_golden, oracle_problem
from oracle.solve import ResidualComputer, design_setup, pin_rows, target_bases

CASES = ["c1_dw_corner_bump", "c1_dw_corner_bump_steer", "c2_macpherson_bump_steer", "c3_rocker_ubar_coilover_roll",
         "c4_tbar_bump", "dw_corner_rocker", "macpherson_axle"]
H = 1e-3   # mm; Richardson on h and 2h leaves ~h^4 x (fifth derivative) ~ 1e-12


class Restatement:
    def __init__(self, sus, sweep, prog):
        self.problem, self.values = oracle_problem(sus, sweep, from_design=True, structure_only=True)
        self.values = np.asarray(self.values, dtype=np.float64)
        self.auth = authored_positions(sus)
        self.prog = prog
        self.keep = [i for i, c in enumerate(self.problem.constraints) if c.family != "point_on_line"]

    def setup(self, p):
        authored = dict(self.auth)
        for i, k in enumerate(self.prog.in_keys):
            authored[k] = p[3 * i: 3 * i + 3]
        pos0, consts = design_setup(self.problem, authored)
        return pos0, consts, target_bases(self.problem, pos0)

    def residual(self, x, p, s):
        pos0, consts, bases = self.setup(p)
        rc = ResidualComputer(self.problem, pos0, consts)
        nc = len(self.problem.constraints)
        r = rc.compute(x, bases + self.values[:, s])
        pins = [float((x[col: col + 3] - p0) @ n) for col, n, p0 in pin_rows(self.problem, consts)]
        return np.concatenate([r[self.keep], pins, r[nc:]])

    def jacobian(self, x, p, s):
        pos0, consts, bases = self.setup(p)
        rc = ResidualComputer(self.problem, pos0, consts)
        nc = len(self.problem.constraints)
        J = rc.compute_jacobian(x, bases + self.values[:, s])
        rows = []
        for col, n, _ in pin_rows(self.problem, consts):
            row = np.zeros(self.problem.n)
            row[col: col + 3] = n
            rows.append(row)
        return np.vstack([J[self.keep], *rows, J[nc:]]) if rows else np.vstack([J[self.keep], J[nc:]])

    def points(self, x, p):
        pos0, consts, _ = self.setup(p)
        rc = ResidualComputer(self.problem, pos0, consts)
        rc._refresh(x)
        return np.array([rc.pos[k] for k in self.prog.out_keys])

    @staticmethod
    def richardson(f, h):
        d1 = (f(h) - f(-h)) / (2 * h)
        d2 = (f(2 * h) - f(-2 * h)) / (4 * h)
        return (4 * d1 - d2) / 3

    def sensitivity(self, x, p, s, coords):
        """[len(coords), n_out, 3] at state x of step s."""
        J = self.jacobian(x, p, s)
        out = []
        for k in coords:
            e = np.zeros_like(p)
            e[k] = 1.0
            dr = self.richardson(lambda t: self.residual(x, p + t * e, s), H)
            dx = -np.linalg.lstsq(J, dr, rcond=None)[0]
            out.append(self.richardson(lambda t: self.points(x + t * dx, p + t * e), H))
        return np.array(out)


def device_state(prog, positions_s):
    pts = {k: positions_s[i] for i, k in enumerate(prog.out_keys)}
    return lambda problem: np.concatenate([pts[k] for k in problem.free_order])


# Bar per entry, relative to max(1, |S|): the Richardson differences leave ~1e-11 (h = 1e-3 mm); the
# oracle's SVD least squares and the device's Cholesky of the normal equations differ by round-off times
# the condition number of A (cond(J)^2 <= 1e7 on these topologies: 1e-9); the device evaluates at its own
# state, the oracle at the same state.  Bar: 1e-8.
REF_TOL = 1e-8


def compare(prog, sus, sweep, hp, out, steps, coords):
    ref = Restatement(sus, sweep, prog)
    worst = 0.0
    for i in range(hp.shape[0]):
        for s in steps:
            x = device_state(prog, out["positions"][i, s])(ref.problem)
            want = ref.sensitivity(x, hp[i], s, coords)
            got = out["hardpoint_sensitivity"][i, s][coords]
            err = np.abs(got - want) / np.maximum(1.0, np.abs(want))
            worst = max(worst, float(err.max()))
    assert worst <= REF_TOL, worst
    return worst


@pytest.mark.parametrize("name", CASES)
def test_golden_sweep_against_restatement_emu(name):
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_suspension
    meta, _ = load_golden(name)
    sus, sweep = build_case(meta)
    prog = compile_suspension(sus, sweep, with_shims=False)
    auth = authored_positions(sus)
    hp = np.concatenate([auth[k] for k in prog.in_keys])[None]
    _, values = sweep_target_values(sweep)
    out = emu_solve(prog, hp, np.asarray(values, dtype=np.float64), want_hardpoint_sensitivity=True)
    assert (out["status"] == 0).all()
    S = out["positions"].shape[1]
    K = len(prog.sensitivity_inputs)
    compare(prog, sus, sweep, hp, out, sorted({0, S // 2, S - 1}), list(range(0, K, max(1, K // 10))))


@pytest.mark.parametrize("name", ["batch256_c1", "batch256_c2", "batch256_c3"])
def test_perturbed_batch_against_restatement_emu(name):
    from open_kinematics_b200.core.solver import sweep_target_values
    from open_kinematics_b200.core.topology import compile_suspension
    from test_batches import batch_inputs
    from helpers import build_suspension, build_sweep
    meta, arr = load_golden(name)
    sus = build_suspension(meta["geometry"])
    sweep = build_sweep(meta["sweep"], sus)
    prog = compile_suspension(sus, sweep, with_shims=False)
    hp, _ = batch_inputs(meta, arr, prog, range(32))
    _, values = sweep_target_values(sweep)
    out = emu_solve(prog, hp, np.asarray(values, dtype=np.float64), want_hardpoint_sensitivity=True)
    assert (out["status"] == 0).all()
    S, K = out["positions"].shape[1], len(prog.sensitivity_inputs)
    compare(prog, sus, sweep, hp, out, [S - 1], list(range(0, K, max(1, K // 4))))
