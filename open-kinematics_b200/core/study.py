"""Tolerance studies: Monte Carlo and full-factorial DoE over hardpoints and params, with the inputs
generated and the per-step statistics reduced on the device (``okin_study``, include/okin.h).

A study moves kilobytes across PCIe whatever the number of instances: it returns, per step and
quantity, the count, mean, standard deviation, extremes with the instances that produced them, an
optional histogram and the failure counts.  ``BatchSolver.study_inputs`` regenerates the inputs of
chosen instances (for example the argmax of a column) so they can be re-solved with
``BatchSolver.solve``.  The sampling contract and the reduction order are in DESIGN.md section 10.
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .primitives.point_ref import PointRef, Side

VARIATE_NORMAL, VARIATE_UNIFORM, VARIATE_GRID, VARIATE_SOBOL_UNIFORM, VARIATE_SOBOL_NORMAL = 0, 1, 2, 3, 4
SEQUENCES = ("philox", "sobol")
QUANTITY_POSITION, QUANTITY_METRIC, QUANTITY_MAX_RESIDUAL, QUANTITY_NFEV = 0, 1, 2, 3
SOLVER_QUANTITIES = ("solver_max_residual", "solver_nfev")
AXES = "xyz"


def _point_name(key) -> str:
    return key.name.lower()


class Sampling:
    """Which input coordinates of a ``BatchSolver``'s model vary in a study, and how.

    Coordinates are the hardpoint coordinates (``3 * input slot + axis``) followed by the params
    (``program.param_names``, e.g. ``"<label>.setup_thickness"`` of a camber shim); every
    coordinate starts at its nominal value (``nominal_hardpoints()``, ``program.param_default``).
    Each ``normal`` / ``uniform`` / ``grid`` call gives every coordinate it names its own variate, in
    the order named; ``coords`` is a point key (all three axes), a ``(key, axis)`` pair, a point or
    param name, ``"all"``, or a list of these.  ``"all"`` is every hardpoint coordinate except
    centre-line y coordinates whose nominal is 0 (the T-bar pivot build validation needs them there).
    With ``mirror_right`` every right-side point with a left twin follows that twin: it shares the
    twin's variate with the y scale negated, and cannot be assigned itself.

    ``normal`` and ``uniform`` draw Philox pseudo-random variates by default; ``sequence="sobol"``
    draws them from a scrambled Sobol' sequence instead (one Sobol' dimension per variate, in the
    order assigned), whose mean and std estimates converge close to ``N^-1`` for smooth responses
    rather than ``N^-1/2``.  They are best at ``N = 2^m`` instances.  The kinds mix freely; with grid
    factors every grid node sees the same Sobol' sample (instance ``i`` takes Sobol' point
    ``i // prod(levels)``), a crossed design."""

    def __init__(self, solver, mirror_right: bool = False):
        prog = solver.program
        self.program = prog
        self.mirror_right = bool(mirror_right)
        self.n_hardpoint_coords = 3 * prog.n_in
        self.nominal = np.concatenate([np.asarray(solver.nominal_hardpoints(), dtype=np.float64),
                                       np.asarray(prog.param_default, dtype=np.float64)])
        self.source = np.full(self.nominal.size, -1, dtype=np.int32)
        self.scale = np.zeros(self.nominal.size)
        self.variate_kind: list = []
        self.grid_levels: list = []
        self._slot = {k: i for i, k in enumerate(prog.in_keys)}
        self._names = {_point_name(k): k for k in prog.in_keys}
        self._twin = {}             # left slot -> right slot
        if self.mirror_right:
            for k, i in self._slot.items():
                if getattr(k, "side", None) is Side.RIGHT and PointRef(Side.LEFT, k.point) in self._slot:
                    self._twin[self._slot[PointRef(Side.LEFT, k.point)]] = i
        self._followers = set(self._twin.values())

    def coordinate_name(self, c: int) -> str:
        if c >= self.n_hardpoint_coords:
            return self.program.param_names[c - self.n_hardpoint_coords]
        return f"{_point_name(self.program.in_keys[c // 3])}_{AXES[c % 3]}"

    def _coords(self, coords) -> list:
        if isinstance(coords, str):
            if coords == "all":
                out = []
                for i, key in enumerate(self.program.in_keys):
                    if i in self._followers:
                        continue
                    for a in range(3):
                        if a == 1 and getattr(key, "side", None) is Side.CENTER and abs(self.nominal[3 * i + 1]) < 1e-9:
                            continue
                        out.append(3 * i + a)
                return out
            if coords in self.program.param_names:
                return [self.n_hardpoint_coords + self.program.param_names.index(coords)]
            if coords.lower() in self._names:
                return self._coords(self._names[coords.lower()])
            raise ValueError(f"Unknown study coordinate {coords!r}")
        try:
            if coords in self._slot:
                return [3 * self._slot[coords] + a for a in range(3)]
        except TypeError:
            pass
        if isinstance(coords, tuple) and len(coords) == 2 and (coords[1] in (0, 1, 2) or coords[1] in tuple(AXES)):
            axis = AXES.index(coords[1]) if isinstance(coords[1], str) else int(coords[1])
            key = self._names.get(coords[0].lower()) if isinstance(coords[0], str) else coords[0]
            if key in self._slot:
                return [3 * self._slot[key] + axis]
        if isinstance(coords, (list, tuple)):
            return [c for item in coords for c in self._coords(item)]
        raise ValueError(f"Unknown study coordinate {coords!r}")

    def _assign(self, coords, kind: int, width, levels: int = 0) -> "Sampling":
        idx = self._coords(coords)
        widths = np.broadcast_to(np.asarray(width, dtype=np.float64), (len(idx),))
        for c, w in zip(idx, widths):
            if c < self.n_hardpoint_coords and c // 3 in self._followers:
                raise ValueError(f"{self.coordinate_name(c)} follows its left twin (mirror_right)")
            if self.source[c] >= 0:
                raise ValueError(f"Study coordinate {self.coordinate_name(c)} assigned twice")
            v = len(self.variate_kind)
            self.variate_kind.append(kind)
            self.grid_levels.append(int(levels))
            self.source[c], self.scale[c] = v, float(w)
            if c < self.n_hardpoint_coords and c // 3 in self._twin:
                r = 3 * self._twin[c // 3] + c % 3
                self.source[r], self.scale[r] = v, -float(w) if c % 3 == 1 else float(w)
        return self

    @staticmethod
    def _kind(sequence: str, philox: int, sobol: int) -> int:
        if sequence not in SEQUENCES:
            raise ValueError(f"Unknown sequence {sequence!r}; expected one of {SEQUENCES}")
        return sobol if sequence == "sobol" else philox

    def normal(self, coords, sigma, sequence: str = "philox") -> "Sampling":
        """Independent normal variation with standard deviation ``sigma`` (scalar or one per coordinate),
        drawn from ``sequence`` (``"philox"`` or ``"sobol"``)."""
        return self._assign(coords, self._kind(sequence, VARIATE_NORMAL, VARIATE_SOBOL_NORMAL), sigma)

    def uniform(self, coords, half_width, sequence: str = "philox") -> "Sampling":
        """Independent uniform variation on ``[nominal - half_width, nominal + half_width)``, drawn
        from ``sequence`` (``"philox"`` or ``"sobol"``)."""
        return self._assign(coords, self._kind(sequence, VARIATE_UNIFORM, VARIATE_SOBOL_UNIFORM), half_width)

    def grid(self, coords, half_range, levels: int) -> "Sampling":
        """Full-factorial factors: ``levels`` equally spaced values on ``nominal +- half_range``.
        Instance ``i`` visits grid node ``i mod prod(levels)``; the first grid coordinate named over
        all ``grid`` calls varies fastest."""
        if int(levels) < 2:
            raise ValueError("A grid factor needs at least 2 levels")
        return self._assign(coords, VARIATE_GRID, half_range, levels)

    def tables(self) -> dict:
        return {"variate_kind": np.asarray(self.variate_kind, dtype=np.int32),
                "grid_levels": np.asarray(self.grid_levels, dtype=np.int32),
                "nominal": np.ascontiguousarray(self.nominal), "source": np.ascontiguousarray(self.source),
                "scale": np.ascontiguousarray(self.scale)}


def study_quantities(program, points=None, metrics=None, solver_quantities=()) -> tuple:
    """``(names, units, kinds, indices)`` of the quantities a study reduces, in the column order of
    ``io.results_writer.batch_table``: solver quantities, metric columns, then ``<point>_{x,y,z}``.
    ``points`` / ``metrics``: a list (point keys or names, metric names) or ``"all"``."""
    from .metrics.registry import metric_unit
    names, units, kinds, indices = [], [], [], []
    for sq in solver_quantities:
        if sq not in SOLVER_QUANTITIES:
            raise ValueError(f"Unknown solver quantity {sq!r}; expected one of {SOLVER_QUANTITIES}")
        names.append(sq)
        units.append("")
        kinds.append(QUANTITY_MAX_RESIDUAL if sq == "solver_max_residual" else QUANTITY_NFEV)
        indices.append(0)
    if metrics is not None:
        wanted = program.metric_names if isinstance(metrics, str) and metrics == "all" else list(metrics)
        if wanted and not program.metric_names:
            raise ValueError("This topology was compiled without a metric program")
        for m in wanted:
            if m not in program.metric_names:
                raise ValueError(f"Unknown metric column {m!r}")
            names.append(m)
            units.append(metric_unit(m))
            kinds.append(QUANTITY_METRIC)
            indices.append(program.metric_names.index(m))
    if points is not None:
        by_name = {_point_name(k): k for k in program.out_keys}
        keys = program.out_keys if isinstance(points, str) and points == "all" else list(points)
        for key in keys:
            key = by_name.get(key.lower()) if isinstance(key, str) else key
            if key not in program.out_keys:
                raise ValueError(f"Unknown output point {key!r}")
            slot = program.out_keys.index(key)
            for a in range(3):
                names.append(f"{_point_name(key)}_{AXES[a]}")
                units.append("mm")
                kinds.append(QUANTITY_POSITION)
                indices.append(3 * slot + a)
    if not names:
        raise ValueError("A study needs at least one quantity (points, metrics or solver_quantities)")
    return names, units, np.asarray(kinds, dtype=np.int32), np.asarray(indices, dtype=np.int32)


@dataclass
class StudyResult:
    """Per-step statistics of a study, ``[n_steps, n_quantities]`` unless noted; columns = ``quantities``.

    count / nonfinite: accepted finite values / accepted NaN or inf values (NaN = the reference's
    None, +inf = a derivative tie marker); a value is accepted when its step was (status OK or
    step < failed_step).  std uses ddof = 1 (NaN below 2 values); min / max / argmin / argmax give
    the extremes and the instance id producing each (smallest id on a tie; NaN / -1 when empty).
    histogram ``[n_steps, n_quantities, bins + 2]``: bin 0 counts values below ``hist_lo``, the
    last bin values at or above ``hist_hi``.  status_counts ``[4]`` counts instances per status
    (0 ok, 1 not converged, 2 residual rejected, 3 invalid geometry), failed_at_step ``[n_steps]``
    instances by first failed step."""

    quantities: list
    units: list
    count: np.ndarray
    nonfinite: np.ndarray
    mean: np.ndarray
    std: np.ndarray
    min: np.ndarray
    max: np.ndarray
    argmin: np.ndarray
    argmax: np.ndarray
    histogram: np.ndarray | None
    status_counts: np.ndarray
    failed_at_step: np.ndarray
    hist_lo: np.ndarray | None = None
    hist_hi: np.ndarray | None = None

    @classmethod
    def from_out(cls, names, units, out: dict, hist_lo=None, hist_hi=None) -> "StudyResult":
        count = out["count"]
        with np.errstate(invalid="ignore", divide="ignore"):
            std = np.where(count >= 2, np.sqrt(out["m2"] / np.maximum(count - 1, 1)), np.nan)
        return cls(list(names), list(units), count, out["nonfinite"], out["mean"], std, out["min"], out["max"],
                   out["argmin"], out["argmax"], out["histogram"], out["status_counts"], out["failed_at_step"],
                   hist_lo, hist_hi)

    def quantile(self, p: float) -> np.ndarray:
        """``[n_steps, n_quantities]`` quantile ``p`` from the histograms, linear inside a bin; NaN
        where the rank lands in the under- or overflow bin, or nothing was counted."""
        if self.histogram is None:
            raise ValueError("quantile needs a study run with histograms")
        if not 0.0 <= p <= 1.0:
            raise ValueError("p must lie in [0, 1]")
        h = self.histogram.astype(np.float64)
        nb = h.shape[-1] - 2
        total = h.sum(-1)
        rank = p * total
        cum = np.cumsum(h, -1)
        hit = (cum >= rank[..., None]) & (h > 0)
        b = np.argmax(hit, axis=-1)
        before = np.take_along_axis(cum - h, b[..., None], -1)[..., 0]
        inside = np.take_along_axis(h, b[..., None], -1)[..., 0]
        width = (self.hist_hi - self.hist_lo) / nb
        with np.errstate(invalid="ignore", divide="ignore"):
            value = self.hist_lo + (b - 1 + (rank - before) / inside) * width
        return np.where((total > 0) & (b >= 1) & (b <= nb), value, np.nan)


def study_request(solver, sampling: Sampling, seed: int, points, metrics, solver_quantities, histograms,
                  bins: int) -> tuple:
    """``(names, units, arrays, desc)`` of a study request; ``arrays`` keeps the buffers ``desc``
    points at alive."""
    from .. import _lib
    if sampling.program is not solver.program:
        raise ValueError("The sampling was built for another solver")
    names, units, kinds, indices = study_quantities(solver.program, points, metrics, solver_quantities)
    arrays = dict(sampling.tables(), quantity_kind=kinds, quantity_index=indices, hist_lo=None, hist_hi=None)
    n_bins = 0
    if histograms is not None:
        missing = [n for n in names if n not in histograms]
        if missing:
            raise ValueError(f"histograms needs a (lo, hi) range for every quantity; missing {missing}")
        arrays["hist_lo"] = np.array([float(histograms[n][0]) for n in names])
        arrays["hist_hi"] = np.array([float(histograms[n][1]) for n in names])
        n_bins = int(bins)
    return names, units, arrays, _lib.StudyDesc.of(arrays, seed=seed, n_bins=n_bins)


def run_study(solver, sampling: Sampling, n_instances: int, seed: int = 0, points=None, metrics=None,
              solver_quantities=(), histograms=None, bins: int = 64, solver_config=None, devices=None) -> StudyResult:
    from .. import _lib
    names, units, arrays, desc = study_request(solver, sampling, seed, points, metrics, solver_quantities,
                                               histograms, bins)
    cfg = _lib.default_cfg(residual_tol=float(solver_config.residual_tolerance)) if solver_config else None
    out = solver.topology.study(solver.values, int(n_instances), desc, cfg, devices=devices)
    return StudyResult.from_out(names, units, out, arrays["hist_lo"], arrays["hist_hi"])


def study_inputs(solver, sampling: Sampling, seed: int, ids, device: int = 0) -> tuple:
    names, units, arrays, desc = study_request(solver, sampling, seed, None, None, SOLVER_QUANTITIES, None, 0)
    return solver.topology.study_sample(desc, ids, device)
