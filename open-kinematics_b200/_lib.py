"""ctypes binding of the C ABI in ``include/okin.h`` (library built from ``csrc/``).

There is no fallback: if ``csrc/libokin.so`` is missing or no CUDA device is
visible, every solve entry point raises.
"""

from __future__ import annotations

import ctypes
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# OKIN_LIB points at an alternative build of the same library (kernel experiments); default in-tree.
LIB_PATH = os.environ.get("OKIN_LIB") or os.path.join(CSRC, "libokin.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_f64p = ctypes.POINTER(ctypes.c_double)


class TopologyDesc(ctypes.Structure):
    _fields_ = [("hdr", c_i32p), ("iblob", c_i32p), ("n_iblob", ctypes.c_int64),
                ("fblob", c_f64p), ("n_fblob", ctypes.c_int64)]


class SolverCfg(ctypes.Structure):
    _fields_ = [("step_tol", ctypes.c_double), ("coarse_tol", ctypes.c_double), ("fine_tol", ctypes.c_double),
                ("residual_tol", ctypes.c_double),
                ("mu_init", ctypes.c_double),
                ("max_iter", ctypes.c_int32), ("use_predictor", ctypes.c_int32)]


class BatchIO(ctypes.Structure):
    """``okin_batch_io``: the buffers of one batch call (host or device addresses)."""

    INPUTS = ("hardpoints", "params", "target_values", "instance_targets")
    OUTPUTS = ("status", "failed_step", "positions", "iters", "max_residual", "tangents", "velocities",
               "tangent_health", "metrics", "design", "diagnostics", "jumps", "worst_row", "hardpoint_sensitivity")
    # field order of the C struct (include/okin.h)
    _fields_ = [(n, ctypes.c_void_p) for n in (
        "hardpoints", "params", "target_values", "status", "failed_step", "positions", "iters", "max_residual",
        "tangents", "velocities", "tangent_health", "metrics", "design", "diagnostics", "jumps",
        "instance_targets", "worst_row", "hardpoint_sensitivity")]

    @classmethod
    def of(cls, **buffers) -> "BatchIO":
        """Build from numpy arrays / integer addresses / None, by field name."""
        io = cls()
        for name, buf in buffers.items():
            if name not in cls.INPUTS + cls.OUTPUTS:
                raise KeyError(name)
            if buf is None:
                continue
            setattr(io, name, buf.ctypes.data if isinstance(buf, np.ndarray) else int(buf))
        return io


class TopologyInfo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "n_points", "n_in_points", "n_out_points", "n_unknowns", "n_targets", "n_rows",
        "smem_bytes_per_instance", "n_levels", "n_metrics", "n_params", "n_diagnostics")]


class StudyDesc(ctypes.Structure):
    """``okin_study_desc``: sampling tables and quantity list of a tolerance study (host addresses)."""
    _fields_ = [("seed", ctypes.c_uint64), ("n_variates", ctypes.c_int32), ("variate_kind", ctypes.c_void_p),
                ("grid_levels", ctypes.c_void_p), ("n_coords", ctypes.c_int32), ("nominal", ctypes.c_void_p),
                ("source", ctypes.c_void_p), ("scale", ctypes.c_void_p), ("n_quantities", ctypes.c_int32),
                ("quantity_kind", ctypes.c_void_p), ("quantity_index", ctypes.c_void_p), ("n_bins", ctypes.c_int32),
                ("hist_lo", ctypes.c_void_p), ("hist_hi", ctypes.c_void_p)]

    @classmethod
    def of(cls, arrays: dict, seed: int = 0, n_bins: int = 0) -> "StudyDesc":
        """From the int32 / float64 arrays ``variate_kind``, ``grid_levels``, ``nominal``, ``source``,
        ``scale``, ``quantity_kind``, ``quantity_index``, ``hist_lo``, ``hist_hi`` (kept alive by the
        caller; missing ones are NULL)."""
        d = cls()
        d.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        d.n_bins = int(n_bins)
        for name, arr in arrays.items():
            if arr is not None:
                setattr(d, name, arr.ctypes.data)
        d.n_variates = len(arrays["variate_kind"])
        d.n_coords = len(arrays["nominal"])
        d.n_quantities = len(arrays["quantity_kind"]) if arrays.get("quantity_kind") is not None else 0
        return d


class StudyOut(ctypes.Structure):
    """``okin_study_out``: host result buffers of ``okin_study``."""
    FIELDS = ("count", "nonfinite", "mean", "m2", "min", "max", "argmin", "argmax", "histogram", "status_counts",
              "failed_at_step")
    _fields_ = [(n, ctypes.c_void_p) for n in FIELDS]


# name -> (restype, argtypes); also the list the "exports every declared symbol" test checks.
SIGNATURES = {
    "okin_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "okin_default_cfg": (ctypes.c_int, [ctypes.POINTER(SolverCfg)]),
    "okin_topology_create": (ctypes.c_int, [ctypes.POINTER(TopologyDesc), ctypes.POINTER(ctypes.c_void_p)]),
    "okin_topology_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "okin_topology_get_info": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(TopologyInfo)]),
    "okin_solve_batch": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.POINTER(SolverCfg), ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(BatchIO),
        ctypes.c_void_p, ctypes.c_int32]),
    "okin_solve_batch_device": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.POINTER(SolverCfg), ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32,
        ctypes.POINTER(BatchIO)]),
    "okin_shard_range": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                        ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "okin_launch_geometry": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, c_i32p, c_i32p, c_i32p, c_i32p]),
    "okin_fp64_peak": (ctypes.c_int, [ctypes.c_int32, c_f64p]),
    "okin_lean_calibration": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, c_i32p, c_f64p, c_f64p]),
    "okin_host_alloc": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(ctypes.c_void_p)]),
    "okin_host_free": (ctypes.c_int, [ctypes.c_void_p]),
    "okin_study": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.POINTER(SolverCfg), ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p,
        ctypes.POINTER(StudyDesc), ctypes.POINTER(StudyOut), ctypes.c_void_p, ctypes.c_int32]),
    "okin_study_sample": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.POINTER(StudyDesc), ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_int32]),
    "okin_last_error": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int32]),
}

_lib = None
_lock = threading.Lock()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile ``csrc/okin_abi.cu`` for sm_100a into ``csrc/libokin.so`` (in-tree)."""
    sources = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    sources.append(os.path.join(_HERE, "..", "include", "okin.h"))
    if not force and os.path.exists(LIB_PATH):
        if os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(s) for s in sources):
            return LIB_PATH
    cmd = ["nvcc", *NVCC_FLAGS, "-o", LIB_PATH, os.path.join(CSRC, "okin_abi.cu")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{proc.stdout}\n{proc.stderr}")
    if verbose:
        print(proc.stderr)
    return LIB_PATH


def load() -> ctypes.CDLL:
    """Load the CUDA library; raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: build the CUDA extension first "
                    "(python -c 'import __graft_entry__ as g; g.build()'); there is no CPU fallback."
                )
            lib = ctypes.CDLL(LIB_PATH)
            for name, (restype, argtypes) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = restype
                fn.argtypes = argtypes
            _lib = lib
    return _lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(1024)
    load().okin_last_error(buf, len(buf))
    return buf.value.decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def device_count() -> int:
    n = ctypes.c_int(0)
    rc = load().okin_device_count(ctypes.byref(n))
    return n.value if rc == 0 else 0


def require_device() -> None:
    if device_count() < 1:
        raise RuntimeError("No CUDA device visible: the solver has no CPU fallback (" + last_error() + ")")


def shard_range(n_instances: int, shard: int, n_shards: int) -> tuple:
    begin, count = ctypes.c_int64(), ctypes.c_int64()
    check(load().okin_shard_range(n_instances, shard, n_shards, ctypes.byref(begin), ctypes.byref(count)),
          "okin_shard_range")
    return begin.value, count.value


def pinned_empty(shape, dtype=np.float64, device: int = 0) -> np.ndarray:
    """Uninitialised array in page-locked host memory (``okin_host_alloc``), placed next to
    ``device``.  Buffers like this keep the H2D / kernel / D2H pipeline of ``okin_solve_batch``
    overlapped; allocate once and reuse (``solve_batch(out=...)``), page-locking is slow."""
    import weakref
    shape = tuple(int(d) for d in (shape if isinstance(shape, (tuple, list)) else (shape,)))
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
    if nbytes == 0:
        return np.empty(shape, dtype)
    ptr = ctypes.c_void_p()
    check(load().okin_host_alloc(nbytes, device, ctypes.byref(ptr)), "okin_host_alloc")
    raw = np.ctypeslib.as_array((ctypes.c_char * nbytes).from_address(ptr.value))
    weakref.finalize(raw, load().okin_host_free, ptr.value)   # views keep ``raw`` alive through .base
    return raw.view(dtype).reshape(shape)


def default_cfg(**overrides) -> SolverCfg:
    cfg = SolverCfg()
    check(load().okin_default_cfg(ctypes.byref(cfg)), "okin_default_cfg")
    for key, value in overrides.items():
        if value is not None:
            setattr(cfg, key, value)
    return cfg


class DeviceTopology:
    """Owns an ``okin_topology*`` created from a compiled ``TopologyProgram``."""

    def __init__(self, program):
        self.program = program
        self._hdr = np.ascontiguousarray(program.hdr, dtype=np.int32)
        self._ib = np.ascontiguousarray(program.iblob, dtype=np.int32)
        self._fb = np.ascontiguousarray(program.fblob, dtype=np.float64)
        desc = TopologyDesc(
            self._hdr.ctypes.data_as(c_i32p), self._ib.ctypes.data_as(c_i32p), self._ib.size,
            self._fb.ctypes.data_as(c_f64p), self._fb.size,
        )
        self.handle = ctypes.c_void_p()
        check(load().okin_topology_create(ctypes.byref(desc), ctypes.byref(self.handle)), "okin_topology_create")

    def info(self) -> TopologyInfo:
        out = TopologyInfo()
        check(load().okin_topology_get_info(self.handle, ctypes.byref(out)), "okin_topology_get_info")
        return out

    def launch_geometry(self, n_instances: int, device: int = 0) -> dict:
        vals = [ctypes.c_int32() for _ in range(4)]
        check(load().okin_launch_geometry(self.handle, device, n_instances, *[ctypes.byref(v) for v in vals]),
              "okin_launch_geometry")
        return dict(zip(("grid", "block", "smem_bytes", "ctas_per_sm"), (v.value for v in vals)))

    def lean_calibration(self, device: int = 0) -> dict:
        """Lean kernel family chosen for this topology on ``device`` (see ``okin_lean_calibration``)."""
        regs, wide, narrow = ctypes.c_int32(), ctypes.c_double(), ctypes.c_double()
        check(load().okin_lean_calibration(self.handle, device, ctypes.byref(regs), ctypes.byref(wide),
                                           ctypes.byref(narrow)), "okin_lean_calibration")
        return {"registers": regs.value, "ms_168": wide.value, "ms_128": narrow.value}

    def close(self) -> None:
        if self.handle:
            load().okin_topology_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    # -- tolerance studies ------------------------------------------------------------
    def study(self, target_values: np.ndarray, n_instances: int, desc: StudyDesc, cfg: SolverCfg | None = None,
              devices=None) -> dict:
        """``okin_study``: generate, solve and reduce ``n_instances`` instances on the device(s).
        Returns the ``okin_study_out`` arrays, ``[n_steps, n_quantities]`` each (``histogram``
        ``[n_steps, n_quantities, n_bins + 2]`` or None, ``status_counts`` [4], ``failed_at_step``
        [n_steps])."""
        require_device()
        tv = np.ascontiguousarray(target_values, dtype=np.float64)
        nt = len(self.program.target_points)
        if tv.ndim != 2 or tv.shape[0] != nt:
            raise ValueError(f"target_values must have shape ({nt}, n_steps), got {tv.shape}")
        S, Q, nb = tv.shape[1], desc.n_quantities, desc.n_bins
        out = {name: np.zeros((S, Q), np.int64 if name in ("count", "nonfinite", "argmin", "argmax") else np.float64)
               for name in StudyOut.FIELDS[:8]}
        out["histogram"] = np.zeros((S, Q, nb + 2), np.int64) if nb > 0 else None
        out["status_counts"] = np.zeros(4, np.int64)
        out["failed_at_step"] = np.zeros(S, np.int64)
        o = StudyOut(**{k: (v.ctypes.data if v is not None else None) for k, v in out.items()})
        dev = np.ascontiguousarray(devices if devices is not None else [0], dtype=np.int32)
        check(load().okin_study(self.handle, ctypes.byref(cfg or default_cfg()), int(n_instances), S, tv.ctypes.data,
                                ctypes.byref(desc), ctypes.byref(o), dev.ctypes.data, dev.size), "okin_study")
        return out

    def study_sample(self, desc: StudyDesc, ids, device: int = 0) -> tuple:
        """``okin_study_sample``: the generated ``(hardpoints [n, n_in*3], params [n, n_params])`` of
        the instances ``ids``."""
        require_device()
        ids = np.ascontiguousarray(ids, dtype=np.int64).reshape(-1)
        hp = np.zeros((ids.size, 3 * self.program.n_in))
        par = np.zeros((ids.size, len(self.program.param_names)))
        check(load().okin_study_sample(self.handle, ctypes.byref(desc), ids.size, ids.ctypes.data, hp.ctypes.data,
                                       par.ctypes.data if par.size else None, device), "okin_study_sample")
        return hp, par

    # -- host buffers ------------------------------------------------------------------
    def solve_batch(self, hardpoints: np.ndarray, target_values: np.ndarray, cfg: SolverCfg | None = None,
                    devices=None, want_positions=True, want_tangents=False, want_metrics=False,
                    want_design=False, params: np.ndarray | None = None, want_velocities=False,
                    want_health=False, want_diagnostics=False, instance_targets: np.ndarray | None = None,
                    want_worst_row=False, out: dict | None = None, pinned: bool = False,
                    want_hardpoint_sensitivity=False) -> dict:
        """hardpoints [n_inst, n_in*3]; target_values [n_targets, n_steps];
        instance_targets optional [n_inst, n_targets, n_steps] (replaces target_values).
        ``out``: a dict returned by an earlier call; arrays of matching shape are overwritten instead
        of allocated (the way to reuse page-locked buffers).  ``pinned``: allocate what is missing in
        page-locked memory next to the first device.  ``want_hardpoint_sensitivity``: d position /
        d hardpoint coordinate ``[n_inst, n_steps, n_sens, n_out, 3]``, rows in the order of
        ``program.sensitivity_inputs`` (not on a topology with camber-shim records)."""
        require_device()
        prog = self.program
        hp = np.ascontiguousarray(hardpoints, dtype=np.float64)
        if hp.ndim != 2 or hp.shape[1] != 3 * prog.n_in:
            raise ValueError(f"hardpoints must have shape (n_instances, {3 * prog.n_in}), got {hp.shape}")
        tv = np.ascontiguousarray(target_values, dtype=np.float64)
        nt = len(prog.target_points)
        if tv.ndim != 2 or tv.shape[0] != nt:
            raise ValueError(f"target_values must have shape ({nt}, n_steps), got {tv.shape}")
        n_inst, n_steps = hp.shape[0], tv.shape[1]
        par = None
        if params is not None:
            par = np.ascontiguousarray(params, dtype=np.float64)
            if par.shape != (n_inst, len(prog.param_names)):
                raise ValueError(f"params must have shape ({n_inst}, {len(prog.param_names)}), got {par.shape}")
            if par.shape[1] == 0:
                par = None
        itv = None
        if instance_targets is not None:
            itv = np.ascontiguousarray(instance_targets, dtype=np.float64)
            if itv.shape != (n_inst, nt, n_steps):
                raise ValueError(f"instance_targets must have shape ({n_inst}, {nt}, {n_steps}), got {itv.shape}")
        cfg = cfg or default_cfg()
        dev = np.ascontiguousarray(devices if devices is not None else [0], dtype=np.int32)
        prev = out or {}

        def buf(name, want, shape, dtype=np.float64):
            if not want:
                return None
            old = prev.get(name)
            if isinstance(old, np.ndarray) and old.shape == tuple(shape) and old.dtype == np.dtype(dtype) \
                    and old.flags.c_contiguous and old.flags.writeable:
                return old
            return pinned_empty(shape, dtype, int(dev[0])) if pinned else np.empty(shape, dtype)

        out = {
            "positions": buf("positions", want_positions, (n_inst, n_steps, prog.n_out, 3)),
            "status": buf("status", True, (n_inst,), np.int32),
            "failed_step": buf("failed_step", True, (n_inst,), np.int32),
            "iters": buf("iters", True, (n_inst, n_steps), np.int32),
            "max_residual": buf("max_residual", True, (n_inst, n_steps)),
            "tangents": buf("tangents", want_tangents, (n_inst, n_steps, nt, prog.n_unknowns)),
            "velocities": buf("velocities", want_velocities, (n_inst, n_steps, nt, prog.n_out, 3)),
            "tangent_health": buf("tangent_health", want_health, (n_inst, n_steps, 2)),
            "metrics": buf("metrics", want_metrics, (n_inst, n_steps, len(prog.metric_names))),
            "design": buf("design", want_design, (n_inst, prog.n_out, 3)),
            "diagnostics": buf("diagnostics", want_diagnostics, (n_inst, n_steps, len(prog.diagnostic_names))),
            "jumps": buf("jumps", want_diagnostics, (n_inst, n_steps, prog.n_unknowns // 3)),
            "worst_row": buf("worst_row", want_worst_row, (n_inst,), np.int32),
            "hardpoint_sensitivity": buf("hardpoint_sensitivity", want_hardpoint_sensitivity,
                                         (n_inst, n_steps, len(prog.sensitivity_inputs), prog.n_out, 3)),
        }
        if want_diagnostics and not prog.diagnostic_names:
            raise ValueError("This topology was compiled without a diagnostic program")
        if want_metrics and not prog.metric_names:
            raise ValueError("This topology was compiled without a metric program")
        io = BatchIO.of(hardpoints=hp, params=par, target_values=tv, instance_targets=itv, **out)
        check(load().okin_solve_batch(self.handle, ctypes.byref(cfg), n_inst, n_steps, ctypes.byref(io),
                                      dev.ctypes.data, dev.size), "okin_solve_batch")
        return out
