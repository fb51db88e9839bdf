/* C ABI of the B200-native batched suspension-kinematics solver.
 *
 * The reference (nickmccleery/open-kinematics, pure Python) has no FFI; its solve-path
 * seams are the Python functions listed below (paths relative to src/kinematics/core/).
 * This header is what a ctypes/cffi binding of those seams binds instead:
 *
 *   okin_topology_create   <- ResidualComputer.__init__ / build_jac_plan (solver.py:187-214,
 *                             :281-500) + DerivedPointsManager.__init__ (points/derived/
 *                             manager.py:95-105): everything computed once per topology.
 *   okin_solve_batch       <- Suspension.initial_state() incl. the camber-shim pre-solve
 *                             (corner/double_wishbone.py:233-257, :501-571, config/shims.py:284-501),
 *                             solve_suspension_sweep (solver.py:654-776), once per instance,
 *                             plus compute_state_tangents (sensitivity.py:57-143) when
 *                             tangents_out is given and Suspension.compute_state_metrics
 *                             (suspensions/base.py:198-204 -> metrics/main.py:63, :145) when
 *                             metrics_out is given.
 *   okin_solve_batch_device   same, on buffers already resident in device memory.
 *
 * Conventions: plain pointers and sizes, caller owns every buffer, every function returns 0 on
 * success and a negative code on error (message via okin_last_error), no exceptions cross the
 * boundary.  A topology handle may be used from several threads as long as each thread uses a
 * different device.  All floating point is IEEE fp64.
 *
 * Buffer layouts ("instance-major": one instance's data is contiguous, so a warp that owns an
 * instance reads and writes coalesced rows and an instance range is one contiguous slab).  This is a
 * deliberate departure from the structure-of-arrays wording of the north star: instance-fastest SoA
 * coalesces for a thread-per-instance kernel; with one warp per instance it would turn every row
 * access into 32 scattered 8-byte accesses (measured DRAM traffic with this layout: 1.06x the
 * algorithmic bytes):
 *   hardpoints      [n_instances][n_in_points*3]     authored positions, slot order = the
 *                                                    compiled topology's input points
 *   params          [n_instances][n_params]          per-instance scalar parameters (camber-shim face
 *                                                    datums, normal and thicknesses per shimmed
 *                                                    corner); NULL = the topology's defaults
 *   target_values   [n_targets][n_steps]             sweep values shared by all instances
 *                                                    (relative displacement or absolute coordinate,
 *                                                    as declared per target)
 *   positions_out   [n_instances][n_steps][n_out_points*3]   NaN after a failed step
 *   iters_out       [n_instances][n_steps]           residual evaluations (SolverInfo.nfev)
 *   max_residual_out[n_instances][n_steps]           max |r| at the solution (SolverInfo.max_residual)
 *   tangents_out    [n_instances][n_steps][n_targets][n_unknowns]  dq/dt_j, reference column order
 *   velocities_out  [n_instances][n_steps][n_targets][n_out_points*3]  TangentField.velocities: first-order
 *                                                    response of every output point (free, fixed = 0,
 *                                                    derived) to each target (sensitivity.py:115-141)
 *   tangent_health_out [n_instances][n_steps][2]     TangentSolveInfo (sensitivity.py:42-55):
 *                                                    {smallest singular value, condition number} of the
 *                                                    pinned Jacobian, by power / inverse iteration with
 *                                                    the Cholesky factor (estimates from inside)
 *   metrics_out     [n_instances][n_steps][n_metrics]  state / mechanism / derivative metric columns in
 *                                                    the reference's flat export order; NaN where the
 *                                                    reference yields None, +inf in a derivative column whose
 *                                                    driver tangents tie (the reference raises there,
 *                                                    metrics/derivatives.py:299-304)
 *   design_out      [n_instances][n_out_points*3]    design (setup) pose after the camber-shim
 *                                                    pre-solve and derived points
 *   diagnostics_out [n_instances][n_steps][n_diagnostics]  sweep diagnostics as per-state reductions
 *                                                    (diagnostics.py:136-226, axle/mechanisms.py:432-549):
 *                                                    column 0 = OKIN_DIAG_* flag bits, 1 = number of free
 *                                                    points that jumped into the step, 2 = largest such
 *                                                    displacement, 3 = its output slot, 4 = its threshold,
 *                                                    then the topology columns (U-bar branch volume and
 *                                                    chirality margin, transmission margins; NaN = None)
 *   jumps_out       [n_instances][n_steps][n_unknowns/3]  row 0: continuity threshold of each free point
 *                                                    (reference column order); row s>0: displacement into
 *                                                    step s where it exceeded the threshold, else 0
 *   instance_targets [n_instances][n_targets][n_steps] per-instance sweep tables (Monte Carlo over the sweep
 *                                                    itself; SURVEY.md section 8b); when given it replaces the
 *                                                    shared target_values
 *   hardpoint_sensitivity [n_instances][n_steps][n_sens][n_out_points*3]  d position / d hardpoint
 *                                                    coordinate: row k is the coordinate the topology lists
 *                                                    k-th among its sensitivity inputs (3 * input slot + axis),
 *                                                    params held fixed.  Free points: the Gauss-Newton
 *                                                    sensitivity -A^-1 J^T dR/dp_k with the factor the tangents
 *                                                    use; fixed points: e_k; derived points: through their op.
 *                                                    NaN after a failed step.  Not available on a topology
 *                                                    with camber-shim records (OKIN_ERR_USAGE)
 *   status_out      [n_instances]                    OKIN_STATUS_*
 *   failed_step_out [n_instances]                    -1 or the first failed step
 *   worst_row_out   [n_instances]                    device row owning max|r| at the failed step, -1 when the
 *                                                    sweep did not fail; the host maps it to the reference's
 *                                                    "Worst residual row" text (describe_worst_residual,
 *                                                    solver.py:640-651) through TopologyProgram.row_source
 * The buffers of one call travel in an okin_batch_io; every output pointer except status /
 * failed_step may be NULL (not wanted).
 */
#ifndef OKIN_H
#define OKIN_H

#ifndef __CUDACC_RTC__
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define OKIN_OK 0
#define OKIN_ERR_USAGE (-1)
#define OKIN_ERR_CUDA (-2)
#define OKIN_ERR_NO_DEVICE (-3)

#define OKIN_STATUS_OK 0
#define OKIN_STATUS_NOT_CONVERGED 1     /* RuntimeError("Solver failed to converge") solver.py:726-730 */
#define OKIN_STATUS_RESIDUAL_REJECTED 2 /* RuntimeError("...did not reach an acceptable residual") solver.py:738-747 */
#define OKIN_STATUS_INVALID_GEOMETRY 3  /* NaN / degenerate design pose */

typedef struct okin_topology okin_topology;

/* Flat program produced by the host topology compiler (open-kinematics_b200/core/topology.py);
 * layout in open-kinematics_b200/csrc/okin_defs.h. */
typedef struct okin_topology_desc {
  const int32_t* hdr;   /* [OKIN_HDR_SIZE] */
  const int32_t* iblob;
  int64_t n_iblob;
  const double* fblob;
  int64_t n_fblob;
} okin_topology_desc;

/* Solver controls.  residual_tol mirrors SolverConfig.residual_tolerance (solver.py:80); the
 * MINPACK ftol/xtol/gtol of the reference have no counterpart: the device solve always runs its
 * Gauss-Newton iteration until a verification step is below step_tol. */
typedef struct okin_solver_cfg {
  double step_tol;       /* mm; the iteration ends when the verification (chord) step, which is also
                            applied, has max|dx| <= step_tol; default 1e-6 (typical size 1e-9) */
  double coarse_tol;     /* mm; an undamped Gauss-Newton step this small triggers the chord step;
                            default 1e-3 */
  double fine_tol;       /* mm; an undamped Gauss-Newton step this small ends the iteration without the
                            chord step (error left ~ curvature x fine_tol^2, i.e. ~1e-10 mm for
                            mm-scale linkages); default 1e-4 */
  double residual_tol;   /* default 1e-3 */
  double mu_init;        /* first Marquardt damping after a rejected step; default 1e-3 */
  int32_t max_iter;      /* factorisations per step; default 50 */
  int32_t use_predictor; /* highest continuation predictor order, 0 = plain warm start; default 4.  Full-output
                            kernels: Adams-Bashforth on the tangents (orders 1..3); lean kernels: backward-
                            difference extrapolation of the solution history (orders 1..4) */
} okin_solver_cfg;

typedef struct okin_topology_info {
  int32_t n_points, n_in_points, n_out_points, n_unknowns, n_targets, n_rows;
  int32_t smem_bytes_per_instance, n_levels, n_metrics, n_params, n_diagnostics;
} okin_topology_info;

/* Buffers of one batch call (layouts in the header comment).  Host pointers for okin_solve_batch,
 * device pointers for okin_solve_batch_device.  Zero-initialise, then set what is wanted. */
typedef struct okin_batch_io {
  const double* hardpoints;     /* required */
  const double* params;         /* optional */
  const double* target_values;  /* required when n_targets * n_steps > 0 */
  int32_t* status;              /* required */
  int32_t* failed_step;         /* required */
  double* positions;
  int32_t* iters;
  double* max_residual;
  double* tangents;
  double* velocities;
  double* tangent_health;
  double* metrics;
  double* design;
  double* diagnostics;
  double* jumps;
  const double* instance_targets; /* optional [n_instances][n_targets][n_steps]; replaces target_values */
  int32_t* worst_row;             /* optional [n_instances] */
  double* hardpoint_sensitivity;  /* optional [n_instances][n_steps][n_sens][n_out_points*3] */
} okin_batch_io;

int okin_device_count(int* out);
int okin_default_cfg(okin_solver_cfg* out);
int okin_topology_create(const okin_topology_desc* desc, okin_topology** out);
int okin_topology_destroy(okin_topology* topo);
int okin_topology_get_info(const okin_topology* topo, okin_topology_info* out);

/* Host buffers; instance range sharded evenly over device_ids (NULL / 0 => device 0), one host
 * thread per device.  Returns after every output has landed in the caller's buffers (also on
 * error: no copy is left in flight). */
int okin_solve_batch(okin_topology* topo, const okin_solver_cfg* cfg, int64_t n_instances, int32_t n_steps,
                     const okin_batch_io* io, const int32_t* device_ids, int32_t n_devices);

/* Device buffers on `device`; enqueues on `stream` (a cudaStream_t, may be NULL) and returns
 * without synchronising. */
int okin_solve_batch_device(okin_topology* topo, const okin_solver_cfg* cfg, int32_t device, void* stream,
                            int64_t n_instances, int32_t n_steps, const okin_batch_io* d_io);

/* Page-locked host memory for the buffers of okin_solve_batch (copies from / to pageable memory are
 * staged by the driver and block; with these the H2D / kernel / D2H pipeline overlaps).  The pages are
 * placed on the NUMA node next to `device` when the box exposes it (device < 0: no preference).
 * Replaces nothing in the reference (its arrays are NumPy allocations, solver.py:187-214). */
int okin_host_alloc(int64_t bytes, int32_t device, void** out);
int okin_host_free(void* ptr);

/* Instance range [begin, begin+count) that shard k of n_shards owns: [k*N/G, (k+1)*N/G).  The
 * same rule splits a host batch over device_ids and a torchrun job over ranks. */
int okin_shard_range(int64_t n_instances, int32_t shard, int32_t n_shards, int64_t* begin, int64_t* count);

/* Launch geometry the library would use for n_instances on `device` (for reporting). */
int okin_launch_geometry(okin_topology* topo, int32_t device, int64_t n_instances, int32_t* grid, int32_t* block,
                         int32_t* smem_bytes, int32_t* ctas_per_sm);

/* Which lean kernel family (positions + solver statistics only) this topology uses on `device`.  The
 * first large batch on a device times the generic 168- and 128-register families and, when the
 * topology has a spec (okin_topology_set_spec) that NVRTC compiles, the same two families specialised
 * to the topology, and keeps the fastest; OKIN_LEAN_REGS = 128 | 168 | spec128 | spec168 pins one. */
typedef struct okin_lean_family {
  int32_t registers;     /* 128 or 168 once chosen on that device, 0 before */
  int32_t specialised;   /* 1: the topology-specialised kernel of that register cap */
  double ms[4];          /* calibration times in ms: generic 168, generic 128, specialised 168, specialised 128
                            (0 when not timed: pinned, not yet run, or the specialised kernels unavailable) */
  double spec_compile_s; /* NVRTC compile time of the specialised kernels (s), 0 when not compiled */
  char spec_error[256];  /* why the specialised kernels are not in use ("" when they compiled and loaded) */
} okin_lean_family;
int okin_lean_calibration(okin_topology* topo, int32_t device, okin_lean_family* out);

/* Source of the topology's generated spec (okin_spec.h, TopologyProgram.spec_source); set before the
 * first lean launch.  Without one only the generic lean kernels run. */
int okin_topology_set_spec(okin_topology* topo, const char* source);

/* Compile the lean kernels of a spec with NVRTC for sm_100a and --ptxas-options=-v, without a device:
 * the log (registers, spills) and the cubin (copied when cubin_capacity suffices). */
int okin_spec_compile(const char* source, int32_t shim, char* log, int32_t log_len, int64_t* cubin_bytes,
                      void* cubin, int64_t cubin_capacity);

/* Dependent-DFMA-chain microbenchmark: measured fp64 FMA peak of `device` in TFLOP/s
 * (the roofline denominator; MEASURED_PEAKS.json carries no fp64 figure). */
int okin_fp64_peak(int32_t device, double* tflops_out);

/* ---- Tolerance studies ---------------------------------------------------------------------
 * okin_study solves n_instances instances whose inputs are generated on the device from
 * (seed, instance id) and reduces every wanted (step, quantity) over the instances on the device;
 * nothing per instance crosses to the host.  Sampling contract (stable: changing it changes every
 * study's draws).  Instance i (global, 0-based) draws n_variates variates z_v:
 *   normal / uniform: one Philox4x32-10 call per variate, key = (lo32(seed), hi32(seed)),
 *     counter = (lo32(i), hi32(i), v, 0) -> words x0..x3; u = ((x1 << 32 | x0) >> 11) * 2^-53,
 *     u' = ((x3 << 32 | x2) >> 11) * 2^-53;
 *     normal: z = sqrt(-2 log(1 - u)) * cospi(2 u');  uniform: z = 2u - 1 in [-1, 1)
 *   grid (full factorial): node = i mod prod(L_g) over the grid variates, the first grid variate
 *     varying fastest; d_g = mixed-radix digit g of node; z = d_g / (L_g - 1) * 2.0 - 1.0
 *   sobol uniform / sobol normal: scrambled Sobol' sequence, 52-bit integers X, bit 51 = the 2^-1
 *     digit.  The Sobol' variates take dimensions d = 0, 1, ... in variate order (counting Sobol'
 *     variates only).  Point index j = i / prod(L_g) over the grid variates (j = i without grid
 *     variates), so every grid node sees the same Sobol' sample (a crossed design).
 *     Unscrambled: direction numbers V[d][0..52) of Joe-Kuo new-joe-kuo-6.21201 (SciPy's table):
 *     poly_d of degree m (bit length - 1), m_k = vinit[d][k] for k < m and, for k >= m,
 *     m_k = m_{k-m} ^ XOR_{l=1..m, bit (m-l) of poly_d set} 2^l m_{k-l};  m_k = 1 for all k when d = 0;
 *     V[d][k] = m_k << (51 - k).  Point j: X = XOR of V[d][k] over the set bits k of j ^ (j >> 1)
 *     (SciPy's order: qmc.Sobol(D, scramble=False, bits=52) gives X * 2^-52).
 *     Scramble (linear matrix scramble + digital shift, per Sobol' variate v, always on): with
 *     W(a) = ((x1 << 32 | x0) >> 12) of Philox4x32-10 under the key above at counter (a, 0, v, 1),
 *     row k < 52 of a lower-triangular GF(2) matrix M_v with unit diagonal is
 *     R_k = (W(k) & ~(2^(51-k) - 1)) | 2^(51-k) (digit k, bit 51 - k, of M x is the parity of
 *     R_k & x), and the shift is S_v = W(52).  Scrambled X = S_v ^ XOR over the same bits k of
 *     M_v V[d][k].  Instance draws use counter word 3 = 0, so the two counter spaces never meet.
 *     sobol uniform: z = X * 2^-51 - 1 (exact, in [-1, 1));
 *     sobol normal: z = PPND16((2X + 1) * 2^-53), Wichura's AS241 inverse normal CDF in fp64.
 *     Limits (usage errors): at most OKIN_SOBOL_MAX_VARIATES Sobol' variates, no saturated grid
 *     period (prod(L_g) >= 2^63), j < 2^52.  Estimates are best at N = 2^m instances (per grid node).
 * Coordinate c (3 * input slot + axis, then the params, n_coords = 3 * n_in_points + n_params) takes
 *   value_c = nominal_c + scale_c * z_{source_c}   (nominal_c when source_c = -1).
 * Reduction: a quantity's value at (instance, step) counts iff the step was accepted (status OK or
 * step < failed_step) and the value is finite; accepted non-finite values (NaN = the reference's None,
 * +inf tie markers) are counted in nonfinite.  Instances are cut into chunks of OKIN_STUDY_CHUNK,
 * dealt round-robin over device_ids; within a chunk the moments are reduced in an order fixed by the
 * instance indices alone and the chunk partials are folded on the host in global chunk order, so a
 * result is bit-identical for any device list and any scheduling.  min / max carry the global id of
 * the instance that produced them (smallest id on a tie).  Histograms: n_bins uniform bins on
 * [hist_lo, hist_hi) plus an underflow (bin 0) and an overflow bin (bin n_bins + 1). */
#define OKIN_STUDY_CHUNK 65536

#define OKIN_VARIATE_NORMAL 0
#define OKIN_VARIATE_UNIFORM 1
#define OKIN_VARIATE_GRID 2
#define OKIN_VARIATE_SOBOL_UNIFORM 3
#define OKIN_VARIATE_SOBOL_NORMAL 4
#define OKIN_SOBOL_MAX_VARIATES 1024
#define OKIN_SOBOL_BITS 52

#define OKIN_QUANTITY_POSITION 0      /* index = 3 * output slot + axis (positions_out column) */
#define OKIN_QUANTITY_METRIC 1        /* index = metric column */
#define OKIN_QUANTITY_MAX_RESIDUAL 2  /* index ignored */
#define OKIN_QUANTITY_NFEV 3          /* index ignored */

typedef struct okin_study_desc {
  uint64_t seed;
  int32_t n_variates;
  const int32_t* variate_kind;    /* [n_variates] OKIN_VARIATE_* */
  const int32_t* grid_levels;     /* [n_variates] L >= 2 for grid variates; ignored for the others */
  int32_t n_coords;               /* 3 * n_in_points + n_params */
  const double* nominal;          /* [n_coords] */
  const int32_t* source;          /* [n_coords] variate index, or -1 = held at nominal */
  const double* scale;            /* [n_coords] */
  int32_t n_quantities;
  const int32_t* quantity_kind;   /* [n_quantities] OKIN_QUANTITY_* */
  const int32_t* quantity_index;  /* [n_quantities] */
  int32_t n_bins;                 /* 0 (no histograms) .. 4096 */
  const double* hist_lo;          /* [n_quantities] when n_bins > 0 */
  const double* hist_hi;          /* [n_quantities] when n_bins > 0, > hist_lo */
} okin_study_desc;

/* Results of okin_study, host buffers, [S][Q] = [n_steps][n_quantities].  m2 = sum of squared
 * deviations from the mean; mean / m2 / min / max are NaN and argmin / argmax -1 where count is 0. */
typedef struct okin_study_out {
  int64_t* count;           /* [S][Q] required */
  int64_t* nonfinite;       /* [S][Q] required */
  double* mean;             /* [S][Q] required */
  double* m2;               /* [S][Q] required */
  double* min;              /* [S][Q] required */
  double* max;              /* [S][Q] required */
  int64_t* argmin;          /* [S][Q] required, global instance id */
  int64_t* argmax;          /* [S][Q] required, global instance id */
  int64_t* histogram;       /* [S][Q][n_bins + 2], required when n_bins > 0 */
  int64_t* status_counts;   /* [4] instances per OKIN_STATUS_*, required */
  int64_t* failed_at_step;  /* [S] instances whose first failed step is s, required */
} okin_study_out;

/* Generate, solve and reduce n_instances instances (positions-only quantities use the lean kernel
 * family, a metric quantity the full one).  Device memory is bounded by the chunk size, host memory
 * by the number of devices; neither grows with n_instances. */
int okin_study(okin_topology* topo, const okin_solver_cfg* cfg, int64_t n_instances, int32_t n_steps,
               const double* target_values, const okin_study_desc* desc, okin_study_out* out,
               const int32_t* device_ids, int32_t n_devices);

/* The inputs okin_study generates for the instances instance_ids[0..n_ids), generated on `device`:
 * hardpoints_out [n_ids][n_in_points*3], params_out [n_ids][n_params] (may be NULL when n_params = 0).
 * The quantity fields of desc are not read. */
int okin_study_sample(okin_topology* topo, const okin_study_desc* desc, int64_t n_ids, const int64_t* instance_ids,
                      double* hardpoints_out, double* params_out, int32_t device);

int okin_last_error(char* buf, int32_t len);

#ifdef __cplusplus
}
#endif
#endif /* OKIN_H */
