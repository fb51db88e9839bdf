// Per-instance solve core: design-constant setup, residual/Jacobian rows, normal-equation
// assembly, 3x3-block sparse Cholesky, Gauss-Newton / Levenberg-Marquardt continuation over a
// sweep, tangent solves.  One *warp* owns one suspension instance; all per-instance state
// lives in that warp's slice of shared memory and the code is a sequence of *phases*:
//
//     OKIN_PHASE_BEGIN  ... body executed by every lane, `lane` in scope ...  OKIN_PHASE_END
//
// A phase ends with __syncwarp(); lanes only communicate through shared memory across phase
// boundaries, and everything outside a phase is warp-uniform.  Under OKIN_LANE_EMU (plain
// g++, used by tests/ only, never by the product library) a phase is a loop over 32 lanes,
// which lets the CPU-only CI run this exact source against the oracle.
//
// What replaces what in the reference (paths relative to src/kinematics/core/):
//   okin_setup        <- Suspension.constraints() design constants (suspensions/corner/*.py,
//                        axle/*.py), convert_targets_to_absolute (solver.py:584-627)
//   okin_eval_rows    <- ResidualComputer.compute / compute_jacobian (solver.py:226-275, :502-581)
//   okin_derived_*    <- DerivedPointsManager.update_in_place / compute_point_jacobian
//                        (points/derived/manager.py:186-197, :271-324), hand-written JVPs
//   okin_solve_step   <- least_squares(method="lm") call (solver.py:124-169, :717-724)
//   okin_sweep        <- solve_suspension_sweep loop (solver.py:716-774); okin_extrapolate is the
//                        predicted start, okin_worst_row <- describe_worst_residual (solver.py:640-651)
//   tangent columns   <- compute_state_tangents (sensitivity.py:57-143): right-hand sides carried through
//                        the Cholesky factorisation of the system linearised at the solution
//                        (okin_tangent_rhs, okin_factor, okin_solve), okin_point_vel for derived points,
//                        okin_tangent_health for rank / sigma_min / cond
//   okin_shim_presolve <- solve_camber_shim_assembly + application (suspensions/config/shims.py:284-501,
//                        corner/double_wishbone.py:501-571)
//   okin_metrics      <- Suspension.compute_state_metrics (metrics/*.py; kernels in okin_metrics.cuh)
//   okin_diagnostics, okin_continuity <- diagnose_sweep (diagnostics.py:118-226) and the U-bar checks
//                        (axle/mechanisms.py:432-549)
#pragma once

#ifndef OKIN_INLINE_HOT
#define OKIN_INLINE_HOT 1
#endif
// Code footprint matters (profiles/README.md, round 2 step f): the interpreter does not fit the
// instruction caches once the warps of a CTA are in different phases.  OKIN_COMPACT_LOOPS 1: lane-strided
// loops (one to three rounds) are not unrolled; 2: nor are the short runtime-count loops of the row
// evaluation.  Measured and rejected: warp reductions and sqrt / rsqrt / atan2 as calls of one shared
// copy each (the calls spill around themselves, and local-memory traffic uses the pipe the kernel is
// bound by).
#ifndef OKIN_COMPACT_LOOPS
#define OKIN_COMPACT_LOOPS 2
#endif
#include <stddef.h>

#include "../../include/okin.h"
#include "okin_defs.h"
#include "okin_gen_constraints.cuh"
#include "okin_metrics.cuh"

// Phase functions are kept out of line on the device: inlining all of them into the sweep loop
// (each is called from several places) costs registers (255/thread) and instruction cache.  The
// three gather-loop phases (assembly, factorisation, triangular solves) are the exception
// (OKIN_FN_HOT): inlined they are scheduled with the caller's registers, +7 % on the flagship and
// +15 % on the corner topologies (profiles/README.md, round 2).
#if defined(__CUDACC__) && !defined(OKIN_LANE_EMU)
#define OKIN_FN __host__ __device__ __noinline__
#if OKIN_INLINE_HOT
#define OKIN_FN_HOT __host__ __device__ __forceinline__
#else
#define OKIN_FN_HOT OKIN_FN
#endif
#else
#define OKIN_FN inline
#define OKIN_FN_HOT inline
#endif

#if defined(__CUDA_ARCH__) && !defined(OKIN_LANE_EMU)
#define OKIN_PHASE_BEGIN { const int lane = (int)(threadIdx.x & 31u);
#define OKIN_PHASE_END } __syncwarp();
#define OKIN_LDG(p) (*(p))   // int32 tables live in shared memory, double constants in global

#else
#define OKIN_PHASE_BEGIN for (int lane = 0; lane < 32; ++lane) {
#define OKIN_PHASE_END }
#define OKIN_LDG(p) (*(p))
#endif

// Address-space hint.  The per-instance state, the header and the hot tables live in the CTA's dynamic
// shared memory, but they reach the (out-of-line) phase functions as generic pointers, for which the
// compiler emits generic loads and 64-bit address arithmetic.  OKIN_SHARED re-derives a pointer from
// the shared array symbol, which lets it prove the address space (LDS/STS, 32-bit addressing).  Only
// for pointers that are in shared memory in the sweep kernel; identity in the lane emulation.
#if defined(__CUDACC__) && !defined(OKIN_LANE_EMU)
extern __shared__ double okin_smem[];
#endif
#if defined(__CUDA_ARCH__) && !defined(OKIN_LANE_EMU)
#define OKIN_SHARED(p)                                                                  \
  (reinterpret_cast<decltype(p)>(reinterpret_cast<char*>(okin_smem) +                   \
                                 (reinterpret_cast<const char*>(p) - reinterpret_cast<const char*>(okin_smem))))
#else
#define OKIN_SHARED(p) (p)
#endif

// Unroll factor of the gather loops over a task's contributions (factor update, triangular solves,
// assembly).  Not unrolled by default: the trip counts are 1-8 and data dependent, and the smaller
// code measured 5 % faster than the compiler's own 4x unrolling (profiles/r01_g_*).
#ifndef OKIN_INNER_UNROLL
#define OKIN_INNER_UNROLL 1
#endif
// Lane-strided loops run one to three rounds; left to itself the compiler unrolls them four times.
#if defined(__CUDA_ARCH__) && OKIN_COMPACT_LOOPS
#define OKIN_LANE_LOOP _Pragma("unroll 1")
#else
#define OKIN_LANE_LOOP
#endif
#if defined(__CUDA_ARCH__) && OKIN_COMPACT_LOOPS >= 2
#define OKIN_SHORT_LOOP _Pragma("unroll 1")
#else
#define OKIN_SHORT_LOOP
#endif
#define OKIN_STR2(x) #x
#define OKIN_STR(x) OKIN_STR2(x)
#if defined(__CUDA_ARCH__)
#define OKIN_UNROLL_INNER _Pragma(OKIN_STR(unroll OKIN_INNER_UNROLL))
#else
#define OKIN_UNROLL_INNER
#endif

// Warp reductions over the per-lane partials a phase left in red[0..32): shuffles on the device
// (every lane ends with the result), a plain loop in the lane emulation.  NaN propagates in max.
#if defined(__CUDA_ARCH__) && !defined(OKIN_LANE_EMU)
OKIN_HD double okin_red_sum(const double* red) {
  double v = red[threadIdx.x & 31u];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
OKIN_HD double okin_red_max(const double* red) {
  double v = red[threadIdx.x & 31u];
  for (int o = 16; o > 0; o >>= 1) {
    const double w = __shfl_xor_sync(0xffffffffu, v, o);
    v = (w > v || w != w) ? w : v;
  }
  return v;
}
#else
OKIN_HD double okin_red_sum(const double* red) {
  double v = 0.0;
  for (int k = 0; k < 32; ++k) v += red[k];
  return v;
}
OKIN_HD double okin_red_max(const double* red) {
  double v = red[0];
  for (int k = 1; k < 32; ++k) v = (red[k] > v || red[k] != red[k]) ? red[k] : v;
  return v;
}
#endif

// Gather loops (factor update, triangular solves, assembly): every operand of a contribution is
// loaded into its own variable before the first FMA.  A warp issues in order, so the shared-memory
// latency is then paid once per contribution (twelve loads in flight) instead of once per FMA -- but
// only if the register allocator is not squeezed: under the 128-register cap of a 16-warp CTA ptxas
// sinks every load back to its use (LDS -> DFMA pairs through one register), which is why the lean
// kernel runs 12 warps per SM at 168 registers (profiles/r02_*; okin_abi.cu OKIN_LEAN_MAX_THREADS).
struct OkinProgram {
  const int32_t* hdr;  // [OKIN_HDR_SIZE]
  const int32_t* ib;   // int32 blob: at least its hot prefix hdr[OKIN_H_NHOT] (shared memory in the kernel)
  const double* fb;    // double blob
  const int32_t* ibc;  // whole int32 blob (global memory); cold sections are read from here
  const int32_t* const* sec;  // [OKIN_S_COUNT] start of every int32 section (hot: in ib, cold: in ibc),
                              // resolved once per CTA by okin_resolve_sections
};

struct OkinSolverCfg {
  double step_tol;      // converged when the verification (chord) step has max|dx| <= step_tol (mm)
  double coarse_tol;    // a Gauss-Newton step with max|dx| <= coarse_tol is followed by the chord step
  double fine_tol;      // a Gauss-Newton step with max|dx| <= fine_tol ends the iteration unverified
                        // (the error left is second order in it)
  double residual_tol;  // accept a state when max|r| <= residual_tol   (reference constants.py:20)
  double mu_init;       // first Marquardt damping factor after a rejected Gauss-Newton step
  int32_t max_iter;     // factorisations per step before "not converged"
  int32_t use_predictor;  // continuation predictor order: 0 warm start only, 1..3 (Adams-Bashforth on the tangents)
};

OKIN_HD const int32_t* okin_sec(const OkinProgram& pr, int s) { return OKIN_SHARED(pr.sec)[s]; }
// Fills table[s] for section s: the hot prefix of the blob lives at ib, the rest at ibc.
OKIN_HD void okin_resolve_section(const int32_t* hdr, const int32_t* ib, const int32_t* ibc, int s,
                                  const int32_t** table) {
  const int off = hdr[OKIN_H_SEC0 + 2 * s];
  table[s] = (off < hdr[OKIN_H_NHOT] ? ib : ibc) + off;
}
OKIN_HD int okin_sec_len(const OkinProgram& pr, int s) { return pr.hdr[OKIN_H_SEC0 + 2 * s + 1]; }
OKIN_HD const double* okin_fsec(const OkinProgram& pr, int s) { return pr.fb + pr.hdr[OKIN_H_FSEC0 + 2 * s]; }

// Warp-uniform scalars kept in registers (identical in every lane).
struct OkinState {
  double f2;    // ||r||^2 over least-squares rows at the current point
  double rmax;  // max|r| over all rows at the current point
  double mu;    // current damping (0 = pure Gauss-Newton)
  int notpd;    // factorisation hit a non-positive pivot
};

// ---------------------------------------------------------------------------------------
// Derived points: value and forward-mode tangent of one op.
// ---------------------------------------------------------------------------------------
OKIN_HD void okin_unit_jvp(const double v[3], const double dv[3], double u[3], double du[3], double* inv_len) {
  const double il = OKIN_RSQRT(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  u[0] = v[0] * il; u[1] = v[1] * il; u[2] = v[2] * il;
  const double ud = u[0] * dv[0] + u[1] * dv[1] + u[2] * dv[2];
  du[0] = (dv[0] - u[0] * ud) * il; du[1] = (dv[1] - u[1] * ud) * il; du[2] = (dv[2] - u[2] * ud) * il;
  *inv_len = il;
}

// out = f(a, b, c; par); dout = J_a da + J_b db + J_c dc.  (definitions.py:24-180)
OKIN_HD void okin_dop_eval(int op, double par, const double* a, const double* b, const double* c,
                           const double* da, const double* db, const double* dc, double out[3], double dout[3]) {
  if (op == OKIN_DOP_MIDPOINT) {
    for (int k = 0; k < 3; ++k) { out[k] = a[k] + (b[k] - a[k]) * 0.5; dout[k] = da[k] + (db[k] - da[k]) * 0.5; }
  } else if (op == OKIN_DOP_ALONG_LINE) {
    double v[3], dv[3], u[3], du[3], il;
    for (int k = 0; k < 3; ++k) { v[k] = b[k] - a[k]; dv[k] = db[k] - da[k]; }
    okin_unit_jvp(v, dv, u, du, &il);
    for (int k = 0; k < 3; ++k) { out[k] = a[k] + u[k] * par; dout[k] = da[k] + du[k] * par; }
  } else {  // OKIN_DOP_CONTACT_PATCH: a = wheel centre, b = axle inboard, c = axle outboard
    double v[3], dv[3], u[3], du[3], il;
    for (int k = 0; k < 3; ++k) { v[k] = c[k] - b[k]; dv[k] = dc[k] - db[k]; }
    okin_unit_jvp(v, dv, u, du, &il);
    // down = (0,0,-1); w = down - (down.u) u
    const double s = -u[2], ds = -du[2];
    double w[3], dw[3], q[3], dq[3];
    for (int k = 0; k < 3; ++k) { w[k] = -s * u[k]; dw[k] = -(ds * u[k] + s * du[k]); }
    w[2] -= 1.0;
    okin_unit_jvp(w, dw, q, dq, &il);
    for (int k = 0; k < 3; ++k) { out[k] = a[k] + q[k] * par; dout[k] = da[k] + dq[k] * par; }
  }
}

// Evaluate derived points into pos[], one dependency level per phase, one lane per op.
// active_only: only the ops referenced by solve rows (wheel centre, strut clamp).
template <typename Dummy = void>
OKIN_FN void okin_derived_update(const OkinProgram& pr, double* sm, bool active_only) {
  sm = OKIN_SHARED(sm);
  const int32_t* dop = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP));
  const int32_t* lev = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP_LEV));
  const int nlev = okin_sec_len(pr, OKIN_S_DOP_LEV) - 1;
  double* pos = sm + pr.hdr[OKIN_H_OFF_POS];
  const double* par = sm + pr.hdr[OKIN_H_OFF_PAR];
  for (int lv = 0; lv < nlev; ++lv) {
    const int b = OKIN_LDG(lev + lv), e = OKIN_LDG(lev + lv + 1);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int d = b + lane; d < e; d += 32) {
      const int32_t* rec = dop + d * OKIN_DOP_STRIDE;
      if (active_only && !OKIN_LDG(rec + 7)) continue;
      const double z[3] = {0.0, 0.0, 0.0};
      const int ia = OKIN_LDG(rec + 2), ib = OKIN_LDG(rec + 3), ic = OKIN_LDG(rec + 4);
      double out[3], dout[3];
      okin_dop_eval(OKIN_LDG(rec + 0), par[OKIN_LDG(rec + 5)], pos + 3 * ia, pos + 3 * (ib < 0 ? ia : ib),
                    pos + 3 * (ic < 0 ? ia : ic), z, z, z, out, dout);
      const int o = OKIN_LDG(rec + 1);
      pos[3 * o] = out[0]; pos[3 * o + 1] = out[1]; pos[3 * o + 2] = out[2];
    }
    OKIN_PHASE_END
  }
}

// Jacobian blocks d(derived)/d(free base point) by seeding one coordinate per task and
// pushing it through the op chain (manager.py:271-324 does the same with dual numbers).
template <typename Dummy = void>
OKIN_FN void okin_derived_jacobians(const OkinProgram& pr, double* sm) {
  sm = OKIN_SHARED(sm);
  const int nad = pr.hdr[OKIN_H_NAD];
  if (nad == 0) return;
  const int32_t* adj = OKIN_SHARED(okin_sec(pr, OKIN_S_ADJ));
  const int32_t* chain = OKIN_SHARED(okin_sec(pr, OKIN_S_ADJ_CHAIN));
  const int32_t* dop = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP));
  const double* pos = sm + pr.hdr[OKIN_H_OFF_POS];
  const double* par = sm + pr.hdr[OKIN_H_OFF_PAR];
  double* dblk = sm + pr.hdr[OKIN_H_OFF_DBLK];
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < nad; t += 32) {
    const int32_t* rec = adj + t * OKIN_ADJ_STRIDE;
    const int base = OKIN_LDG(rec + 1), comp = OKIN_LDG(rec + 2), off = OKIN_LDG(rec + 3);
    const int cb = OKIN_LDG(rec + 4), ce = OKIN_LDG(rec + 5);
    int tp[OKIN_MAX_CHAIN];
    double tv[OKIN_MAX_CHAIN][3];
    int nt = 0;
    double seed[3] = {0.0, 0.0, 0.0};
    seed[comp] = 1.0;
    const double z[3] = {0.0, 0.0, 0.0};
    double dout[3] = {0.0, 0.0, 0.0};
    OKIN_SHORT_LOOP
    for (int q = cb; q < ce; ++q) {
      const int32_t* op = dop + OKIN_LDG(chain + q) * OKIN_DOP_STRIDE;
      const int in[3] = {OKIN_LDG(op + 2), OKIN_LDG(op + 3), OKIN_LDG(op + 4)};
      const double* dv[3];
      for (int s = 0; s < 3; ++s) {
        dv[s] = z;
        if (in[s] == base) dv[s] = seed;
        for (int k = 0; k < nt; ++k)
          if (tp[k] == in[s]) dv[s] = tv[k];
      }
      double out[3];
      const int ia = in[0], ib = in[1] < 0 ? in[0] : in[1], ic = in[2] < 0 ? in[0] : in[2];
      okin_dop_eval(OKIN_LDG(op + 0), par[OKIN_LDG(op + 5)], pos + 3 * ia, pos + 3 * ib, pos + 3 * ic,
                    dv[0], dv[1], dv[2], out, dout);
      tp[nt] = OKIN_LDG(op + 1);
      tv[nt][0] = dout[0]; tv[nt][1] = dout[1]; tv[nt][2] = dout[2];
      ++nt;
    }
    dblk[off + 0 + comp] = dout[0];
    dblk[off + 3 + comp] = dout[1];
    dblk[off + 6 + comp] = dout[2];
  }
  OKIN_PHASE_END
}

// ---------------------------------------------------------------------------------------
// Camber-shim assembly pre-solve: moves the design pose to the setup pose before anything else is
// derived from it (double_wishbone.py:501-571, config/shims.py:284-501).  One lane per shimmed
// corner: Gauss-Newton on 7(+1) unknowns / 10(+1) residuals from x = 0 with a forward-mode
// Jacobian (the reference uses SciPy's finite differences; both converge to the same root of the
// consistent system, 1e-13 apart in the reference's own default-vs-tight runs).
// ---------------------------------------------------------------------------------------
template <typename Dummy = void>
OKIN_FN void okin_shim_presolve(const OkinProgram& pr, double* sm, const double* params, int* invalid) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nshim = hdr[OKIN_H_NSHIM];
  if (nshim == 0) return;
  const int32_t* recs = okin_sec(pr, OKIN_S_SHIM);
  const int32_t* lists = okin_sec(pr, OKIN_S_SHIM_PTS);
  double* pos = sm + hdr[OKIN_H_OFF_POS];
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  red[lane] = 0.0;
  if (lane < nshim) {
    const int32_t* rec = recs + lane * OKIN_SHIM_STRIDE;
    const double* q = params + OKIN_LDG(rec + 11);
    const double t_design = q[9], t_setup = q[10];
    if (fabs(t_setup - t_design) >= OKIN_GEOM_EPS) {
      double* ubj = pos + 3 * OKIN_LDG(rec + 0);
      const double* lbj = pos + 3 * OKIN_LDG(rec + 1);
      const double* uwf = pos + 3 * OKIN_LDG(rec + 2);
      const double* uwr = pos + 3 * OKIN_LDG(rec + 3);
      const double* hli = pos + 3 * OKIN_LDG(rec + 4);
      const double* hlo = pos + 3 * OKIN_LDG(rec + 5);
      OkinShimCtx c;
      c.t_setup = t_setup;
      const double half = 0.5 * t_design;
      double wl = 0.0, hl = 0.0;
      for (int k = 0; k < 3; ++k) {
        c.n[k] = q[6 + k];
        c.wb_axis[k] = uwr[k] - uwf[k]; wl += c.wb_axis[k] * c.wb_axis[k];
        c.hl_in[k] = hli[k]; c.lbj[k] = lbj[k]; c.uwf[k] = uwf[k];
        c.uwf_to_ubj[k] = ubj[k] - uwf[k];
        c.ubj_to_a[k] = q[k] - half * q[6 + k] - ubj[k];
        c.ubj_to_b[k] = q[3 + k] - half * q[6 + k] - ubj[k];
        c.lbj_to_a[k] = q[k] + half * q[6 + k] - lbj[k];
        c.lbj_to_b[k] = q[3 + k] + half * q[6 + k] - lbj[k];
        c.lbj_to_hl_out[k] = hlo[k] - lbj[k];
        hl += (hlo[k] - hli[k]) * (hlo[k] - hli[k]);
      }
      wl = 1.0 / sqrt(wl);
      for (int k = 0; k < 3; ++k) c.wb_axis[k] *= wl;
      c.hl_len = sqrt(hl);
      c.has_rocker = OKIN_LDG(rec + 6);
      const double* ra = pos;
      if (c.has_rocker) {
        ra = pos + 3 * OKIN_LDG(rec + 7);
        const double* rb = pos + 3 * OKIN_LDG(rec + 8);
        const double* pi = pos + 3 * OKIN_LDG(rec + 9);
        const double* po = pos + 3 * OKIN_LDG(rec + 10);
        double al = 0.0, pl = 0.0;
        for (int k = 0; k < 3; ++k) {
          c.rk_axis_pt[k] = ra[k];
          c.rk_axis[k] = rb[k] - ra[k]; al += c.rk_axis[k] * c.rk_axis[k];
          c.rk_to_pr_in[k] = pi[k] - ra[k];
          c.lbj_to_pr_out[k] = po[k] - lbj[k];
          pl += (po[k] - pi[k]) * (po[k] - pi[k]);
        }
        al = 1.0 / sqrt(al);
        for (int k = 0; k < 3; ++k) c.rk_axis[k] *= al;
        c.pr_len = sqrt(pl);
      }
      const int n = 7 + c.has_rocker, m = 10 + c.has_rocker;
      double x[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      bool ok = false;
      for (int it = 0; it < 40 && !ok; ++it) {
        double J[11][8], r[11];
        for (int col = 0; col < n; ++col) {
          OkinDual xd[8], rd[11];
          for (int k = 0; k < 8; ++k) xd[k] = OkinDual{x[k], k == col ? 1.0 : 0.0};
          okin_shim_residuals<OkinDual>(c, xd, rd);
          for (int i = 0; i < m; ++i) { J[i][col] = rd[i].d; r[i] = rd[i].v; }
        }
        // normal equations + dense Cholesky (8x8)
        double A[8][8], g[8];
        for (int a = 0; a < n; ++a) {
          g[a] = 0.0;
          for (int i = 0; i < m; ++i) g[a] -= J[i][a] * r[i];
          for (int b = 0; b <= a; ++b) {
            double acc = 0.0;
            for (int i = 0; i < m; ++i) acc += J[i][a] * J[i][b];
            A[a][b] = acc;
          }
        }
        bool pd = true;
        for (int a = 0; a < n; ++a) {
          for (int b = 0; b <= a; ++b) {
            double acc = A[a][b];
            for (int k = 0; k < b; ++k) acc -= A[a][k] * A[b][k];
            if (a == b) { pd = pd && acc > 0.0; A[a][a] = sqrt(acc); }
            else A[a][b] = acc / A[b][b];
          }
        }
        if (!pd) break;
        for (int a = 0; a < n; ++a) {
          double acc = g[a];
          for (int k = 0; k < a; ++k) acc -= A[a][k] * g[k];
          g[a] = acc / A[a][a];
        }
        double hmax = 0.0;
        for (int a = n - 1; a >= 0; --a) {
          double acc = g[a];
          for (int k = a + 1; k < n; ++k) acc -= A[k][a] * g[k];
          g[a] = acc / A[a][a];
          x[a] += g[a];
          hmax = fabs(g[a]) > hmax ? fabs(g[a]) : hmax;
        }
        ok = hmax <= 1e-13;
      }
      double rfin[11];
      okin_shim_residuals<double>(c, x, rfin);
      double rmax = 0.0;
      for (int i = 0; i < m; ++i) rmax = fabs(rfin[i]) > rmax ? fabs(rfin[i]) : rmax;
      if (!ok || !(rmax <= 1e-3)) {
        red[lane] = 1.0;  // shims.py:451-462 raises: flag the instance invalid
      } else {
        // apply (double_wishbone.py:546-571)
        const double z3[3] = {0.0, 0.0, 0.0};
        const OkinV3<double> wb = {c.wb_axis[0] * x[0], c.wb_axis[1] * x[0], c.wb_axis[2] * x[0]};
        const OkinV3<double> nu = okin_rodrigues(okin_lift(c.uwf_to_ubj, z3, 0.0), wb);
        ubj[0] = c.uwf[0] + nu.x; ubj[1] = c.uwf[1] + nu.y; ubj[2] = c.uwf[2] + nu.z;
        const double ang = sqrt(x[4] * x[4] + x[5] * x[5] + x[6] * x[6]);
        if (ang > OKIN_GEOM_EPS) {
          const double axis[3] = {x[4] / ang, x[5] / ang, x[6] / ang};
          for (int k = OKIN_LDG(rec + 12); k < OKIN_LDG(rec + 13); ++k)
            okin_rotate_about_axis(pos + 3 * OKIN_LDG(lists + k), c.lbj, axis, ang);
        }
        if (c.has_rocker)
          for (int k = OKIN_LDG(rec + 14); k < OKIN_LDG(rec + 15); ++k)
            okin_rotate_about_axis(pos + 3 * OKIN_LDG(lists + k), c.rk_axis_pt, c.rk_axis, x[7]);
      }
    }
  }
  OKIN_PHASE_END
  if (okin_red_sum(red) != 0.0) *invalid = 1;
}

// ---------------------------------------------------------------------------------------
// Setup: inputs -> pos, derived parameters, design pose, per-instance constants.
// ---------------------------------------------------------------------------------------
template <bool SHIM>
OKIN_FN void okin_setup(const OkinProgram& pr, double* sm, const double* __restrict__ hardpoints,
                        const double* __restrict__ params, int* invalid, bool keep_design) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  double* pos = sm + hdr[OKIN_H_OFF_POS];
  double* cst = sm + hdr[OKIN_H_OFF_CST];
  double* par = sm + hdr[OKIN_H_OFF_PAR];
  const int nin = hdr[OKIN_H_NIN];
  const int32_t* in_point = okin_sec(pr, OKIN_S_IN_POINT);
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < 3 * nin; t += 32) pos[3 * OKIN_LDG(in_point + t / 3) + t % 3] = hardpoints[t];
  OKIN_PHASE_END
  if (SHIM) okin_shim_presolve(pr, sm, params ? params : okin_fsec(pr, OKIN_F_PARAM_DEFAULT), invalid);

  // Derived-op parameters.  A design projection reads the *authored* position of the derived
  // point (macpherson.py:199-204), which is what pos[] still holds at this moment.
  const int ndop = hdr[OKIN_H_NDOP];
  const int32_t* dop = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP));
  const int32_t* par_mode = okin_sec(pr, OKIN_S_PAR_MODE);
  const double* par_val = okin_fsec(pr, OKIN_F_PAR_VAL);
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int d = lane; d < ndop; d += 32) {
    const int32_t* rec = dop + d * OKIN_DOP_STRIDE;
    const int p = OKIN_LDG(rec + 5);
    double value = OKIN_LDG(par_val + p);
    if (OKIN_LDG(par_mode + p) == OKIN_PAR_DESIGN_PROJECTION) {
      const double* a = pos + 3 * OKIN_LDG(rec + 2);
      const double* b = pos + 3 * OKIN_LDG(rec + 3);
      const double* o = hardpoints + 3 * OKIN_LDG(rec + 6);
      const double v[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
      const double il = OKIN_RSQRT(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
      value = ((o[0] - a[0]) * v[0] + (o[1] - a[1]) * v[1] + (o[2] - a[2]) * v[2]) * il;
    }
    par[p] = value;
  }
  OKIN_PHASE_END

  okin_derived_update(pr, sm, false);

  if (keep_design) {  // design positions kept for the metrics (travel references, rotation datums)
    const int ndsn = hdr[OKIN_H_NDSN];
    const int32_t* dpt = okin_sec(pr, OKIN_S_DESIGN_PT);
    double* dsn = sm + hdr[OKIN_H_OFF_DSN];
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < 3 * ndsn; t += 32) dsn[t] = pos[3 * OKIN_LDG(dpt + t / 3) + t % 3];
    OKIN_PHASE_END
  }

  // Per-instance constants: each row's own quantity at the design pose (true norms, no
  // softnorm: vector_utils/geometric.py:17-28, :71-104, :197-214).
  const int nrows = hdr[OKIN_H_NROW] + hdr[OKIN_H_NREP];
  const int32_t* rows = okin_sec(pr, OKIN_S_ROW);
  const double* cst_init = okin_fsec(pr, OKIN_F_CST_INIT);
  const int ncst = hdr[OKIN_H_NCST];
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < ncst; t += 32) cst[t] = OKIN_LDG(cst_init + t);
  OKIN_PHASE_END
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < nrows; t += 32) {
    const int32_t* rec = rows + t * OKIN_ROW_STRIDE;
    const int rule = OKIN_LDG(rec + OKIN_R_RULE);
    if (rule == OKIN_RULE_EXPLICIT) continue;
    const int fam = OKIN_LDG(rec + OKIN_R_FAM);
    double* c = cst + OKIN_LDG(rec + OKIN_R_CST);
    const double* p0 = pos + 3 * OKIN_LDG(rec + OKIN_R_P0);
    if (rule == OKIN_RULE_DESIGN_POINT) {
      c[0] = p0[0]; c[1] = p0[1]; c[2] = p0[2];
    } else if (rule == OKIN_RULE_TARGET_BASE) {
      c[3] = c[0] * p0[0] + c[1] * p0[1] + c[2] * p0[2];
    } else if (fam == OKIN_FAM_DISTANCE) {
      const double* p1 = pos + 3 * OKIN_LDG(rec + OKIN_R_P1);
      const double dx = p1[0] - p0[0], dy = p1[1] - p0[1], dz = p1[2] - p0[2];
      c[0] = sqrt(dx * dx + dy * dy + dz * dz);
    } else if (fam == OKIN_FAM_ANGLE) {
      // compute_vector_vector_angle on unit vectors (geometric.py:94-104)
      const double* p1 = pos + 3 * OKIN_LDG(rec + OKIN_R_P1);
      const double* p2 = pos + 3 * OKIN_LDG(rec + OKIN_R_P2);
      const double* p3 = pos + 3 * OKIN_LDG(rec + OKIN_R_P3);
      double a[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]};
      double b[3] = {p3[0] - p2[0], p3[1] - p2[1], p3[2] - p2[2]};
      const double na = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
      const double nb = sqrt(b[0] * b[0] + b[1] * b[1] + b[2] * b[2]);
      for (int k = 0; k < 3; ++k) { a[k] /= na; b[k] /= nb; }
      const double cx = a[1] * b[2] - a[2] * b[1], cy = a[2] * b[0] - a[0] * b[2], cz = a[0] * b[1] - a[1] * b[0];
      c[0] = atan2(sqrt(cx * cx + cy * cy + cz * cz), a[0] * b[0] + a[1] * b[1] + a[2] * b[2]);
    } else if (fam == OKIN_FAM_SCALAR_TRIPLE) {
      const double* p1 = pos + 3 * OKIN_LDG(rec + OKIN_R_P1);
      const double* p2 = pos + 3 * OKIN_LDG(rec + OKIN_R_P2);
      const double* p3 = pos + 3 * OKIN_LDG(rec + OKIN_R_P3);
      const double a[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]};
      const double b[3] = {p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2]};
      const double d[3] = {p3[0] - p0[0], p3[1] - p0[1], p3[2] - p0[2]};
      const double v = a[0] * (b[1] * d[2] - b[2] * d[1]) + a[1] * (b[2] * d[0] - b[0] * d[2]) +
                       a[2] * (b[0] * d[1] - b[1] * d[0]);
      c[0] = v;
      c[1] = 1.0 / fabs(v);
    }
  }
  OKIN_PHASE_END
}

// ---------------------------------------------------------------------------------------
// Row evaluation: residuals (and gradients mapped to effective free blocks).
// ---------------------------------------------------------------------------------------
template <typename Dummy = void>
OKIN_FN void okin_eval_rows(const OkinProgram& pr, double* sm, const double* tval, bool with_grad, OkinState& st) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  okin_derived_update(pr, sm, true);
  if (with_grad) okin_derived_jacobians(pr, sm);
  const int nls = hdr[OKIN_H_NROW];
  const int nrows = nls + hdr[OKIN_H_NREP];
  const int32_t* rows = OKIN_SHARED(okin_sec(pr, OKIN_S_ROW_HOT));
  const int32_t* der = OKIN_SHARED(okin_sec(pr, OKIN_S_DER));
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* cst = sm + hdr[OKIN_H_OFF_CST];
  const double* dblk = sm + hdr[OKIN_H_OFF_DBLK];
  double* r = sm + hdr[OKIN_H_OFF_R];
  double* rg = sm + hdr[OKIN_H_OFF_RG];
  double* red = sm + hdr[OKIN_H_OFF_RED];
  const int32_t* drow = OKIN_SHARED(okin_sec(pr, OKIN_S_DROW));
  const int ndrow = hdr[OKIN_H_NDROW], ngrow = hdr[OKIN_H_NGROW];
  OKIN_PHASE_BEGIN
  double sq = 0.0;
  // Fast path: plain distance rows (most of every shipped topology).  r = sqrt(s + eps^2) - eps - L,
  // u = (p2 - p1)/sqrt(s + eps^2) is the whole gradient (dR/dp2 = u, dR/dp1 = -u).
  OKIN_LANE_LOOP
  for (int slot = lane; slot < ndrow; slot += 32) {
    const uint32_t pp = (uint32_t)OKIN_LDG(drow + slot), oo = (uint32_t)OKIN_LDG(drow + ndrow + slot);
    const double* a = pos + 3 * (pp & 0xffffu);
    const double* b = pos + 3 * (pp >> 16);
    const double dx = b[0] - a[0], dy = b[1] - a[1], dz = b[2] - a[2];
    const double s2 = dx * dx + dy * dy + dz * dz + OKIN_EPS_SQ;
    const double inv = OKIN_RSQRT(s2);
    const double res = s2 * inv - OKIN_EPS - cst[oo & 0xffffu];
    r[OKIN_LDG(drow + 2 * ndrow + slot)] = res;
    sq += res * res;
    if (with_grad) {
      double* u = rg + (oo >> 16);
      u[0] = dx * inv; u[1] = dy * inv; u[2] = dz * inv;
    }
  }
  OKIN_LANE_LOOP
  for (int slot = lane; slot < ngrow; slot += 32) {
    const int32_t* rec = rows + slot * OKIN_ROW_STRIDE;
    const int t = OKIN_LDG(rec + OKIN_R_ROWID);
    const int fam = OKIN_LDG(rec + OKIN_R_FAM);
    const double* c = cst + OKIN_LDG(rec + OKIN_R_CST);
    double p[12], g[12];
    int np = 0;
    for (int s = 0; s < 4; ++s) {
      const int pi = OKIN_LDG(rec + OKIN_R_P0 + s);
      if (pi < 0) break;
      p[3 * s] = pos[3 * pi]; p[3 * s + 1] = pos[3 * pi + 1]; p[3 * s + 2] = pos[3 * pi + 2];
      np = s + 1;
    }
    const bool grad = with_grad && t < nls;
    double res;
    if (fam == OKIN_FAM_TARGET) {
      res = c[0] * p[0] + c[1] * p[1] + c[2] * p[2] - (c[3] + tval[OKIN_LDG(rec + OKIN_R_AUX)]);
      g[0] = c[0]; g[1] = c[1]; g[2] = c[2];
    } else if (grad) {
      res = okin_family_resgrad(fam, p, c, g);
    } else {
      res = okin_family_res(fam, p, c);
    }
    r[t] = res;
    if (t < nls) sq += res * res;
    if (grad) {
      double* out = rg + OKIN_LDG(rec + OKIN_R_RG);
      const int neff = OKIN_LDG(rec + OKIN_R_NEFF);
      for (int e = 0; e < 3 * neff; ++e) out[e] = 0.0;
      OKIN_SHORT_LOOP
      for (int s = 0; s < np; ++s) {
        const int m = OKIN_LDG(rec + OKIN_R_S0 + s);
        if (m < 0) continue;
        const double gx = g[3 * s], gy = g[3 * s + 1], gz = g[3 * s + 2];
        if (m < OKIN_SLOT_DER) {
          out[3 * m] += gx; out[3 * m + 1] += gy; out[3 * m + 2] += gz;
        } else {
          const int32_t* dd = der + (m - OKIN_SLOT_DER) * OKIN_DER_STRIDE;
          const int nd = OKIN_LDG(dd);
          OKIN_SHORT_LOOP
          for (int q = 0; q < nd; ++q) {
            const double* B = dblk + OKIN_LDG(dd + 1 + 2 * q);
            const int e = OKIN_LDG(dd + 2 + 2 * q);
            out[3 * e] += gx * B[0] + gy * B[3] + gz * B[6];
            out[3 * e + 1] += gx * B[1] + gy * B[4] + gz * B[7];
            out[3 * e + 2] += gx * B[2] + gy * B[5] + gz * B[8];
          }
        }
      }
    }
  }
  red[lane] = sq;
  OKIN_PHASE_END
  const double f2 = okin_red_sum(red);
  // max|r| in a second sweep over r[] so that the reduction scratch stays one value per lane
  OKIN_PHASE_BEGIN
  double mx = 0.0;
  OKIN_LANE_LOOP
  for (int t = lane; t < nrows; t += 32) {
    const double ar = fabs(r[t]);
    mx = (ar > mx || ar != ar) ? ar : mx;
  }
  red[lane] = mx;
  OKIN_PHASE_END
  const double rmax = okin_red_max(red);
  st.f2 = f2;
  st.rmax = rmax;
}

// ---------------------------------------------------------------------------------------
// Normal equations: A = J^T J (+ mu diag(A)) into the factor storage, g = J^T r into vec[0].
// ---------------------------------------------------------------------------------------
template <typename Dummy = void>
OKIN_FN_HOT void okin_assemble(const OkinProgram& pr, double* sm, double mu, bool g_only) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nat = hdr[OKIN_H_NAT];
  const int nf = hdr[OKIN_H_NF];
  const int32_t* aptr = OKIN_SHARED(okin_sec(pr, OKIN_S_ASM_PTR));
  const int32_t* atask = OKIN_SHARED(okin_sec(pr, OKIN_S_ASM_TASK));
  const int32_t* acon = OKIN_SHARED(okin_sec(pr, OKIN_S_ASM_CON));
  const int32_t* gptr = OKIN_SHARED(okin_sec(pr, OKIN_S_G_PTR));
  const int32_t* gcon = OKIN_SHARED(okin_sec(pr, OKIN_S_G_CON));
  const double* rg = sm + hdr[OKIN_H_OFF_RG];
  const double* r = sm + hdr[OKIN_H_OFF_R];
  double* Lb = sm + hdr[OKIN_H_OFF_LB];
  double* vec = sm + hdr[OKIN_H_OFF_VEC];
  const double damp = 1.0 + mu, lev = mu * 1e-9;
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = (g_only ? nat : 0) + lane; t < nat + nf; t += 32) {
    if (t < nat) {
      // one 3x3 block of A: sum of outer products ga gb^T over the rows coupling the two points
      const int b = OKIN_LDG(aptr + t), e = OKIN_LDG(aptr + t + 1);
      double a00 = 0, a01 = 0, a02 = 0, a10 = 0, a11 = 0, a12 = 0, a20 = 0, a21 = 0, a22 = 0;
      OKIN_UNROLL_INNER
      for (int q = b; q < e; ++q) {
        const uint32_t w = (uint32_t)OKIN_LDG(acon + q);
        const double* ga = rg + ((w >> 16) & 0x7fffu);
        const double* gb = rg + (w & 0xffffu);
        const double sg = (w & OKIN_CON_NEG) ? -1.0 : 1.0;
        const double p0 = ga[0], p1 = ga[1], p2 = ga[2], y0 = gb[0], y1 = gb[1], y2 = gb[2];
        const double x0 = sg * p0, x1 = sg * p1, x2 = sg * p2;
        a00 = fma(x0, y0, a00); a01 = fma(x0, y1, a01); a02 = fma(x0, y2, a02);
        a10 = fma(x1, y0, a10); a11 = fma(x1, y1, a11); a12 = fma(x1, y2, a12);
        a20 = fma(x2, y0, a20); a21 = fma(x2, y1, a21); a22 = fma(x2, y2, a22);
      }
      const int task = OKIN_LDG(atask + t);
      // Marquardt scaling plus a small Levenberg shift: a row whose gradient vanishes at the current
      // point (a spherical joint that is exactly closed) leaves a zero diagonal that scaling alone never
      // makes positive; MINPACK substitutes 1 for a zero column norm there (lmder, diag(j) = 1).
      if (task & OKIN_ASM_DIAG) { a00 = a00 * damp + lev; a11 = a11 * damp + lev; a22 = a22 * damp + lev; }
      double* dst = Lb + 9 * (task & 0xffff);
      dst[0] = a00; dst[1] = a01; dst[2] = a02; dst[3] = a10; dst[4] = a11; dst[5] = a12;
      dst[6] = a20; dst[7] = a21; dst[8] = a22;
    } else {
      const int j = t - nat;
      const int b = OKIN_LDG(gptr + j), e = OKIN_LDG(gptr + j + 1);
      double g0 = 0, g1 = 0, g2 = 0;
      OKIN_UNROLL_INNER
      for (int q = b; q < e; ++q) {
        const uint32_t w = (uint32_t)OKIN_LDG(gcon + q);
        const double* ga = rg + ((w >> 16) & 0x7fffu);
        const double res = (w & OKIN_CON_NEG) ? -r[w & 0xffffu] : r[w & 0xffffu];
        g0 = fma(ga[0], res, g0); g1 = fma(ga[1], res, g1); g2 = fma(ga[2], res, g2);
      }
      vec[3 * j] = -g0; vec[3 * j + 1] = -g1; vec[3 * j + 2] = -g2;  // right-hand side of A h = -g
    }
  }
  OKIN_PHASE_END
}

// ---------------------------------------------------------------------------------------
// 3x3-block sparse Cholesky, left-looking, level-scheduled over the elimination tree.
// A finished column's diagonal block holds its factor {l00,l10,l11,l20,l21,l22, 1/l00, 1/l11, 1/l22}.
// ---------------------------------------------------------------------------------------
OKIN_HD bool okin_chol3(const double* d, double f[9]) {
  // d: 3x3 row-major block, lower part valid.
  const double d00 = d[0], d10 = d[3], d11 = d[4], d20 = d[6], d21 = d[7], d22 = d[8];
  const double i00 = OKIN_RSQRT(d00);
  const double l00 = d00 * i00, l10 = d10 * i00, l20 = d20 * i00;
  const double t11 = d11 - l10 * l10;
  const double i11 = OKIN_RSQRT(t11);
  const double l11 = t11 * i11;
  const double l21 = (d21 - l20 * l10) * i11;
  const double t22 = d22 - l20 * l20 - l21 * l21;
  const double i22 = OKIN_RSQRT(t22);
  const double l22 = t22 * i22;
  f[0] = l00; f[1] = l10; f[2] = l11; f[3] = l20; f[4] = l21; f[5] = l22; f[6] = i00; f[7] = i11; f[8] = i22;
  return d00 > 0.0 && t11 > 0.0 && t22 > 0.0;
}

// Once a column's diagonal block has received its updates nothing reads its raw entries again, so the
// factor {l00,l10,l11,l20,l21,l22, 1/l00,1/l11,1/l22} is written over it.
OKIN_HD void okin_write_diag_factor(double* sm, int doff, double* red, int lane) {
  sm = OKIN_SHARED(sm);
  double f[9];
  const bool ok = okin_chol3(sm + doff, f);
  double* o = sm + doff;
  for (int k = 0; k < 9; ++k) o[k] = f[k];
  if (!ok) red[lane] = 1.0;
}

// carry_tangents: also run the update / scale tasks of the tangent right-hand sides vec[1..NT]
// (ordered last in every level by the host compiler).
template <typename Dummy = void>
OKIN_FN_HOT void okin_factor(const OkinProgram& pr, double* sm, OkinState& st, bool carry_tangents) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nlev = hdr[OKIN_H_NLEV];
  const int32_t* lev_upd = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_UPD));
  const int32_t* lev_upd_mid = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_UPD_MID));
  const int32_t* udst = OKIN_SHARED(okin_sec(pr, OKIN_S_UPD_DST));
  const int32_t* uptr = OKIN_SHARED(okin_sec(pr, OKIN_S_UPD_PTR));
  const int32_t* ucon = OKIN_SHARED(okin_sec(pr, OKIN_S_UPD_CON));
  const int32_t* lev_scl = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_SCL));
  const int32_t* lev_scl_mid = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_SCL_MID));
  const int32_t* scl = OKIN_SHARED(okin_sec(pr, OKIN_S_SCL));
  const int32_t* lcp = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_COL_PTR));
  const int32_t* lcol = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_COL));
  const int32_t* doffs = OKIN_SHARED(okin_sec(pr, OKIN_S_DIAG_OFF));
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  red[lane] = 0.0;
  OKIN_PHASE_END
  for (int lv = 0; lv < nlev; ++lv) {
    const int ub = OKIN_LDG(lev_upd + lv), ue = carry_tangents ? OKIN_LDG(lev_upd + lv + 1) : OKIN_LDG(lev_upd_mid + lv);
    if (ue > ub) {
      OKIN_PHASE_BEGIN
      // left-looking update of one block row (or of a carried right-hand side), two contributions per trip
      OKIN_LANE_LOOP
      for (int t = ub + lane; t < ue; t += 32) {
        const int b = OKIN_LDG(uptr + t), e = OKIN_LDG(uptr + t + 1);
        double* dst = sm + OKIN_LDG(udst + t);
        double c0 = dst[0], c1 = dst[1], c2 = dst[2];
        OKIN_UNROLL_INNER
        for (int q = b; q < e; ++q) {
          const uint32_t w = (uint32_t)OKIN_LDG(ucon + q);
          const double* a = sm + (w >> 16);
          const double* B = sm + (w & 0xffffu);
          const double a0 = a[0], a1 = a[1], a2 = a[2];
          const double b0 = B[0], b1 = B[1], b2 = B[2], b3 = B[3], b4 = B[4], b5 = B[5], b6 = B[6], b7 = B[7], b8 = B[8];
          c0 = fma(-a0, b0, c0); c1 = fma(-a0, b3, c1); c2 = fma(-a0, b6, c2);
          c0 = fma(-a1, b1, c0); c1 = fma(-a1, b4, c1); c2 = fma(-a1, b7, c2);
          c0 = fma(-a2, b2, c0); c1 = fma(-a2, b5, c1); c2 = fma(-a2, b8, c2);
        }
        dst[0] = c0; dst[1] = c1; dst[2] = c2;
      }
      OKIN_PHASE_END
    }
    // The level's diagonal blocks are final: factor each once, in place (one lane per column), so that
    // the scale tasks below and the triangular solves later read the factor instead of recomputing it.
    const int wb = OKIN_LDG(lcp + lv), we = OKIN_LDG(lcp + lv + 1);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int c = wb + lane; c < we; c += 32)
      okin_write_diag_factor(sm, OKIN_LDG(doffs + OKIN_LDG(lcol + c)), red, lane);
    OKIN_PHASE_END
    const int sb = OKIN_LDG(lev_scl + lv), se = carry_tangents ? OKIN_LDG(lev_scl + lv + 1) : OKIN_LDG(lev_scl_mid + lv);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = sb + lane; t < se; t += 32) {
      const uint32_t w = (uint32_t)OKIN_LDG(scl + t);
      const double* f = sm + (w & 0xffffu);
      double* b = sm + (w >> 16);
      const double x0 = b[0] * f[6];
      const double x1 = (b[1] - x0 * f[1]) * f[7];
      const double x2 = (b[2] - x0 * f[3] - x1 * f[4]) * f[8];
      b[0] = x0; b[1] = x1; b[2] = x2;
    }
    OKIN_PHASE_END
  }
  st.notpd = okin_red_sum(red) != 0.0;
}

// Solve A X = B for nrhs right-hand sides stored at vec[first .. first+nrhs) (elimination order),
// in place.  skip_forward: vec[first] already holds L^{-1} b (the factorisation carries vec[0]
// as an extra row).
template <typename Dummy = void>
OKIN_FN_HOT void okin_solve(const OkinProgram& pr, double* sm, int first, int nrhs, bool skip_forward) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nlev = hdr[OKIN_H_NLEV];
  const int n = 3 * hdr[OKIN_H_NF];
  const int32_t* lcp = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_COL_PTR));
  const int32_t* lcol = OKIN_SHARED(okin_sec(pr, OKIN_S_LEV_COL));
  const int32_t* fptr = OKIN_SHARED(okin_sec(pr, OKIN_S_FW_PTR));
  const int32_t* fcon = OKIN_SHARED(okin_sec(pr, OKIN_S_FW_CON));
  const int32_t* bptr = OKIN_SHARED(okin_sec(pr, OKIN_S_BW_PTR));
  const int32_t* bcon = OKIN_SHARED(okin_sec(pr, OKIN_S_BW_CON));
  const double* Lb = sm;
  const int32_t* doffs = OKIN_SHARED(okin_sec(pr, OKIN_S_DIAG_OFF));
  double* vec = sm + hdr[OKIN_H_OFF_VEC] + first * n;
  for (int lv = 0; lv < (skip_forward ? 0 : nlev); ++lv) {  // L y = b
    const int cb = OKIN_LDG(lcp + lv), ce = OKIN_LDG(lcp + lv + 1);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < (ce - cb) * nrhs; t += 32) {
      const int j = OKIN_LDG(lcol + cb + t / nrhs);
      double* v = vec + (t % nrhs) * n;
      double t0 = v[3 * j], t1 = v[3 * j + 1], t2 = v[3 * j + 2];
      OKIN_UNROLL_INNER
      for (int q = OKIN_LDG(fptr + j); q < OKIN_LDG(fptr + j + 1); ++q) {
        const uint32_t w = (uint32_t)OKIN_LDG(fcon + q);
        const double* B = Lb + (w >> 16);
        const double* y = v + (w & 0xffffu);
        const double y0 = y[0], y1 = y[1], y2 = y[2];
        const double b0 = B[0], b1 = B[1], b2 = B[2], b3 = B[3], b4 = B[4], b5 = B[5], b6 = B[6], b7 = B[7], b8 = B[8];
        t0 = fma(-b0, y0, t0); t1 = fma(-b3, y0, t1); t2 = fma(-b6, y0, t2);
        t0 = fma(-b1, y1, t0); t1 = fma(-b4, y1, t1); t2 = fma(-b7, y1, t2);
        t0 = fma(-b2, y2, t0); t1 = fma(-b5, y2, t1); t2 = fma(-b8, y2, t2);
      }
      const double* f = sm + OKIN_LDG(doffs + j);
      const double y0 = t0 * f[6];
      const double y1 = (t1 - f[1] * y0) * f[7];
      const double y2 = (t2 - f[3] * y0 - f[4] * y1) * f[8];
      v[3 * j] = y0; v[3 * j + 1] = y1; v[3 * j + 2] = y2;
    }
    OKIN_PHASE_END
  }
  for (int lv = nlev - 1; lv >= 0; --lv) {  // L^T x = y
    const int cb = OKIN_LDG(lcp + lv), ce = OKIN_LDG(lcp + lv + 1);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < (ce - cb) * nrhs; t += 32) {
      const int j = OKIN_LDG(lcol + cb + t / nrhs);
      double* v = vec + (t % nrhs) * n;
      double t0 = v[3 * j], t1 = v[3 * j + 1], t2 = v[3 * j + 2];
      OKIN_UNROLL_INNER
      for (int q = OKIN_LDG(bptr + j); q < OKIN_LDG(bptr + j + 1); ++q) {
        const uint32_t w = (uint32_t)OKIN_LDG(bcon + q);
        const double* B = Lb + (w >> 16);
        const double* x = v + (w & 0xffffu);
        const double x0 = x[0], x1 = x[1], x2 = x[2];
        const double b0 = B[0], b1 = B[1], b2 = B[2], b3 = B[3], b4 = B[4], b5 = B[5], b6 = B[6], b7 = B[7], b8 = B[8];
        t0 = fma(-b0, x0, t0); t1 = fma(-b1, x0, t1); t2 = fma(-b2, x0, t2);
        t0 = fma(-b3, x1, t0); t1 = fma(-b4, x1, t1); t2 = fma(-b5, x1, t2);
        t0 = fma(-b6, x2, t0); t1 = fma(-b7, x2, t1); t2 = fma(-b8, x2, t2);
      }
      const double* f = sm + OKIN_LDG(doffs + j);
      const double x2 = t2 * f[8];
      const double x1 = (t1 - f[4] * x2) * f[7];
      const double x0 = (t0 - f[1] * x1 - f[3] * x2) * f[6];
      v[3 * j] = x0; v[3 * j + 1] = x1; v[3 * j + 2] = x2;
    }
    OKIN_PHASE_END
  }
}

// pos[free] += scale * vec[which]; returns max|vec[which]| (warp-uniform).
template <typename Dummy = void>
OKIN_FN double okin_apply_step(const OkinProgram& pr, double* sm, int which, double scale, bool save) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int n = 3 * hdr[OKIN_H_NF];
  const int32_t* ep = OKIN_SHARED(okin_sec(pr, OKIN_S_ELIM_POINT));
  double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* v = sm + hdr[OKIN_H_OFF_VEC] + which * n;
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  double mx = 0.0;
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) {
    const int idx = 3 * OKIN_LDG(ep + u / 3) + u % 3;
    const double x = pos[idx];
    const double h = v[u];
    pos[idx] = x + scale * h;
    const double ah = fabs(h);
    mx = (ah > mx || ah != ah) ? ah : mx;
  }
  red[lane] = mx;
  OKIN_PHASE_END
  return okin_red_max(red);
}

template <typename Dummy = void>
OKIN_FN void okin_restore(const OkinProgram& pr, double* sm) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int n = 3 * hdr[OKIN_H_NF];
  const int32_t* ep = OKIN_SHARED(okin_sec(pr, OKIN_S_ELIM_POINT));
  double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* h = sm + hdr[OKIN_H_OFF_VEC];   // the step just applied (vec[0], scale 1)
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) pos[3 * OKIN_LDG(ep + u / 3) + u % 3] -= h[u];
  OKIN_PHASE_END
}

// max|vec[which]| (warp-uniform).
template <typename Dummy = void>
OKIN_FN double okin_vec_max(const OkinProgram& pr, double* sm, int which) {
  sm = OKIN_SHARED(sm);
  const int n = 3 * pr.hdr[OKIN_H_NF];
  const double* v = sm + pr.hdr[OKIN_H_OFF_VEC] + which * n;
  double* red = sm + pr.hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  double mx = 0.0;
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) {
    const double a = fabs(v[u]);
    mx = (a > mx || a != a) ? a : mx;
  }
  red[lane] = mx;
  OKIN_PHASE_END
  return okin_red_max(red);
}

// Continuation predictor (no tangents needed): with the last accepted
// solutions x_k (in pos), x_{k-1} (xprev) and the two older increments d1 = x_{k-1} - x_{k-2},
// d2 = x_{k-2} - x_{k-3} (float32: they only shape the starting point), the next increment for
// uniform target steps is the Newton backward-difference extrapolation
//   order 1: d0      order 2: 2 d0 - d1      order 3: 3 d0 - 3 d1 + d2,      d0 = x_k - x_{k-1}.
// Always shifts the history and leaves xprev = x_k: the start of the step, which is also what a failed
// predicted start is retried from (the reference's plain warm start, solver.py:774).
template <typename Dummy = void>
OKIN_FN void okin_extrapolate(const OkinProgram& pr, double* sm, int order) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int n = 3 * hdr[OKIN_H_NF];
  const int32_t* ep = OKIN_SHARED(okin_sec(pr, OKIN_S_ELIM_POINT));
  double* pos = sm + hdr[OKIN_H_OFF_POS];
  double* xprev = sm + hdr[OKIN_H_OFF_XPREV];
  float* h1 = reinterpret_cast<float*>(sm + hdr[OKIN_H_OFF_DHIST]);
  float* h2 = h1 + 2 * ((n + 1) / 2);
  float* h3 = h2 + 2 * ((n + 1) / 2);
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) {
    const int idx = 3 * OKIN_LDG(ep + u / 3) + u % 3;
    const double x = pos[idx];
    const double d0 = x - xprev[u];
    const double d1 = (double)h1[u], d2 = (double)h2[u], d3 = (double)h3[u];
    double step = 0.0;
    if (order == 1) step = d0;
    if (order == 2) step = 2.0 * d0 - d1;
    if (order == 3) step = 3.0 * (d0 - d1) + d2;
    if (order >= 4) step = 4.0 * (d0 + d2) - 6.0 * d1 - d3;
    h3[u] = h2[u];
    h2[u] = h1[u];
    h1[u] = (float)d0;
    xprev[u] = x;
    pos[idx] = x + step;
  }
  OKIN_PHASE_END
}

// Right-hand sides of the tangent systems A dq/dt_j = J_target_j^T into vec[1..NT]
// (sensitivity.py:89-101 solved through the normal equations: with full column rank
// lstsq([J; pins], e_j) == (J^T J)^{-1} J^T e_j).  Uses the target rows of rg[].
template <typename Dummy = void>
OKIN_FN void okin_tangent_rhs(const OkinProgram& pr, double* sm) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nt = hdr[OKIN_H_NT];
  const int n = 3 * hdr[OKIN_H_NF];
  const int32_t* sptr = OKIN_SHARED(okin_sec(pr, OKIN_S_TGT_SC_PTR));
  const int32_t* sc = OKIN_SHARED(okin_sec(pr, OKIN_S_TGT_SC));
  const double* rg = sm + hdr[OKIN_H_OFF_RG];
  double* vec = sm + hdr[OKIN_H_OFF_VEC] + n;
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < nt * n; t += 32) vec[t] = 0.0;
  OKIN_PHASE_END
  OKIN_PHASE_BEGIN
  for (int j = 0; j < nt; ++j)
    for (int q = OKIN_LDG(sptr + j) + lane; q < OKIN_LDG(sptr + j + 1); q += 32) {
      const uint32_t w = (uint32_t)OKIN_LDG(sc + q);
      vec[j * n + (w & 0xffffu)] = rg[w >> 16];
    }
  OKIN_PHASE_END
}

// Residuals of the linear model at the step just taken: r <- r + J h (J = the row gradients of the
// linearisation the step came from, h = vec[0]); report rows from their two pins.  For a final step
// |h| <= fine_tol this differs from the residuals at the new point by the second-order term
// (curvature x |h|^2, ~1e-10 mm), so the lean kernel reports it as max|r| instead of paying a second
// row evaluation per state.  Sets st.f2 / st.rmax like okin_eval_rows.
template <typename Dummy = void>
OKIN_FN void okin_linear_residuals(const OkinProgram& pr, double* sm, OkinState& st) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nls = hdr[OKIN_H_NROW], nrep = hdr[OKIN_H_NREP];
  const int32_t* jptr = OKIN_SHARED(okin_sec(pr, OKIN_S_JH_PTR));
  const int32_t* jcon = OKIN_SHARED(okin_sec(pr, OKIN_S_JH_CON));
  const int32_t* rpin = OKIN_SHARED(okin_sec(pr, OKIN_S_REP_PINS));
  const double* rg = sm + hdr[OKIN_H_OFF_RG];
  const double* h = sm + hdr[OKIN_H_OFF_VEC];
  double* r = sm + hdr[OKIN_H_OFF_R];
  double* red = sm + hdr[OKIN_H_OFF_RED];
  double sq = 0.0, mx = 0.0;
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < nls; t += 32) {
    double acc = r[t];
    for (int q = OKIN_LDG(jptr + t), e = OKIN_LDG(jptr + t + 1); q < e; ++q) {
      const uint32_t w = (uint32_t)OKIN_LDG(jcon + q);
      const double* g = rg + ((w >> 16) & 0x7fffu);
      const double* x = h + (w & 0xffffu);
      const double g0 = g[0], g1 = g[1], g2 = g[2], x0 = x[0], x1 = x[1], x2 = x[2];
      const double dot = fma(g0, x0, fma(g1, x1, g2 * x2));
      acc += (w & OKIN_CON_NEG) ? -dot : dot;
    }
    r[t] = acc;
  }
  OKIN_PHASE_END
  OKIN_PHASE_BEGIN
  double lsq = 0.0, lmx = 0.0;
  OKIN_LANE_LOOP
  for (int t = lane; t < nls; t += 32) {
    const double v = r[t], a = fabs(v);
    lsq += v * v;
    lmx = (a > lmx || a != a) ? a : lmx;
  }
  OKIN_LANE_LOOP
  for (int t = lane; t < nrep; t += 32) {
    const double p1 = r[OKIN_LDG(rpin + 2 * t)], p2 = r[OKIN_LDG(rpin + 2 * t + 1)];
    const double v = sqrt(p1 * p1 + p2 * p2 + OKIN_EPS_SQ) - OKIN_EPS;
    r[nls + t] = v;
    lmx = (v > lmx || v != v) ? v : lmx;
  }
  red[lane] = lsq;
  sq = lsq; mx = lmx;
  OKIN_PHASE_END
#if defined(__CUDA_ARCH__) && !defined(OKIN_LANE_EMU)
  st.f2 = okin_red_sum(red);
  OKIN_PHASE_BEGIN
  red[lane] = mx;
  OKIN_PHASE_END
  st.rmax = okin_red_max(red);
  (void)sq;
#else
  // lane emulation: the phase body ran once per lane; redo the reductions serially
  double f2 = 0.0, rm = 0.0;
  for (int t = 0; t < nls + nrep; ++t) {
    const double a = fabs(r[t]);
    if (t < nls) f2 += r[t] * r[t];
    rm = (a > rm || a != a) ? a : rm;
  }
  st.f2 = f2;
  st.rmax = rm;
  (void)sq; (void)mx;
#endif
}

// ---------------------------------------------------------------------------------------
// One sweep step: Gauss-Newton on the pinned least-squares system, Marquardt damping only
// after a step that fails to reduce ||r||^2.  A step below fine_tol ends the iteration (error
// second order in it); a step below coarse_tol is verified and finished by a chord step.
// Returns the number of residual evaluations (the SolverInfo.nfev analogue).  On return r[] holds
// the residuals at (within step_tol of) the final point; *gradients_at_solution: rg[] holds the row
// gradients there too (only asked for when the caller linearises at the solution afterwards).
// ---------------------------------------------------------------------------------------
template <typename Dummy = void>
OKIN_HD int okin_solve_step(const OkinProgram& pr, double* sm, const double* tval, const OkinSolverCfg& cfg,
                            OkinState& st, bool* converged, bool relinearise, bool* gradients_at_solution) {
  *gradients_at_solution = false;
  sm = OKIN_SHARED(sm);
  int nfev = 0;
  st.mu = 0.0;
  double nu = 2.0;
  bool gn_rejected = false;  // an undamped step of this solve has been rejected
  okin_eval_rows(pr, sm, tval, true, st);
  ++nfev;
  *converged = false;
  for (int it = 0; it < cfg.max_iter; ++it) {
    // The factorisation carries the step right-hand side as an extra block row, so the forward
    // substitution is part of it and one backward pass yields the step.  (The tangent right-hand sides
    // ride along only when the caller linearises at a solution for the exported tangents / metrics.)
    okin_assemble(pr, sm, st.mu, false);
    okin_factor(pr, sm, st, false);
    if (st.notpd) {  // rank-deficient normal matrix: damp and retry from the same point
      st.mu = st.mu > 0.0 ? st.mu * 10.0 : cfg.mu_init;
      if (st.mu > 1e12) break;
      continue;
    }
    okin_solve(pr, sm, 0, 1, true);
    const double hmax = okin_apply_step(pr, sm, 0, 1.0, true);
    if (!(hmax == hmax)) {  // NaN step: invalid geometry
      okin_restore(pr, sm);
      break;
    }
    const double f2_old = st.f2;
    if (st.mu == 0.0 && hmax <= cfg.coarse_tol) {
      // Residuals at the new point (also the reported max|r|).  When the caller will relinearise at
      // the solution anyway (exported tangents / metrics) and this step already ends the iteration,
      // the row gradients are evaluated in the same pass.
      const bool last = hmax <= cfg.fine_tol;
      if (last && !relinearise) {
        // final step of a solve that needs nothing at the solution but max|r|: residuals of the linear
        // model instead of a second row evaluation (error of second order in hmax)
        okin_linear_residuals(pr, sm, st);
        *converged = true;
        break;
      }
      okin_eval_rows(pr, sm, tval, relinearise && last, st);
      ++nfev;
      if (last) {                                // error left ~ k hmax^2: done without verification
        *gradients_at_solution = relinearise;
        *converged = true;
        break;
      }
      // Verify with a chord step h2 = -(J0^T J0)^{-1} J0^T r(x1) that reuses the factor and the row
      // gradients of the linearisation (g-only assembly, one forward/backward pass).
      okin_assemble(pr, sm, 0.0, true);
      okin_solve(pr, sm, 0, 1, false);
      const double h2 = okin_apply_step(pr, sm, 0, 1.0, true);
      if (h2 <= cfg.step_tol) {
        *converged = true;
        break;
      }
      okin_restore(pr, sm);
      // Not contracting fast enough: relinearise at the current point.
      okin_eval_rows(pr, sm, tval, true, st);
      ++nfev;
      continue;
    }
    // Damped step: ||r + J h||^2, the linear model's prediction (r[] and rg[] still hold the old point),
    // for the gain ratio below.
    double f2_model = 0.0;
    if (st.mu > 0.0) {
      okin_linear_residuals(pr, sm, st);
      f2_model = st.f2;
    }
    okin_eval_rows(pr, sm, tval, true, st);
    ++nfev;
    if (hmax <= cfg.step_tol && !gn_rejected) {
      // Tiny step under damping: drop the damping and let undamped steps confirm.  (Not after a rejected
      // undamped step: that would cycle rejected -> mu_init -> tiny -> 0 -> rejected until max_iter;
      // such a step goes through the acceptance test below, where it ends the iteration as stagnation.)
      st.mu = 0.0;
      nu = 2.0;
    } else if (st.f2 <= f2_old * (1.0 + 1e-12) + 1e-300) {
      // Accepted.  A damped step that no longer reduces ||r||^2 means the iteration sits at a
      // least-squares compromise of an unreachable target, or at a root the undamped steps overshoot
      // (MINPACK's ftol exit, reference SolverConfig.ftol); report it converged so that the residual
      // test decides exactly like solver.py:735-747.
      if (st.mu > 0.0 && f2_old - st.f2 <= 1e-7 * f2_old) { *converged = true; break; }
      if (st.mu > 0.0) {
        // Gain-ratio update (Nielsen): rho = actual / predicted reduction; mu / 3 for a step the model
        // predicted well, up to mu * 2 for one it did not.  Towards pure Gauss-Newton, but not back to it
        // once an undamped step of this solve has been rejected.
        const double rho = (f2_old - st.f2) / fmax(f2_old - f2_model, 1e-300);
        const double t = 2.0 * rho - 1.0;
        st.mu *= fmax(1.0 / 3.0, 1.0 - t * t * t);
        if (st.mu < 1e-10 && !gn_rejected) st.mu = 0.0;
      }
      nu = 2.0;
    } else {
      okin_restore(pr, sm);
      okin_eval_rows(pr, sm, tval, true, st);
      ++nfev;
      gn_rejected = gn_rejected || st.mu == 0.0;
      st.mu = st.mu > 0.0 ? st.mu * nu : cfg.mu_init;
      nu *= 2.0;
      if (st.mu > 1e12) break;
    }
    // A damped iteration (after a rejected undamped step) that used up its budget has stagnated: it
    // creeps along a weak direction towards a root or a least-squares compromise.  Report it converged,
    // like the compromise exit above, so that the residual test decides on the current point.
    if (gn_rejected && it == cfg.max_iter - 1) *converged = true;
  }
  return nfev;
}

// ---------------------------------------------------------------------------------------
// Metrics (csrc/okin_metrics.cuh holds the response kernels and record layouts).
// ---------------------------------------------------------------------------------------
// Velocity of point p along tangent j: free points read the tangent vector, fixed points are at
// rest, derived points push their inputs' velocities through the op (sensitivity.py:118-141).
// Derived inputs of derived points are supported one level deep (contact patch <- wheel centre).
OKIN_HD void okin_point_vel_base(const OkinProgram& pr, const double* sm, int p, int j, double v[3]) {
  sm = OKIN_SHARED(sm);
  v[0] = v[1] = v[2] = 0.0;
  if (p < 0) return;
  const int e = OKIN_LDG(OKIN_SHARED(okin_sec(pr, OKIN_S_POINT_ELIM)) + p);
  if (e < 0) return;
  const double* V = sm + pr.hdr[OKIN_H_OFF_VEC] + (1 + j) * 3 * pr.hdr[OKIN_H_NF] + 3 * e;
  v[0] = V[0]; v[1] = V[1]; v[2] = V[2];
}
OKIN_HD void okin_point_vel_op(const OkinProgram& pr, const double* sm, int d, const double* da, const double* db,
                               const double* dc, double v[3]) {
  sm = OKIN_SHARED(sm);
  const int32_t* rec = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP)) + d * OKIN_DOP_STRIDE;
  const int ia = OKIN_LDG(rec + 2), ib = OKIN_LDG(rec + 3), ic = OKIN_LDG(rec + 4);
  const double* pos = sm + pr.hdr[OKIN_H_OFF_POS];
  const double* par = sm + pr.hdr[OKIN_H_OFF_PAR];
  double out[3];
  okin_dop_eval(OKIN_LDG(rec + 0), par[OKIN_LDG(rec + 5)], pos + 3 * ia, pos + 3 * (ib < 0 ? ia : ib),
                pos + 3 * (ic < 0 ? ia : ic), da, db, dc, out, v);
}
OKIN_HD void okin_point_vel1(const OkinProgram& pr, const double* sm, int p, int j, double v[3]) {
  sm = OKIN_SHARED(sm);
  const int d = p < 0 ? -1 : OKIN_LDG(OKIN_SHARED(okin_sec(pr, OKIN_S_POINT_DOP)) + p);
  if (d < 0) { okin_point_vel_base(pr, sm, p, j, v); return; }
  const int32_t* rec = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP)) + d * OKIN_DOP_STRIDE;
  double da[3], db[3], dc[3];
  okin_point_vel_base(pr, sm, OKIN_LDG(rec + 2), j, da);
  okin_point_vel_base(pr, sm, OKIN_LDG(rec + 3), j, db);
  okin_point_vel_base(pr, sm, OKIN_LDG(rec + 4), j, dc);
  okin_point_vel_op(pr, sm, d, da, db, dc, v);
}
OKIN_HD void okin_point_vel(const OkinProgram& pr, const double* sm, int p, int j, double v[3]) {
  sm = OKIN_SHARED(sm);
  const int d = p < 0 ? -1 : OKIN_LDG(OKIN_SHARED(okin_sec(pr, OKIN_S_POINT_DOP)) + p);
  if (d < 0) { okin_point_vel_base(pr, sm, p, j, v); return; }
  const int32_t* rec = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP)) + d * OKIN_DOP_STRIDE;
  double da[3], db[3], dc[3];
  okin_point_vel1(pr, sm, OKIN_LDG(rec + 2), j, da);
  okin_point_vel1(pr, sm, OKIN_LDG(rec + 3), j, db);
  okin_point_vel1(pr, sm, OKIN_LDG(rec + 4), j, dc);
  okin_point_vel_op(pr, sm, d, da, db, dc, v);
}

// One generic response on T in {double, OkinDual}; vel == nullptr for plain values.
template <typename T>
OKIN_HD T okin_response(const OkinProgram& pr, const double* sm, const int32_t* rec, int j) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* dsn = sm + hdr[OKIN_H_OFF_DSN];
  const double* fc = okin_fsec(pr, OKIN_F_MCONST) + OKIN_LDG(rec + 12);
  const int rtype = OKIN_LDG(rec + 1);
  OkinV3<T> P[4];
  for (int k = 0; k < 4; ++k) {
    const int p = OKIN_LDG(rec + 2 + k);
    double v[3] = {0.0, 0.0, 0.0};
    if (p >= 0 && j >= 0) okin_point_vel(pr, sm, p, j, v);
    P[k] = okin_lift(pos + 3 * (p < 0 ? 0 : p), v, T());
  }
  const int d0 = OKIN_LDG(rec + 6), d1 = OKIN_LDG(rec + 7);
  switch (rtype) {
    case OKIN_R_COORD: return P[0].x * fc[0] + P[0].y * fc[1] + P[0].z * fc[2];
    case OKIN_R_DIST: return okin_distance(P[0], P[1]);
    case OKIN_R_CAMBER: return okin_camber_deg(P[0], P[1], fc[0]);
    case OKIN_R_TOE: return okin_toe_deg(P[0], P[1], fc[0]);
    case OKIN_R_CASTER: return okin_caster_deg(P[0], P[1]);
    case OKIN_R_KPI: return okin_kpi_deg(P[0], P[1], fc[0]);
    case OKIN_R_ROTATION: {
      const double* a = pos + 3 * OKIN_LDG(rec + 3);
      const double* b = pos + 3 * OKIN_LDG(rec + 4);
      return okin_rotation_deg(P[0], dsn + 3 * d0, a, b) * fc[0];
    }
    case OKIN_R_ROTATION_DIFF: {
      const double* a = pos + 3 * OKIN_LDG(rec + 3);
      const double* b = pos + 3 * OKIN_LDG(rec + 4);
      return okin_rotation_deg(P[0], dsn + 3 * d0, a, b) - okin_rotation_deg(P[3], dsn + 3 * d1, a, b);
    }
    case OKIN_R_MID_X: return P[0].x + (P[1].x - P[0].x) * 0.5;
    case OKIN_R_TBAR_TWIST_DEG: return okin_tbar_twist_rad(P[0], P[1], P[2]) * OKIN_RAD2DEG;
    case OKIN_R_TBAR_TWIST_DELTA: {
      const double z[3] = {0.0, 0.0, 0.0};
      const double design = okin_tbar_twist_rad(okin_lift(dsn + 3 * d0, z, 0.0), okin_lift(dsn + 3 * d1, z, 0.0),
                                                okin_lift(pos + 3 * OKIN_LDG(rec + 4), z, 0.0));
      return (okin_tbar_twist_rad(P[0], P[1], P[2]) - okin_const(design, T())) * OKIN_RAD2DEG;
    }
    case OKIN_R_TBAR_HEAVE: {
      // signed angle of the crossbar centre about (pivot, +Y) from its design position
      const T half = okin_const(0.5, T());
      const OkinV3<T> center = P[0] + okin_scale(P[1] - P[0], half);
      double dc[3];
      for (int k = 0; k < 3; ++k) dc[k] = dsn[3 * d0 + k] + (dsn[3 * d1 + k] - dsn[3 * d0 + k]) * 0.5;
      const double* pivot = pos + 3 * OKIN_LDG(rec + 4);
      const double pivot_b[3] = {pivot[0], pivot[1] + 1.0, pivot[2]};
      return okin_rotation_deg(center, dc, pivot, pivot_b);
    }
    default: return okin_const(NAN, T());
  }
}

// 19 corner state metrics of catalog.py:86-159 for one corner; one lane.
OKIN_HD void okin_corner_metrics(const OkinProgram& pr, double* sm, const int32_t* rec, double* out, double* ctx) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* dsn = sm + hdr[OKIN_H_OFF_DSN];
  const double* fc = okin_fsec(pr, OKIN_F_MCONST) + OKIN_LDG(rec + 18);
  const double side = fc[0], cg_z = fc[1], wheelbase = fc[2], bias = fc[3];
  const int flags = OKIN_LDG(rec + 19);
  const double* ai = pos + 3 * OKIN_LDG(rec + 0);
  const double* ao = pos + 3 * OKIN_LDG(rec + 1);
  const double* wc = pos + 3 * OKIN_LDG(rec + 2);
  const double* cp = pos + 3 * OKIN_LDG(rec + 3);
  const double* lo = pos + 3 * OKIN_LDG(rec + 4);
  const double* up = pos + 3 * OKIN_LDG(rec + 5);
  double* o = out + OKIN_LDG(rec + 17);
  const double z3[3] = {0.0, 0.0, 0.0};
  const OkinV3<double> AI = okin_lift(ai, z3, 0.0), AO = okin_lift(ao, z3, 0.0);
  const OkinV3<double> LO = okin_lift(lo, z3, 0.0), UP = okin_lift(up, z3, 0.0);
  o[0] = okin_camber_deg(AI, AO, side);
  o[1] = okin_caster_deg(LO, UP);
  o[2] = okin_kpi_deg(LO, UP, side);
  o[5] = okin_toe_deg(AI, AO, side);
  // steering axis / ground plane at the contact-patch height (context.py:118-141)
  const double sd[3] = {up[0] - lo[0], up[1] - lo[1], up[2] - lo[2]};
  double ax[3] = {ao[0] - ai[0], ao[1] - ai[1], ao[2] - ai[2]};
  const double ial = 1.0 / sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
  ax[0] *= ial; ax[1] *= ial; ax[2] *= ial;
  if (fabs(sd[2]) < OKIN_GEOM_EPS) {
    o[3] = NAN; o[4] = NAN;
  } else {
    const double t = (cp[2] - lo[2]) / sd[2];
    const double gp[3] = {lo[0] + t * sd[0], lo[1] + t * sd[1], lo[2] + t * sd[2]};
    const double wl = 1.0 / sqrt(ax[0] * ax[0] + ax[1] * ax[1]);
    o[3] = -((gp[0] - cp[0]) * ax[0] * wl + (gp[1] - cp[1]) * ax[1] * wl);  // scrub radius
    o[4] = gp[0] - cp[0];                                                  // mechanical trail
  }
  // instant axis = intersection of two planes n.x + d = 0 (geometric.py:216-302)
  double n1[3] = {1.0, 0.0, 0.0}, n2[3] = {0.0, 1.0, 0.0}, d1 = 0.0, d2 = 0.0;
  const int ic_kind = OKIN_LDG(rec + 6);
  bool ok = ic_kind != OKIN_IC_NONE;
  if (ok) {
    const double* a = pos + 3 * OKIN_LDG(rec + 7);
    const double* b = pos + 3 * OKIN_LDG(rec + 8);
    const double* c = pos + 3 * OKIN_LDG(rec + 9);
    const double u[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, w[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
    n1[0] = u[1] * w[2] - u[2] * w[1]; n1[1] = u[2] * w[0] - u[0] * w[2]; n1[2] = u[0] * w[1] - u[1] * w[0];
    const double m = sqrt(n1[0] * n1[0] + n1[1] * n1[1] + n1[2] * n1[2]);
    ok = ok && m >= OKIN_GEOM_EPS;
    n1[0] /= m; n1[1] /= m; n1[2] /= m;
    d1 = -(n1[0] * a[0] + n1[1] * a[1] + n1[2] * a[2]);
  }
  if (ic_kind == OKIN_IC_DW) {
    const double* a = pos + 3 * OKIN_LDG(rec + 10);
    const double* b = pos + 3 * OKIN_LDG(rec + 11);
    const double* c = pos + 3 * OKIN_LDG(rec + 12);
    const double u[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, w[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
    n2[0] = u[1] * w[2] - u[2] * w[1]; n2[1] = u[2] * w[0] - u[0] * w[2]; n2[2] = u[0] * w[1] - u[1] * w[0];
    const double m = sqrt(n2[0] * n2[0] + n2[1] * n2[1] + n2[2] * n2[2]);
    ok = ok && m >= OKIN_GEOM_EPS;
    n2[0] /= m; n2[1] /= m; n2[2] /= m;
    d2 = -(n2[0] * a[0] + n2[1] * a[1] + n2[2] * a[2]);
  } else if (ic_kind == OKIN_IC_MAC) {  // plane through the strut top normal to the strut axis (macpherson.py:346-355)
    const double* ball = pos + 3 * OKIN_LDG(rec + 9);
    const double* top = pos + 3 * OKIN_LDG(rec + 10);
    n2[0] = top[0] - ball[0]; n2[1] = top[1] - ball[1]; n2[2] = top[2] - ball[2];
    const double m = sqrt(n2[0] * n2[0] + n2[1] * n2[1] + n2[2] * n2[2]);
    n2[0] /= m; n2[1] /= m; n2[2] /= m;
    d2 = -(n2[0] * top[0] + n2[1] * top[1] + n2[2] * top[2]);
  }
  double dir[3] = {n1[1] * n2[2] - n1[2] * n2[1], n1[2] * n2[0] - n1[0] * n2[2], n1[0] * n2[1] - n1[1] * n2[0]};
  const double dm2 = dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2];
  ok = ok && dm2 >= OKIN_GEOM_EPS * OKIN_GEOM_EPS;
  const double q[3] = {d2 * n1[0] - d1 * n2[0], d2 * n1[1] - d1 * n2[1], d2 * n1[2] - d1 * n2[2]};
  const double pt[3] = {(q[1] * dir[2] - q[2] * dir[1]) / dm2, (q[2] * dir[0] - q[0] * dir[2]) / dm2,
                        (q[0] * dir[1] - q[1] * dir[0]) / dm2};
  const double idm = 1.0 / sqrt(dm2);
  dir[0] *= idm; dir[1] *= idm; dir[2] *= idm;
  const bool sv_ok = ok && fabs(dir[1]) >= OKIN_GEOM_EPS;  // y = wc.y plane (double_wishbone.py:352-376)
  const bool fv_ok = ok && fabs(dir[0]) >= OKIN_GEOM_EPS;  // x = wc.x plane (:405-431)
  double svic[3] = {NAN, NAN, NAN}, fvic[3] = {NAN, NAN, NAN};
  if (sv_ok) {
    const double t = (wc[1] - pt[1]) / dir[1];
    for (int k = 0; k < 3; ++k) svic[k] = pt[k] + t * dir[k];
  }
  if (fv_ok) {
    const double t = (wc[0] - pt[0]) / dir[0];
    for (int k = 0; k < 3; ++k) fvic[k] = pt[k] + t * dir[k];
  }
  o[6] = svic[0]; o[7] = svic[2];
  o[8] = sv_ok ? svic[0] - cp[0] : NAN;
  o[9] = fvic[1]; o[10] = fvic[2];
  if (fv_ok) {
    const double dy = fvic[1] - cp[1], dz = fvic[2] - cp[2];
    const double sgn = dy > 0.0 ? 1.0 : (dy < 0.0 ? -1.0 : 0.0);
    o[11] = sqrt(dy * dy + dz * dz) * (-side * sgn);
  } else {
    o[11] = NAN;
  }
  o[12] = wc[2] - dsn[3 * OKIN_LDG(rec + 15) + 2];
  o[13] = fabs(cp[1]);
  const int dt = OKIN_LDG(rec + 13), db = OKIN_LDG(rec + 14);
  if (dt >= 0) {
    const double* a = pos + 3 * dt;
    const double* b = pos + 3 * db;
    o[14] = sqrt((a[0] - b[0]) * (a[0] - b[0]) + (a[1] - b[1]) * (a[1] - b[1]) + (a[2] - b[2]) * (a[2] - b[2]));
  } else {
    o[14] = NAN;
  }
  // anti geometry (anti_geometry.py:33-206)
  const double run_cp = svic[0] - cp[0];
  o[15] = (sv_ok && fabs(run_cp) >= OKIN_GEOM_EPS) ? atan((svic[2] - cp[2]) / run_cp) * OKIN_RAD2DEG : NAN;
  const double height = cg_z - cp[2];
  const bool h_ok = height > OKIN_GEOM_EPS;
  o[16] = NAN; o[17] = NAN; o[18] = NAN;
  if ((flags & OKIN_MF_FRONT) && (flags & OKIN_MF_HAS_BIAS) && sv_ok && fabs(run_cp) >= OKIN_GEOM_EPS && h_ok)
    o[16] = 100.0 * bias * (wheelbase / height) * ((svic[2] - cp[2]) / (cp[0] - svic[0]));
  if ((flags & OKIN_MF_REAR) && (flags & OKIN_MF_HAS_BIAS) && sv_ok && fabs(run_cp) >= OKIN_GEOM_EPS && h_ok)
    o[17] = 100.0 * (1.0 - bias) * (wheelbase / height) * ((svic[2] - cp[2]) / run_cp);
  if ((flags & OKIN_MF_DRIVEN_HERE) && sv_ok && h_ok) {
    const double run = (flags & OKIN_MF_FRONT) ? wc[0] - svic[0] : svic[0] - wc[0];
    if (fabs(run) >= OKIN_GEOM_EPS) o[18] = 100.0 * (wheelbase / height) * ((svic[2] - wc[2]) / run);
  }
  ctx[0] = fvic[1]; ctx[1] = fvic[2]; ctx[2] = fv_ok ? 1.0 : 0.0;
}

// All metric columns of one state into out[NM].
template <typename Dummy = void>
OKIN_FN void okin_metrics(const OkinProgram& pr, double* sm, double* out) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nmc = hdr[OKIN_H_NMC], nmop = hdr[OKIN_H_NMOP];
  const int32_t* corners = OKIN_SHARED(okin_sec(pr, OKIN_S_MCORNER));
  const int32_t* mops = OKIN_SHARED(okin_sec(pr, OKIN_S_MOP));
  double* ctx = sm + hdr[OKIN_H_OFF_MCTX];
  const int nt = hdr[OKIN_H_NT];
  OKIN_PHASE_BEGIN
  if (lane < nmc) okin_corner_metrics(pr, sm, corners + lane * OKIN_MCORNER_STRIDE, out, ctx + 4 * lane);
  for (int t = lane - nmc; t < nmop; t += 32 - nmc) {
    if (t < 0) continue;
    const int32_t* rec = mops + t * OKIN_MOP_STRIDE;
    double value;
    if (OKIN_LDG(rec + 0) == OKIN_MOP_VALUE) {
      value = okin_response<double>(pr, sm, rec, -1);
    } else {
      // select the tangent with the strongest driver rate (derivatives.py:273-309)
      const int dp = OKIN_LDG(rec + 8), da = OKIN_LDG(rec + 9), mask = OKIN_LDG(rec + 10);
      int best = -1;
      double strongest = 0.0, best_rate = 0.0;
      bool tied = false;
      for (int j = 0; j < nt; ++j) {
        if (!((mask >> j) & 1)) continue;
        double v[3];
        okin_point_vel(pr, sm, dp, j, v);
        const double rate = fabs(v[da]);
        if (rate > strongest + OKIN_GEOM_EPS) { best = j; strongest = rate; best_rate = v[da]; tied = false; }
        else if (rate >= OKIN_GEOM_EPS && fabs(rate - strongest) <= OKIN_GEOM_EPS) tied = true;
      }
      if (best < 0 || strongest < OKIN_GEOM_EPS) {
        value = NAN;            // no driver tangent: the reference's None
      } else if (tied) {
        value = INFINITY;       // equal-strength drivers: the reference raises (derivatives.py:299-304)
      } else {
        const OkinDual resp = okin_response<OkinDual>(pr, sm, rec, best);
        value = resp.d / best_rate;
      }
    }
    out[OKIN_LDG(rec + 11)] = value;
  }
  OKIN_PHASE_END
  if (hdr[OKIN_H_NMAXLE]) {
    // axle-level state metrics (axle_metrics.py:18-95)
    const int32_t* rec = OKIN_SHARED(okin_sec(pr, OKIN_S_MAXLE));
    const double* pos = sm + hdr[OKIN_H_OFF_POS];
    const double* dsn = sm + hdr[OKIN_H_OFF_DSN];
    OKIN_PHASE_BEGIN
    if (lane == 0) {
      const double* wcL = pos + 3 * OKIN_LDG(rec + 0);
      const double* wcR = pos + 3 * OKIN_LDG(rec + 1);
      const double* cpL = pos + 3 * OKIN_LDG(rec + 2);
      const double* cpR = pos + 3 * OKIN_LDG(rec + 3);
      const double lz = wcL[2] - dsn[3 * OKIN_LDG(rec + 4) + 2], rz = wcR[2] - dsn[3 * OKIN_LDG(rec + 5) + 2];
      const double clz = cpL[2] - dsn[3 * OKIN_LDG(rec + 6) + 2], crz = cpR[2] - dsn[3 * OKIN_LDG(rec + 7) + 2];
      const double track = fabs(cpL[1] - cpR[1]);
      double* o = out + OKIN_LDG(rec + 10);
      o[0] = 0.5 * (lz + rz);
      o[1] = atan2(lz - rz, track) * OKIN_RAD2DEG;
      o[2] = -0.5 * (clz + crz);
      o[3] = track;
      o[4] = NAN; o[5] = NAN;
      if (ctx[2] != 0.0 && ctx[6] != 0.0) {
        const double l2 = ctx[0] - cpL[1], l3 = ctx[1] - cpL[2], r2 = ctx[4] - cpR[1], r3 = ctx[5] - cpR[2];
        const double den = l2 * r3 - l3 * r2;
        if (fabs(den) >= OKIN_GEOM_EPS) {
          const double par = ((cpR[1] - cpL[1]) * r3 - (cpR[2] - cpL[2]) * r2) / den;
          o[4] = cpL[1] + par * l2;
          o[5] = cpL[2] + par * l3;
        }
      }
      const int rack = OKIN_LDG(rec + 8);
      o[6] = rack >= 0 ? pos[3 * rack + 1] - dsn[3 * OKIN_LDG(rec + 9) + 1] : NAN;
    }
    OKIN_PHASE_END
  }
}



// ---------------------------------------------------------------------------------------
// Sweep diagnostics.  Topology checks are evaluated per state inside the sweep (the state is in
// shared memory); the continuity check needs a point's whole displacement history and runs as a
// second pass over the instance's position rows (okin_continuity).
// ---------------------------------------------------------------------------------------
#define OKIN_TRANSMISSION_WARN 0.15   // axle/mechanisms.py:70
#define OKIN_JUMP_FLOOR_MM 5.0        // diagnostics.py:30-31
#define OKIN_JUMP_MEDIAN_FACTOR 4.0

OKIN_HD double okin_stp(const double* o, const double* a, const double* b, const double* c) {
  const double ax = a[0] - o[0], ay = a[1] - o[1], az = a[2] - o[2];
  const double bx = b[0] - o[0], by = b[1] - o[1], bz = b[2] - o[2];
  const double cx = c[0] - o[0], cy = c[1] - o[1], cz = c[2] - o[2];
  return ax * (by * cz - bz * cy) + ay * (bz * cx - bx * cz) + az * (bx * cy - by * cx);
}

// One state's diagnostic row: flags + topology columns (the jump columns are zeroed here and
// filled by okin_continuity).  ok: the state was accepted; status: the instance status so far.
template <typename Dummy = void>
OKIN_FN void okin_diagnostics(const OkinProgram& pr, double* sm, double* row, bool ok, int status) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nd = hdr[OKIN_H_NDIAG], nop = hdr[OKIN_H_NDGOP];
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* dsn = sm + hdr[OKIN_H_OFF_DSN];
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < nd; t += 32) row[t] = t == 3 ? -1.0 : (t < OKIN_DIAG_BASE || ok ? 0.0 : NAN);
  red[lane] = 0.0;
  OKIN_PHASE_END
  if (ok) {
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < nop; t += 32) {
      const int32_t* rec = okin_sec(pr, OKIN_S_DGOP) + t * OKIN_DGOP_STRIDE;
      const int col = OKIN_LDG(rec + 6);
      int flags = 0;
      if (OKIN_LDG(rec) == OKIN_DG_CHIRALITY) {
        const double* a = pos + 3 * OKIN_LDG(rec + 1);
        const double* b = pos + 3 * OKIN_LDG(rec + 2);
        const double* r = pos + 3 * OKIN_LDG(rec + 3);
        const double* u = pos + 3 * OKIN_LDG(rec + 4);
        const double vol = okin_stp(a, b, r, u);
        const double design = okin_stp(dsn + 3 * OKIN_LDG(rec + 7), dsn + 3 * OKIN_LDG(rec + 8),
                                       dsn + 3 * OKIN_LDG(rec + 9), dsn + 3 * OKIN_LDG(rec + 10));
        double n[3] = {0.0, 0.0, 0.0};
        const double* q[3] = {b, r, u};
        for (int k = 0; k < 3; ++k)
          n[k] = sqrt((q[k][0] - a[0]) * (q[k][0] - a[0]) + (q[k][1] - a[1]) * (q[k][1] - a[1]) +
                      (q[k][2] - a[2]) * (q[k][2] - a[2]));
        const double scale = n[0] * n[1] * n[2];
        const double margin = scale <= OKIN_GEOM_EPS ? 0.0 : vol / scale;
        const int sv = (vol > 0.0) - (vol < 0.0), sd = (design > 0.0) - (design < 0.0);
        if (fabs(margin) <= OKIN_GEOM_EPS) flags = OKIN_DIAG_CHIRALITY_BOUNDARY;
        else if (sv != sd) flags = OKIN_DIAG_CHIRALITY_INVERTED;
        row[col] = vol;
        row[col + 1] = margin;
        row[col + 2] = flags == OKIN_DIAG_CHIRALITY_BOUNDARY ? 1.0 : (flags ? 2.0 : 0.0);
      } else {  // OKIN_DG_TRANSMISSION (axle/mechanisms.py:143-163)
        const double* drv = pos + 3 * OKIN_LDG(rec + 1);
        const double* a = pos + 3 * OKIN_LDG(rec + 2);
        const double* b = pos + 3 * OKIN_LDG(rec + 3);
        const double* l0 = pos + 3 * OKIN_LDG(rec + 4);
        const double* l1 = pos + 3 * OKIN_LDG(rec + 5);
        double ax[3], lk[3], rad[3];
        for (int k = 0; k < 3; ++k) { ax[k] = b[k] - a[k]; lk[k] = l1[k] - l0[k]; rad[k] = drv[k] - a[k]; }
        const double an = sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
        const double ln = sqrt(lk[0] * lk[0] + lk[1] * lk[1] + lk[2] * lk[2]);
        double margin = NAN;
        if (an != 0.0 && ln != 0.0) {
          for (int k = 0; k < 3; ++k) ax[k] /= an;
          const double along = rad[0] * ax[0] + rad[1] * ax[1] + rad[2] * ax[2];
          for (int k = 0; k < 3; ++k) rad[k] -= ax[k] * along;
          const double tg[3] = {ax[1] * rad[2] - ax[2] * rad[1], ax[2] * rad[0] - ax[0] * rad[2],
                                ax[0] * rad[1] - ax[1] * rad[0]};
          const double tn = sqrt(tg[0] * tg[0] + tg[1] * tg[1] + tg[2] * tg[2]);
          if (tn != 0.0) margin = fabs((lk[0] * tg[0] + lk[1] * tg[1] + lk[2] * tg[2]) / (ln * tn));
        }
        if (margin < OKIN_TRANSMISSION_WARN) flags = OKIN_DIAG_TRANSMISSION;
        row[col] = margin;
      }
      red[t & 31] = (double)((int)red[t & 31] | flags);
    }
    OKIN_PHASE_END
  }
  OKIN_PHASE_BEGIN
  if (lane == 0) {
    int flags = 0;
    for (int k = 0; k < 32; ++k) flags |= (int)red[k];
    if (!ok && status == OKIN_STATUS_RESIDUAL_REJECTED) flags |= OKIN_DIAG_RESIDUAL;
    else if (!ok && status != OKIN_STATUS_OK) flags |= OKIN_DIAG_NOT_CONVERGED;
    row[0] = (double)flags;
  }
  OKIN_PHASE_END
}

// Continuity check of one instance (diagnostics.py:176-226): per free point the Euclidean
// displacement of every sweep transition, the median of the non-zero ones, threshold
// max(5 mm, 4 x median); displacements above it are jumps into the later step.
//   scratch   [32][stride] doubles + [32] thresholds + [32] slots (stride >= n_steps - 1)
//   positions [n_steps][NOUT*3] of this instance; n_ok solved states lead the rows
//   diag      [n_steps][NDIAG] rows of this instance (columns 0..4 updated)
//   jumps     optional [n_steps][NF]: row 0 = each point's threshold, row s>0 = displacement into
//             step s where it exceeded the threshold, else 0
template <typename Dummy = void>
OKIN_HD void okin_continuity(const OkinProgram& pr, double* scratch, int stride, const double* positions,
                             int n_steps, int n_ok, double* diag, double* jumps) {
  const int32_t* hdr = pr.hdr;   // global memory in the continuity kernel
  const int nf = hdr[OKIN_H_NF], nout3 = 3 * hdr[OKIN_H_NOUT], nd = hdr[OKIN_H_NDIAG];
  const int32_t* free_out = okin_sec(pr, OKIN_S_FREE_OUT);
  const int ntr = n_ok > 1 ? n_ok - 1 : 0;
  double* thr = scratch + 32 * stride;
  double* slots = thr + 32;
  if (jumps) {
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < n_steps * nf; t += 32) jumps[t] = 0.0;
    OKIN_PHASE_END
  }
  for (int base = 0; base < nf; base += 32) {
    OKIN_PHASE_BEGIN     // lane = free point: displacement history, median, threshold
    const int k = base + lane;
    const int slot = k < nf ? OKIN_LDG(free_out + k) : -1;
    double* d = scratch + lane * stride;
    double threshold = INFINITY;
    if (slot >= 0 && ntr > 0) {
      const double* p = positions + 3 * slot;
      double px = p[0], py = p[1], pz = p[2];
      int nz = 0;
      for (int t = 0; t < ntr; ++t) {
        const double* c = p + (size_t)(t + 1) * nout3;
        const double dx = c[0] - px, dy = c[1] - py, dz = c[2] - pz;
        d[t] = sqrt(dx * dx + dy * dy + dz * dz);
        nz += d[t] > 0.0;
        px = c[0]; py = c[1]; pz = c[2];
      }
      double med = 0.0;
      if (nz > 0) {  // statistics.median of the non-zero displacements
        const int lo = (nz - 1) / 2, hi = nz / 2;
        double vlo = 0.0, vhi = 0.0;
        for (int i = 0; i < ntr; ++i) {
          const double di = d[i];
          if (!(di > 0.0)) continue;
          int rank = 0;
          for (int j = 0; j < ntr; ++j) {
            const double dj = d[j];
            rank += (dj > 0.0) && (dj < di || (dj == di && j < i));
          }
          if (rank == lo) vlo = di;
          if (rank == hi) vhi = di;
        }
        med = 0.5 * (vlo + vhi);
      }
      threshold = fmax(OKIN_JUMP_FLOOR_MM, OKIN_JUMP_MEDIAN_FACTOR * med);
      if (jumps) {
        jumps[k] = threshold;
        for (int t = 0; t < ntr; ++t)
          if (d[t] > threshold) jumps[(size_t)(t + 1) * nf + k] = d[t];
      }
    }
    thr[lane] = threshold;
    slots[lane] = (double)slot;
    OKIN_PHASE_END
    OKIN_PHASE_BEGIN     // lane = transition: fold this group of points into the step's row
    OKIN_LANE_LOOP
    for (int t = lane; t < ntr; t += 32) {
      double* row = diag + (size_t)(t + 1) * nd;
      double count = row[1], worst = row[2], wslot = row[3], wthr = row[4];
      for (int q = 0; q < 32; ++q) {
        if (slots[q] < 0.0) continue;
        const double v = scratch[q * stride + t];
        if (v > thr[q]) {
          count += 1.0;
          if (v > worst) { worst = v; wslot = slots[q]; wthr = thr[q]; }
        }
      }
      if (count > row[1]) {
        row[0] = (double)((int)row[0] | OKIN_DIAG_JUMP);
        row[1] = count; row[2] = worst; row[3] = wslot; row[4] = wthr;
      }
    }
    OKIN_PHASE_END
  }
}

// z = L^T x (lt) or x = L z (plain) with the block factor; returns |result|^2 (warp-uniform).
template <typename Dummy = void>
OKIN_FN double okin_factor_multiply(const OkinProgram& pr, double* sm, const double* src, double* dst, bool lt) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nf = hdr[OKIN_H_NF];
  const int32_t* ptr = okin_sec(pr, lt ? OKIN_S_BW_PTR : OKIN_S_FW_PTR);
  const int32_t* con = okin_sec(pr, lt ? OKIN_S_BW_CON : OKIN_S_FW_CON);
  const int32_t* doffs = OKIN_SHARED(okin_sec(pr, OKIN_S_DIAG_OFF));
  const double* Lb = sm;
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  double acc = 0.0;
  OKIN_LANE_LOOP
  for (int j = lane; j < nf; j += 32) {
    const double* f = sm + OKIN_LDG(doffs + j);   // {l00,l10,l11,l20,l21,l22,...}
    const double x0 = src[3 * j], x1 = src[3 * j + 1], x2 = src[3 * j + 2];
    double t0, t1, t2;
    if (lt) { t0 = f[0] * x0 + f[1] * x1 + f[3] * x2; t1 = f[2] * x1 + f[4] * x2; t2 = f[5] * x2; }
    else { t0 = f[0] * x0; t1 = f[1] * x0 + f[2] * x1; t2 = f[3] * x0 + f[4] * x1 + f[5] * x2; }
    for (int q = OKIN_LDG(ptr + j); q < OKIN_LDG(ptr + j + 1); ++q) {
      const uint32_t w = (uint32_t)OKIN_LDG(con + q);
      const double* B = Lb + (w >> 16);
      const double* y = src + (w & 0xffffu);
      if (lt) {
        t0 += B[0] * y[0] + B[3] * y[1] + B[6] * y[2];
        t1 += B[1] * y[0] + B[4] * y[1] + B[7] * y[2];
        t2 += B[2] * y[0] + B[5] * y[1] + B[8] * y[2];
      } else {
        t0 += B[0] * y[0] + B[1] * y[1] + B[2] * y[2];
        t1 += B[3] * y[0] + B[4] * y[1] + B[5] * y[2];
        t2 += B[6] * y[0] + B[7] * y[1] + B[8] * y[2];
      }
    }
    dst[3 * j] = t0; dst[3 * j + 1] = t1; dst[3 * j + 2] = t2;
    acc += t0 * t0 + t1 * t1 + t2 * t2;
  }
  red[lane] = acc;
  OKIN_PHASE_END
  return okin_red_sum(red);
}

// v *= s; returns nothing.  |v|^2 helper below.
template <typename Dummy = void>
OKIN_FN double okin_scale_norm2(const OkinProgram& pr, double* sm, double* v, double s) {
  sm = OKIN_SHARED(sm);
  const int n = 3 * pr.hdr[OKIN_H_NF];
  double* red = sm + pr.hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  double acc = 0.0;
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) {
    const double x = v[u] * s;
    v[u] = x;
    acc += x * x;
  }
  red[lane] = acc;
  OKIN_PHASE_END
  return okin_red_sum(red);
}

// a . b (warp-uniform).
template <typename Dummy = void>
OKIN_FN double okin_dot(const OkinProgram& pr, double* sm, const double* a, const double* b) {
  sm = OKIN_SHARED(sm);
  const int n = 3 * pr.hdr[OKIN_H_NF];
  double* red = sm + pr.hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  double acc = 0.0;
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) acc += a[u] * b[u];
  red[lane] = acc;
  OKIN_PHASE_END
  return okin_red_sum(red);
}

template <typename Dummy = void>
OKIN_FN void okin_copy(const OkinProgram& pr, double* dst, const double* src) {
  const int n = 3 * pr.hdr[OKIN_H_NF];
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) dst[u] = src[u];
  OKIN_PHASE_END
}

struct OkinGram2 { double aa, ab, bb; };

// Gram-Schmidt on the pair {a, b} in place; returns their Gram matrix from before.
template <typename Dummy = void>
OKIN_FN OkinGram2 okin_orthonormalise2(const OkinProgram& pr, double* sm, double* a, double* b) {
  sm = OKIN_SHARED(sm);
  const int n = 3 * pr.hdr[OKIN_H_NF];
  double* red = sm + pr.hdr[OKIN_H_OFF_RED];
  OkinGram2 g;
  g.aa = okin_dot(pr, sm, a, a);
  g.ab = okin_dot(pr, sm, a, b);
  const double p = g.ab / g.aa, s = 1.0 / sqrt(g.aa);
  OKIN_PHASE_BEGIN
  double acc = 0.0;
  OKIN_LANE_LOOP
  for (int u = lane; u < n; u += 32) {
    const double w = b[u] - p * a[u];
    b[u] = w;
    a[u] *= s;
    acc += w * w;
  }
  red[lane] = acc;
  OKIN_PHASE_END
  const double bb = okin_red_sum(red);
  g.bb = bb + p * g.ab;
  okin_scale_norm2(pr, sm, b, 1.0 / sqrt(bb));
  return g;
}

// Largest eigenvalue of the symmetric [[a, b], [b, d]] and its unit eigenvector (c0, c1).
OKIN_HD double okin_sym2_top(double a, double b, double d, double* c0, double* c1) {
  const double h = 0.5 * (a - d), r = sqrt(h * h + b * b);
  const double u = h >= 0.0 ? h + r : b, v = h >= 0.0 ? b : r - h;   // (t - d, b) or (b, t - a)
  const double nrm = sqrt(u * u + v * v);
  *c0 = nrm > 0.0 ? u / nrm : 1.0;
  *c1 = nrm > 0.0 ? v / nrm : 0.0;
  return 0.5 * (a + d) + r;
}

// Numerical health of the tangent system at the current factorisation (TangentSolveInfo,
// sensitivity.py:42-55, :97-113): the extreme singular values of the pinned Jacobian are the
// square roots of the extreme eigenvalues of A = L L^T.  sigma_max by subspace iteration with
// A (the factor), sigma_min by subspace iteration with A^{-1} (the triangular solves), each on
// two vectors with a Rayleigh-Ritz step: the extreme eigenvalues of the shipped mechanisms come
// in near-degenerate pairs (left / right of an axle: 2e-5 .. 2e-2 apart), which a single vector
// separates only over thousands of steps, while two vectors span the pair and converge at the
// ratio to the third eigenvalue.  The Ritz values are estimates from inside (sigma_max from
// below, sigma_min from above).  Each iteration stops once the residual of its top Ritz pair
// (theta, u), |B u - theta u|^2 = |B u|^2 - theta^2 (B = A or A^{-1}), is below
// OKIN_HEALTH_TOL * theta: an eigenvalue of B then lies within that distance of theta, so the
// eigenvalue error is at most OKIN_HEALTH_TOL relative however close its neighbours are.
// out2 = {sigma_min, sigma_max / sigma_min}.  Scratch: the row-gradient storage (dead until the
// next row evaluation; two vectors) and vec[0] (staging of one vector).
#define OKIN_HEALTH_TOL 1e-5
#define OKIN_HEALTH_MAX_ITERS 200
template <typename Dummy = void>
OKIN_FN void okin_tangent_health(const OkinProgram& pr, double* sm, bool notpd, double* out2) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int n = 3 * hdr[OKIN_H_NF];
  double* x1 = sm + hdr[OKIN_H_OFF_RG];
  double* x2 = x1 + n;
  double* v0 = sm + hdr[OKIN_H_OFF_VEC];
  const double tol2 = OKIN_HEALTH_TOL * OKIN_HEALTH_TOL;
  double theta[2] = {0.0, 0.0};     // top Ritz values of A and of A^{-1}
  for (int inverse = 0; inverse < 2 && !notpd; ++inverse) {
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int u = lane; u < n; u += 32) {
      // deterministic start vectors: one positive, one signed
      const uint32_t hsh = ((uint32_t)u + 1u) * 2654435761u;
      x1[u] = 1.0 + 0.37 * (double)((hsh >> 16) & 0xffu) / 256.0;
      x2[u] = (double)((hsh >> 12) & 0xffffu) / 65536.0 - 0.5;
    }
    OKIN_PHASE_END
    double th = 0.0, c0 = 1.0, c1 = 0.0;
    for (int it = 0; it < OKIN_HEALTH_MAX_ITERS; ++it) {
      // {x1, x2} = B X of the previous iteration: its Gram matrix gives |B u|^2 = c^T G c
      const OkinGram2 g = okin_orthonormalise2(pr, sm, x1, x2);
      if (it > 0) {
        const double r2 = c0 * c0 * g.aa + 2.0 * c0 * c1 * g.ab + c1 * c1 * g.bb - th * th;
        if (!(r2 > tol2 * th * th)) break;   // (NaN stops too)
      }
      double h11, h12, h22;     // X^T B X, with X <- B X in place
      if (!inverse) {
        h11 = okin_factor_multiply(pr, sm, x1, v0, true);     // |L^T x1|^2
        okin_factor_multiply(pr, sm, v0, x1, false);          // x1 <- A x1
        h12 = okin_dot(pr, sm, x1, x2);
        h22 = okin_factor_multiply(pr, sm, x2, v0, true);
        okin_factor_multiply(pr, sm, v0, x2, false);
      } else {
        okin_copy(pr, v0, x1);
        okin_solve(pr, sm, 0, 1, false);                      // v0 <- A^{-1} x1
        h11 = okin_dot(pr, sm, x1, v0);
        h12 = okin_dot(pr, sm, x2, v0);
        okin_copy(pr, x1, v0);
        okin_copy(pr, v0, x2);
        okin_solve(pr, sm, 0, 1, false);
        h22 = okin_dot(pr, sm, x2, v0);
        okin_copy(pr, x2, v0);
      }
      th = okin_sym2_top(h11, h12, h22, &c0, &c1);
    }
    theta[inverse] = th;
  }
  const double smax2 = theta[0], smin2 = 1.0 / theta[1];
  const bool good = !notpd && smin2 == smin2 && smin2 > 0.0 && smin2 < INFINITY && smax2 == smax2;
  OKIN_PHASE_BEGIN
  if (lane == 0) {
    out2[0] = good ? sqrt(smin2) : 0.0;
    out2[1] = good ? sqrt(smax2 / smin2) : INFINITY;
  }
  OKIN_PHASE_END
}

// ---------------------------------------------------------------------------------------
// Hardpoint sensitivities: d pos_o / d p_k for the hardpoint coordinates p_k listed in OKIN_S_SENS_IN
// (k = 3 * input slot + axis), params held fixed.  At an accepted state x*(p),
//   dx*/dp_k = -A^{-1} J_x^T dR/dp_k,   A = J_x^T J_x the factor the tangents use (Gauss-Newton: the
//   sum r_i Hess(r_i) is dropped, as for the tangents),
//   dR/dp_k = (dR/dpos) (dpos/dp_k)|_x + (dR/dc) (dc/dp_k),
// where c are the per-instance design constants (okin_setup rules) and derived-op parameters depend on
// p through the design pose.  The part that depends on p alone (dc/dp, dpar/dp) is evaluated once per
// instance at the design pose; the rest per accepted state, after every other output of the state.
// Per-warp scratch in global memory (okin_sens_ws_doubles):
//   dcst [NSENS][NCST]   dc/dp_k of every per-instance constant (0 for explicit ones)
//   dpar [NSENS][NPAR]   d(derived-op parameter)/dp_k
//   grad [NROW][13]      dR/d(row point s), s = 0..3, and R of every least-squares row at the state
//   tan  [3P]            tangent of every point for the column being processed
// ---------------------------------------------------------------------------------------
OKIN_HD const int32_t* okin_sec_cold(const OkinProgram& pr, int s) { return pr.ibc + pr.hdr[OKIN_H_SEC0 + 2 * s]; }
OKIN_HD size_t okin_sens_ws_doubles(const int32_t* hdr) {
  return (size_t)hdr[OKIN_H_NSENS] * (hdr[OKIN_H_NCST] + hdr[OKIN_H_NPAR]) + 13 * (size_t)hdr[OKIN_H_NROW] +
         3 * (size_t)hdr[OKIN_H_P];
}

// d out / d par of a derived op: the unit direction its parameter scales (okin_dop_eval).
OKIN_HD void okin_dop_par_dir(int op, const double* a, const double* b, const double* c, double dir[3]) {
  dir[0] = dir[1] = dir[2] = 0.0;
  if (op == OKIN_DOP_MIDPOINT) return;
  const double z[3] = {0.0, 0.0, 0.0};
  double v[3], u[3], du[3], il;
  if (op == OKIN_DOP_ALONG_LINE) {
    for (int k = 0; k < 3; ++k) v[k] = b[k] - a[k];
    okin_unit_jvp(v, z, dir, du, &il);
    return;
  }
  for (int k = 0; k < 3; ++k) v[k] = c[k] - b[k];
  okin_unit_jvp(v, z, u, du, &il);
  const double s = -u[2];
  double w[3] = {-s * u[0], -s * u[1], -s * u[2] - 1.0};
  okin_unit_jvp(w, z, dir, du, &il);
}

// Tangent of every point along hardpoint coordinate `coord` into tan[3P], one derived level per
// phase.  Fixed points move with their hardpoint (e_k); free points take free[] (elimination order)
// when given, their hardpoint when `design` (the design pose is the authored one), else stay;
// derived points push their inputs' tangents and dpar[] through the op at the current pos[].  An input
// slot holding a derived point's authored position acts only through dpar.
template <typename Dummy = void>
OKIN_FN void okin_sens_points(const OkinProgram& pr, double* sm, int coord, const double* dpar, const double* free,
                              bool design, double* tan) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int np = hdr[OKIN_H_P];
  const int32_t* kind = okin_sec(pr, OKIN_S_POINT_KIND);
  const int32_t* pelim = OKIN_SHARED(okin_sec(pr, OKIN_S_POINT_ELIM));
  const int moved = OKIN_LDG(okin_sec(pr, OKIN_S_IN_POINT) + coord / 3), axis = coord % 3;
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < 3 * np; t += 32) {
    const int q = t / 3, kq = OKIN_LDG(kind + q);
    double v = 0.0;
    if (kq == OKIN_PT_FIXED || (kq == OKIN_PT_FREE && design)) v = (q == moved && t % 3 == axis) ? 1.0 : 0.0;
    else if (kq == OKIN_PT_FREE && free) v = free[3 * OKIN_LDG(pelim + q) + t % 3];
    tan[t] = v;
  }
  OKIN_PHASE_END
  const int32_t* dop = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP));
  const int32_t* lev = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP_LEV));
  const int nlev = okin_sec_len(pr, OKIN_S_DOP_LEV) - 1;
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* par = sm + hdr[OKIN_H_OFF_PAR];
  for (int lv = 0; lv < nlev; ++lv) {
    const int b = OKIN_LDG(lev + lv), e = OKIN_LDG(lev + lv + 1);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int d = b + lane; d < e; d += 32) {
      const int32_t* rec = dop + d * OKIN_DOP_STRIDE;
      const int op = OKIN_LDG(rec + 0), pi = OKIN_LDG(rec + 5);
      const int ia = OKIN_LDG(rec + 2), ib = OKIN_LDG(rec + 3) < 0 ? ia : OKIN_LDG(rec + 3);
      const int ic = OKIN_LDG(rec + 4) < 0 ? ia : OKIN_LDG(rec + 4);
      double out[3], dout[3], dir[3];
      okin_dop_eval(op, par[pi], pos + 3 * ia, pos + 3 * ib, pos + 3 * ic, tan + 3 * ia, tan + 3 * ib, tan + 3 * ic,
                    out, dout);
      okin_dop_par_dir(op, pos + 3 * ia, pos + 3 * ib, pos + 3 * ic, dir);
      const double dp = dpar[pi];
      double* o = tan + 3 * OKIN_LDG(rec + 1);
      o[0] = dout[0] + dp * dir[0]; o[1] = dout[1] + dp * dir[1]; o[2] = dout[2] + dp * dir[2];
    }
    OKIN_PHASE_END
  }
}

// Once per instance, at the design pose okin_setup left in pos[]: dpar/dp_k and dc/dp_k of every
// sensitivity column (forward mode through the okin_setup rules).
template <typename Dummy = void>
OKIN_FN void okin_sens_setup(const OkinProgram& pr, double* sm, const double* __restrict__ hardpoints, double* ws) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nsens = hdr[OKIN_H_NSENS], ncst = hdr[OKIN_H_NCST], npar = hdr[OKIN_H_NPAR];
  const int ndop = hdr[OKIN_H_NDOP], nls = hdr[OKIN_H_NROW];
  const int32_t* sens_in = okin_sec_cold(pr, OKIN_S_SENS_IN);
  const int32_t* in_point = okin_sec(pr, OKIN_S_IN_POINT);
  const int32_t* dop = OKIN_SHARED(okin_sec(pr, OKIN_S_DOP));
  const int32_t* par_mode = okin_sec(pr, OKIN_S_PAR_MODE);
  const int32_t* rows = okin_sec(pr, OKIN_S_ROW);
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* cst = sm + hdr[OKIN_H_OFF_CST];
  double* tan = ws + (size_t)nsens * (ncst + npar) + 13 * (size_t)nls;
  for (int k = 0; k < nsens; ++k) {
    const int coord = OKIN_LDG(sens_in + k), moved = OKIN_LDG(in_point + coord / 3), axis = coord % 3;
    double* dpar = ws + (size_t)nsens * ncst + (size_t)k * npar;
    double* dc_all = ws + (size_t)k * ncst;
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int d = lane; d < ndop; d += 32) {  // design projection (okin_setup): (o - a) . unit(b - a)
      const int32_t* rec = dop + d * OKIN_DOP_STRIDE;
      const int p = OKIN_LDG(rec + 5);
      double value = 0.0;
      if (OKIN_LDG(par_mode + p) == OKIN_PAR_DESIGN_PROJECTION) {
        const int ia = OKIN_LDG(rec + 2), ib = OKIN_LDG(rec + 3), io = OKIN_LDG(rec + 6);
        const double* a = pos + 3 * ia;
        const double* b = pos + 3 * ib;
        const double* o = hardpoints + 3 * io;
        double v[3], u[3], du[3], dv[3], il, dd[3];
        for (int c = 0; c < 3; ++c) {
          const double da = (ia == moved && c == axis) ? 1.0 : 0.0, db = (ib == moved && c == axis) ? 1.0 : 0.0;
          v[c] = b[c] - a[c];
          dv[c] = db - da;
          dd[c] = ((coord / 3 == io && c == axis) ? 1.0 : 0.0) - da;
        }
        okin_unit_jvp(v, dv, u, du, &il);
        for (int c = 0; c < 3; ++c) value += dd[c] * u[c] + (o[c] - a[c]) * du[c];
      }
      dpar[p] = value;
    }
    OKIN_LANE_LOOP
    for (int t = lane; t < ncst; t += 32) dc_all[t] = 0.0;
    OKIN_PHASE_END
    okin_sens_points(pr, sm, coord, dpar, nullptr, true, tan);
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < nls; t += 32) {
      const int32_t* rec = rows + t * OKIN_ROW_STRIDE;
      const int rule = OKIN_LDG(rec + OKIN_R_RULE);
      if (rule == OKIN_RULE_EXPLICIT) continue;
      const int fam = OKIN_LDG(rec + OKIN_R_FAM);
      const double* c = cst + OKIN_LDG(rec + OKIN_R_CST);
      double* dc = dc_all + OKIN_LDG(rec + OKIN_R_CST);
      OkinDual q[4][3];
      for (int s = 0; s < 4; ++s) {
        const int pi = OKIN_LDG(rec + OKIN_R_P0 + s);
        for (int m = 0; m < 3; ++m) q[s][m] = pi < 0 ? OkinDual{0.0, 0.0} : OkinDual{pos[3 * pi + m], tan[3 * pi + m]};
      }
      if (rule == OKIN_RULE_DESIGN_POINT) {
        dc[0] = q[0][0].d; dc[1] = q[0][1].d; dc[2] = q[0][2].d;
      } else if (rule == OKIN_RULE_TARGET_BASE) {
        dc[3] = c[0] * q[0][0].d + c[1] * q[0][1].d + c[2] * q[0][2].d;
      } else if (fam == OKIN_FAM_DISTANCE) {
        OkinDual s2 = {0.0, 0.0};
        for (int m = 0; m < 3; ++m) s2 = s2 + (q[1][m] - q[0][m]) * (q[1][m] - q[0][m]);
        dc[0] = okin_sqrt(s2).d;
      } else if (fam == OKIN_FAM_ANGLE) {
        OkinDual a[3], b[3], na = {0.0, 0.0}, nb = {0.0, 0.0};
        for (int m = 0; m < 3; ++m) { a[m] = q[1][m] - q[0][m]; b[m] = q[3][m] - q[2][m]; na = na + a[m] * a[m]; nb = nb + b[m] * b[m]; }
        na = okin_sqrt(na); nb = okin_sqrt(nb);
        for (int m = 0; m < 3; ++m) { a[m] = a[m] / na; b[m] = b[m] / nb; }
        const OkinDual cx = a[1] * b[2] - a[2] * b[1], cy = a[2] * b[0] - a[0] * b[2], cz = a[0] * b[1] - a[1] * b[0];
        dc[0] = okin_atan2(okin_sqrt(cx * cx + cy * cy + cz * cz), a[0] * b[0] + a[1] * b[1] + a[2] * b[2]).d;
      } else if (fam == OKIN_FAM_SCALAR_TRIPLE) {
        OkinDual a[3], b[3], e[3];
        for (int m = 0; m < 3; ++m) { a[m] = q[1][m] - q[0][m]; b[m] = q[2][m] - q[0][m]; e[m] = q[3][m] - q[0][m]; }
        const OkinDual v = a[0] * (b[1] * e[2] - b[2] * e[1]) + a[1] * (b[2] * e[0] - b[0] * e[2]) +
                           a[2] * (b[0] * e[1] - b[1] * e[0]);
        dc[0] = v.d;
        dc[1] = -(v.v > 0.0 ? 1.0 : -1.0) * v.d / (v.v * v.v);   // c[1] = 1/|V|
      }
    }
    OKIN_PHASE_END
  }
}

// One accepted state: d pos_o / d p_k of every output point for every sensitivity column into
// dst[NSENS][NOUT*3].  Needs the factor of A at the state (okin_factor) and pos[] at the state; the
// right-hand sides use vec[0 .. NT] (the tangents have been exported by then).
template <typename Dummy = void>
OKIN_FN void okin_sens_state(const OkinProgram& pr, double* sm, const double* tval, double* ws, double* dst) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nsens = hdr[OKIN_H_NSENS], ncst = hdr[OKIN_H_NCST], npar = hdr[OKIN_H_NPAR];
  const int nls = hdr[OKIN_H_NROW], nout = hdr[OKIN_H_NOUT], n = 3 * hdr[OKIN_H_NF];
  const int group = 1 + hdr[OKIN_H_NT];
  const int32_t* sens_in = okin_sec_cold(pr, OKIN_S_SENS_IN);
  const int32_t* rows = okin_sec(pr, OKIN_S_ROW);
  const int32_t* out_point = OKIN_SHARED(okin_sec(pr, OKIN_S_OUT_POINT));
  const double* pos = sm + hdr[OKIN_H_OFF_POS];
  const double* cst = sm + hdr[OKIN_H_OFF_CST];
  double* r = sm + hdr[OKIN_H_OFF_R];
  double* vec = sm + hdr[OKIN_H_OFF_VEC];
  double* grad = ws + (size_t)nsens * (ncst + npar);
  double* tan = grad + 13 * (size_t)nls;
  // Row gradients J_x at the state (the tangent health uses their storage as scratch), and the
  // per-point gradients of every least-squares row.
  OkinState scratch_state;
  okin_eval_rows(pr, sm, tval, true, scratch_state);
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int t = lane; t < nls; t += 32) {
    const int32_t* rec = rows + t * OKIN_ROW_STRIDE;
    const int fam = OKIN_LDG(rec + OKIN_R_FAM);
    const double* c = cst + OKIN_LDG(rec + OKIN_R_CST);
    double p[12], g[12];
    for (int m = 0; m < 12; ++m) { p[m] = 0.0; g[m] = 0.0; }
    for (int s = 0; s < 4; ++s) {
      const int pi = OKIN_LDG(rec + OKIN_R_P0 + s);
      if (pi < 0) break;
      p[3 * s] = pos[3 * pi]; p[3 * s + 1] = pos[3 * pi + 1]; p[3 * s + 2] = pos[3 * pi + 2];
    }
    if (fam == OKIN_FAM_TARGET) { g[0] = c[0]; g[1] = c[1]; g[2] = c[2]; }
    else okin_family_resgrad(fam, p, c, g);
    double* o = grad + 13 * (size_t)t;
    for (int m = 0; m < 12; ++m) o[m] = g[m];
    o[12] = r[t];
  }
  OKIN_PHASE_END
  for (int k0 = 0; k0 < nsens; k0 += group) {
    const int m = nsens - k0 < group ? nsens - k0 : group;
    for (int j = m - 1; j >= 0; --j) {  // vec[0] last: the gather below writes it
      const int k = k0 + j, coord = OKIN_LDG(sens_in + k);
      const double* dc_all = ws + (size_t)k * ncst;
      okin_sens_points(pr, sm, coord, ws + (size_t)nsens * ncst + (size_t)k * npar, nullptr, false, tan);
      OKIN_PHASE_BEGIN
      OKIN_LANE_LOOP
      for (int t = lane; t < nls; t += 32) {  // r[t] <- dR_t/dp_k
        const int32_t* rec = rows + t * OKIN_ROW_STRIDE;
        const double* g = grad + 13 * (size_t)t;
        double acc = 0.0;
        for (int s = 0; s < 4; ++s) {
          const int pi = OKIN_LDG(rec + OKIN_R_P0 + s);
          if (pi < 0) break;
          acc += g[3 * s] * tan[3 * pi] + g[3 * s + 1] * tan[3 * pi + 1] + g[3 * s + 2] * tan[3 * pi + 2];
        }
        const int rule = OKIN_LDG(rec + OKIN_R_RULE);
        const double* c = cst + OKIN_LDG(rec + OKIN_R_CST);
        const double* dc = dc_all + OKIN_LDG(rec + OKIN_R_CST);
        if (rule == OKIN_RULE_DESIGN_POINT) {          // linear pin n.(p - anchor)
          acc -= g[0] * dc[0] + g[1] * dc[1] + g[2] * dc[2];
        } else if (rule == OKIN_RULE_TARGET_BASE) {    // dir.p - (base + value)
          acc -= dc[3];
        } else if (rule == OKIN_RULE_DESIGN_VALUE) {
          if (OKIN_LDG(rec + OKIN_R_FAM) == OKIN_FAM_SCALAR_TRIPLE) acc += -c[1] * dc[0] + g[12] / c[1] * dc[1];
          else acc -= dc[0];                            // quantity - design value
        }
        r[t] = acc;
      }
      OKIN_PHASE_END
      okin_assemble(pr, sm, 0.0, true);  // vec[0] = -J_x^T dR/dp_k
      if (j > 0) okin_copy(pr, vec + j * n, vec);
    }
    okin_solve(pr, sm, 0, m, false);
    for (int j = 0; j < m; ++j) {
      const int k = k0 + j;
      okin_sens_points(pr, sm, OKIN_LDG(sens_in + k), ws + (size_t)nsens * ncst + (size_t)k * npar, vec + j * n,
                       false, tan);
      double* o = dst + (size_t)k * 3 * nout;
      OKIN_PHASE_BEGIN
      OKIN_LANE_LOOP
      for (int t = lane; t < 3 * nout; t += 32) o[t] = tan[3 * OKIN_LDG(out_point + t / 3) + t % 3];
      OKIN_PHASE_END
    }
  }
}

struct OkinOutputs {
  double* positions;      // [n_steps][NOUT*3] or null
  int32_t* iters;         // [n_steps] or null
  double* max_residual;   // [n_steps] or null
  double* tangents;       // [n_steps][NT][3*NF] (reference column order) or null
  double* velocities;     // [n_steps][NT][NOUT*3] velocity of every output point per target, or null
  double* health;         // [n_steps][2] {sigma_min, cond} of the tangent system, or null
  double* metrics;        // [n_steps][NM] or null (NaN == the reference's None)
  double* design;         // [NOUT*3] design (setup) pose or null
  double* diagnostics;    // [n_steps][NDIAG] or null
  int32_t* status;        // [1]
  int32_t* failed_step;   // [1]
  int32_t* worst_row;     // [1] or null: row owning max|r| at the failed step (solver.py:640-651), else -1
  double* sensitivity;    // [n_steps][NSENS][NOUT*3] hardpoint sensitivities or null (SENS instantiation only)
  double* sens_ws;        // okin_sens_ws_doubles scratch of the warp (SENS instantiation only)
};

// Index of the row with the largest |r| in r[0 .. nrows) (first one on ties, like np.argmax;
// a NaN row wins).  Warp-uniform result.  Only runs when a sweep fails.
template <typename Dummy = void>
OKIN_FN int okin_worst_row(const OkinProgram& pr, double* sm) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nrows = hdr[OKIN_H_NROW] + hdr[OKIN_H_NREP];
  const double* r = sm + hdr[OKIN_H_OFF_R];
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  double mx = -1.0;
  OKIN_LANE_LOOP
  for (int t = lane; t < nrows; t += 32) {
    const double ar = fabs(r[t]);
    if (ar > mx || ar != ar) mx = ar;
  }
  red[lane] = mx;
  OKIN_PHASE_END
  const double rmax = okin_red_max(red);
  OKIN_PHASE_BEGIN
  int first = 1 << 30;
  OKIN_LANE_LOOP
  for (int t = lane; t < nrows; t += 32) {
    const double ar = fabs(r[t]);
    if ((ar == rmax || (ar != ar && rmax != rmax)) && t < first) first = t;
  }
  red[lane] = (double)first;
  OKIN_PHASE_END
  OKIN_PHASE_BEGIN
  if (lane == 0) {
    double lo = red[0];
    for (int k = 1; k < 32; ++k) lo = red[k] < lo ? red[k] : lo;
    red[0] = lo;
  }
  OKIN_PHASE_END
  const int row = (int)red[0];
  return row < nrows ? row : -1;
}

// Whole sweep for one instance (solver.py:716-774).  tvals: [NT][n_steps] relative/absolute
// sweep values shared by all instances of the launch.
// FULL: tangents / velocities / health / metrics / diagnostics outputs are compiled in (the lean
// instantiation only writes positions, solver statistics and the design pose: the throughput
// path, whose code footprint matters -- see profiles/r01_g_*).  SHIM: the topology has camber-shim
// records (the pre-solve is a large, once-per-instance piece of code).  SENS (with FULL, without SHIM):
// the hardpoint-sensitivity output is compiled in.
template <bool FULL, bool SHIM, bool SENS = false>
OKIN_HD void okin_sweep(const OkinProgram& pr, double* sm, const double* __restrict__ hardpoints,
                        const double* __restrict__ params, const double* __restrict__ tvals, int n_steps,
                        const OkinSolverCfg& cfg, const OkinOutputs& out) {
  sm = OKIN_SHARED(sm);
  const int32_t* hdr = OKIN_SHARED(pr.hdr);
  const int nt = hdr[OKIN_H_NT];
  const int n = 3 * hdr[OKIN_H_NF];
  const int nout = hdr[OKIN_H_NOUT];
  const int32_t* out_point = OKIN_SHARED(okin_sec(pr, OKIN_S_OUT_POINT));
  const int32_t* ecol = okin_sec(pr, OKIN_S_ELIM_COL);
  const int32_t* elim_point = OKIN_SHARED(okin_sec(pr, OKIN_S_ELIM_POINT));
  double* pos = sm + hdr[OKIN_H_OFF_POS];
  double* vec = sm + hdr[OKIN_H_OFF_VEC];
  const double* xprev = sm + hdr[OKIN_H_OFF_XPREV];
  // outputs only the full instantiation knows about
  double* const o_tangents = FULL ? out.tangents : nullptr;
  double* const o_velocities = FULL ? out.velocities : nullptr;
  double* const o_health = FULL ? out.health : nullptr;
  double* const o_metrics = FULL ? out.metrics : nullptr;
  double* const o_diagnostics = FULL ? out.diagnostics : nullptr;
  double* const o_sens = SENS ? out.sensitivity : nullptr;
  int invalid = 0;
  okin_setup<SHIM>(pr, sm, hardpoints, params, &invalid, FULL);
  if (SENS && o_sens && !invalid) okin_sens_setup(pr, sm, hardpoints, out.sens_ws);
  if (out.design) {  // design (setup) pose of every output point
    OKIN_PHASE_BEGIN
    OKIN_LANE_LOOP
    for (int t = lane; t < 3 * nout; t += 32) out.design[t] = pos[3 * OKIN_LDG(out_point + t / 3) + t % 3];
    OKIN_PHASE_END
  }

  OkinState st;
  st.f2 = 0.0; st.rmax = 0.0; st.mu = 0.0; st.notpd = 0;
  int status = invalid ? OKIN_STATUS_INVALID_GEOMETRY : OKIN_STATUS_OK, failed = invalid ? 0 : -1;
  // Target values of the current step, their increments and the previous increments live in shared
  // memory (runtime-indexed per-thread arrays would be local memory).
  double* tcur = sm + hdr[OKIN_H_OFF_TGT];
  double* dt = tcur + OKIN_MAX_TARGETS;
  double* red = sm + hdr[OKIN_H_OFF_RED];
  OKIN_PHASE_BEGIN
  OKIN_LANE_LOOP
  for (int j = lane; j < 2 * OKIN_MAX_TARGETS; j += 32) tcur[j] = 0.0;
  {   // increment history of the extrapolation predictor
    float* h = reinterpret_cast<float*>(sm + hdr[OKIN_H_OFF_DHIST]);
    OKIN_LANE_LOOP
    for (int u = lane; u < 6 * ((n + 1) / 2); u += 32) h[u] = 0.0f;
  }
  OKIN_PHASE_END
  int run = 0;      // consecutive sweep steps (ending at the current one) with the same target increments
  int worst = -1;

  for (int s = 0; s < n_steps; ++s) {
    if (status == OKIN_STATUS_OK) {
      OKIN_PHASE_BEGIN
      double changed = 0.0;
      if (lane < nt) {
        const double cur = OKIN_LDG(tvals + lane * n_steps + s);
        const double d = cur - tcur[lane], dprev = dt[lane];
        tcur[lane] = cur;
        if (fabs(d - dprev) > 1e-9 * (fabs(d) + fabs(dprev))) changed = 1.0;
        dt[lane] = d;
      }
      red[lane] = changed;
      OKIN_PHASE_END
      const bool same = okin_red_sum(red) == 0.0;
      run = s == 0 ? 0 : (same && run > 0 ? run + 1 : 1);
      // Predicted start: extrapolation of the solution history (first increment known at step 2, order
      // limited by the run of equal target increments).
      int order = run - 1 < cfg.use_predictor ? run - 1 : cfg.use_predictor;
      if (order < 0) order = 0;
      okin_extrapolate(pr, sm, order);
      const bool predicted = order > 0;
      bool conv = false;
      const bool relinearise = o_tangents || o_velocities || o_health || o_metrics || o_sens;
      bool at_solution = false;
      int nfev = 0;
      bool valid = true;
      // The reference starts every step from the previous solution (solver.py:717-774, x_0 = result.x).
      // The predicted start is an optimisation only: if the step fails from it, the previous solution
      // is restored and the step is solved again from the plain warm start before it is flagged.
      for (int attempt = 0; attempt < 2; ++attempt) {
        if (attempt == 1) {
          OKIN_PHASE_BEGIN
          OKIN_LANE_LOOP
          for (int u = lane; u < n; u += 32) pos[3 * OKIN_LDG(elim_point + u / 3) + u % 3] = xprev[u];
          OKIN_PHASE_END
          run = 1;
        }
        nfev += okin_solve_step(pr, sm, tcur, cfg, st, &conv, relinearise, &at_solution);
        valid = st.rmax == st.rmax;
        if ((conv && valid && st.rmax <= cfg.residual_tol) || !predicted) break;
      }
      if (!conv || !valid) {
        status = valid ? OKIN_STATUS_NOT_CONVERGED : OKIN_STATUS_INVALID_GEOMETRY;
        failed = s;
      } else if (st.rmax > cfg.residual_tol) {
        status = OKIN_STATUS_RESIDUAL_REJECTED;
        failed = s;
      }
      if (status != OKIN_STATUS_OK && out.worst_row) worst = okin_worst_row(pr, sm);
      OKIN_PHASE_BEGIN
      if (lane == 0) {
        if (out.iters) out.iters[s] = nfev;
        if (out.max_residual) out.max_residual[s] = st.rmax;
      }
      OKIN_PHASE_END
      if (status == OKIN_STATUS_OK) {
        if (FULL && relinearise) {
          // Exported tangents are taken at the solution itself: linearise there, carrying the tangent
          // right-hand sides through the factorisation (the iteration itself never needs them).
          if (!at_solution) {
            const double rmax = st.rmax;
            okin_eval_rows(pr, sm, tcur, true, st);
            st.rmax = rmax;
          }
          okin_assemble(pr, sm, 0.0, false);
          okin_tangent_rhs(pr, sm);
          okin_factor(pr, sm, st, true);
          okin_solve(pr, sm, 1, nt, true);
        }
        okin_derived_update(pr, sm, false);
      }
    } else {
      OKIN_PHASE_BEGIN
      if (lane == 0) {
        if (out.iters) out.iters[s] = 0;
        if (out.max_residual) out.max_residual[s] = NAN;
      }
      OKIN_PHASE_END
    }
    const bool ok = status == OKIN_STATUS_OK;
    if (out.positions) {
      double* dst = out.positions + (size_t)s * 3 * nout;
      OKIN_PHASE_BEGIN
      OKIN_LANE_LOOP
      for (int t = lane; t < 3 * nout; t += 32)
        dst[t] = ok ? pos[3 * OKIN_LDG(out_point + t / 3) + t % 3] : NAN;
      OKIN_PHASE_END
    }
    if (FULL && o_metrics) {
      const int nm = hdr[OKIN_H_NM];
      double* dst = o_metrics + (size_t)s * nm;
      if (ok) {
        okin_metrics(pr, sm, dst);
      } else {
        OKIN_PHASE_BEGIN
        OKIN_LANE_LOOP
        for (int t = lane; t < nm; t += 32) dst[t] = NAN;
        OKIN_PHASE_END
      }
    }
    if (FULL && o_velocities) {  // TangentField.velocities (sensitivity.py:115-141)
      double* dst = o_velocities + (size_t)s * nt * 3 * nout;
      OKIN_PHASE_BEGIN
      OKIN_LANE_LOOP
      for (int t = lane; t < nt * nout; t += 32) {
        double v[3] = {NAN, NAN, NAN};
        if (ok) okin_point_vel(pr, sm, OKIN_LDG(out_point + t % nout), t / nout, v);
        dst[3 * t] = v[0]; dst[3 * t + 1] = v[1]; dst[3 * t + 2] = v[2];
      }
      OKIN_PHASE_END
    }
    if (FULL && o_tangents) {
      double* dst = o_tangents + (size_t)s * nt * n;
      OKIN_PHASE_BEGIN
      OKIN_LANE_LOOP
      for (int t = lane; t < nt * n; t += 32) {
        const int j = t / n, u = t % n;  // u: elimination-ordered unknown
        dst[j * n + 3 * OKIN_LDG(ecol + u / 3) + u % 3] = ok ? vec[n + j * n + u] : NAN;
      }
      OKIN_PHASE_END
    }
    if (FULL && o_diagnostics && hdr[OKIN_H_NDIAG])
      okin_diagnostics(pr, sm, o_diagnostics + (size_t)s * hdr[OKIN_H_NDIAG], ok,
                       failed == s ? status : OKIN_STATUS_OK);
    if (FULL && o_health) {
      if (ok) {
        okin_tangent_health(pr, sm, st.notpd != 0, o_health + 2 * s);
      } else {
        OKIN_PHASE_BEGIN
        if (lane == 0) { o_health[2 * s] = NAN; o_health[2 * s + 1] = NAN; }
        OKIN_PHASE_END
      }
    }
    if (SENS && o_sens) {
      const int nsens = hdr[OKIN_H_NSENS];
      double* dst = o_sens + (size_t)s * nsens * 3 * nout;
      if (ok) {
        okin_sens_state(pr, sm, tcur, out.sens_ws, dst);
      } else {
        OKIN_PHASE_BEGIN
        OKIN_LANE_LOOP
        for (int t = lane; t < nsens * 3 * nout; t += 32) dst[t] = NAN;
        OKIN_PHASE_END
      }
    }
  }
  OKIN_PHASE_BEGIN
  if (lane == 0) {
    out.status[0] = status;
    out.failed_step[0] = failed;
    if (out.worst_row) out.worst_row[0] = worst;
  }
  OKIN_PHASE_END
}

// ---- per-instance slices of the batch buffers (okin_batch_io, include/okin.h) -------------------
// okin_batch_io without its last field: the kernels take the sensitivity output as a trailing
// parameter instead, so that the parameter layout (and the code) of the instantiations that never
// write it stays what it was before that output existed.
struct OkinKernelIO {
  const double* hardpoints;
  const double* params;
  const double* target_values;
  int32_t* status;
  int32_t* failed_step;
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
  const double* instance_targets;
  int32_t* worst_row;
};
static_assert(sizeof(OkinKernelIO) == offsetof(okin_batch_io, hardpoint_sensitivity), "OkinKernelIO layout");

// The fields of okin_batch_io in struct order.
enum okin_io_field {
  OKIN_IO_HARDPOINTS = 0, OKIN_IO_PARAMS, OKIN_IO_TARGET_VALUES, OKIN_IO_STATUS, OKIN_IO_FAILED_STEP,
  OKIN_IO_POSITIONS, OKIN_IO_ITERS, OKIN_IO_MAX_RESIDUAL, OKIN_IO_TANGENTS, OKIN_IO_VELOCITIES,
  OKIN_IO_TANGENT_HEALTH, OKIN_IO_METRICS, OKIN_IO_DESIGN, OKIN_IO_DIAGNOSTICS, OKIN_IO_JUMPS,
  OKIN_IO_INSTANCE_TARGETS, OKIN_IO_WORST_ROW, OKIN_IO_HARDPOINT_SENSITIVITY, OKIN_IO_COUNT
};

// The counts of the header every instance's slices depend on, read once (the sweep kernel keeps
// them in registers across its instance loop); the counts of optional fields are read from hdr when
// the field is wanted.
struct OkinIOShape {
  int32_t nin, nout, nt, n;   // input points, output points, targets, unknowns (3 * NF)
  const int32_t* hdr;
};
OKIN_HD OkinIOShape okin_io_shape(const int32_t* hdr) {
  return {hdr[OKIN_H_NIN], hdr[OKIN_H_NOUT], hdr[OKIN_H_NT], 3 * hdr[OKIN_H_NF], hdr};
}

// Elements of field f that belong to one instance (int32 for status, failed_step, iters and
// worst_row, double otherwise); 0 for target_values, which all instances share.
OKIN_HD size_t okin_io_count(int f, const OkinIOShape& h, int n_steps) {
  const size_t S = (size_t)n_steps;
  switch (f) {
    case OKIN_IO_HARDPOINTS: return 3 * (size_t)h.nin;
    case OKIN_IO_PARAMS: return (size_t)h.hdr[OKIN_H_NPARAM];
    case OKIN_IO_POSITIONS: return S * 3 * h.nout;
    case OKIN_IO_ITERS:
    case OKIN_IO_MAX_RESIDUAL: return S;
    case OKIN_IO_TANGENTS: return S * h.nt * h.n;
    case OKIN_IO_VELOCITIES: return S * h.nt * 3 * h.nout;
    case OKIN_IO_TANGENT_HEALTH: return S * 2;
    case OKIN_IO_METRICS: return S * h.hdr[OKIN_H_NM];
    case OKIN_IO_DESIGN: return 3 * (size_t)h.nout;
    case OKIN_IO_DIAGNOSTICS: return S * h.hdr[OKIN_H_NDIAG];
    case OKIN_IO_JUMPS: return S * (h.n / 3);
    case OKIN_IO_INSTANCE_TARGETS: return (size_t)h.nt * S;
    case OKIN_IO_HARDPOINT_SENSITIVITY: return S * h.hdr[OKIN_H_NSENS] * 3 * h.nout;
    case OKIN_IO_TARGET_VALUES: return 0;
    default: return 1;   // status, failed_step, worst_row
  }
}

// Full instantiation when a per-state tangent / metric / diagnostic output is wanted, else lean.
OKIN_HD bool okin_wants_full(const okin_batch_io& io) {
  return io.tangents || io.velocities || io.tangent_health || io.metrics || io.diagnostics;
}

// Instance i's outputs in the batch buffers (null where the batch does not want a field; sens_out:
// the hardpoint_sensitivity buffer or null) and its inputs: hardpoints, params (null = defaults) and
// sweep targets (its own row of instance_targets when given, else the shared target_values).
OKIN_HD void okin_instance_io(const OkinKernelIO& io, double* sens_out, const OkinIOShape& shape, int n_steps,
                              long long i, OkinOutputs& out, const double*& hardpoints, const double*& params,
                              const double*& targets) {
#define OKIN_SLICE(p, f) ((p) ? (p) + (size_t)i * okin_io_count(f, shape, n_steps) : nullptr)
  out.positions = OKIN_SLICE(io.positions, OKIN_IO_POSITIONS);
  out.iters = OKIN_SLICE(io.iters, OKIN_IO_ITERS);
  out.max_residual = OKIN_SLICE(io.max_residual, OKIN_IO_MAX_RESIDUAL);
  out.tangents = OKIN_SLICE(io.tangents, OKIN_IO_TANGENTS);
  out.velocities = OKIN_SLICE(io.velocities, OKIN_IO_VELOCITIES);
  out.health = OKIN_SLICE(io.tangent_health, OKIN_IO_TANGENT_HEALTH);
  out.metrics = OKIN_SLICE(io.metrics, OKIN_IO_METRICS);
  out.design = OKIN_SLICE(io.design, OKIN_IO_DESIGN);
  out.diagnostics = OKIN_SLICE(io.diagnostics, OKIN_IO_DIAGNOSTICS);
  out.status = io.status + i;
  out.failed_step = io.failed_step + i;
  out.worst_row = OKIN_SLICE(io.worst_row, OKIN_IO_WORST_ROW);
  out.sensitivity = OKIN_SLICE(sens_out, OKIN_IO_HARDPOINT_SENSITIVITY);
  hardpoints = io.hardpoints + (size_t)i * okin_io_count(OKIN_IO_HARDPOINTS, shape, n_steps);
  params = OKIN_SLICE(io.params, OKIN_IO_PARAMS);
  targets = io.instance_targets ? OKIN_SLICE(io.instance_targets, OKIN_IO_INSTANCE_TARGETS) : io.target_values;
#undef OKIN_SLICE
}
