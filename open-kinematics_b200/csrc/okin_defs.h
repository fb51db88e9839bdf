// Shared definitions of the device core, the C ABI and (by value) core/topology.py.
// Plain C so that include/okin.h users and the g++ lane-emulation test harness can
// include it too.
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define OKIN_HD __host__ __device__ __forceinline__
#else
#define OKIN_HD inline
#endif

#if defined(__CUDA_ARCH__)
#define OKIN_RSQRT(x) rsqrt(x)
#else
#define OKIN_RSQRT(x) (1.0 / sqrt(x))
#endif

// softnorm(s) = sqrt(s + EPS_SQ) - EPS   (reference core/primitives/soft_math.py:16-27)
#define OKIN_EPS 1e-6
#define OKIN_EPS_SQ 1e-12

// Constraint-family codes (order = FAMILIES in tools/generate_jacobians.py).
#define OKIN_FAM_DISTANCE 0
#define OKIN_FAM_SPHERICAL 1
#define OKIN_FAM_ANGLE 2
#define OKIN_FAM_THREE_POINT_ANGLE 3
#define OKIN_FAM_VECTORS_PARALLEL 4
#define OKIN_FAM_VECTORS_PERPENDICULAR 5
#define OKIN_FAM_EQUAL_DISTANCE 6
#define OKIN_FAM_POINT_ON_LINE 7
#define OKIN_FAM_LINEAR_POINT 8
#define OKIN_FAM_MIDPOINT_ON_PLANE 9
#define OKIN_FAM_COPLANAR 10
#define OKIN_FAM_SCALAR_TRIPLE 11
// Sweep-target row: dir.p - value(step); c = [dir(3), base] with value = base + sweep value.
#define OKIN_FAM_TARGET 12

// Point kinds.
#define OKIN_PT_FIXED 0
#define OKIN_PT_FREE 1
#define OKIN_PT_DERIVED 2

// Derived-point ops (reference core/points/derived/definitions.py:24-180).
#define OKIN_DOP_MIDPOINT 1      // out = a + (b - a)/2
#define OKIN_DOP_ALONG_LINE 2    // out = a + unit(b - a) * param
#define OKIN_DOP_CONTACT_PATCH 3 // out = a + unit(down - (down.u)u) * param, u = unit(c - b), down = -Z

// Parameter modes of a derived op.
#define OKIN_PAR_SHARED 0            // value from the topology
#define OKIN_PAR_DESIGN_PROJECTION 1 // dot(authored_out - a, unit(b - a)) at the design pose

// Per-row design-constant rules evaluated once per instance (setup phase).
#define OKIN_RULE_EXPLICIT 0     // constants come from the topology (cst_init)
#define OKIN_RULE_DESIGN_VALUE 1 // family's own quantity at the design pose (length, angle, volume)
#define OKIN_RULE_DESIGN_POINT 2 // c[0..2] = design position of the row's point (line / pin anchor)
#define OKIN_RULE_TARGET_BASE 3  // c[3] = dir . design position (relative target), else 0

// Per-instance status (okin_solve_batch status_out).
// Sweep diagnostics (reference core/diagnostics.py:136-226, axle/mechanisms.py:119-163, :432-549).
// Per state: column 0 = OKIN_DIAG_* flag bits (as a double), 1 = number of free points that jumped
// into this step, 2 = largest such displacement (mm), 3 = its output point slot, 4 = its
// threshold; then the topology columns of the diagnostic ops.
#define OKIN_DIAG_BASE 5
#define OKIN_DIAG_NOT_CONVERGED 1
#define OKIN_DIAG_RESIDUAL 2
#define OKIN_DIAG_JUMP 4
#define OKIN_DIAG_CHIRALITY_BOUNDARY 8
#define OKIN_DIAG_CHIRALITY_INVERTED 16
#define OKIN_DIAG_TRANSMISSION 32
// diagnostic op record: {kind, p0..p4, column, design slots d0..d3}
#define OKIN_DGOP_STRIDE 12
#define OKIN_DG_CHIRALITY 0      // points axis_a, axis_b, rocker pickup, bar pickup -> (signed volume, margin, 0 ok | 1 boundary | 2 inverted)
#define OKIN_DG_TRANSMISSION 1   // points driven, axis_a, axis_b, link_from, link_to -> margin (NaN = undefined)

#define OKIN_STATUS_OK 0
#define OKIN_STATUS_NOT_CONVERGED 1
#define OKIN_STATUS_RESIDUAL_REJECTED 2
#define OKIN_STATUS_INVALID_GEOMETRY 3

// ---------------------------------------------------------------------------
// Compiled topology program = int32 header + one int32 blob + one double blob.
// hdr[0 .. OKIN_H_SEC0)            counts and shared-memory offsets (enum below)
// hdr[OKIN_H_SEC0 + 2*s, +1]       (offset, length) of int32 section s in the int blob
// hdr[OKIN_H_FSEC0 + 2*s, +1]      (offset, length) of double section s in the double blob
// ---------------------------------------------------------------------------
enum okin_hdr_slot {
  OKIN_H_MAGIC = 0,
  OKIN_H_P,        // points
  OKIN_H_NF,       // free points (unknowns = 3*NF)
  OKIN_H_NIN,      // input points per instance
  OKIN_H_NDOP,     // derived ops
  OKIN_H_NPAR,     // derived-op parameters
  OKIN_H_NROW,     // least-squares rows (constraints with pins, then targets)
  OKIN_H_NREP,     // report-only rows (original point-on-line residuals), stored after the LS rows
  OKIN_H_NT,       // targets
  OKIN_H_NCST,     // per-instance constants (doubles)
  OKIN_H_NRG,      // row-gradient storage (doubles)
  OKIN_H_NAD,      // derived-Jacobian column tasks
  OKIN_H_NDB,      // derived-Jacobian block storage (doubles)
  OKIN_H_NB,       // factor blocks (3x3)
  OKIN_H_NLEV,     // elimination-tree levels
  OKIN_H_NAT,      // assembly tasks (scalar entries of A)
  OKIN_H_NOUT,     // output points
  OKIN_H_TROW0,    // first target row
  // shared-memory layout (offsets in doubles from the instance's base)
  OKIN_H_OFF_POS, OKIN_H_OFF_CST, OKIN_H_OFF_R, OKIN_H_OFF_RG, OKIN_H_OFF_DBLK, OKIN_H_OFF_LB,
  OKIN_H_OFF_VEC, OKIN_H_OFF_RED, OKIN_H_OFF_PAR,
  OKIN_H_UNUSED0,
  OKIN_H_SMEM_DOUBLES, // shared-memory doubles per instance
  // metric program (csrc/okin_metrics.cuh)
  OKIN_H_NM,       // metric columns per state
  OKIN_H_NMC,      // corner records
  OKIN_H_NMOP,     // generic metric ops
  OKIN_H_NMAXLE,   // 0 or 1 axle record
  OKIN_H_NDSN,     // design-pose slots kept for the metrics
  OKIN_H_OFF_DSN, OKIN_H_OFF_MCTX,
  OKIN_H_NSHIM,    // camber-shim pre-solve records (one per shimmed corner)
  OKIN_H_NPARAM,   // per-instance scalar parameters (doubles)
  OKIN_H_NDROW,    // distance rows on the fast evaluation path
  OKIN_H_NGROW,    // rows on the generic evaluation path (ROW_ORDER entries)
  OKIN_H_UNUSED1,
  OKIN_H_OFF_TGT,  // [2][OKIN_MAX_TARGETS] target values of the current step and their last increments
  OKIN_H_NHOT,     // int32 words of the hot prefix of the int blob (sections used inside the
                   // iteration; the kernel keeps them in shared memory, the rest stays in global memory)
  OKIN_H_NDIAG,    // diagnostic columns per state (OKIN_DIAG_BASE + topology columns), 0 = no program
  OKIN_H_NDGOP,    // topology diagnostic ops
  OKIN_H_FREE_ALL_OUT,  // 1 when every free point is an output point (ELIM_OUT has no -1)
  OKIN_H_OFF_XPREV,  // previous accepted solution (3*NF doubles, elimination order)
  OKIN_H_OFF_DHIST,  // three older solution increments as float32 vectors (extrapolation predictor)
  OKIN_H_SMEM_DOUBLES_LEAN,  // slice size of an instance solved without tangents / metrics / diagnostics
  OKIN_H_NSENS,    // hardpoint-sensitivity rows (entries of OKIN_S_SENS_IN)
  OKIN_H_SEC0 = 64,                      // room for 64 scalar slots,
  OKIN_H_FSEC0 = 64 + 2 * 64,            // 64 int32 sections
  OKIN_HDR_SIZE = 64 + 2 * 64 + 2 * 8    // and 8 double sections
};
#define OKIN_MAGIC 0x4f4b494e  // "OKIN"

// int32 sections
enum okin_isec {
  // hot sections: read inside the iteration; the sweep kernel keeps them in shared memory and the
  // device code addresses them as shared (OKIN_SHARED)
  OKIN_S_DOP = 0,            // [NDOP][OKIN_DOP_STRIDE]
  OKIN_S_ADJ,            // [NAD][OKIN_ADJ_STRIDE]
  OKIN_S_ADJ_CHAIN,      // derived-op indices, referenced by ADJ
  OKIN_S_DER,            // [..][OKIN_DER_STRIDE]
  OKIN_S_ASM_PTR,        // [NAT+1] contribution ranges per assembly task (one task per 3x3 block)
  OKIN_S_ASM_TASK,       // [NAT] block id | OKIN_ASM_DIAG flag, heaviest task first
  OKIN_S_ASM_CON,        // (ia << 16) | ib: rg[] offsets of the two 3-vectors whose outer product is added
  OKIN_S_G_PTR,          // [NF+1]  (elimination-ordered block columns)
  OKIN_S_G_CON,          // (irg << 16) | row: g_j += rg[irg..irg+3) * r[row]
  OKIN_S_LEV_UPD_MID,    // [NLEV] end of the level's update tasks that do not belong to tangent right-hand sides
  OKIN_S_LEV_SCL_MID,    // [NLEV] same for the scale tasks
  OKIN_S_JH_PTR,         // [NROW+1] ranges into JH_CON: the Jacobian row of each least-squares row
  OKIN_S_JH_CON,         // (rg offset << 16) | 3 * elimination position (| OKIN_CON_NEG): r_t += rg . h_j
  OKIN_S_REP_PINS,       // [NREP][2] the two pin rows of each report (point-on-line) row
  OKIN_S_LEV_UPD,        // [NLEV+1] ranges into UPD_DST/UPD_PTR
  OKIN_S_UPD_DST,        // shared-memory offset of the 3-entry row being updated
  OKIN_S_UPD_PTR,        // [n_upd+1]
  OKIN_S_UPD_CON,        // (offA << 16) | offB : acc[c] -= sum_t sm[offA+t]*sm[offB+3c+t]
  OKIN_S_LEV_SCL,        // [NLEV+1] ranges into SCL
  OKIN_S_SCL,            // [..] = diag block offset | row offset << 16 (shared-memory offsets)
  OKIN_S_LEV_COL_PTR,    // [NLEV+1]
  OKIN_S_LEV_COL,        // elimination columns of each level
  OKIN_S_SOLVE_LEV,      // [2][NLEV+1] task ranges of the forward phases (levels upwards), then of the
                         // backward phases (levels from the root down)
  OKIN_S_SOLVE_TASK,     // (first contribution << 16) | OKIN_SOLVE_FIN | column; the next word's first
                         // contribution ends the range (one extra word after the last task)
  OKIN_S_SOLVE_CON,      // (block offset << 16) | (3 * source column)
  OKIN_S_ELIM_POINT,     // [NF] elimination position -> point index
  OKIN_S_TGT_SC_PTR,     // [NT+1]
  OKIN_S_TGT_SC,         // (rg index << 16) | unknown index (elimination order)
  OKIN_S_OUT_POINT,      // [NOUT]
  OKIN_S_DOP_LEV,        // [n_derived_levels+1] ranges of DOP evaluated in one parallel phase
  OKIN_S_DROW,           // [3][NDROW] = {p0 | p1 << 16}, {cst_off | rg_off << 16}, {row}: plain distance rows
  OKIN_S_DIAG_OFF,       // [NF] shared-memory offset of the diagonal block of elimination column j
  OKIN_S_ROW_HOT,        // [NGROW][OKIN_ROW_STRIDE] records of the generic-path rows in evaluation order
                         // (grouped by family), each carrying its row index in OKIN_R_ROWID
  // metric program and the point maps its velocity look-ups walk: read once per state by the
  // full-output kernels (pointer chasing through global memory cost more than the solve itself)
  OKIN_S_POINT_ELIM,     // [P] elimination position of a free point, else -1
  OKIN_S_POINT_DOP,      // [P] derived-op index of a derived point, else -1
  OKIN_S_MCORNER,        // [NMC][OKIN_MCORNER_STRIDE]
  OKIN_S_MOP,            // [NMOP][OKIN_MOP_STRIDE]
  OKIN_S_MAXLE,          // [NMAXLE][OKIN_MAXLE_STRIDE]
  // cold sections (index >= OKIN_S_COLD0): set-up rules, outputs requested per state, metrics,
  // diagnostics, shims; they stay in global memory
  OKIN_S_COLD0,
  OKIN_S_ROW = OKIN_S_COLD0,            // [NROW+NREP][OKIN_ROW_STRIDE]
  OKIN_S_ROW_ORDER,      // [NROW+NREP] evaluation order (rows grouped by family)
  OKIN_S_IN_POINT,       // [NIN] input slot -> point
  OKIN_S_PAR_MODE,       // [NPAR]
  OKIN_S_POINT_KIND, // [P]
  OKIN_S_DESIGN_PT,      // [NDSN] points whose design position is kept for the metrics
  OKIN_S_SHIM,           // [NSHIM][OKIN_SHIM_STRIDE]
  OKIN_S_SHIM_PTS,       // point lists referenced by SHIM (upright attachments, rocker group)
  OKIN_S_FREE_OUT,       // [NF] output slot of free point k (reference column order), -1 = not exported
  OKIN_S_DGOP,           // [NDGOP][OKIN_DGOP_STRIDE] topology diagnostic ops
  OKIN_S_ELIM_COL,       // [NF] elimination position -> reference column block (sorted free-point order)
  OKIN_S_ELIM_OUT,       // [NF] elimination position -> output slot of that free point, -1 = not exported
  OKIN_S_FW_PTR,         // [NF+1] per-column lists of L z (okin_factor_multiply)
  OKIN_S_FW_CON,         // (block offset << 16) | (3*K)
  OKIN_S_BW_PTR,         // [NF+1] per-column lists of L^T z
  OKIN_S_BW_CON,         // (block offset << 16) | (3*I)
  OKIN_S_COUNT,
  // Sections from here on are not in the per-CTA section table (okin_resolve_section), so the kernels
  // that never read them keep their shared-memory layout; device code reaches them with okin_sec_cold.
  OKIN_S_SENS_IN = OKIN_S_COUNT,  // [NSENS] hardpoint coordinate 3 * input slot + axis of each sensitivity row
  OKIN_S_COUNT_ALL
};
#define OKIN_ASM_DIAG 0x40000000
// Solve task flag: the visit finalises its column (3x3 diagonal solve after the contributions).
#define OKIN_SOLVE_FIN 0x8000
// Contribution words carry a negate flag: the product enters with a minus sign (a fast distance
// row stores u = dR/dp2 once, dR/dp1 = -u).
#define OKIN_CON_NEG 0x80000000

// double sections
enum okin_fsec { OKIN_F_PAR_VAL = 0, OKIN_F_CST_INIT, OKIN_F_MCONST, OKIN_F_PARAM_DEFAULT, OKIN_F_COUNT };

// Row record: int32[OKIN_ROW_STRIDE]
enum okin_row_slot {
  OKIN_R_FAM = 0,
  OKIN_R_P0, OKIN_R_P1, OKIN_R_P2, OKIN_R_P3, // point indices (-1 unused)
  OKIN_R_CST,   // offset of the row's constants in cst[]
  OKIN_R_RG,    // offset of the row's effective-gradient storage in rg[]
  OKIN_R_NEFF,  // number of effective free blocks
  OKIN_R_RULE,  // design-constant rule
  OKIN_R_S0, OKIN_R_S1, OKIN_R_S2, OKIN_R_S3, // slot map: -1 none, <OKIN_SLOT_DER direct eff index, else derived descriptor
  OKIN_R_AUX,   // target index for target rows
  OKIN_R_ROWID, // row index (OKIN_S_ROW_HOT records)
  OKIN_ROW_STRIDE = 17   // odd: lanes reading the same field of consecutive rows hit distinct banks
};
#define OKIN_SLOT_DER 64

// Derived-slot descriptor: int32[8] = {ndeps, dblk_off0, eff0, dblk_off1, eff1, dblk_off2, eff2, 0}
#define OKIN_DER_STRIDE 8
// Derived op record: int32[8] = {op, out, a, b, c, par, authored_input_slot, active}
#define OKIN_DOP_STRIDE 8
// Derived-Jacobian column task: int32[8] = {D, B, comp, dblk_off, chain_begin, chain_end, 0, 0}
#define OKIN_ADJ_STRIDE 8
#define OKIN_MAX_CHAIN 4
#define OKIN_MAX_TARGETS 4

// Camber-shim record: int32[OKIN_SHIM_STRIDE] =
//   {ubj, lbj, upper_wishbone_inboard_front, upper_wishbone_inboard_rear, heading_in, heading_out,
//    has_rocker, rocker_axis_a, rocker_axis_b, pushrod_in, pushrod_out, param_off,
//    upright_list_begin, upright_list_end, rocker_list_begin, rocker_list_end}
// params[param_off ..] = {face_a(3), face_b(3), face_normal(3), design_thickness, setup_thickness}
#define OKIN_SHIM_STRIDE 16
#define OKIN_SHIM_NPARAM 11
