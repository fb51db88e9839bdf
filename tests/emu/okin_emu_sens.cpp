// Lane-emulation build of the hardpoint-sensitivity instantiation of the device core
// (okin_sweep<FULL = true, SHIM = false, SENS = true>) for CPU-only tests; never linked into the
// product library.  Same conventions as okin_emu.cpp.
#define OKIN_LANE_EMU 1
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/okin.h"
#include "okin_core.cuh"

// Returns -3 (the library's OKIN_ERR_USAGE) on a topology with camber-shim records.
extern "C" int okin_emu_sens_sweep(const int32_t* hdr, const int32_t* ib, const double* fb, long n_instances,
                                   int n_steps, const okin_solver_cfg* c, const okin_batch_io* io) {
  if (hdr[OKIN_H_MAGIC] != OKIN_MAGIC) return -1;
  if (hdr[OKIN_H_NSHIM] > 0) return -3;
  if (!io->hardpoint_sensitivity) return -4;
  const int32_t* sec[OKIN_S_COUNT];
  for (int s = 0; s < OKIN_S_COUNT; ++s) okin_resolve_section(hdr, ib, ib, s, sec);
  OkinProgram pr{hdr, ib, fb, ib, sec};
  OkinSolverCfg cfg{c->step_tol, c->coarse_tol, c->fine_tol, c->residual_tol, c->mu_init, c->max_iter,
                    c->use_predictor};
  const int nin = hdr[OKIN_H_NIN], nout = hdr[OKIN_H_NOUT], nt = hdr[OKIN_H_NT], n = 3 * hdr[OKIN_H_NF];
  std::vector<double> sm(hdr[OKIN_H_SMEM_DOUBLES]);
  std::vector<double> ws(okin_sens_ws_doubles(hdr));
  for (long i = 0; i < n_instances; ++i) {
    std::fill(sm.begin(), sm.end(), 0.0);
    OkinOutputs out;
    out.positions = io->positions ? io->positions + (size_t)i * n_steps * 3 * nout : nullptr;
    out.iters = io->iters ? io->iters + (size_t)i * n_steps : nullptr;
    out.max_residual = io->max_residual ? io->max_residual + (size_t)i * n_steps : nullptr;
    out.tangents = io->tangents ? io->tangents + (size_t)i * n_steps * nt * n : nullptr;
    out.velocities = io->velocities ? io->velocities + (size_t)i * n_steps * nt * 3 * nout : nullptr;
    out.health = io->tangent_health ? io->tangent_health + (size_t)i * n_steps * 2 : nullptr;
    out.metrics = io->metrics ? io->metrics + (size_t)i * n_steps * hdr[OKIN_H_NM] : nullptr;
    out.design = io->design ? io->design + (size_t)i * 3 * nout : nullptr;
    const int nd = hdr[OKIN_H_NDIAG];
    out.diagnostics = (io->diagnostics && nd) ? io->diagnostics + (size_t)i * n_steps * nd : nullptr;
    out.status = io->status + i;
    out.failed_step = io->failed_step + i;
    out.worst_row = io->worst_row ? io->worst_row + i : nullptr;
    out.sensitivity = io->hardpoint_sensitivity + (size_t)i * n_steps * hdr[OKIN_H_NSENS] * 3 * nout;
    out.sens_ws = ws.data();
    const double* tv = io->instance_targets ? io->instance_targets + (size_t)i * nt * n_steps : io->target_values;
    okin_sweep<true, false, true>(pr, sm.data(), io->hardpoints + (size_t)i * 3 * nin, nullptr, tv, n_steps, cfg, out);
    if (out.diagnostics && n_steps > 0) {  // continuity pass, as the product's second kernel does
      const int stride = (n_steps - 1) | 1;
      std::vector<double> scratch((size_t)32 * stride + 64);
      const int failed = io->failed_step[i];
      okin_continuity(pr, scratch.data(), stride, io->positions + (size_t)i * n_steps * 3 * nout, n_steps,
                      failed < 0 ? n_steps : failed, out.diagnostics,
                      io->jumps ? io->jumps + (size_t)i * n_steps * (n / 3) : nullptr);
    }
  }
  return 0;
}
