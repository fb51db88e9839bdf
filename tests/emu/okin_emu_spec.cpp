// Lane-emulation build of the topology-specialised lean kernel for CPU-only tests: csrc/okin_core.cuh
// compiled with -DOKIN_SPEC and a topology's generated okin_spec.h (core/topology.py spec_source) on
// the include path.  A spec describes the lean instantiation's phases only, so this harness runs the
// lean sweep, the way okin_emu.cpp runs it for a batch without tangent / metric / diagnostic outputs.
#define OKIN_LANE_EMU 1
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/okin.h"
#include "okin_core.cuh"

// Returns -1 for a bad header, -4 for a batch that wants the full instantiation, -2 when the lean
// instantiation wrote outside its slice.
extern "C" int okin_emu_sweep(const int32_t* hdr, const int32_t* ib, const double* fb, long n_instances,
                              int n_steps, const okin_solver_cfg* c, const okin_batch_io* io) {
  if (hdr[OKIN_H_MAGIC] != OKIN_MAGIC) return -1;
  if (io->hardpoint_sensitivity || okin_wants_full(*io)) return -4;
  const int32_t* sec[OKIN_S_COUNT];
  for (int s = 0; s < OKIN_S_COUNT; ++s) okin_resolve_section(hdr, ib, ib, s, sec);
  OkinProgram pr{hdr, ib, fb, ib, sec};
  pr.spec = okin_spec_words;
  OkinSolverCfg cfg{c->step_tol, c->coarse_tol, c->fine_tol, c->residual_tol, c->mu_init, c->max_iter,
                    c->use_predictor};
  OkinKernelIO kio;
  std::memcpy(&kio, io, sizeof(kio));
  const OkinIOShape shape = okin_io_shape(hdr);
  std::vector<double> sm(hdr[OKIN_H_SMEM_DOUBLES]);
  const size_t live = (size_t)hdr[OKIN_H_SMEM_DOUBLES_LEAN];
  for (long i = 0; i < n_instances; ++i) {
    std::fill(sm.begin(), sm.begin() + live, 0.0);
    std::fill(sm.begin() + live, sm.end(), NAN);
    OkinOutputs out;
    const double *hp, *par, *tv;
    okin_instance_io(kio, nullptr, shape, n_steps, i, out, hp, par, tv);
    okin_sweep<false, true>(pr, sm.data(), hp, par, tv, n_steps, cfg, out);
    for (size_t k = live; k < sm.size(); ++k)
      if (sm[k] == sm[k]) return -2;
  }
  return 0;
}
