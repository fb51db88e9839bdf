// Lane-emulation build of the device core for CPU-only tests (never linked into the product
// library): every phase of csrc/okin_core.cuh runs as a loop over 32 lanes.  The batch entry point
// slices the batch buffers and picks the instantiation the way the library's kernels and launch()
// do; the study entry points run the generator, the sweep and the reduction order of okin_study.
#define OKIN_LANE_EMU 1
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/okin.h"
#include "okin_core.cuh"
#include "okin_study.cuh"

// Returns -3 (the library's OKIN_ERR_USAGE) for hardpoint sensitivities on a topology with
// camber-shim records, -2 when a lean instantiation wrote outside its slice.
extern "C" int okin_emu_sweep(const int32_t* hdr, const int32_t* ib, const double* fb, long n_instances,
                              int n_steps, const okin_solver_cfg* c, const okin_batch_io* io) {
  if (hdr[OKIN_H_MAGIC] != OKIN_MAGIC) return -1;
  const bool sens = io->hardpoint_sensitivity != nullptr;
  if (sens && hdr[OKIN_H_NSHIM] > 0) return -3;
  const int32_t* sec[OKIN_S_COUNT];
  for (int s = 0; s < OKIN_S_COUNT; ++s) okin_resolve_section(hdr, ib, ib, s, sec);
  OkinProgram pr{hdr, ib, fb, ib, sec};
  OkinSolverCfg cfg{c->step_tol, c->coarse_tol, c->fine_tol, c->residual_tol, c->mu_init, c->max_iter,
                    c->use_predictor};
  OkinKernelIO kio;
  std::memcpy(&kio, io, sizeof(kio));
  const OkinIOShape shape = okin_io_shape(hdr);
  const bool full = sens || okin_wants_full(*io);
  std::vector<double> sm(hdr[OKIN_H_SMEM_DOUBLES]);
  std::vector<double> ws(sens ? okin_sens_ws_doubles(hdr) : 0);
  // the lean instantiation only owns the lean part of the slice
  const size_t live = full ? (size_t)hdr[OKIN_H_SMEM_DOUBLES] : (size_t)hdr[OKIN_H_SMEM_DOUBLES_LEAN];
  for (long i = 0; i < n_instances; ++i) {
    std::fill(sm.begin(), sm.begin() + live, 0.0);
    std::fill(sm.begin() + live, sm.end(), NAN);     // a lean run must not touch the rest
    OkinOutputs out;
    const double *hp, *par, *tv;
    okin_instance_io(kio, io->hardpoint_sensitivity, shape, n_steps, i, out, hp, par, tv);
    out.sens_ws = ws.data();
    if (sens)
      okin_sweep<true, false, true>(pr, sm.data(), hp, par, tv, n_steps, cfg, out);
    else if (full)
      okin_sweep<true, true>(pr, sm.data(), hp, par, tv, n_steps, cfg, out);
    else
      okin_sweep<false, true>(pr, sm.data(), hp, par, tv, n_steps, cfg, out);
    for (size_t k = live; k < sm.size(); ++k)
      if (sm[k] == sm[k]) return -2;                   // lean instantiation wrote outside its slice
  }
  if (io->diagnostics && hdr[OKIN_H_NDIAG] && n_steps > 0) {   // continuity pass, as the library's second kernel
    const int stride = (n_steps - 1) | 1;
    std::vector<double> scratch((size_t)32 * stride + 64);
    for (long i = 0; i < n_instances; ++i) {
      const int failed = io->failed_step[i];
      okin_continuity(pr, scratch.data(), stride, io->positions + i * okin_io_count(OKIN_IO_POSITIONS, shape, n_steps),
                      n_steps, failed < 0 ? n_steps : failed,
                      io->diagnostics + i * okin_io_count(OKIN_IO_DIAGNOSTICS, shape, n_steps),
                      io->jumps ? io->jumps + i * okin_io_count(OKIN_IO_JUMPS, shape, n_steps) : nullptr);
    }
  }
  return 0;
}

// One constraint row of the generated family functions (csrc/okin_gen_constraints.cuh): residual via
// both entry points and the gradient, for the family-row golden vectors.
extern "C" int okin_emu_family(int fam, const double* p, const double* c, double* res, double* res_only, double* g) {
  for (int k = 0; k < 12; ++k) g[k] = 0.0;
  *res = okin_family_resgrad(fam, p, c, g);
  *res_only = okin_family_res(fam, p, c);
  return 0;
}

// ---- tolerance studies --------------------------------------------------------------------------
// No validation: the library validates before anything runs.
namespace {

OkinStudyTables tables_of(const okin_study_desc* desc, std::vector<uint64_t>& stride) {
  stride.assign(desc->n_variates + 1, 0);
  uint64_t period = 0;
  okin_study_grid_places(desc->n_variates, desc->variate_kind, desc->grid_levels, stride.data(), &period);
  return OkinStudyTables{desc->seed, period, desc->n_coords, desc->nominal, desc->scale, desc->source,
                         desc->variate_kind, desc->grid_levels, stride.data()};
}

void generate(const OkinStudyTables& t, const int32_t* hdr, long long n_ids, const long long* ids, long long base,
              double* hp, double* par) {
  const int nin3 = 3 * hdr[OKIN_H_NIN], npar = hdr[OKIN_H_NPARAM];
  for (long long r = 0; r < n_ids; ++r)
    for (int c = 0; c < t.n_coords; ++c) {
      const double v = okin_study_coord(t, (uint64_t)(ids ? ids[r] : base + r), c);
      if (c < nin3) hp[r * nin3 + c] = v;
      else par[r * npar + (c - nin3)] = v;
    }
}

}  // namespace

extern "C" int okin_emu_study_sample(const int32_t* hdr, const okin_study_desc* desc, long long n_ids,
                                     const long long* ids, double* hp, double* par) {
  std::vector<uint64_t> stride;
  generate(tables_of(desc, stride), hdr, n_ids, ids, 0, hp, par);
  return 0;
}

// okin_study with the chunk size as an argument, so that small studies cross several chunks.  Chunks
// are dealt round-robin over `n_devices` emulated devices, which run one after another; their chunk
// partials are folded in global chunk order and their integer counts summed, as the library does.
extern "C" int okin_emu_study(const int32_t* hdr, const int32_t* ib, const double* fb, long long n, int S,
                              const double* tv, const okin_solver_cfg* c, const okin_study_desc* desc,
                              okin_study_out* out, long long chunk, int n_devices) {
  std::vector<uint64_t> stride;
  const OkinStudyTables t = tables_of(desc, stride);
  const OkinIOShape shape = okin_io_shape(hdr);
  const int nout3 = 3 * hdr[OKIN_H_NOUT], nm = hdr[OKIN_H_NM], Q = desc->n_quantities, SQ = S * Q;
  const int nb = desc->n_bins, nb2 = nb + 2;
  bool want_pos = false, want_met = false;
  for (int q = 0; q < Q; ++q) {
    want_pos |= desc->quantity_kind[q] == OKIN_QUANTITY_POSITION;
    want_met |= desc->quantity_kind[q] == OKIN_QUANTITY_METRIC;
  }
  // one chunk's buffers, as the library allocates a pipeline slot
  auto buffer = [&](int f) { return std::vector<double>(std::max<size_t>(chunk * okin_io_count(f, shape, S), 1)); };
  auto ibuffer = [&](int f) { return std::vector<int32_t>(chunk * okin_io_count(f, shape, S)); };
  std::vector<double> hp = buffer(OKIN_IO_HARDPOINTS), par = buffer(OKIN_IO_PARAMS), pos = buffer(OKIN_IO_POSITIONS),
                      met = buffer(OKIN_IO_METRICS), res = buffer(OKIN_IO_MAX_RESIDUAL);
  std::vector<int32_t> iters = ibuffer(OKIN_IO_ITERS), st = ibuffer(OKIN_IO_STATUS), failed = ibuffer(OKIN_IO_FAILED_STEP);
  okin_batch_io io{};
  io.hardpoints = hp.data();
  io.params = hdr[OKIN_H_NPARAM] ? par.data() : nullptr;
  io.target_values = tv;
  io.status = st.data();
  io.failed_step = failed.data();
  io.positions = want_pos ? pos.data() : nullptr;
  io.iters = iters.data();
  io.max_residual = res.data();
  io.metrics = want_met ? met.data() : nullptr;
  const OkinStudyChunk ch{io.positions, io.metrics, iters.data(), res.data(), st.data(), failed.data(), S, nout3, nm};
  const long long n_chunks = (n + chunk - 1) / chunk;
  // per emulated device: integer accumulators; per chunk: the partial, folded in chunk order below
  std::vector<std::vector<unsigned long long>> hist(n_devices, std::vector<unsigned long long>((size_t)SQ * nb2, 0));
  std::vector<std::vector<unsigned long long>> status(n_devices, std::vector<unsigned long long>(4, 0));
  std::vector<std::vector<unsigned long long>> failed_at(n_devices, std::vector<unsigned long long>(S, 0));
  std::vector<std::vector<OkinMoments>> partial(n_chunks, std::vector<OkinMoments>(SQ));
  for (int dev = 0; dev < n_devices; ++dev)
    for (long long k = dev; k < n_chunks; k += n_devices) {
      const long long base = k * chunk, rows = std::min(chunk, n - base);
      generate(t, hdr, rows, nullptr, base, hp.data(), par.data());
      const int rc = okin_emu_sweep(hdr, ib, fb, rows, S, c, &io);
      if (rc) return rc;
      for (int j = 0; j < SQ; ++j) {
        const int s = j / Q, q = j - s * Q, kind = desc->quantity_kind[q], index = desc->quantity_index[q];
        const double lo = nb ? desc->hist_lo[q] : 0.0, hi = nb ? desc->hist_hi[q] : 0.0;
        OkinMoments chunk_m;
        okin_moments_clear(chunk_m);
        for (int g = 0; g < OKIN_STUDY_GROUPS; ++g) {
          OkinMoments group_m;
          okin_moments_clear(group_m);
          for (int y = 0; y < OKIN_STUDY_GROUP; ++y) {
            OkinMoments m;
            okin_moments_clear(m);
            okin_study_partition(ch, kind, index, s, g * OKIN_STUDY_GROUP + y, rows, base, nb, lo, hi, m,
                                 [&](int b) { ++hist[dev][(size_t)j * nb2 + b]; });
            if (y == 0) group_m = m;
            else okin_moments_merge(group_m, m);
          }
          if (g == 0) chunk_m = group_m;
          else okin_moments_merge(chunk_m, group_m);
        }
        partial[k][j] = chunk_m;
      }
      for (long long r = 0; r < rows; ++r) {
        if (st[r] >= 0 && st[r] < 4) ++status[dev][st[r]];
        if (failed[r] >= 0 && failed[r] < S) ++failed_at[dev][failed[r]];
      }
    }
  std::vector<OkinMoments> acc(SQ);
  for (OkinMoments& m : acc) okin_moments_clear(m);
  for (long long k = 0; k < n_chunks; ++k)
    for (int j = 0; j < SQ; ++j) okin_moments_merge(acc[j], partial[k][j]);
  std::vector<OkinStudyCounts> counts;
  for (int dev = 0; dev < n_devices; ++dev) counts.push_back({hist[dev].data(), status[dev].data(), failed_at[dev].data()});
  okin_study_fold(acc.data(), S, SQ, nb, counts.data(), n_devices, out);
  return 0;
}

// Philox4x32-10 on one counter / key, for the known-answer tests.
extern "C" void okin_emu_philox(uint32_t* ctr, const uint32_t* key) { okin_philox4x32_10(ctr, key[0], key[1]); }
