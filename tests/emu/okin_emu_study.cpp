// Lane-emulation study driver for CPU-only tests (never linked into the product library): the
// generator, the sweep and the reduction of okin_study (csrc/okin_abi.cu) with the chunk size as an
// argument, so that small studies cross several chunks.  Chunks are dealt round-robin over
// `n_devices` emulated devices, which run one after another; their chunk partials are folded in
// global chunk order and their integer counts summed, as the library does.  No validation: the
// library validates before anything runs.
#define OKIN_LANE_EMU 1
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/okin.h"
#include "okin_core.cuh"
#include "okin_study.cuh"

namespace {

OkinStudyTables tables_of(const okin_study_desc* desc, std::vector<uint64_t>& stride) {
  stride.assign(desc->n_variates + 1, 0);
  uint64_t period = 0;
  okin_study_grid_places(desc->n_variates, desc->variate_kind, desc->grid_levels, stride.data(), &period);
  return OkinStudyTables{desc->seed, period, desc->n_coords, desc->nominal, desc->scale, desc->source,
                         desc->variate_kind, desc->grid_levels, stride.data()};
}

}  // namespace

extern "C" int okin_emu_study_sample(const int32_t* hdr, const okin_study_desc* desc, long long n_ids,
                                     const long long* ids, double* hp, double* par) {
  std::vector<uint64_t> stride;
  const OkinStudyTables t = tables_of(desc, stride);
  const int nin3 = 3 * hdr[OKIN_H_NIN], npar = hdr[OKIN_H_NPARAM];
  for (long long r = 0; r < n_ids; ++r)
    for (int c = 0; c < t.n_coords; ++c) {
      const double v = okin_study_coord(t, (uint64_t)ids[r], c);
      if (c < nin3) hp[r * nin3 + c] = v;
      else par[r * npar + (c - nin3)] = v;
    }
  return 0;
}

extern "C" int okin_emu_study(const int32_t* hdr, const int32_t* ib, const double* fb, long long n, int S,
                              const double* tv, const okin_solver_cfg* c, const okin_study_desc* desc,
                              okin_study_out* out, long long chunk, int n_devices) {
  if (hdr[OKIN_H_MAGIC] != OKIN_MAGIC) return -1;
  const int32_t* sec[OKIN_S_COUNT];
  for (int s = 0; s < OKIN_S_COUNT; ++s) okin_resolve_section(hdr, ib, ib, s, sec);
  OkinProgram pr{hdr, ib, fb, ib, sec};
  OkinSolverCfg cfg{c->step_tol, c->coarse_tol, c->fine_tol, c->residual_tol, c->mu_init, c->max_iter,
                    c->use_predictor};
  std::vector<uint64_t> stride;
  const OkinStudyTables t = tables_of(desc, stride);
  const int nin3 = 3 * hdr[OKIN_H_NIN], npar = hdr[OKIN_H_NPARAM], nout3 = 3 * hdr[OKIN_H_NOUT];
  const int nm = hdr[OKIN_H_NM], Q = desc->n_quantities, SQ = S * Q, nb = desc->n_bins, nb2 = nb + 2;
  bool full = false;
  for (int q = 0; q < Q; ++q) full |= desc->quantity_kind[q] == OKIN_QUANTITY_METRIC;
  const long long n_chunks = (n + chunk - 1) / chunk;
  // per emulated device: integer accumulators; per chunk: the partial, folded in chunk order below
  std::vector<std::vector<int64_t>> hist(n_devices, std::vector<int64_t>((size_t)SQ * nb2, 0));
  std::vector<std::vector<int64_t>> status(n_devices, std::vector<int64_t>(4, 0));
  std::vector<std::vector<int64_t>> failed_at(n_devices, std::vector<int64_t>(S, 0));
  std::vector<std::vector<OkinMoments>> partial(n_chunks, std::vector<OkinMoments>(SQ));
  std::vector<double> sm(hdr[OKIN_H_SMEM_DOUBLES]);
  std::vector<double> hp(chunk * nin3), par(chunk * (npar ? npar : 1)), pos((size_t)chunk * S * nout3),
      met((size_t)chunk * S * (nm ? nm : 1)), res((size_t)chunk * S);
  std::vector<int32_t> iters((size_t)chunk * S), st(chunk), failed(chunk);
  for (int dev = 0; dev < n_devices; ++dev)
    for (long long k = dev; k < n_chunks; k += n_devices) {
      const long long base = k * chunk, rows = std::min(chunk, n - base);
      for (long long r = 0; r < rows; ++r) {
        for (int cc = 0; cc < t.n_coords; ++cc) {
          const double v = okin_study_coord(t, (uint64_t)(base + r), cc);
          if (cc < nin3) hp[r * nin3 + cc] = v;
          else par[r * npar + (cc - nin3)] = v;
        }
        std::fill(sm.begin(), sm.end(), 0.0);
        OkinOutputs o{};
        o.positions = pos.data() + (size_t)r * S * nout3;
        o.iters = iters.data() + (size_t)r * S;
        o.max_residual = res.data() + (size_t)r * S;
        o.metrics = full ? met.data() + (size_t)r * S * nm : nullptr;
        o.status = st.data() + r;
        o.failed_step = failed.data() + r;
        const double* pp = npar ? par.data() + (size_t)r * npar : nullptr;
        if (full) okin_sweep<true, true>(pr, sm.data(), hp.data() + r * nin3, pp, tv, S, cfg, o);
        else okin_sweep<false, true>(pr, sm.data(), hp.data() + r * nin3, pp, tv, S, cfg, o);
      }
      const OkinStudyChunk ch{pos.data(), met.data(), iters.data(), res.data(), st.data(), failed.data(), S, nout3, nm};
      for (int j = 0; j < SQ; ++j) {
        const int s = j / Q, q = j - s * Q, kind = desc->quantity_kind[q], index = desc->quantity_index[q];
        OkinMoments chunk_m;
        okin_moments_clear(chunk_m);
        for (int g = 0; g < OKIN_STUDY_GROUPS; ++g) {
          OkinMoments group_m;
          okin_moments_clear(group_m);
          for (int y = 0; y < OKIN_STUDY_GROUP; ++y) {
            OkinMoments m;
            okin_moments_clear(m);
            for (long long r = g * OKIN_STUDY_GROUP + y; r < rows; r += OKIN_STUDY_PARTS) {
              double x;
              if (!okin_study_fetch(ch, kind, index, r, s, &x)) continue;
              okin_moments_push(m, x, base + r);
              if (nb && isfinite(x)) ++hist[dev][(size_t)j * nb2 + okin_study_bin(x, desc->hist_lo[q], desc->hist_hi[q], nb)];
            }
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
  for (int j = 0; j < SQ; ++j) {
    const OkinMoments& m = acc[j];
    const bool empty = m.count == 0;
    out->count[j] = m.count;
    out->nonfinite[j] = m.nonfinite;
    out->mean[j] = empty ? NAN : m.mean;
    out->m2[j] = empty ? NAN : m.m2;
    out->min[j] = empty ? NAN : m.min;
    out->max[j] = empty ? NAN : m.max;
    out->argmin[j] = empty ? -1 : m.argmin;
    out->argmax[j] = empty ? -1 : m.argmax;
  }
  for (int k = 0; k < 4; ++k) out->status_counts[k] = 0;
  for (int s = 0; s < S; ++s) out->failed_at_step[s] = 0;
  if (nb) std::fill(out->histogram, out->histogram + (size_t)SQ * nb2, (int64_t)0);
  for (int dev = 0; dev < n_devices; ++dev) {
    for (int k = 0; k < 4; ++k) out->status_counts[k] += status[dev][k];
    for (int s = 0; s < S; ++s) out->failed_at_step[s] += failed_at[dev][s];
    if (nb)
      for (size_t k = 0; k < (size_t)SQ * nb2; ++k) out->histogram[k] += hist[dev][k];
  }
  return 0;
}

// Philox4x32-10 on one counter / key, for the known-answer tests.
extern "C" void okin_emu_philox(uint32_t* ctr, const uint32_t* key) { okin_philox4x32_10(ctr, key[0], key[1]); }
