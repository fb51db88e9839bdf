// Test-only entry points into the Sobol' part of csrc/okin_study.cuh (never linked into the product
// library): the scrambled tables okin_study uploads to the device, and AS241.
#include <cstring>

#include "okin_study.cuh"

// Ranks, scrambled direction numbers dirs[n_sobol][52] and shifts[n_sobol] of n_variates validated
// variates under `seed`, as okin_study builds them; returns n_sobol (dirs / shift sized by the caller
// for n_variates Sobol' variates).
extern "C" int okin_emu_sobol_tables(uint64_t seed, int n_variates, const int32_t* kind, const int32_t* levels,
                                     int32_t* rank, uint64_t* dirs, uint64_t* shift) {
  OkinStudyHostTables h;
  h.index(n_variates, kind, levels);
  h.scramble(seed, n_variates);
  std::memcpy(rank, h.sobol_rank.data(), n_variates * sizeof(int32_t));
  std::memcpy(dirs, h.sobol_dirs.data(), (size_t)h.n_sobol * OKIN_SOBOL_BITS * sizeof(uint64_t));
  std::memcpy(shift, h.sobol_shift.data(), h.n_sobol * sizeof(uint64_t));
  return h.n_sobol;
}

extern "C" void okin_emu_ppnd16(const double* p, double* z, long long n) {
  for (long long k = 0; k < n; ++k) z[k] = okin_ppnd16(p[k]);
}
