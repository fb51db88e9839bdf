// Tolerance studies: the input generator and the reduction arithmetic, shared by the device kernels
// (okin_abi.cu) and the lane-emulation study driver of the tests.  The sampling contract and the
// reduction order are stated in include/okin.h and DESIGN.md section 10.
#pragma once

#include <math.h>
#include <stdint.h>

#include <vector>

#include "../../include/okin.h"
#include "okin_sobol.h"

#if defined(__CUDACC__)
#define OKIN_STUDY_HD __host__ __device__
#else
#define OKIN_STUDY_HD
#endif

// Reduction order inside a chunk: row r of the chunk belongs to partition r % OKIN_STUDY_PARTS.  A
// partition is reduced by Welford in row order; partitions are merged (Chan) in groups of
// OKIN_STUDY_GROUP consecutive ones, then the groups in order.  Nothing depends on which warp solved
// which instance.
#define OKIN_STUDY_GROUP 8
#define OKIN_STUDY_PARTS 512
#define OKIN_STUDY_GROUPS (OKIN_STUDY_PARTS / OKIN_STUDY_GROUP)

// Philox4x32-10 (Salmon et al., SC 2011), in place on the counter.
OKIN_STUDY_HD inline void okin_philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    c[0] = n0;
    c[1] = (uint32_t)p1;
    c[2] = n2;
    c[3] = (uint32_t)p0;
  }
}

// cos(pi x) for x in [0, 2).  The device uses the library's cospi; the host reduces to [0, 1/4]
// with exact steps (Sterbenz) and evaluates cos or sin of pi r there.
OKIN_STUDY_HD inline double okin_cospi(double x) {
#if defined(__CUDA_ARCH__)
  return cospi(x);
#else
  double r = x >= 1.0 ? 2.0 - x : x, sign = 1.0;
  if (r > 0.5) {
    r = 1.0 - r;
    sign = -1.0;
  }
  return r > 0.25 ? sign * sin(M_PI * (0.5 - r)) : sign * cos(M_PI * r);
#endif
}

// nominal + scale * z, rounded twice (never contracted to an FMA), like the two array operations it
// replaces in earlier drivers.
OKIN_STUDY_HD inline double okin_study_axpy(double scale, double z, double nominal) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(__dmul_rn(scale, z), nominal);
#else
  return scale * z + nominal;
#endif
}

// Generator tables (device or host addresses).  stride[v] / period: mixed-radix place value of grid
// variate v and the product of all grid levels; 0 = beyond 2^63 (that digit is 0, no wrap).
// sobol_rank[v]: Sobol' dimension of variate v (-1 for the other kinds); sobol_dirs[d][k] and
// sobol_shift[d]: the scrambled direction numbers and the digital shift of dimension d.  The device
// reads these three; the host (the lane emulation) derives the same integers from the seed.
struct OkinStudyTables {
  uint64_t seed, period;
  int32_t n_coords;
  const double* nominal;
  const double* scale;
  const int32_t* source;
  const int32_t* kind;
  const int32_t* levels;
  const uint64_t* stride;
  const int32_t* sobol_rank;
  const uint64_t* sobol_dirs;
  const uint64_t* sobol_shift;
};

// Host: V[d][0..52) of the unscrambled Sobol' sequence (include/okin.h), d < OKIN_SOBOL_DIMS.
inline void okin_sobol_directions(int d, uint64_t V[OKIN_SOBOL_BITS]) {
  uint64_t m[OKIN_SOBOL_BITS];
  const uint32_t poly = okin_sobol_poly[d];
  int deg = 0;
  while (poly >> (deg + 1)) ++deg;
  for (int k = 0; k < OKIN_SOBOL_BITS; ++k) {
    if (d == 0) {
      m[k] = 1;
    } else if (k < deg) {
      m[k] = okin_sobol_vinit[d][k];
    } else {
      uint64_t x = m[k - deg];
      for (int l = 1; l <= deg; ++l)
        if ((poly >> (deg - l)) & 1u) x ^= m[k - l] << l;
      m[k] = x;
    }
  }
  for (int k = 0; k < OKIN_SOBOL_BITS; ++k) V[k] = m[k] << (OKIN_SOBOL_BITS - 1 - k);
}

// Host: 52-bit word W(a) of Sobol' variate v's scramble stream (counter (a, 0, v, 1)).
inline uint64_t okin_sobol_scramble_word(uint64_t seed, int v, uint32_t a) {
  uint32_t c[4] = {a, 0u, (uint32_t)v, 1u};
  okin_philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return (((uint64_t)c[1] << 32) | c[0]) >> (64 - OKIN_SOBOL_BITS);
}

// Host: rows R_k of the scramble matrix M_v of Sobol' variate v, lower triangular in digit order
// (digit k = bit 51 - k) with unit diagonal.
inline void okin_sobol_matrix(uint64_t seed, int v, uint64_t row[OKIN_SOBOL_BITS]) {
  for (int k = 0; k < OKIN_SOBOL_BITS; ++k) {
    const uint64_t diag = UINT64_C(1) << (OKIN_SOBOL_BITS - 1 - k);
    row[k] = (okin_sobol_scramble_word(seed, v, (uint32_t)k) & ~(diag - 1)) | diag;
  }
}

// Host: M x; digit k of the result is the parity of R_k & x.
inline uint64_t okin_sobol_apply(const uint64_t row[OKIN_SOBOL_BITS], uint64_t x) {
  uint64_t y = 0;
  for (int k = 0; k < OKIN_SOBOL_BITS; ++k)
    y |= (uint64_t)(__builtin_popcountll(row[k] & x) & 1) << (OKIN_SOBOL_BITS - 1 - k);
  return y;
}

// x XOR dir[k] over the set bits k of g.
OKIN_STUDY_HD inline uint64_t okin_sobol_gray_xor(const uint64_t* dir, uint64_t g, uint64_t x) {
  for (; g; g &= g - 1) {
#if defined(__CUDA_ARCH__)
    x ^= dir[__ffsll((long long)g) - 1];
#else
    x ^= dir[__builtin_ctzll(g)];
#endif
  }
  return x;
}

// Wichura, Algorithm AS 241 (PPND16): the standard normal quantile of p in (0, 1), relative error
// about 1e-16.  The polynomials are evaluated with explicit fma so host and device round alike.
OKIN_STUDY_HD inline double okin_ppnd16(double p) {
  const double q = p - 0.5;
  if (fabs(q) <= 0.425) {
    const double r = fma(-q, q, 0.180625);
    const double num =
        fma(fma(fma(fma(fma(fma(fma(2.5090809287301226727e+3, r, 3.3430575583588128105e+4), r,
                                    6.7265770927008700853e+4), r, 4.5921953931549871457e+4), r,
                        1.3731693765509461125e+4), r, 1.9715909503065514427e+3), r, 1.3314166789178437745e+2), r,
            3.3871328727963666080e+0);
    const double den =
        fma(fma(fma(fma(fma(fma(fma(5.2264952788528545610e+3, r, 2.8729085735721942674e+4), r,
                                    3.9307895800092710610e+4), r, 2.1213794301586595867e+4), r,
                        5.3941960214247511077e+3), r, 6.8718700749205790830e+2), r, 4.2313330701600911252e+1), r,
            1.0);
    return q * num / den;
  }
  double r = sqrt(-log(q < 0.0 ? p : 1.0 - p)), z;
  if (r <= 5.0) {
    r -= 1.6;
    const double num =
        fma(fma(fma(fma(fma(fma(fma(7.74545014278341407640e-4, r, 2.27238449892691845833e-2), r,
                                    2.41780725177450611770e-1), r, 1.27045825245236838258e+0), r,
                        3.64784832476320460504e+0), r, 5.76949722146069140550e+0), r, 4.63033784615654529590e+0), r,
            1.42343711074968357734e+0);
    const double den =
        fma(fma(fma(fma(fma(fma(fma(1.05075007164441684324e-9, r, 5.47593808499534494600e-4), r,
                                    1.51986665636164571966e-2), r, 1.48103976427480074590e-1), r,
                        6.89767334985100004550e-1), r, 1.67638483018380384940e+0), r, 2.05319162663775882187e+0), r,
            1.0);
    z = num / den;
  } else {
    r -= 5.0;
    const double num =
        fma(fma(fma(fma(fma(fma(fma(2.01033439929228813265e-7, r, 2.71155556874348757815e-5), r,
                                    1.24266094738807843860e-3), r, 2.65321895265761230930e-2), r,
                        2.96560571828504891230e-1), r, 1.78482653991729133580e+0), r, 5.46378491116411436990e+0), r,
            6.65790464350110377720e+0);
    const double den =
        fma(fma(fma(fma(fma(fma(fma(2.04426310338993978564e-15, r, 1.42151175831644588870e-7), r,
                                    1.84631831751005468180e-5), r, 7.86869131145613259100e-4), r,
                        1.48753612908506148525e-2), r, 1.36929880922735805310e-1), r, 5.99832206555887937690e-1), r,
            1.0);
    z = num / den;
  }
  return q < 0.0 ? -z : z;
}

// Host: the place values and period above for validated variates (grid levels >= 2).
inline void okin_study_grid_places(int n_variates, const int32_t* kind, const int32_t* levels, uint64_t* stride,
                                   uint64_t* period) {
  uint64_t place = 1;
  bool saturated = false;
  for (int v = 0; v < n_variates; ++v) {
    stride[v] = 0;
    if (kind[v] != OKIN_VARIATE_GRID) continue;
    stride[v] = saturated ? 0 : place;
    if (!saturated && place > (UINT64_C(1) << 63) / (uint64_t)levels[v]) saturated = true;
    else if (!saturated) place *= (uint64_t)levels[v];
  }
  *period = saturated ? 0 : place;
}

// Host: the generator tables of validated variates that okin_study builds once per call and uploads:
// grid place values and period, Sobol' ranks, and the scrambled direction numbers
// dirs[rank][0..52) = M_v V[rank][k] and shifts shift[rank] = S_v of every Sobol' variate v.
struct OkinStudyHostTables {
  std::vector<uint64_t> stride, sobol_dirs, sobol_shift;
  std::vector<int32_t> sobol_rank;
  uint64_t period = 0;
  int n_sobol = 0;

  // Place values, period and ranks (cheap; the caller checks n_sobol before scramble()).
  void index(int n_variates, const int32_t* kind, const int32_t* levels) {
    stride.assign(n_variates + 1, 0);
    okin_study_grid_places(n_variates, kind, levels, stride.data(), &period);
    sobol_rank.assign(n_variates + 1, -1);
    n_sobol = 0;
    for (int v = 0; v < n_variates; ++v)
      if (kind[v] == OKIN_VARIATE_SOBOL_UNIFORM || kind[v] == OKIN_VARIATE_SOBOL_NORMAL) sobol_rank[v] = n_sobol++;
  }

  // The scramble of every Sobol' variate under `seed` (n_sobol <= OKIN_SOBOL_DIMS).
  void scramble(uint64_t seed, int n_variates) {
    sobol_dirs.assign((size_t)n_sobol * OKIN_SOBOL_BITS + 1, 0);
    sobol_shift.assign(n_sobol + 1, 0);
    for (int v = 0; v < n_variates; ++v) {
      const int d = sobol_rank[v];
      if (d < 0) continue;
      uint64_t row[OKIN_SOBOL_BITS], V[OKIN_SOBOL_BITS];
      okin_sobol_matrix(seed, v, row);
      okin_sobol_directions(d, V);
      for (int k = 0; k < OKIN_SOBOL_BITS; ++k)
        sobol_dirs[(size_t)d * OKIN_SOBOL_BITS + k] = okin_sobol_apply(row, V[k]);
      sobol_shift[d] = okin_sobol_scramble_word(seed, v, OKIN_SOBOL_BITS);
    }
  }
};

OKIN_STUDY_HD inline double okin_study_variate(const OkinStudyTables& t, uint64_t i, int v) {
  if (t.kind[v] == OKIN_VARIATE_GRID) {
    const uint64_t node = t.period ? i % t.period : i;
    const int64_t L = t.levels[v];
    const uint64_t d = t.stride[v] ? (node / t.stride[v]) % (uint64_t)L : 0;
    return (double)d / (double)(L - 1) * 2.0 - 1.0;
  }
  if (t.kind[v] == OKIN_VARIATE_SOBOL_UNIFORM || t.kind[v] == OKIN_VARIATE_SOBOL_NORMAL) {
    const uint64_t j = i / t.period, g = j ^ (j >> 1);
#if defined(__CUDA_ARCH__)
    const int d = t.sobol_rank[v];
    const uint64_t x = okin_sobol_gray_xor(t.sobol_dirs + (size_t)d * OKIN_SOBOL_BITS, g, t.sobol_shift[d]);
#else
    // M_v (XOR of V[d][k]) ^ S_v from the definition: by linearity over GF(2) the same integer as the
    // device's XOR of the scrambled direction numbers.
    int d = 0;
    for (int w = 0; w < v; ++w)
      d += t.kind[w] == OKIN_VARIATE_SOBOL_UNIFORM || t.kind[w] == OKIN_VARIATE_SOBOL_NORMAL;
    uint64_t V[OKIN_SOBOL_BITS], row[OKIN_SOBOL_BITS];
    okin_sobol_directions(d, V);
    okin_sobol_matrix(t.seed, v, row);
    const uint64_t x =
        okin_sobol_apply(row, okin_sobol_gray_xor(V, g, 0)) ^ okin_sobol_scramble_word(t.seed, v, OKIN_SOBOL_BITS);
#endif
    if (t.kind[v] == OKIN_VARIATE_SOBOL_UNIFORM) return (double)x * 0x1p-51 - 1.0;
    return okin_ppnd16((double)(2 * x + 1) * 0x1p-53);
  }
  uint32_t c[4] = {(uint32_t)i, (uint32_t)(i >> 32), (uint32_t)v, 0u};
  okin_philox4x32_10(c, (uint32_t)t.seed, (uint32_t)(t.seed >> 32));
  const double u = (double)((((uint64_t)c[1] << 32) | c[0]) >> 11) * 0x1p-53;
  if (t.kind[v] == OKIN_VARIATE_UNIFORM) return 2.0 * u - 1.0;
  const double u2 = (double)((((uint64_t)c[3] << 32) | c[2]) >> 11) * 0x1p-53;
  return sqrt(-2.0 * log(1.0 - u)) * okin_cospi(2.0 * u2);
}

OKIN_STUDY_HD inline double okin_study_coord(const OkinStudyTables& t, uint64_t i, int c) {
  const int v = t.source[c];
  return v < 0 ? t.nominal[c] : okin_study_axpy(t.scale[c], okin_study_variate(t, i, v), t.nominal[c]);
}

// Moments and extremes of one (step, quantity) over a set of instances.  argmin < 0: empty.
struct OkinMoments {
  int64_t count, nonfinite;
  double mean, m2, min, max;
  int64_t argmin, argmax;
};

OKIN_STUDY_HD inline void okin_moments_clear(OkinMoments& a) {
  a.count = a.nonfinite = 0;
  a.mean = a.m2 = a.min = a.max = 0.0;
  a.argmin = a.argmax = -1;
}

OKIN_STUDY_HD inline void okin_moments_push(OkinMoments& a, double x, int64_t id) {
  if (!isfinite(x)) {
    ++a.nonfinite;
    return;
  }
  ++a.count;
  const double d = x - a.mean;
  a.mean += d / (double)a.count;
  a.m2 += d * (x - a.mean);
  if (a.argmin < 0 || x < a.min || (x == a.min && id < a.argmin)) { a.min = x; a.argmin = id; }
  if (a.argmax < 0 || x > a.max || (x == a.max && id < a.argmax)) { a.max = x; a.argmax = id; }
}

// a <- a (+) b, Chan et al.; the extremes compare (value, id), so they are independent of the order.
OKIN_STUDY_HD inline void okin_moments_merge(OkinMoments& a, const OkinMoments& b) {
  a.nonfinite += b.nonfinite;
  if (b.count == 0) return;
  if (a.count == 0) {
    a.count = b.count;
    a.mean = b.mean;
    a.m2 = b.m2;
  } else {
    const int64_t n = a.count + b.count;
    const double d = b.mean - a.mean;
    a.mean += d * ((double)b.count / (double)n);
    a.m2 += b.m2 + d * d * ((double)a.count * (double)b.count / (double)n);
    a.count = n;
  }
  if (a.argmin < 0 || b.min < a.min || (b.min == a.min && b.argmin < a.argmin)) { a.min = b.min; a.argmin = b.argmin; }
  if (a.argmax < 0 || b.max > a.max || (b.max == a.max && b.argmax < a.argmax)) { a.max = b.max; a.argmax = b.argmax; }
}

// One chunk's per-instance solver outputs (instance-major, as okin_batch_io lays them out).
struct OkinStudyChunk {
  const double* positions;
  const double* metrics;
  const int32_t* iters;
  const double* max_residual;
  const int32_t* status;
  const int32_t* failed_step;
  int32_t n_steps, nout3, n_metrics;
};

// Value of quantity (kind, index) at row r, step s; false when the step was not accepted.
OKIN_STUDY_HD inline bool okin_study_fetch(const OkinStudyChunk& ch, int kind, int index, int64_t r, int s,
                                           double* x) {
  if (ch.status[r] != OKIN_STATUS_OK && s >= ch.failed_step[r]) return false;
  const size_t rs = (size_t)r * ch.n_steps + s;
  switch (kind) {
    case OKIN_QUANTITY_POSITION: *x = ch.positions[rs * ch.nout3 + index]; break;
    case OKIN_QUANTITY_METRIC: *x = ch.metrics[rs * ch.n_metrics + index]; break;
    case OKIN_QUANTITY_MAX_RESIDUAL: *x = ch.max_residual[rs]; break;
    default: *x = (double)ch.iters[rs]; break;
  }
  return true;
}

// Histogram bin of a finite value: 0 below lo, n_bins + 1 at or above hi.
OKIN_STUDY_HD inline int okin_study_bin(double x, double lo, double hi, int n_bins) {
  if (x < lo) return 0;
  if (x >= hi) return n_bins + 1;
  const int b = (int)((x - lo) / (hi - lo) * (double)n_bins);
  return 1 + (b < n_bins - 1 ? b : n_bins - 1);
}

// Rows p, p + OKIN_STUDY_PARTS, ... < rows of one column (step s, quantity (kind, index)) of a chunk
// whose first row is instance `base`: pushed in row order into m; count_bin(b) records a finite
// value in histogram bin b (n_bins > 0; lo, hi: the quantity's range).
template <class CountBin>
OKIN_STUDY_HD inline void okin_study_partition(const OkinStudyChunk& ch, int kind, int index, int s, long long p,
                                               long long rows, long long base, int n_bins, double lo, double hi,
                                               OkinMoments& m, CountBin count_bin) {
  for (long long r = p; r < rows; r += OKIN_STUDY_PARTS) {
    double x;
    if (!okin_study_fetch(ch, kind, index, r, s, &x)) continue;
    okin_moments_push(m, x, base + r);
    if (n_bins && isfinite(x)) count_bin(okin_study_bin(x, lo, hi, n_bins));
  }
}

// Integer results of one device: hist [SQ][n_bins + 2] (unused when n_bins == 0), status [4],
// failed_at [n_steps].  Exact in any order, summed over the devices.
struct OkinStudyCounts {
  const unsigned long long* hist;
  const unsigned long long* status;
  const unsigned long long* failed_at;
};

// Host: the study result of the accumulated moments acc[SQ] (NaN moments and extremes and -1
// arguments in an empty column) and of the counts of n_devices devices.
inline void okin_study_fold(const OkinMoments* acc, int n_steps, int SQ, int n_bins, const OkinStudyCounts* devices,
                            int n_devices, okin_study_out* out) {
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
  const size_t n_hist = n_bins ? (size_t)SQ * (n_bins + 2) : 0;
  for (size_t k = 0; k < n_hist; ++k) out->histogram[k] = 0;
  for (int k = 0; k < 4; ++k) out->status_counts[k] = 0;
  for (int s = 0; s < n_steps; ++s) out->failed_at_step[s] = 0;
  for (int d = 0; d < n_devices; ++d) {
    for (size_t k = 0; k < n_hist; ++k) out->histogram[k] += (int64_t)devices[d].hist[k];
    for (int k = 0; k < 4; ++k) out->status_counts[k] += (int64_t)devices[d].status[k];
    for (int s = 0; s < n_steps; ++s) out->failed_at_step[s] += (int64_t)devices[d].failed_at[s];
  }
}
