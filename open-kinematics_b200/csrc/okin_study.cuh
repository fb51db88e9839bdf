// Tolerance studies: the input generator and the reduction arithmetic, shared by the device kernels
// (okin_abi.cu) and the lane-emulation study driver of the tests.  The sampling contract and the
// reduction order are stated in include/okin.h and DESIGN.md section 10.
#pragma once

#include <math.h>
#include <stdint.h>

#include "../../include/okin.h"

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
struct OkinStudyTables {
  uint64_t seed, period;
  int32_t n_coords;
  const double* nominal;
  const double* scale;
  const int32_t* source;
  const int32_t* kind;
  const int32_t* levels;
  const uint64_t* stride;
};

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

OKIN_STUDY_HD inline double okin_study_variate(const OkinStudyTables& t, uint64_t i, int v) {
  if (t.kind[v] == OKIN_VARIATE_GRID) {
    const uint64_t node = t.period ? i % t.period : i;
    const int64_t L = t.levels[v];
    const uint64_t d = t.stride[v] ? (node / t.stride[v]) % (uint64_t)L : 0;
    return (double)d / (double)(L - 1) * 2.0 - 1.0;
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
