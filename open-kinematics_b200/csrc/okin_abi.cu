// C ABI (include/okin.h) and the sm_100a kernels behind it.
//
// Kernel mapping: one warp per suspension instance, W instances per CTA (W chosen per topology and
// kernel family by ensure_device), each warp working in its own slice of dynamic shared memory next
// to one shared copy of the hot topology tables; the grid is persistent (SM count x resident CTAs
// per SM) and its warps claim instances from a global counter.  The work is irregular fp64 on
// systems of tens of unknowns (SURVEY.md section 8d; measured: the shared-memory data pipe is the
// binding unit, profiles/r02_d_*), so tensor cores and TMA have nothing to act on; the only global
// traffic is the coalesced instance-major hardpoint read and state write.
// okin_sweep_kernel<FULL, SHIM, MAX_THREADS, SENS> has seven instantiations: full outputs (128 registers)
// and two lean families (128 / 168 registers), each with / without the camber-shim pre-solve, plus the
// full outputs with hardpoint sensitivities (no pre-solve); the continuity pass of the diagnostics is a
// second kernel on the same stream.
#include <cuda_runtime.h>

#include <pthread.h>
#include <sched.h>

#include <algorithm>
#include <condition_variable>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/okin.h"
#include "okin_core.cuh"
#include "okin_study.cuh"

// Kernel families.  The register cap follows from the CTA size limit (65536 / threads):
//   full outputs        512 threads -> 128 registers, up to 16 warps per SM
//   lean, 128 registers 512 threads                    (small topologies, long sweeps: occupancy wins)
//   lean, 168 registers 384 threads -> up to 12 warps  (ptxas only keeps the twelve operand loads of a
//                       gather-loop trip in flight when it is not squeezed for registers; at 128 it sinks
//                       every LDS to its DFMA, profiles/r02_*)
// Which lean family is faster depends on the topology (measured: flagship axle 168, corners and the
// 101-step T-bar axle 128), so the first large launch of a topology on a device times both.
#define OKIN_MAX_THREADS 512
#define OKIN_LEAN_WIDE_THREADS 384
enum { OKIN_FAM_LEAN_WIDE = 0, OKIN_FAM_FULL = 1, OKIN_FAM_LEAN = 2, OKIN_FAM_SENS = 3, OKIN_FAM_COUNT = 4 };
#ifndef OKIN_DRIFT
#define OKIN_DRIFT 1             // how many instances a warp may run ahead of the slowest warp of its CTA
#endif
#define OKIN_MAX_DEVICES 16
#define OKIN_PIPE_SLOTS 3        // streams / workspace slots of the host-buffer pipeline
#define OKIN_PIPE_CHUNK 32768   // instances per pipelined chunk

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

#define OKIN_CUDA(call)                                                                            \
  do {                                                                                             \
    cudaError_t err__ = (call);                                                                    \
    if (err__ != cudaSuccess)                                                                      \
      return fail(OKIN_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(err__));           \
  } while (0)

// cudaFuncSetAttribute + launch of the (process-wide) kernel functions must not interleave between
// threads driving different topologies on the same device.
std::mutex g_launch_mu[OKIN_MAX_DEVICES];

struct DeviceCopy {
  int device = 0;
  bool ready = false;
  int32_t* hdr = nullptr;
  int32_t* ib = nullptr;
  double* fb = nullptr;
  int num_sms = 0;
  // launch shape per kernel family (OKIN_FAM_*)
  struct Shape { int ctas_per_sm = 0, warps_per_cta = 0, smem_bytes = 0; } shape[OKIN_FAM_COUNT];
  int lean_family = -1;          // OKIN_FAM_LEAN or OKIN_FAM_LEAN_WIDE once timed on this device, -1 before
  double lean_tune_ms[2] = {0.0, 0.0};   // calibration times {wide, 128-register}
  int table_doubles = 0;
  int smem_optin = 0;
  // grow-only workspace for the host-buffer entry point
  void* ws = nullptr;
  size_t ws_bytes = 0;
  cudaStream_t streams[OKIN_PIPE_SLOTS] = {};
};

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

}  // namespace

struct okin_topology {
  std::vector<int32_t> hdr, ib;
  std::vector<double> fb;
  DeviceCopy dev[OKIN_MAX_DEVICES];
  std::mutex mu;
};

// Shared memory of a CTA = [topology tables (int32 blob)] [one state slice per warp].  The tables are
// copied once per (persistent) CTA so that every index lookup of the interpreter is a shared-memory
// load instead of a global one (ncu round 1: long-scoreboard stalls on __ldg were the top stall).
// SENS: sens_out = [n_instances][n_steps][NSENS][NOUT*3], sens_ws = okin_sens_ws_doubles per resident warp.
template <bool FULL, bool SHIM, int MAX_THREADS, bool SENS = false>
__global__ void __launch_bounds__(MAX_THREADS, 1)
okin_sweep_kernel(const int32_t* __restrict__ hdr, const int32_t* __restrict__ ib, const double* __restrict__ fb,
                  long long n_instances, int n_steps, OkinSolverCfg cfg, OkinKernelIO io, int n_iblob,
                  int table_doubles, unsigned long long* __restrict__ counter, double* sens_out, double* sens_ws) {
  // [section pointers][header][hot tables][one state slice per warp]
  const int32_t** sec = reinterpret_cast<const int32_t**>(okin_smem);
  int32_t* shdr = reinterpret_cast<int32_t*>(okin_smem + OKIN_S_COUNT);
  int32_t* tab = shdr + OKIN_HDR_SIZE;
  for (int i = threadIdx.x; i < OKIN_HDR_SIZE; i += blockDim.x) shdr[i] = hdr[i];
  const int n_hot = hdr[OKIN_H_NHOT];
  for (int i = threadIdx.x; i < n_hot; i += blockDim.x) tab[i] = ib[i];
  for (int i = threadIdx.x; i < OKIN_S_COUNT; i += blockDim.x) okin_resolve_section(hdr, tab, ib, i, sec);
  __syncthreads();
  hdr = shdr;
  OkinProgram pr{shdr, tab, fb, ib, sec};
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  double* sm = okin_smem + table_doubles + (size_t)warp * hdr[FULL ? OKIN_H_SMEM_DOUBLES : OKIN_H_SMEM_DOUBLES_LEAN];
  const int nin = hdr[OKIN_H_NIN], nout = hdr[OKIN_H_NOUT], nt = hdr[OKIN_H_NT], n = 3 * hdr[OKIN_H_NF];
  // Instances are claimed one at a time from a global counter (no static partition: a warp whose
  // instance is slow -- a failing sweep costs a few normal ones -- simply claims fewer).  The warps of
  // a CTA are kept loosely in step instead of meeting at a barrier: before claiming, a warp compares its
  // own count of finished instances with the slowest live warp of the CTA and waits only while it is
  // more than OKIN_DRIFT - 1 instances ahead.  The slowest warp never waits, so one slow instance delays
  // nobody until the others are OKIN_DRIFT instances ahead of it; and because the warps stay within a
  // few instances of each other they run the same code regions at about the same time, which keeps the
  // (large) interpreter in the instruction cache (round 1 measured -10 % at 1 M instances without any
  // coupling; a barrier per instance, OKIN_DRIFT == 1, cost 27 % on a batch with 0.8 % failing instances).
  __shared__ int s_done[OKIN_MAX_THREADS / 32];
  if ((threadIdx.x & 31) == 0) s_done[warp] = 0;
  __syncthreads();
  int mine = 0;
  for (;;) {
    // wait while too far ahead of the slowest live warp (finished warps park at INT_MAX)
    for (;;) {
      // (progress counters are read and written with shared-memory atomics: a defined cross-warp handshake)
      int v = (int)(threadIdx.x & 31) < warps_per_cta ? atomicOr(&s_done[threadIdx.x & 31], 0) : 0x7fffffff;
      for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
      if (mine - v < OKIN_DRIFT) break;
      __nanosleep(256);
    }
    long long i = 0;
    if ((threadIdx.x & 31) == 0) i = (long long)atomicAdd(counter, 1ull);
    i = __shfl_sync(0xffffffffu, i, 0);
    if (i >= n_instances) break;
    {
      OkinOutputs out;
      out.positions = io.positions ? io.positions + (size_t)i * n_steps * 3 * nout : nullptr;
      out.iters = io.iters ? io.iters + (size_t)i * n_steps : nullptr;
      out.max_residual = io.max_residual ? io.max_residual + (size_t)i * n_steps : nullptr;
      out.tangents = io.tangents ? io.tangents + (size_t)i * n_steps * nt * n : nullptr;
      out.velocities = io.velocities ? io.velocities + (size_t)i * n_steps * nt * 3 * nout : nullptr;
      out.health = io.tangent_health ? io.tangent_health + (size_t)i * n_steps * 2 : nullptr;
      out.metrics = io.metrics ? io.metrics + (size_t)i * n_steps * hdr[OKIN_H_NM] : nullptr;
      out.design = io.design ? io.design + (size_t)i * 3 * nout : nullptr;
      out.diagnostics = io.diagnostics ? io.diagnostics + (size_t)i * n_steps * hdr[OKIN_H_NDIAG] : nullptr;
      out.status = io.status + i;
      out.failed_step = io.failed_step + i;
      out.worst_row = io.worst_row ? io.worst_row + i : nullptr;
      if (SENS) {
        out.sensitivity = sens_out ? sens_out + (size_t)i * n_steps * hdr[OKIN_H_NSENS] * 3 * nout : nullptr;
        out.sens_ws = sens_ws + ((size_t)blockIdx.x * warps_per_cta + warp) * okin_sens_ws_doubles(hdr);
      }
      okin_sweep<FULL, SHIM, SENS>(pr, sm, io.hardpoints + (size_t)i * 3 * nin,
                 io.params ? io.params + (size_t)i * hdr[OKIN_H_NPARAM] : nullptr,
                 io.instance_targets ? io.instance_targets + (size_t)i * nt * n_steps : io.target_values, n_steps,
                 cfg, out);
      __syncwarp();
    }
    ++mine;
    if ((threadIdx.x & 31) == 0) atomicExch(&s_done[warp], mine);
  }
  if ((threadIdx.x & 31) == 0) atomicExch(&s_done[warp], 0x7fffffff);
}

// Second pass of the sweep diagnostics: one warp per instance walks the instance's position rows
// (okin_continuity).  Shared memory per warp: 32 displacement histories + thresholds + slots.
__global__ void okin_continuity_kernel(const int32_t* __restrict__ hdr, const int32_t* __restrict__ ib,
                                       long long n_instances, int n_steps, int stride,
                                       const double* __restrict__ positions, const int32_t* __restrict__ failed_step,
                                       double* diag, double* jumps) {
  const int32_t** sec = reinterpret_cast<const int32_t**>(okin_smem);
  for (int i = threadIdx.x; i < OKIN_S_COUNT; i += blockDim.x) okin_resolve_section(hdr, ib, ib, i, sec);
  __syncthreads();
  OkinProgram pr{hdr, ib, nullptr, ib, sec};
  const int warp = threadIdx.x >> 5, warps_per_cta = blockDim.x >> 5;
  double* scratch = okin_smem + OKIN_S_COUNT + (size_t)warp * (32 * stride + 64);
  const size_t nout3 = 3 * (size_t)hdr[OKIN_H_NOUT], nd = hdr[OKIN_H_NDIAG], nf = hdr[OKIN_H_NF];
  for (long long i = (long long)blockIdx.x * warps_per_cta + warp; i < n_instances;
       i += (long long)gridDim.x * warps_per_cta) {
    const int failed = failed_step[i];
    okin_continuity(pr, scratch, stride, positions + (size_t)i * n_steps * nout3, n_steps,
                    failed < 0 ? n_steps : failed, diag + (size_t)i * n_steps * nd,
                    jumps ? jumps + (size_t)i * n_steps * nf : nullptr);
    __syncwarp();
  }
}

// fp64 peak: 8 independent dependent-FMA chains per thread, enough threads to fill the chip.
__global__ void okin_dfma_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x * 1e-9, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6,
         x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

// ---- tolerance studies (okin_study.cuh) ------------------------------------------------------
// Inputs of instances base + r (ids == NULL) or ids[r], r < count: one thread per coordinate.
__global__ void okin_study_generate(OkinStudyTables t, long long base, const long long* __restrict__ ids,
                                    long long count, int nin3, int npar, double* __restrict__ hp,
                                    double* __restrict__ par) {
  const long long total = count * t.n_coords;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total;
       k += (long long)gridDim.x * blockDim.x) {
    const long long r = k / t.n_coords;
    const int c = (int)(k - r * t.n_coords);
    const double v = okin_study_coord(t, (uint64_t)(ids ? ids[r] : base + r), c);
    if (c < nin3) hp[r * nin3 + c] = v;
    else par[r * npar + (c - nin3)] = v;
  }
}

// Grid (ceil(S*Q / 32), OKIN_STUDY_GROUPS), block (32, OKIN_STUDY_GROUP): lane x owns column
// j = s * Q + q of the block's 32, row y of the block partition blockIdx.y * GROUP + y, which it
// reduces over the chunk rows p, p + PARTS, ...; the block then merges its GROUP partitions in order
// into groups[blockIdx.y][j].  Histogram counts go to `hist` through a per-block shared copy when
// `hist_shared` (n_bins small enough), else directly; status counts are taken by column block 0.
__global__ void __launch_bounds__(32 * OKIN_STUDY_GROUP)
okin_study_reduce(OkinStudyChunk ch, long long rows, long long base, int Q, const int32_t* __restrict__ qkind,
                  const int32_t* __restrict__ qindex, int n_bins, const double* __restrict__ lo,
                  const double* __restrict__ hi, int hist_shared, OkinMoments* __restrict__ groups,
                  unsigned long long* hist, unsigned long long* status_counts, unsigned long long* failed_at_step) {
  __shared__ OkinMoments part[OKIN_STUDY_GROUP][32];
  unsigned long long* sh = reinterpret_cast<unsigned long long*>(okin_smem);
  const int SQ = ch.n_steps * Q, tx = threadIdx.x, ty = threadIdx.y, nb2 = n_bins + 2;
  const int j = blockIdx.x * 32 + tx, p = blockIdx.y * OKIN_STUDY_GROUP + ty;
  if (hist_shared)
    for (int k = ty * 32 + tx; k < 32 * nb2; k += 32 * OKIN_STUDY_GROUP) sh[k] = 0ull;
  __syncthreads();
  OkinMoments m;
  okin_moments_clear(m);
  if (j < SQ) {
    const int s = j / Q, q = j - s * Q, kind = qkind[q], index = qindex[q];
    const double l = n_bins ? lo[q] : 0.0, h = n_bins ? hi[q] : 0.0;
    for (long long r = p; r < rows; r += OKIN_STUDY_PARTS) {
      double x;
      if (!okin_study_fetch(ch, kind, index, r, s, &x)) continue;
      okin_moments_push(m, x, base + r);
      if (n_bins && isfinite(x)) {
        const int b = okin_study_bin(x, l, h, n_bins);
        if (hist_shared) atomicAdd(&sh[tx * nb2 + b], 1ull);
        else atomicAdd(&hist[(size_t)j * nb2 + b], 1ull);
      }
    }
  }
  part[ty][tx] = m;
  if (blockIdx.x == 0 && tx == 0) {
    unsigned long long sc[4] = {0ull, 0ull, 0ull, 0ull};
    for (long long r = p; r < rows; r += OKIN_STUDY_PARTS) {
      const int st = ch.status[r], f = ch.failed_step[r];
      if (st >= 0 && st < 4) ++sc[st];
      if (f >= 0 && f < ch.n_steps) atomicAdd(&failed_at_step[f], 1ull);
    }
    for (int k = 0; k < 4; ++k)
      if (sc[k]) atomicAdd(&status_counts[k], sc[k]);
  }
  __syncthreads();
  if (ty == 0 && j < SQ) {
    OkinMoments g = part[0][tx];
    for (int k = 1; k < OKIN_STUDY_GROUP; ++k) okin_moments_merge(g, part[k][tx]);
    groups[(size_t)blockIdx.y * SQ + j] = g;
  }
  if (hist_shared)
    for (int k = ty * 32 + tx; k < 32 * nb2; k += 32 * OKIN_STUDY_GROUP) {
      const int col = blockIdx.x * 32 + k / nb2;
      if (sh[k] && col < SQ) atomicAdd(&hist[(size_t)col * nb2 + k % nb2], sh[k]);
    }
}

// chunk[j] = groups[0][j] (+) groups[1][j] (+) ... in group order.
__global__ void okin_study_merge(const OkinMoments* __restrict__ groups, int SQ, OkinMoments* __restrict__ chunk) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= SQ) return;
  OkinMoments g = groups[j];
  for (int k = 1; k < OKIN_STUDY_GROUPS; ++k) okin_moments_merge(g, groups[(size_t)k * SQ + j]);
  chunk[j] = g;
}

namespace {

const void* kernel_of(int fam, bool shim) {
  switch (fam) {
    case OKIN_FAM_SENS:
      return (const void*)okin_sweep_kernel<true, false, OKIN_MAX_THREADS, true>;
    case OKIN_FAM_FULL:
      return shim ? (const void*)okin_sweep_kernel<true, true, OKIN_MAX_THREADS>
                  : (const void*)okin_sweep_kernel<true, false, OKIN_MAX_THREADS>;
    case OKIN_FAM_LEAN:
      return shim ? (const void*)okin_sweep_kernel<false, true, OKIN_MAX_THREADS>
                  : (const void*)okin_sweep_kernel<false, false, OKIN_MAX_THREADS>;
    default:
      return shim ? (const void*)okin_sweep_kernel<false, true, OKIN_LEAN_WIDE_THREADS>
                  : (const void*)okin_sweep_kernel<false, false, OKIN_LEAN_WIDE_THREADS>;
  }
}

int ensure_device(okin_topology* t, int device, DeviceCopy** out) {
  if (device < 0 || device >= OKIN_MAX_DEVICES) return fail(OKIN_ERR_USAGE, "device id out of range");
  std::lock_guard<std::mutex> lock(t->mu);
  DeviceCopy& d = t->dev[device];
  if (!d.ready) {
    d.device = device;
    OKIN_CUDA(cudaSetDevice(device));
    OKIN_CUDA(cudaMalloc(&d.hdr, t->hdr.size() * sizeof(int32_t)));
    OKIN_CUDA(cudaMalloc(&d.ib, std::max<size_t>(t->ib.size(), 1) * sizeof(int32_t)));
    OKIN_CUDA(cudaMalloc(&d.fb, std::max<size_t>(t->fb.size(), 1) * sizeof(double)));
    OKIN_CUDA(cudaMemcpy(d.hdr, t->hdr.data(), t->hdr.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    OKIN_CUDA(cudaMemcpy(d.ib, t->ib.data(), t->ib.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    OKIN_CUDA(cudaMemcpy(d.fb, t->fb.data(), t->fb.size() * sizeof(double), cudaMemcpyHostToDevice));
    cudaDeviceProp prop;
    OKIN_CUDA(cudaGetDeviceProperties(&prop, device));
    d.num_sms = prop.multiProcessorCount;
    d.smem_optin = (int)prop.sharedMemPerBlockOptin;
    // CTA shape: W warps sharing one copy of the tables; pick the W that keeps the most warps resident
    // (shared memory, the 64K-register file at the instantiation's register cap, 1 KB per-CTA
    // reservation).  The lean instantiations own a shorter slice than the full ones.
    d.table_doubles =
        OKIN_S_COUNT + (int)((((size_t)t->hdr[OKIN_H_NHOT] + OKIN_HDR_SIZE) * sizeof(int32_t) + 7) / 8);
    const size_t table_bytes = (size_t)d.table_doubles * 8;
    const size_t sm_budget = prop.sharedMemPerMultiprocessor;
    for (int fam = 0; fam < OKIN_FAM_COUNT; ++fam) {
      const bool full = fam == OKIN_FAM_FULL || fam == OKIN_FAM_SENS;
      const size_t slice_bytes =
          (size_t)t->hdr[full ? OKIN_H_SMEM_DOUBLES : OKIN_H_SMEM_DOUBLES_LEAN] * sizeof(double);
      const int max_threads = fam == OKIN_FAM_LEAN_WIDE ? OKIN_LEAN_WIDE_THREADS : OKIN_MAX_THREADS;
      const int regs_per_thread = (int)(prop.regsPerMultiprocessor / max_threads) & ~7;
      int best_w = 0, best_ctas = 0;
      const char* forced = getenv("OKIN_WARPS_PER_CTA");     // kernel experiments
      for (int w = 1; w <= max_threads / 32; ++w) {
        if (forced && atoi(forced) > 0 && w != atoi(forced)) continue;
        const size_t cta_bytes = table_bytes + w * slice_bytes;
        if (cta_bytes > prop.sharedMemPerBlockOptin) break;
        int ctas = (int)(sm_budget / (cta_bytes + 1024));
        ctas = std::min(ctas, (int)(prop.regsPerMultiprocessor / (regs_per_thread * 32 * w)));
        ctas = std::min(ctas, 32);
        // most resident warps; on a tie the CTA shape closest to 6-8 warps (measured: 6 x 2 CTAs beats
        // 3 x 4 -- fewer copies of the tables -- and 12 x 1 -- a barrier group of 12 warps)
        const bool better_shape = best_w == 0 || (w <= 8 && w > best_w) || (best_w > 8 && w < best_w);
        if (ctas * w > best_w * best_ctas || (ctas * w == best_w * best_ctas && ctas * w > 0 && better_shape)) {
          best_w = w;
          best_ctas = ctas;
        }
      }
      if (best_w == 0 || best_ctas == 0)
        return fail(OKIN_ERR_USAGE, "topology needs more shared memory per CTA than the device offers");
      DeviceCopy::Shape& sh = d.shape[fam];
      sh.warps_per_cta = best_w;
      sh.smem_bytes = (int)(table_bytes + best_w * slice_bytes);
      sh.ctas_per_sm = 1 << 30;
      for (int shim = 0; shim < (fam == OKIN_FAM_SENS ? 1 : 2); ++shim) {
        const void* kernel = kernel_of(fam, shim != 0);
        OKIN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sh.smem_bytes));
        int ctas = 0;
        OKIN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, kernel, best_w * 32, sh.smem_bytes));
        sh.ctas_per_sm = std::min(sh.ctas_per_sm, ctas);
      }
      if (sh.ctas_per_sm < 1) return fail(OKIN_ERR_CUDA, "kernel does not fit on an SM");
    }
    if (const char* fixed = getenv("OKIN_LEAN_REGS"))        // 128 | 168: skip the calibration
      d.lean_family = atoi(fixed) == 128 ? OKIN_FAM_LEAN : OKIN_FAM_LEAN_WIDE;
    for (int k = 0; k < OKIN_PIPE_SLOTS; ++k)
      OKIN_CUDA(cudaStreamCreateWithFlags(&d.streams[k], cudaStreamNonBlocking));
    d.ready = true;
  }
  *out = &d;
  return OKIN_OK;
}

// One launch of a kernel family over [0, n_instances) on `stream`.
int launch_family(okin_topology* t, DeviceCopy* d, int fam, const OkinSolverCfg& c, cudaStream_t stream,
                  int64_t n_instances, int32_t n_steps, const okin_batch_io& io) {
  const DeviceCopy::Shape& sh = d->shape[fam];
  const int w = sh.warps_per_cta;
  const int64_t needed = (n_instances + w - 1) / w;
  const int64_t resident = (int64_t)d->num_sms * sh.ctas_per_sm;
  const int grid = (int)std::min<int64_t>(needed, resident);
  const void* kernel = kernel_of(fam, t->hdr[OKIN_H_NSHIM] > 0);
  // The attribute belongs to the kernel function of this device context, not to a topology: another
  // live topology may have lowered it since ensure_device ran, so it is set before every launch.
  std::lock_guard<std::mutex> launch_lock(g_launch_mu[d->device]);
  OKIN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sh.smem_bytes));
  // instance queue head of this launch (stream-ordered allocation: concurrent launches on other
  // streams have their own)
  unsigned long long* counter = nullptr;
  OKIN_CUDA(cudaMallocAsync(&counter, sizeof(unsigned long long), stream));
  OKIN_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream));
  long long n = (long long)n_instances;
  int n_iblob = (int)t->ib.size();
  OkinSolverCfg cfg = c;
  OkinKernelIO kio;
  std::memcpy(&kio, &io, sizeof(kio));
  // per-resident-warp scratch of the sensitivity phase (stream-ordered, like the counter)
  double* sens_out = io.hardpoint_sensitivity;
  double* sens_ws = nullptr;
  if (fam == OKIN_FAM_SENS)
    OKIN_CUDA(cudaMallocAsync(&sens_ws, (size_t)grid * w * okin_sens_ws_doubles(t->hdr.data()) * sizeof(double) + 8,
                              stream));
  void* args[] = {&d->hdr, &d->ib, &d->fb, &n, &n_steps, &cfg, &kio, &n_iblob, &d->table_doubles, &counter,
                  &sens_out, &sens_ws};
  const cudaError_t launch_err = cudaLaunchKernel(kernel, dim3(grid), dim3(w * 32), args, sh.smem_bytes, stream);
  OKIN_CUDA(cudaFreeAsync(counter, stream));
  if (sens_ws) OKIN_CUDA(cudaFreeAsync(sens_ws, stream));
  OKIN_CUDA(launch_err);
  return OKIN_OK;
}

int launch(okin_topology* t, DeviceCopy* d, const okin_solver_cfg* cfg, cudaStream_t stream, int64_t n_instances,
           int32_t n_steps, const okin_batch_io& io) {
  if (n_instances == 0) return OKIN_OK;
  OkinSolverCfg c{cfg->step_tol, cfg->coarse_tol, cfg->fine_tol, cfg->residual_tol, cfg->mu_init, cfg->max_iter,
                  cfg->use_predictor};
  // lean instantiation when no per-state tangent / metric / diagnostic output is wanted
  const bool full = io.tangents || io.velocities || io.tangent_health || io.metrics || io.diagnostics;
  int fam = io.hardpoint_sensitivity ? OKIN_FAM_SENS : OKIN_FAM_FULL;
  if (!full && !io.hardpoint_sensitivity) {
    fam = d->lean_family;
    const int64_t sample = 4 * (int64_t)d->num_sms * std::max(d->shape[OKIN_FAM_LEAN].ctas_per_sm * d->shape[OKIN_FAM_LEAN].warps_per_cta,
                                                              d->shape[OKIN_FAM_LEAN_WIDE].ctas_per_sm * d->shape[OKIN_FAM_LEAN_WIDE].warps_per_cta);
    if (fam < 0 && n_instances >= 2 * sample) {
      // Calibration, once per (topology, device): both lean families solve the same leading instances
      // of this batch (their results are identical; the batch launch below overwrites them again).
      cudaEvent_t e[2];
      OKIN_CUDA(cudaEventCreate(&e[0]));
      OKIN_CUDA(cudaEventCreate(&e[1]));
      const int order[2] = {OKIN_FAM_LEAN_WIDE, OKIN_FAM_LEAN};
      for (int k = 0; k < 2; ++k) {
        int rc = launch_family(t, d, order[k], c, stream, sample, n_steps, io);   // warm-up (code, tables)
        if (rc) return rc;
        OKIN_CUDA(cudaEventRecord(e[0], stream));
        rc = launch_family(t, d, order[k], c, stream, sample, n_steps, io);
        if (rc) return rc;
        OKIN_CUDA(cudaEventRecord(e[1], stream));
        OKIN_CUDA(cudaEventSynchronize(e[1]));
        float ms = 0.f;
        OKIN_CUDA(cudaEventElapsedTime(&ms, e[0], e[1]));
        d->lean_tune_ms[k] = ms;
      }
      cudaEventDestroy(e[0]);
      cudaEventDestroy(e[1]);
      d->lean_family = fam = d->lean_tune_ms[1] < d->lean_tune_ms[0] ? OKIN_FAM_LEAN : OKIN_FAM_LEAN_WIDE;
    }
    if (fam < 0) fam = OKIN_FAM_LEAN_WIDE;      // small batch: not worth timing, not recorded
  }
  int rc = launch_family(t, d, fam, c, stream, n_instances, n_steps, io);
  if (rc) return rc;
  if (io.diagnostics && t->hdr[OKIN_H_NDIAG] && n_steps > 0) {
    // continuity pass over the position rows the sweep kernel just wrote (same stream)
    const int stride = (n_steps - 1) | 1;   // odd: lanes walk their histories on different banks
    const size_t per_warp = ((size_t)32 * stride + 64) * sizeof(double);
    const size_t fixed = OKIN_S_COUNT * sizeof(double);   // section pointer table
    int cw = 4;
    while (cw > 1 && fixed + cw * per_warp > (size_t)d->smem_optin) cw >>= 1;
    if (fixed + cw * per_warp > (size_t)d->smem_optin)
      return fail(OKIN_ERR_USAGE, "too many sweep steps for the continuity diagnostics");
    OKIN_CUDA(cudaFuncSetAttribute(okin_continuity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(fixed + cw * per_warp)));
    const int cgrid = (int)std::min<int64_t>((n_instances + cw - 1) / cw, (int64_t)d->num_sms * 8);
    okin_continuity_kernel<<<cgrid, cw * 32, fixed + cw * per_warp, stream>>>(
        d->hdr, d->ib, (long long)n_instances, n_steps, stride, io.positions, io.failed_step, io.diagnostics,
        io.jumps);
    OKIN_CUDA(cudaGetLastError());
  }
  return OKIN_OK;
}

int check_common(const okin_topology* t, const okin_solver_cfg* cfg, int64_t n_instances, int32_t n_steps,
                 const okin_batch_io* io) {
  if (!t || !cfg || !io) return fail(OKIN_ERR_USAGE, "null topology, config or io");
  const void *hp = io->hardpoints, *tv = io->target_values, *status = io->status, *failed = io->failed_step;
  if (n_instances < 0 || n_steps < 0) return fail(OKIN_ERR_USAGE, "negative size");
  if (n_instances > 0 && (!hp || !status || !failed)) return fail(OKIN_ERR_USAGE, "null required buffer");
  if (n_steps > 0 && t->hdr[OKIN_H_NT] > 0 && !tv && !io->instance_targets)
    return fail(OKIN_ERR_USAGE, "null target_values (and no instance_targets)");
  if ((io->diagnostics || io->jumps) && !t->hdr[OKIN_H_NDIAG])
    return fail(OKIN_ERR_USAGE, "topology was compiled without a diagnostic program");
  if (io->jumps && !io->diagnostics) return fail(OKIN_ERR_USAGE, "jumps output needs the diagnostics output");
  if (io->hardpoint_sensitivity && t->hdr[OKIN_H_NSHIM] > 0)
    return fail(OKIN_ERR_USAGE, "hardpoint sensitivities are not available on a topology with camber-shim records "
                                "(the shim pre-solve is not differentiated)");
  if (cfg->max_iter < 1 || !(cfg->step_tol > 0.0) || !(cfg->coarse_tol >= cfg->step_tol)) return fail(OKIN_ERR_USAGE, "invalid solver config");
  return OKIN_OK;
}

// ---- host-buffer path ------------------------------------------------------------------------
// Every per-instance array of a call is one "lane" of a pipeline slot: (host pointer, bytes per
// instance).  scratch: device buffer needed although the caller does not want the array back.
struct Lane { const void* host; size_t per_inst; bool input; bool scratch; size_t bytes; };
constexpr int kLanes = 17;

struct HostBatch {
  Lane lanes[kLanes];
  size_t chunk, b_tv, slot_bytes, tv_count;
  const okin_batch_io* io;
  int32_t n_steps;
  HostBatch(const okin_topology* t, int64_t n_instances, int32_t n_steps_, const okin_batch_io* io_) : io(io_), n_steps(n_steps_) {
    const int32_t* h = t->hdr.data();
    const size_t nin3 = 3 * (size_t)h[OKIN_H_NIN], nout3 = 3 * (size_t)h[OKIN_H_NOUT];
    const size_t nt = h[OKIN_H_NT], n = 3 * (size_t)h[OKIN_H_NF];
    const size_t nm = (size_t)h[OKIN_H_NM], npar = (size_t)h[OKIN_H_NPARAM], nd = (size_t)h[OKIN_H_NDIAG];
    const size_t S = (size_t)n_steps;
    const Lane init[kLanes] = {
        {io->hardpoints, nin3 * 8, true, false, 0},
        {(io->params && npar) ? io->params : nullptr, npar * 8, true, false, 0},
        {io->status, 4, false, false, 0},
        {io->failed_step, 4, false, false, 0},
        {io->positions, S * nout3 * 8, false, io->diagnostics && !io->positions, 0},
        {io->iters, S * 4, false, false, 0},
        {io->max_residual, S * 8, false, false, 0},
        {io->tangents, S * nt * n * 8, false, false, 0},
        {io->velocities, S * nt * nout3 * 8, false, false, 0},
        {io->tangent_health, S * 2 * 8, false, false, 0},
        {(io->metrics && nm) ? io->metrics : nullptr, S * nm * 8, false, false, 0},
        {io->design, nout3 * 8, false, false, 0},
        {io->diagnostics, S * nd * 8, false, false, 0},
        {io->jumps, S * (n / 3) * 8, false, false, 0},
        {(io->instance_targets && nt * S) ? io->instance_targets : nullptr, nt * S * 8, true, false, 0},
        {io->worst_row, 4, false, false, 0},
        {io->hardpoint_sensitivity, S * (size_t)h[OKIN_H_NSENS] * nout3 * 8, false, false, 0},
    };
    std::memcpy(lanes, init, sizeof(init));
    chunk = (size_t)std::min<int64_t>(std::max<int64_t>(n_instances, 1), OKIN_PIPE_CHUNK);
    tv_count = nt * S;
    b_tv = align(std::max<size_t>(tv_count, 1) * 8);
    slot_bytes = b_tv;
    for (Lane& l : lanes) {
      l.bytes = (l.host || l.scratch) ? align(chunk * std::max<size_t>(l.per_inst, 1)) : 0;
      slot_bytes += l.bytes;
    }
  }
  static size_t align(size_t b) { return (b + 255) & ~(size_t)255; }
};

struct Shard {
  int device = 0;
  DeviceCopy* d = nullptr;
  int64_t begin = 0, count = 0;
  int rc = OKIN_OK;
  std::string err;
};

// Moves the calling thread onto the CPUs of the NUMA node `device` hangs off (sysfs); false when
// the box does not say (virtual machines often report node -1).
bool bind_thread_near_device(int device) {
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return false;
  for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
  int node = -1;
  {
    std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/numa_node");
    if (!(f >> node) || node < 0) return false;
  }
  std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
  std::string list;
  if (!std::getline(f, list) || list.empty()) return false;
  cpu_set_t set;
  CPU_ZERO(&set);
  size_t pos = 0;
  int n_set = 0;
  while (pos < list.size()) {
    size_t end = list.find(',', pos);
    if (end == std::string::npos) end = list.size();
    const std::string tok = list.substr(pos, end - pos);
    const size_t dash = tok.find('-');
    const int lo = std::atoi(tok.c_str());
    const int hi = dash == std::string::npos ? lo : std::atoi(tok.c_str() + dash + 1);
    for (int c = lo; c <= hi && c < CPU_SETSIZE; ++c) { CPU_SET(c, &set); ++n_set; }
    pos = end + 1;
  }
  if (n_set == 0) return false;
  // keep only CPUs this process may run on
  cpu_set_t allowed;
  if (sched_getaffinity(0, sizeof(allowed), &allowed) == 0) {
    cpu_set_t both;
    CPU_AND(&both, &set, &allowed);
    if (CPU_COUNT(&both) == 0) return false;
    set = both;
  }
  return pthread_setaffinity_np(pthread_self(), sizeof(set), &set) == 0;
}

// One device's instance range: chunks rotate over OKIN_PIPE_SLOTS streams, so the H2D copy of chunk
// k+1 and the D2H copy of chunk k-1 overlap the kernel of chunk k.  Whatever happens, the streams are
// drained before returning: no copy may still be writing into caller buffers after the call.
void run_shard(okin_topology* t, const okin_solver_cfg* cfg, const HostBatch& hb, Shard& sh) {
  DeviceCopy* d = sh.d;
  auto drain = [&] {
    for (int k = 0; k < OKIN_PIPE_SLOTS; ++k) cudaStreamSynchronize(d->streams[k]);
  };
  auto cuda_fail = [&](const char* what, cudaError_t err) {
    drain();
    sh.rc = OKIN_ERR_CUDA;
    sh.err = std::string(what) + ": " + cudaGetErrorString(err);
  };
#define OKIN_SHARD_CUDA(call)                                  \
  do {                                                         \
    cudaError_t err__ = (call);                                \
    if (err__ != cudaSuccess) { cuda_fail(#call, err__); return; } \
  } while (0)
  OKIN_SHARD_CUDA(cudaSetDevice(sh.device));
  const size_t chunk = hb.chunk;
  const int slots = (int)std::min<int64_t>(OKIN_PIPE_SLOTS, (sh.count + (int64_t)chunk - 1) / (int64_t)chunk);
  if (hb.slot_bytes * slots > d->ws_bytes) {
    if (d->ws) OKIN_SHARD_CUDA(cudaFree(d->ws));
    d->ws = nullptr;
    d->ws_bytes = 0;
    OKIN_SHARD_CUDA(cudaMalloc(&d->ws, hb.slot_bytes * slots));
    d->ws_bytes = hb.slot_bytes * slots;
  }
  int64_t done = 0;
  for (int ck = 0; done < sh.count; ++ck, done += (int64_t)chunk) {
    const int slot = ck % slots;
    const size_t c = (size_t)std::min<int64_t>((int64_t)chunk, sh.count - done);
    const size_t b0 = (size_t)(sh.begin + done);
    cudaStream_t st = d->streams[slot];
    char* p = (char*)d->ws + hb.slot_bytes * slot;
    void* dev[kLanes];
    double* w_tv = (double*)p;
    p += hb.b_tv;
    for (int l = 0; l < kLanes; ++l) {
      dev[l] = hb.lanes[l].bytes ? p : nullptr;
      p += hb.lanes[l].bytes;
    }
    for (int l = 0; l < kLanes; ++l)
      if (dev[l] && hb.lanes[l].input)
        OKIN_SHARD_CUDA(cudaMemcpyAsync(dev[l], (const char*)hb.lanes[l].host + b0 * hb.lanes[l].per_inst,
                                        c * hb.lanes[l].per_inst, cudaMemcpyHostToDevice, st));
    if (hb.tv_count && hb.io->target_values && ck < slots)
      OKIN_SHARD_CUDA(cudaMemcpyAsync(w_tv, hb.io->target_values, hb.tv_count * 8, cudaMemcpyHostToDevice, st));
    okin_batch_io dio{};
    dio.hardpoints = (const double*)dev[0];
    dio.params = (const double*)dev[1];
    dio.target_values = hb.io->target_values ? w_tv : nullptr;
    dio.status = (int32_t*)dev[2];
    dio.failed_step = (int32_t*)dev[3];
    dio.positions = (double*)dev[4];
    dio.iters = (int32_t*)dev[5];
    dio.max_residual = (double*)dev[6];
    dio.tangents = (double*)dev[7];
    dio.velocities = (double*)dev[8];
    dio.tangent_health = (double*)dev[9];
    dio.metrics = (double*)dev[10];
    dio.design = (double*)dev[11];
    dio.diagnostics = (double*)dev[12];
    dio.jumps = (double*)dev[13];
    dio.instance_targets = (const double*)dev[14];
    dio.worst_row = (int32_t*)dev[15];
    dio.hardpoint_sensitivity = (double*)dev[16];
    const int rc = launch(t, d, cfg, st, (int64_t)c, hb.n_steps, dio);
    if (rc) {
      drain();
      sh.rc = rc;
      sh.err = g_last_error;
      return;
    }
    for (int l = 0; l < kLanes; ++l)
      if (dev[l] && hb.lanes[l].host && !hb.lanes[l].input && hb.lanes[l].per_inst)
        OKIN_SHARD_CUDA(cudaMemcpyAsync((char*)const_cast<void*>(hb.lanes[l].host) + b0 * hb.lanes[l].per_inst, dev[l],
                                        c * hb.lanes[l].per_inst, cudaMemcpyDeviceToHost, st));
  }
  for (int k = 0; k < OKIN_PIPE_SLOTS; ++k) OKIN_SHARD_CUDA(cudaStreamSynchronize(d->streams[k]));
#undef OKIN_SHARD_CUDA
}

// ---- tolerance studies ------------------------------------------------------------------------
// Generator part of a study descriptor; fills the mixed-radix place values of the grid variates.
int study_check_generator(const okin_topology* t, const okin_study_desc* desc, std::vector<uint64_t>* stride,
                          uint64_t* period) {
  if (!t || !desc) return fail(OKIN_ERR_USAGE, "null topology or study descriptor");
  const int32_t* h = t->hdr.data();
  const int nc = 3 * h[OKIN_H_NIN] + h[OKIN_H_NPARAM], nv = desc->n_variates;
  if (desc->n_coords != nc) return fail(OKIN_ERR_USAGE, "study n_coords must be 3 * n_in_points + n_params");
  if (nv < 0) return fail(OKIN_ERR_USAGE, "negative n_variates");
  if (!desc->nominal || !desc->source || !desc->scale || (nv > 0 && (!desc->variate_kind || !desc->grid_levels)))
    return fail(OKIN_ERR_USAGE, "null study generator table");
  for (int v = 0; v < nv; ++v) {
    const int kind = desc->variate_kind[v];
    if (kind < OKIN_VARIATE_NORMAL || kind > OKIN_VARIATE_GRID) return fail(OKIN_ERR_USAGE, "unknown variate kind");
    if (kind == OKIN_VARIATE_GRID && desc->grid_levels[v] < 2)
      return fail(OKIN_ERR_USAGE, "a grid variate needs at least 2 levels");
  }
  stride->assign(nv + 1, 0);
  okin_study_grid_places(nv, desc->variate_kind, desc->grid_levels, stride->data(), period);
  for (int c = 0; c < nc; ++c) {
    if (desc->source[c] < -1 || desc->source[c] >= nv) return fail(OKIN_ERR_USAGE, "study source out of range");
    if (!std::isfinite(desc->nominal[c]) || !std::isfinite(desc->scale[c]))
      return fail(OKIN_ERR_USAGE, "non-finite study nominal or scale");
  }
  return OKIN_OK;
}

int study_check_quantities(const okin_topology* t, int32_t n_steps, const okin_study_desc* desc,
                           const okin_study_out* out) {
  const int32_t* h = t->hdr.data();
  const int Q = desc->n_quantities;
  if (Q < 1) return fail(OKIN_ERR_USAGE, "a study needs at least one quantity");
  if (!desc->quantity_kind || !desc->quantity_index) return fail(OKIN_ERR_USAGE, "null study quantity table");
  for (int q = 0; q < Q; ++q) {
    const int kind = desc->quantity_kind[q], index = desc->quantity_index[q];
    if (kind == OKIN_QUANTITY_POSITION) {
      if (index < 0 || index >= 3 * h[OKIN_H_NOUT]) return fail(OKIN_ERR_USAGE, "study position quantity out of range");
    } else if (kind == OKIN_QUANTITY_METRIC) {
      if (!h[OKIN_H_NM]) return fail(OKIN_ERR_USAGE, "metric quantity on a topology compiled without a metric program");
      if (index < 0 || index >= h[OKIN_H_NM]) return fail(OKIN_ERR_USAGE, "study metric quantity out of range");
    } else if (kind != OKIN_QUANTITY_MAX_RESIDUAL && kind != OKIN_QUANTITY_NFEV) {
      return fail(OKIN_ERR_USAGE, "unknown study quantity kind");
    }
  }
  if (desc->n_bins < 0 || desc->n_bins > 4096) return fail(OKIN_ERR_USAGE, "n_bins must lie in 0..4096");
  if (desc->n_bins > 0) {
    if (!desc->hist_lo || !desc->hist_hi) return fail(OKIN_ERR_USAGE, "null histogram range");
    for (int q = 0; q < Q; ++q)
      if (!std::isfinite(desc->hist_lo[q]) || !std::isfinite(desc->hist_hi[q]) || !(desc->hist_lo[q] < desc->hist_hi[q]))
        return fail(OKIN_ERR_USAGE, "histogram range needs finite lo < hi");
  }
  if (!out || !out->count || !out->nonfinite || !out->mean || !out->m2 || !out->min || !out->max || !out->argmin ||
      !out->argmax || !out->status_counts || !out->failed_at_step || (desc->n_bins > 0 && !out->histogram))
    return fail(OKIN_ERR_USAGE, "null study output");
  (void)n_steps;
  return OKIN_OK;
}

// Device allocations of one study call on one device, released together.
struct DeviceAllocs {
  std::vector<void*> dev, host;
  ~DeviceAllocs() {
    for (void* p : dev) cudaFree(p);
    for (void* p : host) cudaFreeHost(p);
  }
  template <class T>
  cudaError_t alloc(T** p, size_t n) {
    *p = nullptr;
    const cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) dev.push_back(*p);
    return e;
  }
  template <class T>
  cudaError_t alloc_host(T** p, size_t n) {
    *p = nullptr;
    const cudaError_t e = cudaHostAlloc((void**)p, std::max<size_t>(n, 1) * sizeof(T), cudaHostAllocPortable);
    if (e == cudaSuccess) host.push_back(*p);
    return e;
  }
};

// The generator tables of `desc` on the current device.
int upload_study_tables(const okin_study_desc* desc, const std::vector<uint64_t>& stride, uint64_t period,
                        DeviceAllocs& a, OkinStudyTables* t) {
  const int nc = desc->n_coords, nv = desc->n_variates;
  double *nominal, *scale;
  int32_t *source, *kind, *levels;
  uint64_t* st;
  OKIN_CUDA(a.alloc(&nominal, nc));
  OKIN_CUDA(a.alloc(&scale, nc));
  OKIN_CUDA(a.alloc(&source, nc));
  OKIN_CUDA(a.alloc(&kind, nv));
  OKIN_CUDA(a.alloc(&levels, nv));
  OKIN_CUDA(a.alloc(&st, nv));
  OKIN_CUDA(cudaMemcpy(nominal, desc->nominal, nc * sizeof(double), cudaMemcpyHostToDevice));
  OKIN_CUDA(cudaMemcpy(scale, desc->scale, nc * sizeof(double), cudaMemcpyHostToDevice));
  OKIN_CUDA(cudaMemcpy(source, desc->source, nc * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (nv > 0) {
    OKIN_CUDA(cudaMemcpy(kind, desc->variate_kind, nv * sizeof(int32_t), cudaMemcpyHostToDevice));
    OKIN_CUDA(cudaMemcpy(levels, desc->grid_levels, nv * sizeof(int32_t), cudaMemcpyHostToDevice));
    OKIN_CUDA(cudaMemcpy(st, stride.data(), nv * sizeof(uint64_t), cudaMemcpyHostToDevice));
  }
  *t = OkinStudyTables{desc->seed, period, nc, nominal, scale, source, kind, levels, st};
  return OKIN_OK;
}

int launch_study_generate(const OkinStudyTables& t, long long base, const long long* ids, long long count, int nin3,
                          int npar, double* hp, double* par, int num_sms, cudaStream_t stream) {
  if (count == 0) return OKIN_OK;
  const long long total = count * t.n_coords;
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)num_sms * 16);
  okin_study_generate<<<grid, 256, 0, stream>>>(t, base, ids, count, nin3, npar, hp, par);
  OKIN_CUDA(cudaGetLastError());
  return OKIN_OK;
}

// State shared by the device threads of one okin_study call.  Chunk k goes to device k % G; a device
// starts chunk k only when k < next + window, so the reorder ring (window = G x slots chunk partials)
// never overflows and host memory does not grow with the number of instances.
struct StudyRun {
  okin_topology* t;
  const okin_solver_cfg* cfg;
  int64_t n;
  int32_t S;
  const double* target_values;
  const okin_study_desc* desc;
  std::vector<uint64_t> stride;
  uint64_t period = 0;
  int Q = 0, SQ = 0, nb = 0, n_devices = 0, slots = 0;
  bool want_pos = false, want_met = false;
  int64_t n_chunks = 0, window = 0;
  std::mutex mu;
  std::condition_variable cv;
  int64_t next = 0;
  bool abort = false;
  std::vector<std::vector<OkinMoments>> ring;
  std::vector<char> have;
  std::vector<OkinMoments> acc;

  void deliver(int64_t k, const OkinMoments* part) {
    std::lock_guard<std::mutex> lock(mu);
    const size_t r = (size_t)(k % window);
    ring[r].assign(part, part + SQ);
    have[r] = 1;
    while (next < n_chunks && have[(size_t)(next % window)]) {
      const size_t rr = (size_t)(next % window);
      for (int j = 0; j < SQ; ++j) okin_moments_merge(acc[j], ring[rr][j]);
      have[rr] = 0;
      ++next;
    }
    cv.notify_all();
  }
  bool wait_window(int64_t k) {
    std::unique_lock<std::mutex> lock(mu);
    cv.wait(lock, [&] { return abort || k < next + window; });
    return !abort;
  }
  void stop() {
    std::lock_guard<std::mutex> lock(mu);
    abort = true;
    cv.notify_all();
  }
};

// Integer results of one device (exact in any order, summed over devices at the end).
struct StudyShard {
  int index = 0, device = 0;
  DeviceCopy* d = nullptr;
  std::vector<unsigned long long> hist, status, failed_at;
  int rc = OKIN_OK;
  std::string err;
};

int run_study_shard_body(StudyRun& run, StudyShard& sh, DeviceAllocs& a) {
  DeviceCopy* d = sh.d;
  OKIN_CUDA(cudaSetDevice(sh.device));
  const int32_t* h = run.t->hdr.data();
  const int nin3 = 3 * h[OKIN_H_NIN], npar = h[OKIN_H_NPARAM], nout3 = 3 * h[OKIN_H_NOUT], nm = h[OKIN_H_NM];
  const int nt = h[OKIN_H_NT], S = run.S, Q = run.Q, SQ = run.SQ, nb = run.nb;
  const size_t CH = OKIN_STUDY_CHUNK;
  const int64_t G = run.n_devices;
  const int64_t n_mine = run.n_chunks > sh.index ? (run.n_chunks - sh.index + G - 1) / G : 0;
  const int slots = (int)std::min<int64_t>(run.slots, n_mine);
  OkinStudyTables tab;
  int rc = upload_study_tables(run.desc, run.stride, run.period, a, &tab);
  if (rc) return rc;
  int32_t *qkind, *qindex;
  double *lo = nullptr, *hi = nullptr, *tv = nullptr;
  OKIN_CUDA(a.alloc(&qkind, Q));
  OKIN_CUDA(a.alloc(&qindex, Q));
  OKIN_CUDA(cudaMemcpy(qkind, run.desc->quantity_kind, Q * sizeof(int32_t), cudaMemcpyHostToDevice));
  OKIN_CUDA(cudaMemcpy(qindex, run.desc->quantity_index, Q * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (nb) {
    OKIN_CUDA(a.alloc(&lo, Q));
    OKIN_CUDA(a.alloc(&hi, Q));
    OKIN_CUDA(cudaMemcpy(lo, run.desc->hist_lo, Q * sizeof(double), cudaMemcpyHostToDevice));
    OKIN_CUDA(cudaMemcpy(hi, run.desc->hist_hi, Q * sizeof(double), cudaMemcpyHostToDevice));
  }
  if ((size_t)nt * S) {
    OKIN_CUDA(a.alloc(&tv, (size_t)nt * S));
    OKIN_CUDA(cudaMemcpy(tv, run.target_values, (size_t)nt * S * sizeof(double), cudaMemcpyHostToDevice));
  }
  const size_t nb2 = (size_t)nb + 2, n_hist = nb ? (size_t)SQ * nb2 : 0;
  unsigned long long *hist = nullptr, *status_counts, *failed_at;
  if (n_hist) OKIN_CUDA(a.alloc(&hist, n_hist));
  OKIN_CUDA(a.alloc(&status_counts, 4));
  OKIN_CUDA(a.alloc(&failed_at, S));
  if (n_hist) OKIN_CUDA(cudaMemset(hist, 0, n_hist * sizeof(unsigned long long)));
  OKIN_CUDA(cudaMemset(status_counts, 0, 4 * sizeof(unsigned long long)));
  OKIN_CUDA(cudaMemset(failed_at, 0, std::max(S, 1) * sizeof(unsigned long long)));
  struct Slot {
    double *hp = nullptr, *par = nullptr, *pos = nullptr, *met = nullptr, *res = nullptr;
    int32_t *iters = nullptr, *status = nullptr, *failed = nullptr;
    OkinMoments *groups = nullptr, *chunk = nullptr, *host = nullptr;
  } slot[OKIN_PIPE_SLOTS];
  for (int k = 0; k < slots; ++k) {
    Slot& s = slot[k];
    OKIN_CUDA(a.alloc(&s.hp, CH * nin3));
    if (npar) OKIN_CUDA(a.alloc(&s.par, CH * npar));
    if (run.want_pos) OKIN_CUDA(a.alloc(&s.pos, CH * S * nout3));
    if (run.want_met) OKIN_CUDA(a.alloc(&s.met, CH * S * nm));
    OKIN_CUDA(a.alloc(&s.res, CH * S));
    OKIN_CUDA(a.alloc(&s.iters, CH * S));
    OKIN_CUDA(a.alloc(&s.status, CH));
    OKIN_CUDA(a.alloc(&s.failed, CH));
    OKIN_CUDA(a.alloc(&s.groups, (size_t)OKIN_STUDY_GROUPS * SQ));
    OKIN_CUDA(a.alloc(&s.chunk, SQ));
    OKIN_CUDA(a.alloc_host(&s.host, SQ));
  }
  const int hist_shared = nb && 32 * nb2 * sizeof(unsigned long long) <= 32 * 1024;
  const size_t hist_smem = hist_shared ? 32 * nb2 * sizeof(unsigned long long) : 0;
  auto finish = [&](int64_t l) -> int {   // deliver the partial of this device's l-th chunk
    OKIN_CUDA(cudaStreamSynchronize(d->streams[l % slots]));
    run.deliver(sh.index + l * G, slot[l % slots].host);
    return OKIN_OK;
  };
  for (int64_t l = 0; l < n_mine; ++l) {
    const int64_t k = sh.index + l * G;
    Slot& s = slot[l % slots];
    cudaStream_t st = d->streams[l % slots];
    if (l >= slots && (rc = finish(l - slots))) return rc;
    if (!run.wait_window(k)) return fail(OKIN_ERR_CUDA, "study stopped by another device's error");
    const long long base = k * (long long)CH, c = std::min<long long>((long long)CH, run.n - base);
    rc = launch_study_generate(tab, base, nullptr, c, nin3, npar, s.hp, s.par, d->num_sms, st);
    if (rc) return rc;
    okin_batch_io io{};
    io.hardpoints = s.hp;
    io.params = s.par;
    io.target_values = tv;
    io.status = s.status;
    io.failed_step = s.failed;
    io.positions = s.pos;
    io.iters = s.iters;
    io.max_residual = s.res;
    io.metrics = s.met;
    rc = launch(run.t, d, run.cfg, st, c, S, io);
    if (rc) return rc;
    const OkinStudyChunk ch{s.pos, s.met, s.iters, s.res, s.status, s.failed, S, nout3, nm};
    okin_study_reduce<<<dim3((SQ + 31) / 32, OKIN_STUDY_GROUPS), dim3(32, OKIN_STUDY_GROUP), hist_smem, st>>>(
        ch, c, base, Q, qkind, qindex, nb, lo, hi, hist_shared, s.groups, hist, status_counts, failed_at);
    OKIN_CUDA(cudaGetLastError());
    okin_study_merge<<<(SQ + 127) / 128, 128, 0, st>>>(s.groups, SQ, s.chunk);
    OKIN_CUDA(cudaGetLastError());
    OKIN_CUDA(cudaMemcpyAsync(s.host, s.chunk, SQ * sizeof(OkinMoments), cudaMemcpyDeviceToHost, st));
  }
  for (int64_t l = std::max<int64_t>(0, n_mine - slots); l < n_mine; ++l)
    if ((rc = finish(l))) return rc;
  sh.hist.assign(n_hist, 0);
  sh.status.assign(4, 0);
  sh.failed_at.assign(S, 0);
  if (n_hist) OKIN_CUDA(cudaMemcpy(sh.hist.data(), hist, n_hist * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  OKIN_CUDA(cudaMemcpy(sh.status.data(), status_counts, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if (S) OKIN_CUDA(cudaMemcpy(sh.failed_at.data(), failed_at, S * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return OKIN_OK;
}

void run_study_shard(StudyRun& run, StudyShard& sh) {
  {
    DeviceAllocs a;
    sh.rc = run_study_shard_body(run, sh, a);
    if (sh.rc) {
      sh.err = g_last_error;
      run.stop();
    }
    // nothing may still run on the buffers `a` releases
    for (int k = 0; k < OKIN_PIPE_SLOTS; ++k) cudaStreamSynchronize(sh.d->streams[k]);
  }
}

}  // namespace

extern "C" {

int okin_last_error(char* buf, int32_t len) {
  if (!buf || len <= 0) return OKIN_ERR_USAGE;
  std::snprintf(buf, (size_t)len, "%s", g_last_error.c_str());
  return OKIN_OK;
}

int okin_device_count(int* out) {
  if (!out) return fail(OKIN_ERR_USAGE, "null out");
  int n = 0;
  cudaError_t err = cudaGetDeviceCount(&n);
  if (err != cudaSuccess) {
    *out = 0;
    return fail(OKIN_ERR_NO_DEVICE, cudaGetErrorString(err));
  }
  *out = n;
  return OKIN_OK;
}

int okin_default_cfg(okin_solver_cfg* out) {
  if (!out) return fail(OKIN_ERR_USAGE, "null out");
  out->step_tol = 1e-6;
  out->coarse_tol = 1e-3;
  out->fine_tol = 1e-4;
  out->residual_tol = 1e-3;
  out->mu_init = 1e-3;
  out->max_iter = 50;
  out->use_predictor = 4;
  return OKIN_OK;
}

int okin_topology_create(const okin_topology_desc* desc, okin_topology** out) {
  if (!desc || !out || !desc->hdr || !desc->iblob || !desc->fblob) return fail(OKIN_ERR_USAGE, "null descriptor");
  if (desc->hdr[OKIN_H_MAGIC] != OKIN_MAGIC) return fail(OKIN_ERR_USAGE, "bad topology magic");
  if (desc->n_iblob < 0 || desc->n_fblob < 0) return fail(OKIN_ERR_USAGE, "negative blob size");
  // every section must lie inside its blob
  for (int s = 0; s < OKIN_S_COUNT_ALL; ++s) {
    const int64_t off = desc->hdr[OKIN_H_SEC0 + 2 * s], len = desc->hdr[OKIN_H_SEC0 + 2 * s + 1];
    if (off < 0 || len < 0 || off + len > desc->n_iblob) return fail(OKIN_ERR_USAGE, "int section out of range");
  }
  if (desc->hdr[OKIN_H_NSENS] != desc->hdr[OKIN_H_SEC0 + 2 * OKIN_S_SENS_IN + 1])
    return fail(OKIN_ERR_USAGE, "sensitivity input count does not match its section");
  for (int k = 0; k < desc->hdr[OKIN_H_NSENS]; ++k) {
    const int32_t coord = desc->iblob[desc->hdr[OKIN_H_SEC0 + 2 * OKIN_S_SENS_IN] + k];
    if (coord < 0 || coord >= 3 * desc->hdr[OKIN_H_NIN]) return fail(OKIN_ERR_USAGE, "sensitivity input out of range");
  }
  for (int s = 0; s < OKIN_F_COUNT; ++s) {
    const int64_t off = desc->hdr[OKIN_H_FSEC0 + 2 * s], len = desc->hdr[OKIN_H_FSEC0 + 2 * s + 1];
    if (off < 0 || len < 0 || off + len > desc->n_fblob) return fail(OKIN_ERR_USAGE, "double section out of range");
  }
  if (desc->hdr[OKIN_H_NHOT] < 0 || desc->hdr[OKIN_H_NHOT] > desc->n_iblob)
    return fail(OKIN_ERR_USAGE, "hot prefix out of range");
  // The device code addresses sections below OKIN_S_COLD0 as shared memory: they must lie in the
  // hot prefix, the others behind it.
  for (int s = 0; s < OKIN_S_COUNT_ALL; ++s) {
    const int64_t off = desc->hdr[OKIN_H_SEC0 + 2 * s], len = desc->hdr[OKIN_H_SEC0 + 2 * s + 1];
    const bool in_hot = off + len <= desc->hdr[OKIN_H_NHOT];
    if (s < OKIN_S_COLD0 ? !in_hot : (len > 0 && off < desc->hdr[OKIN_H_NHOT]))
      return fail(OKIN_ERR_USAGE, "section on the wrong side of the hot prefix");
  }
  if (desc->hdr[OKIN_H_NT] > OKIN_MAX_TARGETS) return fail(OKIN_ERR_USAGE, "too many targets");
  okin_topology* t = new okin_topology();
  t->hdr.assign(desc->hdr, desc->hdr + OKIN_HDR_SIZE);
  t->ib.assign(desc->iblob, desc->iblob + desc->n_iblob);
  t->fb.assign(desc->fblob, desc->fblob + desc->n_fblob);
  *out = t;
  return OKIN_OK;
}

int okin_topology_destroy(okin_topology* t) {
  if (!t) return OKIN_OK;
  for (int dev = 0; dev < OKIN_MAX_DEVICES; ++dev) {
    DeviceCopy& d = t->dev[dev];
    if (!d.ready) continue;
    cudaSetDevice(dev);
    cudaFree(d.hdr);
    cudaFree(d.ib);
    cudaFree(d.fb);
    if (d.ws) cudaFree(d.ws);
    for (int k = 0; k < OKIN_PIPE_SLOTS; ++k)
      if (d.streams[k]) cudaStreamDestroy(d.streams[k]);
  }
  delete t;
  return OKIN_OK;
}

int okin_topology_get_info(const okin_topology* t, okin_topology_info* out) {
  if (!t || !out) return fail(OKIN_ERR_USAGE, "null argument");
  const int32_t* h = t->hdr.data();
  out->n_points = h[OKIN_H_P];
  out->n_in_points = h[OKIN_H_NIN];
  out->n_out_points = h[OKIN_H_NOUT];
  out->n_unknowns = 3 * h[OKIN_H_NF];
  out->n_targets = h[OKIN_H_NT];
  out->n_rows = h[OKIN_H_NROW];
  out->smem_bytes_per_instance = h[OKIN_H_SMEM_DOUBLES] * (int32_t)sizeof(double);
  out->n_levels = h[OKIN_H_NLEV];
  out->n_metrics = h[OKIN_H_NM];
  out->n_params = h[OKIN_H_NPARAM];
  out->n_diagnostics = h[OKIN_H_NDIAG];
  return OKIN_OK;
}

int okin_launch_geometry(okin_topology* t, int32_t device, int64_t n_instances, int32_t* grid, int32_t* block,
                         int32_t* smem_bytes, int32_t* ctas_per_sm) {
  if (!t) return fail(OKIN_ERR_USAGE, "null topology");
  DeviceCopy* d = nullptr;
  int rc = ensure_device(t, device, &d);
  if (rc) return rc;
  // the lean family in use (positions + solver statistics), the wide one before any calibration
  const DeviceCopy::Shape& sh = d->shape[d->lean_family >= 0 ? d->lean_family : OKIN_FAM_LEAN_WIDE];
  const int64_t needed = (n_instances + sh.warps_per_cta - 1) / sh.warps_per_cta;
  if (grid) *grid = (int32_t)std::min<int64_t>(needed, (int64_t)d->num_sms * sh.ctas_per_sm);
  if (block) *block = sh.warps_per_cta * 32;
  if (smem_bytes) *smem_bytes = sh.smem_bytes;
  if (ctas_per_sm) *ctas_per_sm = sh.ctas_per_sm;
  return OKIN_OK;
}

int okin_lean_calibration(okin_topology* t, int32_t device, int32_t* registers, double* ms_wide, double* ms_128) {
  if (!t) return fail(OKIN_ERR_USAGE, "null topology");
  DeviceCopy* d = nullptr;
  int rc = ensure_device(t, device, &d);
  if (rc) return rc;
  if (registers) *registers = d->lean_family < 0 ? 0 : (d->lean_family == OKIN_FAM_LEAN ? 128 : 168);
  if (ms_wide) *ms_wide = d->lean_tune_ms[0];
  if (ms_128) *ms_128 = d->lean_tune_ms[1];
  return OKIN_OK;
}

int okin_solve_batch_device(okin_topology* t, const okin_solver_cfg* cfg, int32_t device, void* stream,
                            int64_t n_instances, int32_t n_steps, const okin_batch_io* d_io) {
  int rc = check_common(t, cfg, n_instances, n_steps, d_io);
  if (rc) return rc;
  if (d_io->diagnostics && !d_io->positions && n_instances > 0)
    return fail(OKIN_ERR_USAGE, "device-buffer diagnostics need the positions output (continuity pass reads it)");
  DeviceCopy* d = nullptr;
  rc = ensure_device(t, device, &d);
  if (rc) return rc;
  OKIN_CUDA(cudaSetDevice(device));
  return launch(t, d, cfg, (cudaStream_t)stream, n_instances, n_steps, *d_io);
}

int okin_shard_range(int64_t n_instances, int32_t shard, int32_t n_shards, int64_t* begin, int64_t* count) {
  if (!begin || !count || n_instances < 0 || n_shards < 1 || shard < 0 || shard >= n_shards)
    return fail(OKIN_ERR_USAGE, "invalid shard arguments");
  *begin = n_instances * shard / n_shards;
  *count = n_instances * (shard + 1) / n_shards - *begin;
  return OKIN_OK;
}

int okin_solve_batch(okin_topology* t, const okin_solver_cfg* cfg, int64_t n_instances, int32_t n_steps,
                     const okin_batch_io* io, const int32_t* device_ids, int32_t n_devices) {
  int rc = check_common(t, cfg, n_instances, n_steps, io);
  if (rc) return rc;
  const int32_t default_dev = 0;
  if (!device_ids || n_devices <= 0) {
    device_ids = &default_dev;
    n_devices = 1;
  }
  if (n_devices > OKIN_MAX_DEVICES) return fail(OKIN_ERR_USAGE, "too many devices");
  for (int a = 0; a < n_devices; ++a)
    for (int b = a + 1; b < n_devices; ++b)
      if (device_ids[a] == device_ids[b]) return fail(OKIN_ERR_USAGE, "device listed twice");
  HostBatch hb(t, n_instances, n_steps, io);

  // Contiguous instance ranges [k*N/G, (k+1)*N/G) per device: the host-side "gather" is the D2H
  // copies.  One host thread per device (copies from / to pageable caller buffers block the
  // issuing thread; with a thread per device the devices still run concurrently).
  std::vector<Shard> shards;
  for (int k = 0; k < n_devices; ++k) {
    Shard sh;
    okin_shard_range(n_instances, k, n_devices, &sh.begin, &sh.count);
    if (sh.count == 0) continue;
    sh.device = device_ids[k];
    rc = ensure_device(t, sh.device, &sh.d);
    if (rc) return rc;
    shards.push_back(sh);
  }
  if (shards.size() == 1) {
    run_shard(t, cfg, hb, shards[0]);
  } else {
    std::vector<std::thread> workers;
    for (Shard& sh : shards) workers.emplace_back([&, psh = &sh] { run_shard(t, cfg, hb, *psh); });
    for (std::thread& w : workers) w.join();
  }
  for (const Shard& sh : shards)
    if (sh.rc) return fail(sh.rc, sh.err);
  return OKIN_OK;
}

int okin_study(okin_topology* t, const okin_solver_cfg* cfg, int64_t n_instances, int32_t n_steps,
               const double* target_values, const okin_study_desc* desc, okin_study_out* out,
               const int32_t* device_ids, int32_t n_devices) {
  StudyRun run;
  int rc = study_check_generator(t, desc, &run.stride, &run.period);
  if (rc) return rc;
  if (!cfg) return fail(OKIN_ERR_USAGE, "null solver config");
  if (n_instances < 0 || n_steps < 0) return fail(OKIN_ERR_USAGE, "negative size");
  if (n_steps == 0) return fail(OKIN_ERR_USAGE, "a study needs at least one sweep step");
  if (t->hdr[OKIN_H_NT] > 0 && !target_values) return fail(OKIN_ERR_USAGE, "null target_values");
  if (cfg->max_iter < 1 || !(cfg->step_tol > 0.0) || !(cfg->coarse_tol >= cfg->step_tol))
    return fail(OKIN_ERR_USAGE, "invalid solver config");
  if ((rc = study_check_quantities(t, n_steps, desc, out))) return rc;
  const int32_t default_dev = 0;
  if (!device_ids || n_devices <= 0) {
    device_ids = &default_dev;
    n_devices = 1;
  }
  if (n_devices > OKIN_MAX_DEVICES) return fail(OKIN_ERR_USAGE, "too many devices");
  for (int a = 0; a < n_devices; ++a)
    for (int b = a + 1; b < n_devices; ++b)
      if (device_ids[a] == device_ids[b]) return fail(OKIN_ERR_USAGE, "device listed twice");
  run.t = t;
  run.cfg = cfg;
  run.n = n_instances;
  run.S = n_steps;
  run.target_values = target_values;
  run.desc = desc;
  run.Q = desc->n_quantities;
  run.SQ = n_steps * run.Q;
  run.nb = desc->n_bins;
  run.n_devices = n_devices;
  run.slots = OKIN_PIPE_SLOTS;
  for (int q = 0; q < run.Q; ++q) {
    run.want_pos |= desc->quantity_kind[q] == OKIN_QUANTITY_POSITION;
    run.want_met |= desc->quantity_kind[q] == OKIN_QUANTITY_METRIC;
  }
  run.n_chunks = (n_instances + OKIN_STUDY_CHUNK - 1) / OKIN_STUDY_CHUNK;
  run.window = (int64_t)n_devices * run.slots;
  run.ring.resize(run.window);
  run.have.assign(run.window, 0);
  run.acc.resize(run.SQ);
  for (OkinMoments& m : run.acc) okin_moments_clear(m);
  std::vector<StudyShard> shards(n_devices);
  for (int k = 0; k < n_devices; ++k) {
    shards[k].index = k;
    shards[k].device = device_ids[k];
    if ((rc = ensure_device(t, device_ids[k], &shards[k].d))) return rc;
  }
  if (n_devices == 1) {
    run_study_shard(run, shards[0]);
  } else {
    std::vector<std::thread> workers;
    for (StudyShard& sh : shards) workers.emplace_back([&, psh = &sh] { run_study_shard(run, *psh); });
    for (std::thread& w : workers) w.join();
  }
  const StudyShard* failed = nullptr;
  for (const StudyShard& sh : shards)
    if (sh.rc && (!failed || failed->err.rfind("study stopped", 0) == 0)) failed = &sh;
  if (failed) return fail(failed->rc, failed->err);
  const size_t SQ = run.SQ, nb2 = (size_t)run.nb + 2;
  for (size_t j = 0; j < SQ; ++j) {
    const OkinMoments& m = run.acc[j];
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
  if (run.nb) std::fill(out->histogram, out->histogram + SQ * nb2, (int64_t)0);
  std::fill(out->status_counts, out->status_counts + 4, (int64_t)0);
  std::fill(out->failed_at_step, out->failed_at_step + n_steps, (int64_t)0);
  for (const StudyShard& sh : shards) {
    for (size_t k = 0; k < sh.hist.size(); ++k) out->histogram[k] += (int64_t)sh.hist[k];
    for (int k = 0; k < 4 && k < (int)sh.status.size(); ++k) out->status_counts[k] += (int64_t)sh.status[k];
    for (size_t k = 0; k < sh.failed_at.size(); ++k) out->failed_at_step[k] += (int64_t)sh.failed_at[k];
  }
  return OKIN_OK;
}

int okin_study_sample(okin_topology* t, const okin_study_desc* desc, int64_t n_ids, const int64_t* instance_ids,
                      double* hardpoints_out, double* params_out, int32_t device) {
  std::vector<uint64_t> stride;
  uint64_t period = 0;
  int rc = study_check_generator(t, desc, &stride, &period);
  if (rc) return rc;
  const int nin3 = 3 * t->hdr[OKIN_H_NIN], npar = t->hdr[OKIN_H_NPARAM];
  if (n_ids < 0) return fail(OKIN_ERR_USAGE, "negative n_ids");
  if (n_ids > 0 && (!instance_ids || !hardpoints_out || (npar > 0 && !params_out)))
    return fail(OKIN_ERR_USAGE, "null study sample buffer");
  for (int64_t r = 0; r < n_ids; ++r)
    if (instance_ids[r] < 0) return fail(OKIN_ERR_USAGE, "negative instance id");
  if (n_ids == 0) return OKIN_OK;
  DeviceCopy* d = nullptr;
  if ((rc = ensure_device(t, device, &d))) return rc;
  OKIN_CUDA(cudaSetDevice(device));
  DeviceAllocs a;
  OkinStudyTables tab;
  if ((rc = upload_study_tables(desc, stride, period, a, &tab))) return rc;
  long long* ids;
  double *hp, *par = nullptr;
  OKIN_CUDA(a.alloc(&ids, n_ids));
  OKIN_CUDA(a.alloc(&hp, (size_t)n_ids * nin3));
  if (npar) OKIN_CUDA(a.alloc(&par, (size_t)n_ids * npar));
  OKIN_CUDA(cudaMemcpy(ids, instance_ids, n_ids * sizeof(long long), cudaMemcpyHostToDevice));
  if ((rc = launch_study_generate(tab, 0, ids, n_ids, nin3, npar, hp, par, d->num_sms, d->streams[0]))) return rc;
  OKIN_CUDA(cudaStreamSynchronize(d->streams[0]));
  OKIN_CUDA(cudaMemcpy(hardpoints_out, hp, (size_t)n_ids * nin3 * sizeof(double), cudaMemcpyDeviceToHost));
  if (npar) OKIN_CUDA(cudaMemcpy(params_out, par, (size_t)n_ids * npar * sizeof(double), cudaMemcpyDeviceToHost));
  return OKIN_OK;
}

int okin_host_alloc(int64_t bytes, int32_t device, void** out) {
  if (!out || bytes < 0) return fail(OKIN_ERR_USAGE, "invalid host allocation request");
  *out = nullptr;
  if (bytes == 0) return OKIN_OK;
  // Page-locked, portable (usable from every device context).  Pages are placed on the NUMA node of
  // the allocating thread, so the thread is moved next to `device` for the duration of the call.
  cpu_set_t saved;
  const bool have_saved = pthread_getaffinity_np(pthread_self(), sizeof(saved), &saved) == 0;
  const bool moved = device >= 0 && have_saved && bind_thread_near_device(device);
  cudaError_t err = cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable);
  if (moved) pthread_setaffinity_np(pthread_self(), sizeof(saved), &saved);
  if (err != cudaSuccess) return fail(OKIN_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(err));
  return OKIN_OK;
}

int okin_host_free(void* p) {
  if (!p) return OKIN_OK;
  OKIN_CUDA(cudaFreeHost(p));
  return OKIN_OK;
}

int okin_fp64_peak(int32_t device, double* tflops_out) {
  if (!tflops_out) return fail(OKIN_ERR_USAGE, "null out");
  OKIN_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  OKIN_CUDA(cudaGetDeviceProperties(&prop, device));
  const int block = 256, grid = prop.multiProcessorCount * 8, iters = 1 << 14;
  double* buf = nullptr;
  OKIN_CUDA(cudaMalloc(&buf, (size_t)grid * block * sizeof(double)));
  cudaEvent_t e0, e1;
  OKIN_CUDA(cudaEventCreate(&e0));
  OKIN_CUDA(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    OKIN_CUDA(cudaEventRecord(e0));
    okin_dfma_kernel<<<grid, block>>>(buf, iters, 0.999999, 1e-7);
    OKIN_CUDA(cudaEventRecord(e1));
    OKIN_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    OKIN_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * (double)iters * grid * block;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(buf);
  *tflops_out = best;
  return OKIN_OK;
}

}  // extern "C"
