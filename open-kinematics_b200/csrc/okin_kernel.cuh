// The sweep kernel, shared by the library (okin_abi.cu, generic instantiations) and the run-time
// compilation of a topology's specialised lean kernel (okin_abi.cu, NVRTC with OKIN_SPEC and the
// topology's okin_spec.h).
#pragma once
#include "okin_core.cuh"

#define OKIN_MAX_THREADS 512
#ifndef OKIN_DRIFT
#define OKIN_DRIFT 1             // how many instances a warp may run ahead of the slowest warp of its CTA
#endif

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
#ifdef OKIN_SPEC
  // the spec's packed task words follow the hot tables (table_doubles counts them)
  int32_t* spec = tab + n_hot;
  for (int i = threadIdx.x; i < OKIN_SPEC_WORDS; i += blockDim.x) spec[i] = okin_spec_words[i];
#endif
  __syncthreads();
  hdr = shdr;
  OkinProgram pr{shdr, tab, fb, ib, sec};
#ifdef OKIN_SPEC
  pr.spec = spec;
#endif
  const int warp = threadIdx.x >> 5;
  const int warps_per_cta = blockDim.x >> 5;
  double* sm = okin_smem + table_doubles + (size_t)warp * hdr[FULL ? OKIN_H_SMEM_DOUBLES : OKIN_H_SMEM_DOUBLES_LEAN];
  const OkinIOShape shape = okin_io_shape(hdr);
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
      const double *hp, *par, *tv;
      if (SENS) out.sens_ws = sens_ws + ((size_t)blockIdx.x * warps_per_cta + warp) * okin_sens_ws_doubles(hdr);
      okin_instance_io(io, SENS ? sens_out : nullptr, shape, n_steps, i, out, hp, par, tv);
      okin_sweep<FULL, SHIM, SENS>(pr, sm, hp, par, tv, n_steps, cfg, out);
      __syncwarp();
    }
    ++mine;
    if ((threadIdx.x & 31) == 0) atomicExch(&s_done[warp], mine);
  }
  if ((threadIdx.x & 31) == 0) atomicExch(&s_done[warp], 0x7fffffff);
}

