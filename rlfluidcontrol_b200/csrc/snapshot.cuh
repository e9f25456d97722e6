// snapshot.cuh -- copies of one environment's complete state to a snapshot slot and back (rlfc_env_snapshot /
// rlfc_env_restore and their _device variants).  Included at the end of solver_kernels.cu.
//
// A state is what the next solver or RL step reads before it writes it, plus what the read-outs return: the three level-0
// fields (u.x, u.y of the step-start buffer A, p = lev[0].x, the MG initial guess) and the scalar record of snap_word.
// The slot layout is solver.h SnapSlots.  One kernel serves both directions: grid (chunks, pairs), each pair moves three
// contiguous blocks of n*P floats (16-byte accesses; stride is a multiple of 32 floats, so every block starts 128-byte
// aligned), and the first chunk of a pair also moves the scalar record and the sensors.
#pragma once
#include "solver.h"

namespace rlfc {
namespace {

constexpr int kSnapThreads = 256;
constexpr int kSnapVec = 8;                    // float4 per thread: 32 KB of one field per CTA
constexpr int kSnapAcc0 = 39, kSnapAcc1 = 44;  // words of the draw() accumulators callLearn, Cd, Cl, obs[2]

struct SnapArgs {
  SnapSlots s;
  EnvScalars sc;
  float4 *ux, *uy, *p;                         // the environments' fields (batch base)
  size_t stride4;                              // level-0 per-environment stride in float4
  int nv;                                      // float4 of one field that are copied (n*P/4)
  int B, nprobe;
  SensorSet sens;                              // the environments' sensors (sens.n = 0: none)
  const int *env, *slot;
  int n, restore, keep;
  int* skip;
};

// word w of environment e's scalar record; nullptr = unused word (probes beyond nprobe)
__device__ __forceinline__ unsigned* snap_word(const EnvScalars& sc, int nprobe, int e, int w) {
  float* f = nullptr;
  int* i = nullptr;
  if (w < 2) f = sc.xi + 2 * e + w;                          // 0, 1    xi
  else if (w == 2) f = sc.t + e;                             // 2       AFCCylinder.t
  else if (w == 3) f = sc.flow_t + e;                        // 3       BDIM.t
  else if (w == 4) f = sc.dt + e;                            // 4       dt
  else if (w < 7) f = sc.force + 2 * e + (w - 5);            // 5, 6    force
  else if (w < 39) {                                         // 7 .. 38 probes
    if (w - 7 >= nprobe) return nullptr;
    f = sc.probes + (size_t)e * nprobe + (w - 7);
  }
  else if (w == 39) i = sc.callLearn + e;                    // 39 .. 43 the draw() accumulators
  else if (w == 40) f = sc.Cd + e;
  else if (w == 41) f = sc.Cl + e;
  else if (w < 44) f = sc.obs + 2 * e + (w - 42);
  else if (w == 44) i = sc.frozen + e;                       // 44      frozen
  else if (w == 45) i = sc.non_finite + e;                   // 45      non_finite
  else if (w < 48) i = sc.iters + 2 * e + (w - 46);          // 46, 47  MG iterations
  return f ? reinterpret_cast<unsigned*>(f) : reinterpret_cast<unsigned*>(i);
}

// Pair k of the device arrays (x[k], y[k]) applies when x[k] is in [0, nx), y[k] in [0, ny) (a negative entry is the way
// to skip a pair) and no later pair in range has the same destination (x if dst_x, else y): of pairs with the same
// destination the last one wins.  Called by every thread of the CTA (one __syncthreads_or); the result is CTA-uniform.
__device__ __forceinline__ bool pair_applies(const int* x, const int* y, int k, int n, int nx, int ny, bool dst_x) {
  const int xk = x[k], yk = y[k];
  if (xk < 0 || xk >= nx || yk < 0 || yk >= ny) return false;
  const int dst = dst_x ? xk : yk;
  int later = 0;
  for (int k2 = k + 1 + (int)threadIdx.x; k2 < n; k2 += kSnapThreads) {
    const int x2 = x[k2], y2 = y[k2];
    if (x2 >= 0 && x2 < nx && y2 >= 0 && y2 < ny && (dst_x ? x2 : y2) == dst) later = 1;
  }
  return !__syncthreads_or(later);
}

// chunk c of one field: kSnapThreads * kSnapVec float4 of nv, streamed (the copy is read once)
__device__ __forceinline__ void copy_chunk(const float4* __restrict__ src, float4* __restrict__ dst, int c, int nv) {
  const int i0 = c * kSnapThreads * kSnapVec + (int)threadIdx.x;
  float4 v[kSnapVec];
#pragma unroll
  for (int u = 0; u < kSnapVec; u++)
    if (i0 + u * kSnapThreads < nv) v[u] = __ldcs(src + i0 + u * kSnapThreads);
#pragma unroll
  for (int u = 0; u < kSnapVec; u++)
    if (i0 + u * kSnapThreads < nv) dst[i0 + u * kSnapThreads] = v[u];
}

__global__ void __launch_bounds__(kSnapThreads) k_snapshot_copy(const __grid_constant__ SnapArgs a) {
  const int S = a.s.S, B = a.B;
  const int cpf = (a.nv + kSnapThreads * kSnapVec - 1) / (kSnapThreads * kSnapVec);   // chunks per field
  const int f = blockIdx.x / cpf, c = blockIdx.x - f * cpf;
  for (int k = blockIdx.y; k < a.n; k += gridDim.y) {
    if (!pair_applies(a.env, a.slot, k, a.n, B, S, a.restore)) continue;
    const int e = a.env[k], s = a.slot[k];
    if (a.restore) {
      // only a written slot of the destination's own parameter tuple (whose geometry and fixed-dt hierarchy it has); no
      // short circuit, so that the eleven loads are independent and issue together
      unsigned diff = a.s.hdr[s] ^ 1u;
#pragma unroll
      for (int w = 0; w < 5; w++) diff |= a.s.hdr[(size_t)(1 + w) * S + s] ^ a.s.env_par[(size_t)w * B + e];
      const bool ok = diff == 0u;
      if (blockIdx.x == 0 && threadIdx.x == 0) {
        a.s.refused[e] = ok ? 0 : 1;
        if (ok && a.skip) a.skip[e] = 0;
      }
      if (!ok) continue;
    }
    float4* ef = (f == 0 ? a.ux : f == 1 ? a.uy : a.p) + (size_t)e * a.stride4;
    float4* sf = reinterpret_cast<float4*>(f == 0 ? a.s.ux : f == 1 ? a.s.uy : a.s.p) + (size_t)s * a.stride4;
    const float4* __restrict__ src = a.restore ? sf : ef;
    float4* __restrict__ dstp = a.restore ? ef : sf;
    copy_chunk(src, dstp, c, a.nv);
    if (blockIdx.x == 0 && threadIdx.x < kSnapWords) {
      const int w = threadIdx.x;
      unsigned* x = snap_word(a.sc, a.nprobe, e, w);
      unsigned* r = a.s.rec + (size_t)w * S + s;
      if (x) {
        if (!a.restore) *r = *x;
        else if (!(a.keep && w >= kSnapAcc0 && w < kSnapAcc1)) *x = *r;
      }
      if (!a.restore && w < kSnapHdr) a.s.hdr[(size_t)w * S + s] = w == 0 ? 1u : a.s.env_par[(size_t)(w - 1) * B + e];
    }
    if (blockIdx.x == 0)
      for (int k2 = threadIdx.x; k2 < a.sens.n; k2 += kSnapThreads) {
        float* x = a.sens.out + (size_t)e * a.sens.n + k2;
        float* r = a.s.sens + (size_t)s * a.sens.n + k2;
        if (a.restore) *x = *r;
        else *r = *x;
      }
  }
}

}  // namespace

int launch_snapshot_copy(const SolverParams& q, const SnapSlots& s, const SensorSet& sens, float* ux, float* uy, const int* d_env,
                         const int* d_slot, int n, int restore, int keep_accumulators, int* skip, cudaStream_t st) {
  if (n <= 0) return 0;
  SnapArgs a{};
  a.s = s;
  a.sc = q.sc;
  a.ux = reinterpret_cast<float4*>(ux);
  a.uy = reinterpret_cast<float4*>(uy);
  a.p = reinterpret_cast<float4*>(q.lev[0].x);
  a.stride4 = q.stride / 4;
  a.nv = q.n * q.P / 4;
  a.B = q.B;
  a.nprobe = q.nprobe;
  a.sens = sens;
  a.env = d_env;
  a.slot = d_slot;
  a.n = n;
  a.restore = restore;
  a.keep = keep_accumulators;
  a.skip = skip;
  const int cpf = (a.nv + kSnapThreads * kSnapVec - 1) / (kSnapThreads * kSnapVec);
  k_snapshot_copy<<<dim3(3 * cpf, n < 65535 ? n : 65535), kSnapThreads, 0, st>>>(a);
  return 1;
}

}  // namespace rlfc
