// param_sets.cuh -- reset environments into the parameter library (rlfc_env_reset_sets and its _device variant).
// Included at the end of solver_kernels.cu, after snapshot.cuh, whose pair resolution and chunk copy it shares.
//
// An applied pair (e, s) points environment e at library set s -- its geometry slot, per-environment scalars and fixed dt --
// and does what rlfc_env_reset does: u and p from the handle's init state, the reset scalars.  The caller then rebuilds the
// Poisson hierarchy of the environments reset (launch_poisson_rebuild* on the skip mask this kernel clears).  Grid (3 fields
// x chunks, pairs), like k_snapshot_copy: each pair copies three contiguous blocks of n*P floats with 16-byte accesses, and
// the first chunk of a pair also writes the scalars.
#pragma once
#include "solver.h"

namespace rlfc {
namespace {

struct ResetSetsArgs {
  ParamLib lib;
  EnvScalars sc;
  int *env_slot, *env_nbx, *env_nby;           // SolverParams' per-environment arrays (the whole batch)
  float *env_nu, *env_dRD;
  unsigned* env_par;                           // [5][B] parameter tuples (nullptr without snapshots or records)
  const float4 *iux, *iuy, *ip;                // the init state (one environment)
  float4 *ux, *uy, *p;                         // the environments' fields (batch base)
  size_t stride4;                              // level-0 per-environment stride in float4
  int nv;                                      // float4 of one field that are copied (n*P/4)
  int B;
  const int *env, *set;
  int n, reset_acc, substeps;
  float init_t;
  int* skip;
};

// rlfc_env_reset's scalars of environment e, with dt = the set's t_step*resolution
__device__ __forceinline__ void reset_scalars(const EnvScalars& sc, int e, float init_t, float dt0, int reset_acc, int substeps) {
  sc.xi[2 * e] = 0.f; sc.xi[2 * e + 1] = 0.f;
  sc.t[e] = 0.f;
  sc.flow_t[e] = init_t;                                 // BDIM.resume: t = stuff[0]
  sc.force[2 * e] = 0.f; sc.force[2 * e + 1] = 0.f;
  sc.frozen[e] = 0;
  sc.non_finite[e] = 0;
  sc.dt[e] = dt0;                                        // t_step*resolution
  if (reset_acc) {
    sc.callLearn[e] = substeps;
    sc.Cd[e] = 0.f; sc.Cl[e] = 0.f;
    sc.obs[2 * e] = 0.f; sc.obs[2 * e + 1] = 0.f;
  }
}

__global__ void __launch_bounds__(kSnapThreads) k_reset_sets(const __grid_constant__ ResetSetsArgs a) {
  const int cpf = (a.nv + kSnapThreads * kSnapVec - 1) / (kSnapThreads * kSnapVec);   // chunks per field
  const int f = blockIdx.x / cpf, c = blockIdx.x - f * cpf;
  for (int k = blockIdx.y; k < a.n; k += gridDim.y) {
    if (!pair_applies(a.env, a.set, k, a.n, a.B, a.lib.L, true)) continue;
    const int e = a.env[k], s = a.set[k];
    const float4* src = f == 0 ? a.iux : f == 1 ? a.iuy : a.ip;
    float4* dst = (f == 0 ? a.ux : f == 1 ? a.uy : a.p) + (size_t)e * a.stride4;
    copy_chunk(src, dst, c, a.nv);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      const LibSet& L = a.lib.sets[s];
      a.env_slot[e] = L.slot;
      a.lib.env_set[e] = s;
      a.env_nu[e] = L.nu;
      a.env_dRD[e] = L.dRD;
      a.env_nbx[e] = L.nbx;
      a.env_nby[e] = L.nby;
      if (a.env_par)
        for (int w = 0; w < 5; w++) a.env_par[(size_t)w * a.B + e] = L.bits[w];
      reset_scalars(a.sc, e, a.init_t, L.dt0, a.reset_acc, a.substeps);
      a.skip[e] = 0;
    }
  }
}

}  // namespace

int launch_reset_sets(const SolverParams& q, const ParamLib& lib, const SnapSlots& snap, const float* init_ux,
                      const float* init_uy, const float* init_p, float init_t, float* ux, float* uy, const int* d_env,
                      const int* d_set, int n, int reset_accumulators, int* skip, cudaStream_t st) {
  if (n <= 0) return 0;
  ResetSetsArgs a{};
  a.lib = lib;
  a.sc = q.sc;
  a.env_slot = const_cast<int*>(q.env_slot);
  a.env_nbx = const_cast<int*>(q.env_nband_x);
  a.env_nby = const_cast<int*>(q.env_nband_y);
  a.env_nu = const_cast<float*>(q.env_nu);
  a.env_dRD = const_cast<float*>(q.env_dRD);
  a.env_par = snap.env_par;
  a.iux = reinterpret_cast<const float4*>(init_ux);
  a.iuy = reinterpret_cast<const float4*>(init_uy);
  a.ip = reinterpret_cast<const float4*>(init_p);
  a.ux = reinterpret_cast<float4*>(ux);
  a.uy = reinterpret_cast<float4*>(uy);
  a.p = reinterpret_cast<float4*>(q.lev[0].x);
  a.stride4 = q.stride / 4;
  a.nv = q.n * q.P / 4;
  a.B = q.B;
  a.env = d_env;
  a.set = d_set;
  a.n = n;
  a.reset_acc = reset_accumulators;
  a.substeps = q.substeps;
  a.init_t = init_t;
  a.skip = skip;
  const int cpf = (a.nv + kSnapThreads * kSnapVec - 1) / (kSnapThreads * kSnapVec);
  k_reset_sets<<<dim3(3 * cpf, n < 65535 ? n : 65535), kSnapThreads, 0, st>>>(a);
  return 1;
}

}  // namespace rlfc
