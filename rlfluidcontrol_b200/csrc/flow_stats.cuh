// flow_stats.cuh -- running float64 sums of the flow of every environment (rlfc_config.stats_every; rlfc.h "Flow
// statistics").  Included at the end of solver_kernels.cu, so it is compiled with --fmad=false like the solver.
//
//   k_flow_stats    grid (chunks of an environment's cells, environments): every CTA of an environment not frozen reads its
//                   step counter; the CTA that takes the environment's last ticket advances it.  On a sampled step each
//                   thread adds two adjacent cells (float2 of u.x, u.y, p; double2 read-modify-write of the seven sums).
//   k_stats_reset   grid (chunks, pairs): zeroes the sums, count and step counter of the listed environments.
//
// Every term is either a float converted to double or the product of two such doubles, which is exact, so each term is
// rounded once, when it is added, and a cell's sum is the same however the compiler schedules the adds.  The sums of one
// cell are added in step order, one launch after the other, so they are reproducible bit for bit.
#pragma once
#include "solver.h"

namespace rlfc {
namespace {

constexpr int kStatThreads = 256;
constexpr int kStatPairs = 4;                                   // cell pairs per thread
constexpr int kStatChunk = kStatThreads * kStatPairs;           // cell pairs per CTA

__global__ void __launch_bounds__(kStatThreads)
k_flow_stats(const FlowStats f, const float* __restrict__ ux_all, const float* __restrict__ uy_all,
             const float* __restrict__ p_all, const int* __restrict__ frozen, int n, int m, int P, size_t stride) {
  __shared__ int s_take;
  const int e = blockIdx.y;
  if (frozen[e]) return;                                        // (the same for every CTA of the environment)
  if (threadIdx.x == 0) {
    // every CTA reads the counter before it takes a ticket; the CTA with the last ticket has seen every other CTA's
    // ticket, so its update cannot be read by any CTA of this launch
    const int c = f.step[e];
    const bool take = c + 1 >= f.every;
    s_take = take;
    __threadfence();
    if (atomicAdd(f.ticket + e, 1u) == gridDim.x - 1) {
      __threadfence();
      f.step[e] = take ? 0 : c + 1;
      if (take) f.count[e] += 1;
      f.ticket[e] = 0;                                          // ready for the next launch
    }
  }
  __syncthreads();
  if (!s_take) return;
  const size_t eo = (size_t)e * stride;
  const float* __restrict__ ux = ux_all + eo;
  const float* __restrict__ uy = uy_all + eo;
  const float* __restrict__ p = p_all + eo;
  double* S = f.sums + (size_t)e * kNumStats * stride;
  const int np = m >> 1, items = n * np;                        // (m is even: the level-0 grid is)
#pragma unroll
  for (int r = 0; r < kStatPairs; r++) {
    const int k = blockIdx.x * kStatChunk + r * kStatThreads + threadIdx.x;
    if (k >= items) break;
    const int i = k / np, j = 2 * (k - i * np);
    const size_t o = (size_t)i * P + j;
    const float2 a = *reinterpret_cast<const float2*>(ux + o);
    const float2 b = *reinterpret_cast<const float2*>(uy + o);
    const float2 c = *reinterpret_cast<const float2*>(p + o);
    double2 v[kNumStats];
#pragma unroll
    for (int s = 0; s < kNumStats; s++) v[s] = __ldcs(reinterpret_cast<const double2*>(S + s * stride + o));
    v[RLFC_STAT_UX].x += (double)a.x;               v[RLFC_STAT_UX].y += (double)a.y;
    v[RLFC_STAT_UY].x += (double)b.x;               v[RLFC_STAT_UY].y += (double)b.y;
    v[RLFC_STAT_P].x += (double)c.x;                v[RLFC_STAT_P].y += (double)c.y;
    v[RLFC_STAT_UXUX].x += (double)a.x * (double)a.x; v[RLFC_STAT_UXUX].y += (double)a.y * (double)a.y;
    v[RLFC_STAT_UYUY].x += (double)b.x * (double)b.x; v[RLFC_STAT_UYUY].y += (double)b.y * (double)b.y;
    v[RLFC_STAT_PP].x += (double)c.x * (double)c.x;   v[RLFC_STAT_PP].y += (double)c.y * (double)c.y;
    if (i >= 1 && i <= n - 2) {
      // cell-centred velocity: ux[i+1][j] from the next row, uy[i][j+1] from within the row
      const float2 an = *reinterpret_cast<const float2*>(ux + o + P);
      if (j >= 1) {                                             // cell j (j even: j >= 2)
        const float ucc = (a.x + an.x) * 0.5f, vcc = (b.x + b.y) * 0.5f;
        v[RLFC_STAT_UV].x += (double)ucc * (double)vcc;
      }
      if (j + 1 <= m - 2) {                                     // cell j + 1
        const float ucc = (a.y + an.y) * 0.5f, vcc = (b.y + uy[o + 2]) * 0.5f;
        v[RLFC_STAT_UV].y += (double)ucc * (double)vcc;
      }
    }
#pragma unroll
    for (int s = 0; s < kNumStats; s++) __stcs(reinterpret_cast<double2*>(S + s * stride + o), v[s]);
  }
}

__global__ void __launch_bounds__(kStatThreads)
k_stats_reset(const FlowStats f, const int* __restrict__ ids, int n, int B, size_t stride) {
  const size_t n2 = kNumStats * stride / 2;                     // (stride is a multiple of 32)
  for (int k = blockIdx.y; k < n; k += gridDim.y) {
    const int e = ids[k];
    if (e < 0 || e >= B) continue;
    if (blockIdx.x == 0 && threadIdx.x == 0) { f.count[e] = 0; f.step[e] = 0; }
    double2* S = reinterpret_cast<double2*>(f.sums + (size_t)e * kNumStats * stride);
    for (size_t q = (size_t)blockIdx.x * kStatThreads + threadIdx.x; q < n2; q += (size_t)gridDim.x * kStatThreads)
      S[q] = make_double2(0.0, 0.0);
  }
}

}  // namespace

int launch_flow_stats(const SolverParams& q, const FlowStats& f, const float* ux, const float* uy, cudaStream_t st) {
  if (f.every <= 0) return 0;
  const int chunks = (q.n * (q.m / 2) + kStatChunk - 1) / kStatChunk;
  k_flow_stats<<<dim3(chunks, q.B), kStatThreads, 0, st>>>(f, ux, uy, q.lev[0].x, q.sc.frozen, q.n, q.m, q.P, q.stride);
  return 1;
}

int launch_stats_reset(const SolverParams& q, const FlowStats& f, const int* d_ids, int n, cudaStream_t st) {
  if (f.every <= 0 || n <= 0) return 0;
  const size_t n2 = kNumStats * q.stride / 2;
  const size_t want = (n2 + kStatThreads * 8 - 1) / (kStatThreads * 8);   // 8 double2 per thread
  const int chunks = (int)(want < 1024 ? want : 1024);
  k_stats_reset<<<dim3(chunks, n < 65535 ? n : 65535), kStatThreads, 0, st>>>(f, d_ids, n, q.B, q.stride);
  return 1;
}

}  // namespace rlfc
