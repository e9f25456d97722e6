// smooth_tiny.cuh -- exact lexicographic Gauss-Seidel smoothing (MG.smooth, MG.pde:79-97) of the SMALL levels of the
// V-cycle (at most 32 columns: 48x24, 24x12, ... cells) by ONE warp, all stages in registers.
//
// The row pipeline of smooth_rows.cuh spends ~450 cycles per step whatever the level's size (CTA barrier, shared-memory
// round trip between the stage warps): for a 48x24 level that is 37 k cycles for 1152 cells.  Here lane L owns column
// j = L + 1 and, at step t, the warp runs every stage of the same schedule at once: stage g works on row t - L - 2g
// (stage 0: d = r*inv; stages 1..4: the four sweeps; then x (+)= d one row behind sweep 4).  Each operand is a register of
// the same lane or of a neighbour lane one step earlier:
//     W = this sweep's own previous result,            S = the lane below's previous result of this sweep (shuffle up),
//     E = the previous stage's previous result,        N = the lane above's previous result of the previous stage (shuffle down),
// so a step is two shuffles and nine float operations per sweep, the four sweeps being independent chains.  The level's
// coefficients and right-hand side are staged ONCE into shared memory by the whole CTA (coalesced), lane-contiguous per
// row, rows 0 and ni+1 zero: a stage outside the domain reads zeros and evaluates to +-0 by itself, exactly as the
// pre-skewed tables of the row pipeline arrange it.  x is staged too and written back by the whole CTA.
// Arithmetic per update, unchanged (MG.pde:85-86):  d = (dW*lxW + dE*lxE + dS*lyS + dN*lyN - r) * (-inv).
// Included by solver_kernels.cu inside namespace rlfc::{anonymous}.
#pragma once

// bytes of dynamic shared memory tiny_smooth needs for a level with ni interior rows
__host__ __device__ inline size_t tiny_smem_bytes(int ni) { return (size_t)(ni + 2) * 32 * (16 + 8 + 4); }
__host__ __device__ inline bool tiny_level(int ni, int mj) { return mj <= 32 && ni >= 1; }

// XMODE 1: x = 0 + d (coarsest level), 2: x = x + d.  Called by ALL threads of the CTA (any block size >= 32).
template <int XMODE>
__device__ __forceinline__ void tiny_smooth(const DevLevel& L, const float* __restrict__ r, float* __restrict__ x,
                                            unsigned char* smem_raw, size_t co) {
  const int ni = L.n - 2, mj = L.m - 2, P = L.P;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4* s_a = reinterpret_cast<float4*>(smem_raw);                       // [ni+2][32] {lxW, lxE, lyS, lyN}
  float2* s_b = reinterpret_cast<float2*>(s_a + (size_t)(ni + 2) * 32);    // [ni+2][32] {-inv, r}
  float* s_x = reinterpret_cast<float*>(s_b + (size_t)(ni + 2) * 32);      // [ni+2][32] x
  const float* __restrict__ lx = L.lx + co;                                // co: this environment's coefficients (adaptive mode)
  const float* __restrict__ ly = L.ly + co;
  const float* __restrict__ inv = L.inv + co;
  // ---- stage: rows 0 .. ni+1, lanes 0 .. 31 (zeros outside the interior) ----
  for (int t = threadIdx.x; t < (ni + 2) * 32; t += blockDim.x) {
    const int i = t >> 5, l = t & 31, j = l + 1;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    float2 b = make_float2(0.f, 0.f);
    float xv = 0.f;
    if (i >= 1 && i <= ni && j <= mj) {
      const int k = IDX(i, j);
      a = make_float4(lx[k], lx[k + P], ly[k], ly[k + 1]);
      b = make_float2(-inv[k], r[k]);
      if (XMODE == 2) xv = x[k];
    }
    s_a[t] = a; s_b[t] = b; s_x[t] = xv;
  }
  __syncthreads();
  if (warp == 0) {
    // previous-step results of stages 0..4 (stage 0 = r*inv) of this lane
    float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f, p4 = 0.f;
    const int t_end = ni + mj + 9;                                       // lane mj-1 finishes row ni of sweep 4 at ni + mj + 7
    auto rowc = [&](int i) { return min(max(i, 0), ni + 1) * 32 + lane; };
    auto sweep = [&](int i, float W, float E, float S, float N) {
      const int k = rowc(i);
      const float4 a = s_a[k];
      const float2 b = s_b[k];
      return (W * a.x + E * a.y + S * a.z + N * a.w - b.y) * b.x;        // MG.pde:85-86
    };
#pragma unroll 2
    for (int t = 1; t <= t_end; t++) {
      const int i0 = t - lane;
      // neighbour-lane operands: results of the PREVIOUS step
      float s1 = __shfl_up_sync(0xffffffffu, p1, 1), s2 = __shfl_up_sync(0xffffffffu, p2, 1);
      float s3 = __shfl_up_sync(0xffffffffu, p3, 1), s4 = __shfl_up_sync(0xffffffffu, p4, 1);
      float n0 = __shfl_down_sync(0xffffffffu, p0, 1), n1 = __shfl_down_sync(0xffffffffu, p1, 1);
      float n2 = __shfl_down_sync(0xffffffffu, p2, 1), n3 = __shfl_down_sync(0xffffffffu, p3, 1);
      if (lane == 0) { s1 = 0.f; s2 = 0.f; s3 = 0.f; s4 = 0.f; }         // ghost column of d acts as 0 during the sweeps
      if (lane == 31) { n0 = 0.f; n1 = 0.f; n2 = 0.f; n3 = 0.f; }        // (the row pipeline's zero 33rd lane)
      const float2 b0 = s_b[rowc(i0)];
      const float q0 = b0.y * (-b0.x);                                   // stage 0: d = r * inv (MG.pde:80)
      const float q1 = sweep(i0 - 2, p1, p0, s1, n0);
      const float q2 = sweep(i0 - 4, p2, p1, s2, n1);
      const float q3 = sweep(i0 - 6, p3, p2, s3, n2);
      const float q4 = sweep(i0 - 8, p4, p3, s4, n3);
      const int i4 = i0 - 8;                                             // the row sweep 4 just finished: x (+)= d (MG.pde:95)
      if (i4 >= 1 && i4 <= ni && lane < mj) {
        float* xs = s_x + i4 * 32 + lane;
        *xs = (XMODE == 1) ? 0.f + q4 : *xs + q4;
      }
      p0 = q0; p1 = q1; p2 = q2; p3 = q3; p4 = q4;
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < ni * 32; t += blockDim.x) {
    const int i = 1 + (t >> 5), l = t & 31;
    if (l < mj) x[IDX(i, l + 1)] = s_x[i * 32 + l];
  }
  __syncthreads();
}
