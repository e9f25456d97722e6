// smooth_chain.cuh -- exact lexicographic Gauss-Seidel smoothing (MG.smooth, MG.pde:79-97) for WIDE levels: a sweep
// spans many warps, CTAs and SMs (and, with peer pointers, GPUs), chained column block to column block through
// global memory.  Included by solver_kernels.cu inside namespace rlfc::{anonymous}.
//
// The serial reference updates d[i][j] in place with i outer, j inner, so cell (i,j) sees NEW values at (i-1,j),
// (i,j-1) and OLD values (previous sweep) at (i+1,j), (i,j+1).  Mapping:
//   * the columns of a level are cut into strips of 32; lane L of strip s owns column j = 32 s + L + 1 and walks
//     down the rows one per step, lanes skewed by one step: at local step t the strip works on ENTRY t = the cells
//     (i = t - L, j) -- W comes from the lane's own previous result, S from lane L-1's previous result (shuffle);
//   * one warp = one (sweep g, strip s); the four sweeps of a smooth(4) are four such warp chains running
//     concurrently, sweep g consuming what sweep g-1 produced.  Every array the sweeps touch is STRIP-SKEWED
//     (solver.h ChainLevel): entry t of a strip is one contiguous line, so E = (i+1,j) and N = (i,j+1) of the
//     previous sweep are lanes L and L+1 of ITS entry t+1, lane 31's N is lane 0 of the next strip's entry t-31 and
//     lane 0's S is lane 31 of the previous strip's entry t+31 of the SAME sweep;
//   * there is no barrier and no flag: every element a sweep writes is an 8-byte {value, launch tag} pair (one
//     store), and a consumer that finds an older tag simply reloads until the tag of THIS launch appears (the LL
//     protocol of NCCL).  How the sweep kernel (smooth_chain3.cuh) fetches and validates its operands is described
//     there;
//   * CTAs take their role (environment, sweep, column block) from a ticket counter, so roles start in dependency
//     order whatever the block scheduler does: a CTA only ever waits for CTAs that have already started;
//   * out-of-domain cells have zero coefficients (host table), so they evaluate to +-0 by themselves; ghosts of d
//     act as 0 during the sweeps (their products with the boundary coefficients are +-0 on every level: level 0
//     r_ghost = 0, coarse levels boundary coefficients = 0, MG.pde:120).
// Arithmetic per update keeps the reference order:
//     d = -(dW*lxW + dE*lxE + dS*lyS + dN*lyN - r) * inv      (the minus sign folded into ninv = -inv: exact)
#pragma once

constexpr unsigned kChSpinMax = 1u << 24;   // bounded reload spin: a tag that never comes is a bug, and a trap beats a hung GPU

__device__ __forceinline__ float ch_lds32(unsigned a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}

// element index of cell (i, j) in a strip-skewed array
__device__ __forceinline__ size_t ch_index(int T, int i, int j) {
  const int s = (j - 1) >> 5, L = (j - 1) & 31;
  return ((size_t)s * T + (i + L)) * 32 + L;
}

constexpr int kC2EdgePad = 32;       // front padding of the edge arrays (smooth_chain3.cuh), entries
// edge array `which` (0 = S edges: lane 31's results, 1 = N edges: lane 0's results) of sweep g, environment e, strip s;
// the element a consumer needs at its step t sits at index t + kC2EdgePad
__device__ __forceinline__ uint2* c2_edge(const ChainLevel& ch, int g, int which, int e, int s) {
  return ch.edge + (size_t)(2 * g + which) * ch.edge_arr + ((size_t)e * ch.NS + s) * ch.TE;
}

// ------------------------------------------------------------------------------------------------
// down pass of a wide coarse level, grid-wide (MG.pde:68-70): smooth(0) + increment + residual restriction
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_chain_down(const __grid_constant__ SolverParams q, int level) {
  const int e = blockIdx.z;
  if (!q.sc.active[e] || slab_skip(blockIdx.y, gridDim.y, q.slab_rank, q.slab_n)) return;
  const DevLevel& L = q.lev[level];
  const DevLevel& C = q.lev[level + 1];
  const int J = blockIdx.x * blockDim.x + threadIdx.x + 1;
  const int I = blockIdx.y * blockDim.y + threadIdx.y + 1;
  if (I > C.n - 2 || J > C.m - 2) return;
  const size_t eo = (size_t)e * L.stride;
  down_block<false>(L, C, L.r + eo, L.d + eo, L.x + eo, C.r + (size_t)e * C.stride, I, J, 0);
}

// ------------------------------------------------------------------------------------------------
// up pass of a chained level, one thread per COARSE cell (MG.pde:75-76,139-152): d = prolongate(coarse.x) incl. its
// setBC, x += d, r -= A d.  The new residual and sweep 0 (d = r*inv, MG.pde:80) go to the strip-skewed arrays.
// LEVEL0: x is the pressure, whose ghost cells are live data (x.plusEq(d) runs over all cells); `r` = the smoothed
// residual the down pass left (level 0: the caller's buffer, coarse levels: L.d).
// ------------------------------------------------------------------------------------------------
template <bool LEVEL0>
__global__ void __launch_bounds__(256)
k_chain_up(const __grid_constant__ SolverParams q, int level, const float* __restrict__ r_all) {
  const int e = blockIdx.z;
  if (!q.sc.active[e] || slab_skip(blockIdx.y, gridDim.y, q.slab_rank, q.slab_n)) return;
  const DevLevel& L0 = q.lev[level];
  const DevLevel& L1 = q.lev[level + 1];
  const ChainLevel& ch = L0.ch;
  const int P = L0.P, n = L0.n, m = L0.m, CPc = L1.P;
  const int nci = L1.n - 2, ncj = L1.m - 2;
  const int J = blockIdx.x * blockDim.x + threadIdx.x + 1;
  const int I = blockIdx.y * blockDim.y + threadIdx.y + 1;
  if (I > nci || J > ncj) return;
  const float* __restrict__ xc = L1.x + (size_t)e * L1.stride;
  const size_t eo = (size_t)e * L0.stride;
  float* __restrict__ x = L0.x + eo;
  const float* __restrict__ r = (LEVEL0 ? r_all : L0.d) + eo;
  float* __restrict__ rsk = ch.rsk + (size_t)e * ch.sk_stride;
  uint2* __restrict__ d0 = ch.dsk[0] + (size_t)e * ch.sk_stride;
  const float dc = xc[I * CPc + J];
  const float dWc = (I > 1) ? xc[(I - 1) * CPc + J] : dc, dEc = (I < nci) ? xc[(I + 1) * CPc + J] : dc;
  const float dSc = (J > 1) ? xc[I * CPc + J - 1] : dc, dNc = (J < ncj) ? xc[I * CPc + J + 1] : dc;
  const int i0 = 2 * I - 1, j0 = 2 * J - 1;
  float xo[2][2], ro[2][2];
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) { xo[a][b] = x[IDX(i0 + a, j0 + b)]; ro[a][b] = r[IDX(i0 + a, j0 + b)]; }
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) {
      const int i = i0 + a, j = j0 + b, k = IDX(i, j);
      const float dW = a ? dc : dWc, dE = a ? dEc : dc, dS = b ? dc : dSc, dN = b ? dNc : dc;
      const float Ad = dc * L0.diag[k] + dW * L0.lx[k] + dE * L0.lx[k + P] + dS * L0.ly[k] + dN * L0.ly[k + 1];
      x[k] = xo[a][b] + dc;
      const float rn = ro[a][b] - Ad;
      const size_t o = ch_index(ch.T, i, j);
      rsk[o] = rn;
      const uint2 d0v = make_uint2(__float_as_uint(rn * L0.inv[k]), 0u);        // MG.pde:80
      d0[o] = d0v;
      // lane-0 columns: the N operand of the previous strip's lane 31 in sweep 1 (consumer step = row + 31)
      if (((j - 1) & 31) == 0) c2_edge(ch, 0, 1, e, (j - 1) >> 5)[i + 31 + kC2EdgePad] = d0v;
      if (LEVEL0) {
        const int di = (i == 1) ? -1 : (i == n - 2 ? 1 : 0), dj = (j == 1) ? -1 : (j == m - 2 ? 1 : 0);
        if (di) x[IDX(i + di, j)] += dc;
        if (dj) x[IDX(i, j + dj)] += dc;
        if (di && dj) x[IDX(i + di, j + dj)] += dc;
      }
    }
}

// ------------------------------------------------------------------------------------------------
// increment after the four sweeps (MG.pde:90-97), threads mapped to the skewed layout: a warp owns a strip and a
// run of kChIncEntries entries, lane L walks its column.  Coarse levels: x += d (the residual update is dead: nothing
// reads r after the last smooth of a level).  LEVEL0: d.setBC (clamped neighbours), x += d on all cells (ghosts
// included), r = r - A d written to the plain residual array, r.r accumulated in double; the last CTA of an
// environment adds the per-CTA partial sums in index order and takes the MGsolver loop decision (MG.pde:32-35).
// ------------------------------------------------------------------------------------------------
constexpr int kChIncEntries = 32;
constexpr int kChIncChunk = 8;
constexpr int kChIncWarps = 4;

template <bool LEVEL0>
__global__ void __launch_bounds__(32 * kChIncWarps)
k_chain_incr(const __grid_constant__ SolverParams q, int level, float* __restrict__ r_out_all, int which) {
  const int e = blockIdx.z;
  if (!q.sc.active[e]) return;
  const DevLevel& Lv = q.lev[level];
  const ChainLevel& ch = Lv.ch;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = Lv.n, m = Lv.m, P = Lv.P, ni = n - 2, mj = m - 2, T = ch.T, NS = ch.NS;
  const int s = blockIdx.y;
#ifndef RLFC_INCR_BY_STRIPS
  // slab mode: blocks are shared out by ROWS (runs of entries), like the row-distributed x and r they update with scattered
  // 4-byte accesses; the strip-distributed skewed arrays are read as whole lines, which travel well over NVLink
  if (slab_skip(blockIdx.x, gridDim.x, q.slab_rank, q.slab_n)) return;
#else
  if (q.slab_n > 1 && (s < ch.s0 || s >= ch.s0 + ch.ns_loc)) return;          // slab mode: the strips this device sweeps
#endif
  const int t0 = (blockIdx.x * kChIncWarps + warp) * kChIncEntries + 1;        // first entry of this warp's run
  const int j = 32 * s + lane + 1;
  const size_t eo = (size_t)e * ch.sk_stride;
  const uint2* __restrict__ d4 = ch.dsk[4] + eo;
  const uint2* dcol = d4 + (size_t)s * T * 32 + lane;
  float* x = Lv.x + (size_t)e * Lv.stride;
  double rr = 0.0;
  if (t0 <= ni + 31) {
    const float4* __restrict__ ct = ch.ct + (size_t)s * T * 32 + lane;
    const float* __restrict__ rsk = ch.rsk + eo + (size_t)s * T * 32 + lane;
    float* __restrict__ r_out = LEVEL0 ? r_out_all + (size_t)e * Lv.stride : nullptr;
    float dW = __uint_as_float(dcol[(size_t)(t0 - 1) * 32].x), dC = __uint_as_float(dcol[(size_t)t0 * 32].x);
    float cxW = LEVEL0 ? ct[(size_t)(t0 - 1) * 32].x : 0.f;
    const int t1 = min(t0 + kChIncEntries - 1, ni + 31);
    // chunks of kChIncChunk entries: every load of a chunk is issued before its first store (the read-modify-write of x
    // would otherwise serialise the loop on one memory round trip per entry)
    for (int tb = t0; tb <= t1; tb += kChIncChunk) {
      float dEv[kChIncChunk], xv[kChIncChunk], rsv[kChIncChunk], dSx[kChIncChunk], dNx[kChIncChunk];
      float4 cv[kChIncChunk];
#pragma unroll
      for (int k = 0; k < kChIncChunk; k++) {
        const int t = tb + k, i = t - lane;
        const bool in = t <= t1, ok = in && i >= 1 && i <= ni && j <= mj;
        dEv[k] = in ? __uint_as_float(dcol[(size_t)(t + 1) * 32].x) : 0.f;
        xv[k] = ok ? x[IDX(i, j)] : 0.f;
        if (LEVEL0) {
          cv[k] = in ? ct[(size_t)t * 32] : make_float4(0.f, 0.f, 0.f, 0.f);
          rsv[k] = ok ? rsk[(size_t)t * 32] : 0.f;
          dSx[k] = (lane == 0 && s > 0 && ok) ? __uint_as_float(d4[((size_t)(s - 1) * T + t + 31) * 32 + 31].x) : 0.f;
          dNx[k] = (lane == 31 && s + 1 < NS && ok) ? __uint_as_float(d4[((size_t)(s + 1) * T + t - 31) * 32].x) : 0.f;
        }
      }
#pragma unroll
      for (int k = 0; k < kChIncChunk; k++) {
        const int t = tb + k, i = t - lane;
        if (t > t1) break;
        const bool ok = i >= 1 && i <= ni && j <= mj;
        const float dE = dEv[k];
        if (LEVEL0) {
          const float4 c = cv[k];
          // S = (i, j-1): lane L-1 of entry t-1 = what that lane holds as dW; N = (i, j+1): lane L+1 of entry t+1 = its dE
          float dS = __shfl_up_sync(0xffffffffu, dW, 1), dN = __shfl_down_sync(0xffffffffu, dE, 1);
          if (lane == 0 && s > 0 && ok) dS = dSx[k];
          if (lane == 31 && s + 1 < NS && ok) dN = dNx[k];
          if (ok) {
            const float w_ = (i == 1) ? dC : dW, e_ = (i == ni) ? dC : dE;          // d.setBC: ghost = adjacent interior
            const float s_ = (j == 1) ? dC : dS, n_ = (j == mj) ? dC : dN;
            const float dg = -(cxW + c.x + c.y + c.z);                              // PoissonMatrix.pde:46-48
            const float Ad = dC * dg + w_ * cxW + e_ * c.x + s_ * c.y + n_ * c.z;   // PoissonMatrix.pde:56-61
            const float rN = rsv[k] - Ad;
            const int kk = IDX(i, j);
            r_out[kk] = rN;
            const float prod = rN * rN;                  // float product, double accumulation (Field.pde:304-307)
            rr += (double)prod;
            x[kk] = xv[k] + dC;
            const int di = (i == 1) ? -1 : (i == ni ? 1 : 0), dj = (j == 1) ? -1 : (j == mj ? 1 : 0);
            if (di) x[IDX(i + di, j)] += dC;
            if (dj) x[IDX(i, j + dj)] += dC;
            if (di && dj) x[IDX(i + di, j + dj)] += dC;
          }
          cxW = c.x;
        } else if (ok) {
          x[IDX(i, j)] = xv[k] + dC;                     // x.plusEq(d), MG.pde:95
        }
        dW = dC; dC = dE;
      }
    }
  }
  if (LEVEL0) {
    // r.r: fixed-order reduction (lanes by shuffle tree, warps in order, CTAs in index order)
    __shared__ double wsum[kChIncWarps];
    __shared__ bool s_last;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rr += __shfl_down_sync(0xffffffffu, rr, o);
    if (lane == 0) wsum[warp] = rr;
    __syncthreads();
    const int nblk = gridDim.x * gridDim.y, blk = blockIdx.y * gridDim.x + blockIdx.x;
    if (threadIdx.x == 0) {
      double sblk = 0;
      for (int w = 0; w < kChIncWarps; w++) sblk += wsum[w];
      q.rr_chain[(size_t)e * q.rr_chain_n + blk] = sblk;
      // (slab mode: the blocks of one environment run on several devices)
      if (q.slab_n > 1) { __threadfence_system(); s_last = atomicAdd_system(q.rr_count + e, 1u) == (unsigned)nblk - 1u; }
      else { __threadfence(); s_last = atomicAdd(q.rr_count + e, 1u) == (unsigned)nblk - 1u; }
    }
    __syncthreads();
    if (s_last) {
      if (q.slab_n > 1) __threadfence_system(); else __threadfence();
      const volatile double* part = q.rr_chain + (size_t)e * q.rr_chain_n;
      double acc = 0;
      for (int k = threadIdx.x; k < nblk; k += blockDim.x) acc += part[k];   // fixed assignment of partial sums to threads
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
      if (lane == 0) wsum[warp] = acc;
      __syncthreads();
      if (threadIdx.x == 0) {
        double sum = 0;
        for (int w = 0; w < kChIncWarps; w++) sum += wsum[w];
        q.rr_count[e] = 0u;
        const int it = ++q.sc.iters[2 * e + which];
        if ((float)sum < q.mg_tol || it >= q.mg_max_iters) q.sc.active[e] = 0;
        else if (q.slab_n > 1) atomicExch_system(q.sc.any_active, 1); else atomicExch(q.sc.any_active, 1);
      }
    }
  }
}
