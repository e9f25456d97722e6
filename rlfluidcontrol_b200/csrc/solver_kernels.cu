// solver_kernels.cu -- hand-written sm_100a kernels of the batched BDIM solver (exact mode).
//
// Compiled with --fmad=false: the reference is Java `float` (one IEEE binary32 rounding per
// operation, no contraction); every expression below keeps the reference's association order so the
// device results are bit-identical to the reference arithmetic.  Reference citations are into
// clientLilypad/.
//
// Kernel inventory (one launch handles the whole batch; blockIdx.z / blockIdx.x = environment):
//   k_advdif      VectorField.AdvDif (QUICK, median-limited)            VectorField.pde:170-222
//   k_band_bc     BDIM blend + mu1 term on the body band, then u.setBC   BDIM.pde:109-122, Field.pde:209-234
//   k_residual    r = div(u) - A p                                      VectorField.pde:56-65, PoissonMatrix.pde:53-68
//   k_mg_down0    level-0 smooth(0) + increment + residual restriction  MG.pde:68-70,79-97,124-137
//   k_mg_coarse   levels >= 1 of the V-cycle in one CTA per env          MG.pde:68-97,124-152
//   k_mg_up0      level-0 prolongation + increment                       MG.pde:75-76,139-152
//   k_smooth0     level-0 smooth(4) + increment + r.r + loop test (strip sweep) MG.pde:30-38,79-97, Field.pde:302-310
//   k_psum        serial float interior sum of p                        Field.pde:311-318
//   k_project_u   gradient of the mean-shifted p, velocity correction   VectorField.pde:136-139
//   k_shift_p     p += -sum(p)/N on all cells                            VectorField.pde:136
//   k_bc          u.setBC after the projection                          VectorField.pde:140
//   k_heun        u = (u + us) * 0.5                                     BDIM.pde:95-96
//   k_force       pressForce + probes + time + draw() accumulation       Body.pde:296-303, SaveScalar.pde:61-72, clientCFD.pde:39-47
#include "solver.h"
#include "smooth_strip.cuh"
#include "smooth_rows.cuh"
#include "smooth_wave.cuh"
#include "exact_sum.cuh"

#ifndef RLFC_DOWN_UNROLL
#define RLFC_DOWN_UNROLL 2      // coarse down pass: blocks in flight per thread
#endif
#ifndef RLFC_UP_ROWS
#define RLFC_UP_ROWS 4          // coarse up pass: rows in flight per warp
#endif
constexpr int kDownUnroll = RLFC_DOWN_UNROLL;

namespace rlfc {
namespace {

__device__ __forceinline__ float pmin(float a, float b) { return (a < b) ? a : b; }   // PApplet.min
__device__ __forceinline__ float pmax(float a, float b) { return (a > b) ? a : b; }   // PApplet.max
__device__ __forceinline__ float med3(float a, float b, float c) {                    // VectorField.pde:221
  return pmax(pmin(a, b), pmin(pmax(a, b), c));
}

// ------------------------------------------------------------------------------------------------
// AdvDif (VectorField.pde:170-222)
//
// The reference evaluates, per cell and component, four limited QUICK face values `bho` (west, east,
// south, north) and forms  adv = (uo*bho_w - ue*bho_e) + (vs*bho_s - vn*bho_n).  The east face of cell
// (i,j) is the west face of cell (i+1,j) with the same face velocity and -- for uf != 0 -- the same
// upwind triple (bc, bd, bu) and the same boundary test, so the product uf*bho is identical; for
// uf == 0 both products are +-0.  Likewise north(i,j) = south(i,j+1).  Each face flux is therefore
// computed once:
//   FXx(i,j) = uo*bho(x,i,j,-1,0,uo)   uo = .5(x[i-1][j] + x[i][j])      (x-faces of the x-component)
//   FXy(i,j) = vs*bho(x,i,j,0,-1,vs)   vs = .5(y[i][j]   + y[i-1][j])
//   FYx(i,j) = uo*bho(y,i,j,-1,0,uo)   uo = .5(x[i][j-1] + x[i][j])      (y-component)
//   FYy(i,j) = vs*bho(y,i,j,0,-1,vs)   vs = .5(y[i][j-1] + y[i][j])
//   adv_x = (FXx(i,j) - FXx(i+1,j)) + (FXy(i,j) - FXy(i,j+1)),  adv_y likewise.
// A warp owns 32 consecutive columns j (28 outputs + 2 halo columns each side, coalesced rows) and
// marches down a chunk of rows with a 4-row register window per component; the i-direction fluxes
// are carried in registers from one row to the next, the j-direction operands and fluxes come from
// neighbouring lanes by shuffle.  PApplet.min/max are realised as FMNMX: they differ from the
// ternaries only in the sign of a zero result, which no later operation can turn into a value change.
// ------------------------------------------------------------------------------------------------
constexpr int kAdvCols = 28;      // output columns per warp
constexpr int kAdvRows = 48;      // rows per chunk

__device__ __forceinline__ float med3f(float a, float b, float c) {                   // VectorField.pde:221
  return fmaxf(fminf(a, b), fminf(fmaxf(a, b), c));
}

// limited QUICK value on the face between cells L and H = L+1 along one direction (VectorField.bho in its
// d = -1 form for cell H): bLL, bL | bH, bHH are the four values along the direction, uf the face velocity,
// `plain_pos` / `plain_neg` say whether the upwind cell (L if uf > 0, else H) fails the bounds test
// `i>n-2 || i<2 || j>m-2 || j<2` (VectorField.pde:212), in which case the plain average is returned.
__device__ __forceinline__ float face_value(float uf, float bLL, float bL, float bH, float bHH, bool plain_pos,
                                            bool plain_neg) {
  const float CF = 1.f / 6.f, S = 10.f;
  float bf = 0.5f * (bL + bH);
  const bool pos = uf > 0;
  const float bc = pos ? bL : bH, bd = pos ? bH : bL, bu = pos ? bLL : bHH;
  const float q = bf - CF * (bd - 2 * bc + bu);
  const float b1 = bu + S * (bc - bu);
  const float lim = med3f(q, bc, med3f(bc, bd, b1));
  return (pos ? plain_pos : plain_neg) ? bf : lim;
}

#ifndef RLFC_ADV_MINB
#define RLFC_ADV_MINB 9      // 56 registers, 9 CTAs per SM: 202 -> 193 us (8: 198, 10 and 12 spill: 201, 217)
#endif
template <bool PREDICTOR>
__global__ void __launch_bounds__(128, RLFC_ADV_MINB)
k_advdif(const float* __restrict__ srcx, const float* __restrict__ srcy, const float* __restrict__ u0x,
         const float* __restrict__ u0y, float* __restrict__ dstx, float* __restrict__ dsty, int n, int m, int P,
         size_t stride, float dt, float nu, const int* __restrict__ frozen, int slab_rank, int slab_n, int chunk_rows) {
  if (frozen[blockIdx.z] || slab_skip(blockIdx.y, gridDim.y, slab_rank, slab_n)) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ni = n - 2, mj = m - 2;
  const int jw0 = 1 + blockIdx.x * kAdvCols;                         // first output column of this warp
  const int ia = 1 + (blockIdx.y * 4 + warp) * chunk_rows;           // first row of this chunk
  if (ia > ni) return;
  const int ib = min(ia + chunk_rows - 1, ni);
  const size_t eo = (size_t)blockIdx.z * stride;
  const float* __restrict__ x = srcx + eo;
  const float* __restrict__ y = srcy + eo;
  const int j = jw0 - 2 + lane;                                      // this lane's column (may be outside the array)
  const int jl = min(max(j, 0), m - 1);                              // clamped for loads
  const bool last_cw = jw0 + kAdvCols > mj;                          // this warp also owns ghost column m-1
  const bool out_lane = lane >= 2 && lane < 2 + kAdvCols && j >= 1 && j <= mj;
  const bool ghost_lane = (j == 0 && jw0 == 1) || (j == m - 1 && last_cw);
  // bounds test of bho along j for this column's south face (upwind column j-1 if v > 0, else j), and the
  // column part of the test for the x-direction faces
  const bool jplain_pos = (j - 1 < 2) || (j - 1 > m - 2), jplain_neg = (j < 2) || (j > m - 2);
  const bool jbad = jplain_neg;
  auto ldx = [&](int i) { return x[IDX(min(max(i, 0), n - 1), jl)]; };
  auto ldy = [&](int i) { return y[IDX(min(max(i, 0), n - 1), jl)]; };
  // register window: rows i-2 .. i+1 (a = i-2, b = i-1, c = i, d = i+1), e = i+2 arrives during the step
  float xa = ldx(ia - 2), xb = ldx(ia - 1), xc = ldx(ia), xd = ldx(ia + 1);
  float ya = ldy(ia - 2), yb = ldy(ia - 1), yc = ldy(ia), yd = ldy(ia + 1);
  if (ia == 1 && (out_lane || ghost_lane)) {                          // ghost row 0 of F keeps u's values
    dstx[eo + IDX(0, j)] = xb;
    dsty[eo + IDX(0, j)] = yb;
  }
  // west fluxes of the first row: faces between rows ia-1 and ia
  float fxw, fyw;
  {
    const bool ip = (ia - 1 < 2) || (ia - 1 > n - 2) || jbad, in_ = (ia < 2) || (ia > n - 2) || jbad;
    const float uox = 0.5f * (xb + xc);
    fxw = uox * face_value(uox, xa, xb, xc, xd, ip, in_);
    const float xcm1 = __shfl_up_sync(0xffffffffu, xc, 1);
    const float uoy = 0.5f * (xcm1 + xc);
    fyw = uoy * face_value(uoy, ya, yb, yc, yd, ip, in_);
  }
#pragma unroll 4
  for (int i = ia; i <= ib; i++) {
    const float xe = ldx(i + 2), ye = ldy(i + 2);
    float u0xv, u0yv;
    if (PREDICTOR) { u0xv = xc; u0yv = yc; }
    else { u0xv = u0x[eo + IDX(i, jl)]; u0yv = u0y[eo + IDX(i, jl)]; }
    // neighbours along j of rows i (c) and i+1 (d), i-1 (b)
    const float xcm2 = __shfl_up_sync(0xffffffffu, xc, 2), xcm1 = __shfl_up_sync(0xffffffffu, xc, 1);
    const float xcp1 = __shfl_down_sync(0xffffffffu, xc, 1);
    const float ycm2 = __shfl_up_sync(0xffffffffu, yc, 2), ycm1 = __shfl_up_sync(0xffffffffu, yc, 1);
    const float ycp1 = __shfl_down_sync(0xffffffffu, yc, 1);
    const float xdm1 = __shfl_up_sync(0xffffffffu, xd, 1);
    // east faces (between rows i and i+1) = west faces of row i+1
    const bool ip = (i < 2) || (i > n - 2) || jbad, in_ = (i + 1 < 2) || (i + 1 > n - 2) || jbad;
    const float uex = 0.5f * (xc + xd);
    const float fxe = uex * face_value(uex, xb, xc, xd, xe, ip, in_);
    const float uey = 0.5f * (xdm1 + xd);
    const float fye = uey * face_value(uey, yb, yc, yd, ye, ip, in_);
    // south faces of this column (between columns j-1 and j) on row i
    const bool ibad = (i < 2) || (i > n - 2);
    const float vsx = 0.5f * (yc + yb);
    const float fxs = vsx * face_value(vsx, xcm2, xcm1, xc, xcp1, jplain_pos || ibad, jplain_neg || ibad);
    const float vsy = 0.5f * (ycm1 + yc);
    const float fys = vsy * face_value(vsy, ycm2, ycm1, yc, ycp1, jplain_pos || ibad, jplain_neg || ibad);
    // north faces = south faces of column j+1
    const float fxn = __shfl_down_sync(0xffffffffu, fxs, 1), fyn = __shfl_down_sync(0xffffffffu, fys, 1);
    const float advx = (fxw - fxe) + (fxs - fxn);
    const float advy = (fyw - fye) + (fys - fyn);
    const float difx = xd + xcp1 - 4 * xc + xb + xcm1;                 // VectorField.pde:198-200
    const float dify = yd + ycp1 - 4 * yc + yb + ycm1;
    if (out_lane) {
      dstx[eo + IDX(i, j)] = (advx + nu * difx) * dt + u0xv;
      dsty[eo + IDX(i, j)] = (advy + nu * dify) * dt + u0yv;
    } else if (ghost_lane) {                                           // ghost columns of F keep u's values
      dstx[eo + IDX(i, j)] = xc;
      dsty[eo + IDX(i, j)] = yc;
    }
    fxw = fxe; fyw = fye;
    xa = xb; xb = xc; xc = xd; xd = xe;
    ya = yb; yb = yc; yc = yd; yd = ye;
  }
  if (ib == ni && (out_lane || ghost_lane)) {                          // ghost row n-1
    dstx[eo + IDX(n - 1, j)] = xc;
    dsty[eo + IDX(n - 1, j)] = yc;
  }
}

// Serial float sum of v[1 .. m-2] in index order (the outflow mean of Field.setBC, Field.pde:216-217) by ONE thread: the
// additions form a dependent chain, the shared-memory loads do not -- sixteen of them are issued ahead of their adds.
__device__ __forceinline__ float serial_sum_interior(const float* v, int m) {
  float s = 0;
  int j = 1;
  for (; j + 16 <= m - 1; j += 16) {
    float t[16];
#pragma unroll
    for (int k = 0; k < 16; k++) t[k] = v[j + k];
#pragma unroll
    for (int k = 0; k < 16; k++) s += t[k];
  }
  for (; j < m - 1; j++) s += v[j];
  return s;
}

// ------------------------------------------------------------------------------------------------
// Field.setBC executed by one CTA (Field.pde:209-234, loop structure and statement order kept)
// ------------------------------------------------------------------------------------------------
__device__ void cta_setBC(float* a, int n, int m, int P, int btype, float bval, bool gexit, float* scol) {
  const int tid = threadIdx.x, nt = blockDim.x;
  __shared__ float s_mean;
  for (int j = tid; j < m; j += nt) {
    a[IDX(0, j)] = a[IDX(1, j)];
    float e = a[IDX(n - 2, j)];
    a[IDX(n - 1, j)] = e;
    if (btype == 1) {
      a[IDX(1, j)] = bval;
      if (gexit) scol[j] = e; else a[IDX(n - 1, j)] = bval;
    }
  }
  __syncthreads();
  if (gexit && tid == 0) {
    const float s = serial_sum_interior(scol, m);       // serial float sum in j order
    s_mean = s / (float)(m - 2);
  }
  for (int i = tid; i < n; i += nt) {
    a[IDX(i, 0)] = a[IDX(i, 1)];
    a[IDX(i, m - 1)] = a[IDX(i, m - 2)];
    if (btype == 2) { a[IDX(i, 1)] = bval; a[IDX(i, m - 1)] = bval; }
  }
  __syncthreads();
  if (gexit) {
    const float s = s_mean;
    for (int j = 1 + tid; j < m - 1; j += nt) a[IDX(n - 1, j)] += bval - s;
  }
  __syncthreads();
}

// body velocity from the static basis (BodyUnion.velocity BodyUnion.pde:84-92, Body.velocity Body.pde:234-240)
__device__ __forceinline__ float ub_x(const SolverParams& q, int k, float dphi1, float dphi2) {
  float u1 = (0.f - q.ry1_x[k] * dphi1) / q.dt;
  float u2 = (0.f - q.ry2_x[k] * dphi2) / q.dt;
  float v = 0.f + u1 * q.w1_x[k];
  return v + u2 * q.w2_x[k];
}
__device__ __forceinline__ float ub_y(const SolverParams& q, int k, float dphi1, float dphi2) {
  float u1 = (0.f + q.rx1_y[k] * dphi1) / q.dt;
  float u2 = (0.f + q.rx2_y[k] * dphi2) / q.dt;
  float v = 0.f + u1 * q.w1_y[k];
  return v + u2 * q.w2_y[k];
}

// BDIM.updateUP blend of one band face (BDIM.pde:109-122): u = del*R - ub*(del + (-1)) + del1 * normalGrad(R - ub)
template <bool XCOMP>
__device__ __forceinline__ float band_face(const SolverParams& q, const float* u, const BandFace& f, float dphi1, float dphi2) {
  const int P = q.P, k = IDX(f.i, f.j);
  auto ub = [&](int kk) { return XCOMP ? ub_x(q, kk, dphi1, dphi2) : ub_y(q, kk, dphi1, dphi2); };
  const float R = u[k], ubc = ub(k);
  const float v = f.del * R - ubc * (f.del + (-1.f));
  const float duE = u[k + P] - ub(k + P), duW = u[k - P] - ub(k - P);
  const float duN = u[k + 1] - ub(k + 1), duS = u[k - 1] - ub(k - 1);
  const float g = 0.5f * (f.wnx * (duE - duW) + f.wny * (duN - duS));         // VectorField.pde:50-51
  return v + f.del1 * g;
}

// the blend for a whole (large) band, grid-wide: values go to band_tmp, k_band_bc<true> writes them back
__global__ void __launch_bounds__(256)
k_band_blend(const __grid_constant__ SolverParams q, const float* ux_all, const float* uy_all) {
  const int e = blockIdx.y, b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= q.nband_x + q.nband_y || q.sc.frozen[e] || slab_skip(blockIdx.x, gridDim.x, q.slab_rank, q.slab_n)) return;
  const float* ux = ux_all + (size_t)e * q.stride;
  const float* uy = uy_all + (size_t)e * q.stride;
  float* tmp = q.band_tmp + (size_t)e * (q.nband_x + q.nband_y);
  const float xi1_m = q.action_scale * q.sc.xi[2 * e], xi2_m = q.action_scale * q.sc.xi[2 * e + 1];   // AFCCylinder.pde:48-49
  const float dphi1 = (2 * xi1_m * q.dt) / q.dRD, dphi2 = (2 * xi2_m * q.dt) / q.dRD;
  tmp[b] = (b < q.nband_x) ? band_face<true>(q, ux, q.band_x[b], dphi1, dphi2)
                           : band_face<false>(q, uy, q.band_y[b - q.nband_x], dphi1, dphi2);
}

// BDIM.updateUP blend on the body band (everywhere else it is the identity), then u.setBC()
template <bool PREBLENDED>
__global__ void __launch_bounds__(1024)
k_band_bc(const __grid_constant__ SolverParams q, float* ux_all, float* uy_all) {
  extern __shared__ float scol[];
  const int e = blockIdx.x, P = q.P;
  if (q.sc.frozen[e]) return;
  float* ux = ux_all + (size_t)e * q.stride;
  float* uy = uy_all + (size_t)e * q.stride;
  float* tmp = q.band_tmp + (size_t)e * (q.nband_x + q.nband_y);
  if (!PREBLENDED) {
    // AFCCylinder.pde:48-49
    const float xi1_m = q.action_scale * q.sc.xi[2 * e], xi2_m = q.action_scale * q.sc.xi[2 * e + 1];
    const float dphi1 = (2 * xi1_m * q.dt) / q.dRD, dphi2 = (2 * xi2_m * q.dt) / q.dRD;
    for (int b = threadIdx.x; b < q.nband_x; b += blockDim.x) tmp[b] = band_face<true>(q, ux, q.band_x[b], dphi1, dphi2);
    for (int b = threadIdx.x; b < q.nband_y; b += blockDim.x) tmp[q.nband_x + b] = band_face<false>(q, uy, q.band_y[b], dphi1, dphi2);
    __syncthreads();
  }
  for (int b = threadIdx.x; b < q.nband_x; b += blockDim.x) ux[IDX(q.band_x[b].i, q.band_x[b].j)] = tmp[b];
  for (int b = threadIdx.x; b < q.nband_y; b += blockDim.x) uy[IDX(q.band_y[b].i, q.band_y[b].j)] = tmp[q.nband_x + b];
  __syncthreads();
  cta_setBC(ux, q.n, q.m, P, 1, 1.f, true, scol);     // u.x: btype 1, bval 1, gradientExit (BDIM.pde:52)
  cta_setBC(uy, q.n, q.m, P, 2, 0.f, false, scol);
}

__global__ void __launch_bounds__(1024)
k_bc(const __grid_constant__ SolverParams q, float* ux_all, float* uy_all) {
  extern __shared__ float scol[];
  const int e = blockIdx.x;
  if (q.sc.frozen[e]) return;
  cta_setBC(ux_all + (size_t)e * q.stride, q.n, q.m, q.P, 1, 1.f, true, scol);
  cta_setBC(uy_all + (size_t)e * q.stride, q.n, q.m, q.P, 2, 0.f, false, scol);
}

// ------------------------------------------------------------------------------------------------
// u.setBC (and optionally the BDIM band blend before it) with TWO global-memory phases per environment: every
// operand Field.setBC reads (rows 1 and n-2, columns 1 and m-2 of both components) is fetched up front, the
// statement sequence of Field.pde:209-234 is then replayed on shared-memory copies (same order, same corner
// hand-offs, same serial outflow sum), and the ghost ring is written in one go.  Valid when no band face lies on
// those four lines (checked on the host; the literal kernels above remain the fallback).
// ------------------------------------------------------------------------------------------------
struct BcLines {            // shared-memory image of one component's boundary lines
  float *r0, *r1, *rn1;     // new rows 0, 1, n-1            [m]
  float *c1, *cm2;          // columns 1 and m-2 as loaded    [n]
};

// phase 1 of one component: rows 1 and n-2, columns 1 and m-2 are read and the shared-memory image is formed (the CTA
// strides over the lines, so they may be longer than the CTA)
__device__ __forceinline__ void bc_stage(const BcLines& s, const float* a, int tid, int nt, int n, int m, int P, int btype,
                                         float bval, bool gexit) {
  for (int j = tid; j < m; j += nt) {
    const float row1 = a[IDX(1, j)], rown2 = a[IDX(n - 2, j)];
    s.r0[j] = row1;                                     // a[0][j] = a[1][j]
    s.rn1[j] = (btype == 1 && !gexit) ? bval : rown2;   // a[n-1][j] = a[n-2][j]; btype 1 without gradientExit: = bval
    s.r1[j] = (btype == 1) ? bval : row1;               // btype 1: a[1][j] = bval
  }
  for (int i = tid; i < n; i += nt) { s.c1[i] = a[IDX(i, 1)]; s.cm2[i] = a[IDX(i, m - 2)]; }
}

// final values after the column loop and the outflow correction; `mean` = s/(m-2) of the gradientExit sum
__device__ __forceinline__ void bc_store(const BcLines& s, float* a, int tid, int nt, int n, int m, int P, int btype, float bval,
                                         bool gexit, float mean) {
  for (int j = 1 + tid; j <= m - 2; j += nt) {          // rows 0, 1, n-1, interior columns
    const bool b2 = btype == 2 && j == 1;               // btype 2: a[i][1] = bval on every row
    a[IDX(0, j)] = b2 ? bval : s.r0[j];
    if (btype == 1 || b2) a[IDX(1, j)] = b2 ? bval : s.r1[j];
    float v = s.rn1[j];
    if (gexit) v += bval - mean;                        // a[n-1][j] += bval - s for interior j
    a[IDX(n - 1, j)] = b2 ? bval : v;
  }
  for (int i = tid; i < n; i += nt) {                   // columns 0, (1), m-1 on every row, corners included
    const float src1 = (i == 0) ? s.r0[1] : (i == 1) ? s.r1[1] : (i == n - 1) ? s.rn1[1] : s.c1[i];
    const float src2 = (i == 0) ? s.r0[m - 2] : (i == 1) ? s.r1[m - 2] : (i == n - 1) ? s.rn1[m - 2] : s.cm2[i];
    a[IDX(i, 0)] = src1;                                // a[i][0] = a[i][1]
    a[IDX(i, m - 1)] = (btype == 2) ? bval : src2;      // a[i][m-1] = a[i][m-2]; btype 2: = bval
    if (btype == 2) a[IDX(i, 1)] = bval;
  }
}

template <bool BAND, bool HEUN>
__global__ void __launch_bounds__(1024)
k_bc2(const __grid_constant__ SolverParams q, float* ux_all, float* uy_all, const float* usx_all, const float* usy_all,
      float* uox_all, float* uoy_all) {
  extern __shared__ float bc_smem[];
  const int e = blockIdx.x, P = q.P, n = q.n, m = q.m, tid = threadIdx.x;
  if (q.sc.frozen[e]) return;
  float* ux = ux_all + (size_t)e * q.stride;
  float* uy = uy_all + (size_t)e * q.stride;
  BcLines sx, sy;
  float* w = bc_smem;
  sx.r0 = w; sx.r1 = w + m; sx.rn1 = w + 2 * m; sx.c1 = w + 3 * m; sx.cm2 = w + 3 * m + n;
  w += 3 * m + 2 * n;
  sy.r0 = w; sy.r1 = w + m; sy.rn1 = w + 2 * m; sy.c1 = w + 3 * m; sy.cm2 = w + 3 * m + n;
  w += 3 * m + 2 * n;
  float* tmp = w;                                        // [nband_x + nband_y] blended band values
  __shared__ float s_mean;
  // ---- phase 1: every load ----
  // u.x: btype 1, bval 1, gradientExit (BDIM.pde:52); u.y: btype 2, bval 0
  bc_stage(sx, ux, tid, blockDim.x, n, m, P, 1, 1.f, true);
  bc_stage(sy, uy, tid, blockDim.x, n, m, P, 2, 0.f, false);
  if (BAND) {
    // BDIM.updateUP blend on the body band (BDIM.pde:109-122), identical arithmetic to k_band_bc
    const float xi1_m = q.action_scale * q.sc.xi[2 * e], xi2_m = q.action_scale * q.sc.xi[2 * e + 1];
    const float dphi1 = (2 * xi1_m * q.dt) / q.dRD, dphi2 = (2 * xi2_m * q.dt) / q.dRD;
    for (int b = tid; b < q.nband_x; b += blockDim.x) {
      const BandFace f = q.band_x[b];
      const int k = IDX(f.i, f.j);
      float R = ux[k], ub = ub_x(q, k, dphi1, dphi2);
      float v = f.del * R - ub * (f.del + (-1.f));
      float duE = ux[k + P] - ub_x(q, k + P, dphi1, dphi2), duW = ux[k - P] - ub_x(q, k - P, dphi1, dphi2);
      float duN = ux[k + 1] - ub_x(q, k + 1, dphi1, dphi2), duS = ux[k - 1] - ub_x(q, k - 1, dphi1, dphi2);
      float g = 0.5f * (f.wnx * (duE - duW) + f.wny * (duN - duS));       // VectorField.pde:50
      tmp[b] = v + f.del1 * g;
    }
    for (int b = tid; b < q.nband_y; b += blockDim.x) {
      const BandFace f = q.band_y[b];
      const int k = IDX(f.i, f.j);
      float R = uy[k], ub = ub_y(q, k, dphi1, dphi2);
      float v = f.del * R - ub * (f.del + (-1.f));
      float duE = uy[k + P] - ub_y(q, k + P, dphi1, dphi2), duW = uy[k - P] - ub_y(q, k - P, dphi1, dphi2);
      float duN = uy[k + 1] - ub_y(q, k + 1, dphi1, dphi2), duS = uy[k - 1] - ub_y(q, k - 1, dphi1, dphi2);
      float g = 0.5f * (f.wnx * (duE - duW) + f.wny * (duN - duS));       // VectorField.pde:51
      tmp[q.nband_x + b] = v + f.del1 * g;
    }
  }
  __syncthreads();
  if (tid == 0) {
    const float s = serial_sum_interior(sx.rn1, m);      // serial float sum in j order (Field.pde:216-217)
    s_mean = s / (float)(m - 2);
  }
  // ---- phase 2: every store ----
  if (BAND) {
    for (int b = tid; b < q.nband_x; b += blockDim.x) ux[IDX(q.band_x[b].i, q.band_x[b].j)] = tmp[b];
    for (int b = tid; b < q.nband_y; b += blockDim.x) uy[IDX(q.band_y[b].i, q.band_y[b].j)] = tmp[q.nband_x + b];
  }
  __syncthreads();
  bc_store(sx, ux, tid, blockDim.x, n, m, P, 1, 1.f, true, s_mean);
  bc_store(sy, uy, tid, blockDim.x, n, m, P, 2, 0.f, false, 0.f);
  if (HEUN) {
    // u = (u + us) * 0.5 on the zone k_project_shift<true> left to us (rows 0, 1, n-2, n-1; the first float4 of every
    // row; the float4s from the one holding column m-2 on): the values the boundary conditions just produced
    __syncthreads();
    const float* usx = usx_all + (size_t)e * q.stride;
    const float* usy = usy_all + (size_t)e * q.stride;
    float* uox = uox_all + (size_t)e * q.stride;
    float* uoy = uoy_all + (size_t)e * q.stride;
    const int jz = 4 * ((m - 2) / 4), wz = 4 + (P - jz);      // zone columns of an interior row: [0, 4) and [jz, P)
    for (int t = tid; t < 4 * P; t += blockDim.x) {           // the four full rows
      const int r = t / P, j = t - r * P;
      const int i = (r < 2) ? r : n - 4 + r;
      const int k = IDX(i, j);
      uox[k] = (ux[k] + usx[k]) * 0.5f;
      uoy[k] = (uy[k] + usy[k]) * 0.5f;
    }
    for (int t = tid; t < (n - 4) * wz; t += blockDim.x) {    // the column strips of rows 2 .. n-3
      const int r = t / wz, c = t - r * wz;
      const int i = 2 + r, j = (c < 4) ? c : jz + (c - 4);
      const int k = IDX(i, j);
      uox[k] = (ux[k] + usx[k]) * 0.5f;
      uoy[k] = (uy[k] + usy[k]) * 0.5f;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// residual r = div(u) - A p   (VectorField.pde:56-65, PoissonMatrix.pde:53-68); also opens the solve
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float apply_A(const float* x, const float* __restrict__ lx, const float* __restrict__ ly,
                                         const float* __restrict__ diag, int P, int k) {
  return x[k] * diag[k] + x[k - P] * lx[k] + x[k + P] * lx[k + P] + x[k - 1] * ly[k] + x[k + 1] * ly[k + 1];
}

__global__ void __launch_bounds__(256)
k_residual(const __grid_constant__ SolverParams q, const float* __restrict__ ux_all, const float* __restrict__ uy_all,
           float* __restrict__ r_all, int which) {
  const int P = q.P;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  const int e = blockIdx.z;
  if (q.sc.frozen[e]) return;                          // (active[e] is 0 after every completed solve: the MG kernels skip it too)
  if (i == 0 && j == 0) { q.sc.active[e] = 1; q.sc.iters[2 * e + which] = 0; }
  if (i < 1 || j < 1 || i > q.n - 2 || j > q.m - 2) return;
  const size_t eo = (size_t)e * q.stride;
  const float* ux = ux_all + eo;
  const float* uy = uy_all + eo;
  const float* p = q.lev[0].x + eo;
  const int k = IDX(i, j);
  float s = ux[k + P] - ux[k] + uy[k + 1] - uy[k];
  r_all[eo + k] = s - apply_A(p, q.lev[0].lx, q.lev[0].ly, q.lev[0].diag, P, k);
}

// ------------------------------------------------------------------------------------------------
// down pass of one level, one thread per coarse cell = 2x2 fine block (MG.pde:68-70):
//   smooth(0): d = r*inv, d.setBC (ghost = clamped interior), x += d, r -= A d;  then restrict r.
// `rin` is read with its 4x4 neighbourhood, so the new residual goes to a different buffer `rout`.
// ------------------------------------------------------------------------------------------------
template <bool LEVEL0>
__device__ __forceinline__ void down_block(const DevLevel& L, const DevLevel& C, const float* __restrict__ rin,
                                           float* __restrict__ rout, float* __restrict__ x, float* __restrict__ rc,
                                           int I, int J) {
  const int P = L.P, n = L.n, m = L.m;
  const int i0 = (I - 1) * 2 + 1, j0 = (J - 1) * 2 + 1;
  float d[4][4], rv[2][2];
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++) {
      if ((a == 0 || a == 3) && (b == 0 || b == 3)) { d[a][b] = 0.f; continue; }
      int ci = min(max(i0 - 1 + a, 1), n - 2), cj = min(max(j0 - 1 + b, 1), m - 2);
      const float rr = rin[IDX(ci, cj)];
      d[a][b] = rr * L.inv[IDX(ci, cj)];
      if (a >= 1 && a <= 2 && b >= 1 && b <= 2) rv[a - 1][b - 1] = rr;       // (the block's own cells are never clamped)
    }
  // the block's face coefficients, each loaded once: lx on rows i0 .. i0+2, ly on columns j0 .. j0+2; the diagonal is
  // their plain sum (PoissonMatrix.pde:46-48; checked against the host table at create time)
  float lxv[3][2], lyv[2][3];
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) lxv[a][b] = L.lx[IDX(i0 + a, j0 + b)];
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 3; b++) lyv[a][b] = L.ly[IDX(i0 + a, j0 + b)];
  float rn[2][2];
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) {
      const int i = i0 + a, j = j0 + b, k = IDX(i, j);
      const float dc = d[a + 1][b + 1];
      const float dg = -(lxv[a][b] + lxv[a + 1][b] + lyv[a][b] + lyv[a][b + 1]);
      float Ad = dc * dg + d[a][b + 1] * lxv[a][b] + d[a + 2][b + 1] * lxv[a + 1][b] + d[a + 1][b] * lyv[a][b] +
                 d[a + 1][b + 2] * lyv[a][b + 1];
      rn[a][b] = rv[a][b] - Ad;
      rout[k] = rn[a][b];
      if (LEVEL0) {
        x[k] += dc;
        // ghosts of x receive the clamped d (x.plusEq(d) runs over all cells, MG.pde:95); p's ghosts are live data
        const int di = (i == 1) ? -1 : (i == n - 2 ? 1 : 0), dj = (j == 1) ? -1 : (j == m - 2 ? 1 : 0);
        if (di) x[IDX(i + di, j)] += dc;
        if (dj) x[IDX(i, j + dj)] += dc;
        if (di && dj) x[IDX(i + di, j + dj)] += dc;
      } else {
        x[k] = 0.f + dc;   // coarse x starts at 0 (MG.pde:56); its ghosts are never read (prolongate's setBC overwrites them)
      }
    }
  // MG.restrict(Field) MG.pde:128-133 (its setBC only fills ghosts, which no later operation reads with a non-zero weight)
  rc[I * C.P + J] = rn[0][0] + rn[0][1] + rn[1][0] + rn[1][1];
}

__global__ void __launch_bounds__(256)
k_mg_down0(const __grid_constant__ SolverParams q, const float* __restrict__ rin_all, float* __restrict__ rout_all) {
  const int e = blockIdx.z;
  if (!q.sc.active[e] || slab_skip(blockIdx.y, gridDim.y, q.slab_rank, q.slab_n)) return;
  const DevLevel& L0 = q.lev[0];
  const DevLevel& L1 = q.lev[1];
  const int J = blockIdx.x * blockDim.x + threadIdx.x + 1;   // coarse interior indices
  const int I = blockIdx.y * blockDim.y + threadIdx.y + 1;
  if (I > L1.n - 2 || J > L1.m - 2) return;
  const size_t eo = (size_t)e * L0.stride;
  down_block<true>(L0, L1, rin_all + eo, rout_all + eo, L0.x + eo, L1.r + (size_t)e * L1.stride, I, J);
}

// ------------------------------------------------------------------------------------------------
// First MG iteration of a solve, level 0, fused:  r = div(u) - A p  (VectorField.pde:56-65,
// PoissonMatrix.pde:53-68), then smooth(0) + increment + residual restriction (MG.pde:68-70,79-97,124-137).
// A CTA owns kRdI x kRdJ coarse cells (= 2*kRdI x 2*kRdJ fine cells); phase 1 forms the residual on that tile
// plus a one-cell halo (clamped to the interior, exactly the operands d.setBC would provide) in shared memory,
// phase 2 is down_block on shared-memory operands.  p is read with a distance-2 halo while it is being
// updated, so the new p goes to the OTHER pressure buffer (p ping-pongs A -> B here and B -> A in
// k_project_shift); the unsmoothed residual never reaches HBM.
// ------------------------------------------------------------------------------------------------
constexpr int kRdI = 8, kRdJ = 32;                       // coarse cells per CTA (one per thread)
constexpr int kRdTI = 2 * kRdI + 2, kRdTJ = 2 * kRdJ + 2;

__global__ void __launch_bounds__(kRdI * kRdJ)
k_resid_down0(const __grid_constant__ SolverParams q, const float* __restrict__ ux_all, const float* __restrict__ uy_all,
              const float* __restrict__ pin_all, float* __restrict__ pout_all, float* __restrict__ rout_all, int which) {
  __shared__ float s_r[kRdTI][kRdTJ + 1];
  __shared__ float s_d[kRdTI][kRdTJ + 1];
  const DevLevel& L = q.lev[0];
  const DevLevel& C = q.lev[1];
  const int P = L.P, n = L.n, m = L.m;
  const int e = blockIdx.z;
  if (q.sc.frozen[e]) return;                          // (active[e] is 0 after every completed solve: the MG kernels skip it too)
  if (slab_skip(blockIdx.y, gridDim.y, q.slab_rank, q.slab_n)) return;
  const int tid = threadIdx.y * kRdJ + threadIdx.x;
  if (blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) { q.sc.active[e] = 1; q.sc.iters[2 * e + which] = 0; }
  const size_t eo = (size_t)e * L.stride;
  const float* __restrict__ ux = ux_all + eo;
  const float* __restrict__ uy = uy_all + eo;
  const float* __restrict__ pin = pin_all + eo;
  const int I0 = blockIdx.y * kRdI + 1, J0 = blockIdx.x * kRdJ + 1;     // first coarse cell of the tile
  const int i0 = (I0 - 1) * 2 + 1, j0 = (J0 - 1) * 2 + 1;              // first fine cell
  // ---- phase 1: r and d = r*inv on the tile + halo, at clamped coordinates ----
  for (int t = tid; t < kRdTI * kRdTJ; t += kRdI * kRdJ) {
    const int a = t / kRdTJ, b = t - a * kRdTJ;
    const int i = min(max(i0 - 1 + a, 1), n - 2), j = min(max(j0 - 1 + b, 1), m - 2);
    const int k = IDX(i, j);
    const float sdiv = ux[k + P] - ux[k] + uy[k + 1] - uy[k];
    const float rv = sdiv - apply_A(pin, L.lx, L.ly, L.diag, P, k);
    s_r[a][b] = rv;
    s_d[a][b] = rv * L.inv[k];
  }
  __syncthreads();
  // ---- phase 2: smooth(0) increment and restriction for this thread's coarse cell ----
  const int I = I0 + threadIdx.y, J = J0 + threadIdx.x;
  if (I > C.n - 2 || J > C.m - 2) return;
  const int fi = (I - 1) * 2 + 1, fj = (J - 1) * 2 + 1;
  const int ta = 2 * threadIdx.y + 1, tb = 2 * threadIdx.x + 1;          // tile coordinates of (fi, fj)
  float* __restrict__ pout = pout_all + eo;
  float* __restrict__ rout = rout_all + eo;
  float rn[2][2];
#pragma unroll
  for (int a = 0; a < 2; a++)
#pragma unroll
    for (int b = 0; b < 2; b++) {
      const int i = fi + a, j = fj + b, k = IDX(i, j);
      const float dc = s_d[ta + a][tb + b];
      const float Ad = dc * L.diag[k] + s_d[ta + a - 1][tb + b] * L.lx[k] + s_d[ta + a + 1][tb + b] * L.lx[k + P] +
                       s_d[ta + a][tb + b - 1] * L.ly[k] + s_d[ta + a][tb + b + 1] * L.ly[k + 1];
      rn[a][b] = s_r[ta + a][tb + b] - Ad;
      rout[k] = rn[a][b];
      pout[k] = pin[k] + dc;
      // ghosts of x receive the clamped d (x.plusEq(d) runs over all cells, MG.pde:95)
      const int di = (i == 1) ? -1 : (i == n - 2 ? 1 : 0), dj = (j == 1) ? -1 : (j == m - 2 ? 1 : 0);
      if (di) pout[IDX(i + di, j)] = pin[IDX(i + di, j)] + dc;
      if (dj) pout[IDX(i, j + dj)] = pin[IDX(i, j + dj)] + dc;
      if (di && dj) pout[IDX(i + di, j + dj)] = pin[IDX(i + di, j + dj)] + dc;
    }
  // MG.restrict(Field) MG.pde:128-133
  C.r[(size_t)e * C.stride + I * C.P + J] = rn[0][0] + rn[0][1] + rn[1][0] + rn[1][1];
}

// ------------------------------------------------------------------------------------------------
// The same fused first MG iteration as a MARCHING kernel (the default; k_resid_down0 above is kept as the cross-check,
// RLFC_RESID=tile): a compute warp owns kRmCols columns (+2 halo lanes on either side, as k_advdif) and marches down
// the CTA's kRmRows rows.  Everything that is shared between neighbouring cells is read ONCE: p, ux, lx travel down the
// rows in registers, the j-neighbours of p, uy, ly and d come from the adjacent lanes by shuffle -- 7 reads, 8 shuffles
// and ~27 float operations per cell.  Row i is finalised one step after its d is formed, when d of row i+1 exists.
// Arithmetic and its order are those of k_resid_down0 / the reference.
//
// Where the operands come from: the kernel streams at HBM speed only with enough bytes in flight, and register-target
// loads cannot provide them (one row per lane in flight at 64 registers and 50 % occupancy: 2.4 TB/s; issuing them a
// row or two ahead needed 88 registers and serialised on the warp's load scoreboards, 176 -> 241 us).  So the rows
// come through a shared-memory ring: one lane of a loader warp bulk-copies (cp.async.bulk, UBLKCP) row q of all seven
// operand arrays -- p, ux, uy and the L2-resident lx, ly, diag, inv -- into slot q % kRmDepth, completing on the
// slot's `full` mbarrier; the compute warps read their lane's column out of the slot with plain shared loads and free
// it through the slot's `empty` mbarrier (one arrival per compute warp) once no later step reads that row.  A CTA of
// kRmWarps compute warps covers kRmWarps*kRmCols = 196 columns, the full width of the default grid (192 columns; one
// 800-byte row per array), so all warps share every staged row and the halo columns of neighbouring warps cost no
// extra copy; wider grids are cut into column windows of that width.  Step s (forming row ia-1+s) reads rows s..s+3 of
// the ring (q = row - ia + 2; s-1 .. s+1 for finishing row ia-2+s) and releases row s-1, so the loader runs
// kRmDepth - 5 rows ahead of the slowest warp.
// ------------------------------------------------------------------------------------------------
constexpr int kRmCols = 28;       // output columns per warp (even: 2x2 restriction pairs start at odd columns)
constexpr int kRmWarps = 7;       // compute warps per CTA (+1 loader warp)
constexpr int kRmRows = 32;       // rows per CTA (even)
constexpr int kRmDepth = 8;       // ring slots
constexpr int kRmMinB = 4;        // CTAs per SM: 4 x 47 KB of ring, at most 64 registers
constexpr int kRmArrays = 7;      // staged arrays: p, ux, uy, lx, ly, diag, inv
constexpr int kRmSeg = 208;       // floats per staged row segment: kRmWarps*kRmCols + 4 halo columns, 16-byte aligned ends
constexpr size_t kRmSmem = (size_t)kRmDepth * kRmArrays * kRmSeg * 4 + 2 * kRmDepth * 8;

__global__ void __launch_bounds__(32 * (kRmWarps + 1), kRmMinB)
k_resid_down0_march(const __grid_constant__ SolverParams q, const float* __restrict__ ux_all, const float* __restrict__ uy_all,
                    const float* __restrict__ pin_all, float* __restrict__ pout_all, float* __restrict__ rout_all, int which) {
  using namespace rows_detail;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* ring = reinterpret_cast<float*>(smem_raw);                  // [kRmDepth][kRmArrays][kRmSeg]
  unsigned long long* full = reinterpret_cast<unsigned long long*>(ring + (size_t)kRmDepth * kRmArrays * kRmSeg);
  unsigned long long* empty = full + kRmDepth;
  const DevLevel& L = q.lev[0];
  const DevLevel& C = q.lev[1];
  const int P = L.P, n = L.n, m = L.m, ni = n - 2, mj = m - 2;
  const int e = blockIdx.z;
  if (q.sc.frozen[e]) return;                          // (active[e] is 0 after every completed solve: the MG kernels skip it too)
  if (slab_skip(blockIdx.y, gridDim.y, q.slab_rank, q.slab_n)) return;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) { q.sc.active[e] = 1; q.sc.iters[2 * e + which] = 0; }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int jc0 = 1 + blockIdx.x * (kRmWarps * kRmCols);             // first output column of this CTA (odd)
  const int c0 = max(jc0 - 2, 0) & ~3;                               // staged columns [c0, c1)
  const int c1 = min(P, (jc0 - 2 + (kRmWarps - 1) * kRmCols + 32 + 3) & ~3);
  const int ia = 1 + blockIdx.y * kRmRows;                           // first row of this chunk (odd)
  const int ib = min(ia + kRmRows - 1, ni);
  const int nq = 2 + 2 * ((ib - ia + 2) / 2) + 3;                    // staged rows ia-2 .. : the prologue's three + one per form
  const size_t eo = (size_t)e * L.stride;
  const float* __restrict__ pin = pin_all + eo;
  auto rowc = [&](int i) { return min(max(i, 0), n - 1); };
  if (threadIdx.x == 0) {
    for (int s = 0; s < kRmDepth; s++) { mbar_init(full + s, 1); mbar_init(empty + s, kRmWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == kRmWarps) {                                            // loader
    if (lane == 0) {
      const float* src[kRmArrays] = {pin, ux_all + eo, uy_all + eo, L.lx, L.ly, L.diag, L.inv};
      const unsigned bytes = (unsigned)(c1 - c0) * 4u;
      for (int qq = 0; qq < nq; qq++) {
        const int s = qq % kRmDepth;
        if (qq >= kRmDepth) mbar_wait(empty + s, (unsigned)(qq / kRmDepth - 1) & 1u);
        const size_t off = (size_t)rowc(ia - 2 + qq) * P + c0;
        mbar_expect_tx(full + s, kRmArrays * bytes);
#pragma unroll
        for (int a = 0; a < kRmArrays; a++) bulk_g2s(ring + ((size_t)s * kRmArrays + a) * kRmSeg, src[a] + off, bytes, full + s);
      }
    }
    return;
  }
  float* __restrict__ pout = pout_all + eo;
  float* __restrict__ rout = rout_all + eo;
  const int jw0 = jc0 + warp * kRmCols;                              // first output column of this warp (odd)
  const int j = jw0 - 2 + lane;                                      // this lane's column (may be outside the array)
  const int cs = min(max(j, 0), m - 1) - c0;                         // its (clamped) column in the staged segments
  const bool out_lane = lane >= 2 && lane < 2 + kRmCols && j <= mj;
  const bool jfirst = j == 1, jlast = j == mj;
  enum { aP, aUX, aUY, aLX, aLY, aDG, aIV };
  auto slot = [&](int qq) { return ring + (size_t)(qq % kRmDepth) * kRmArrays * kRmSeg + cs; };
  auto wait_row = [&](int qq) { mbar_wait(full + qq % kRmDepth, (unsigned)(qq / kRmDepth) & 1u); };
  auto release_row = [&](int qq) {
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sm_addr(empty + qq % kRmDepth)) : "memory");
  };
  // rolling rows: p of rows ir-1, ir, ir+1; ux and lx of rows ir, ir+1
  int ir = ia - 1;                                                   // the row whose r and d are formed next
  int qr = 1;                                                        // its ring row
  wait_row(0); wait_row(1); wait_row(2);
  float p_m = slot(0)[aP * kRmSeg], p_c = slot(1)[aP * kRmSeg], p_n = slot(2)[aP * kRmSeg];
  float ux_c = slot(1)[aUX * kRmSeg], lx_c = slot(1)[aLX * kRmSeg];
  // what finalising a row needs from the two rows formed before it
  float d_1 = 0.f, d_2 = 0.f, r_1 = 0.f, pq_1 = 0.f, pq_2 = 0.f, diag_1 = 0.f, lxw_1 = 0.f, ly_1 = 0.f, lyn_1 = 0.f;
  float acc = 0.f;
  // forms r and d of row ir (garbage outside the interior, never used there) and advances the rolling rows
  auto form = [&](float& r_out, float& d_out, float& diag_o, float& lxw_o, float& ly_o, float& lyn_o) {
    wait_row(qr + 2);
    const float* sc = slot(qr);
    const float* sn = slot(qr + 1);
    const float ux_n = sn[aUX * kRmSeg], lx_n = sn[aLX * kRmSeg];
    const float uy_c = sc[aUY * kRmSeg], ly_c = sc[aLY * kRmSeg], dg = sc[aDG * kRmSeg], iv = sc[aIV * kRmSeg];
    const float p_s = __shfl_up_sync(0xffffffffu, p_c, 1), p_nn = __shfl_down_sync(0xffffffffu, p_c, 1);
    const float uy_n = __shfl_down_sync(0xffffffffu, uy_c, 1), ly_n = __shfl_down_sync(0xffffffffu, ly_c, 1);
    const float sdiv = ux_n - ux_c + uy_n - uy_c;                    // VectorField.pde:56-65
    const float Ap = p_c * dg + p_m * lx_c + p_n * lx_n + p_s * ly_c + p_nn * ly_n;   // PoissonMatrix.pde:56-61
    r_out = sdiv - Ap;
    d_out = r_out * iv;                                              // MG.pde:80
    diag_o = dg; lxw_o = lx_c; ly_o = ly_c; lyn_o = ly_n;
    // advance: ir -> ir + 1
    ux_c = ux_n; lx_c = lx_n;
    p_m = p_c; p_c = p_n;
    ir++; qr++;
    p_n = slot(qr + 1)[aP * kRmSeg];
  };
  // finalises row i = ir - 2 (its d is d_1, the rows around it d_2 and d_0): smooth(0) increment, new p, restriction;
  // then row i - 1 is no longer read
  auto finish = [&](int i, float d_0, float lxe, float p_e, bool odd) {
    const float dc = d_1;
    const float dW = (i == 1) ? dc : d_2, dE = (i == ni) ? dc : d_0;             // d.setBC: ghost = adjacent interior value
    const float dSs = __shfl_up_sync(0xffffffffu, dc, 1), dNs = __shfl_down_sync(0xffffffffu, dc, 1);
    const float dS = jfirst ? dc : dSs, dN = jlast ? dc : dNs;
    const float Ad = dc * diag_1 + dW * lxw_1 + dE * lxe + dS * ly_1 + dN * lyn_1;
    const float rn = r_1 - Ad;
    const float rnN = __shfl_down_sync(0xffffffffu, rn, 1);
    acc = odd ? rn + rnN : (acc + rn) + rnN;                         // MG.restrict(Field) MG.pde:128-133: rn00 + rn01 + rn10 + rn11
    if (out_lane) {
      const int k = IDX(i, j);
      rout[k] = rn;
      pout[k] = pq_1 + dc;
      // ghosts of x receive the clamped d (x.plusEq(d) runs over all cells, MG.pde:95); p's ghosts are live data
      const int di = (i == 1) ? -1 : (i == ni ? 1 : 0), dj = jfirst ? -1 : (jlast ? 1 : 0);
      if (di) pout[IDX(i + di, j)] = ((di < 0) ? pq_2 : p_e) + dc;
      if (dj) pout[IDX(i, j + dj)] = slot(qr - 2)[aP * kRmSeg + dj] + dc;
      if (di && dj) pout[IDX(i + di, j + dj)] = slot(qr - 2 + di)[aP * kRmSeg + dj] + dc;
      if (!odd && !(lane & 1)) C.r[(size_t)e * C.stride + (i >> 1) * C.P + ((j + 1) >> 1)] = acc;
    }
    release_row(qr - 3);
  };
  // prologue: rows ia-1 and ia
  {
    float r0, d0, g0, w0, y0, yn0;
    pq_2 = p_m;                                                       // (p of row ia - 2: only used as a ghost row, never)
    form(r0, d0, g0, w0, y0, yn0);                                    // row ia - 1
    d_2 = d0; pq_2 = p_m;                                             // p_m is now p of row ia - 1
    form(r_1, d_1, diag_1, lxw_1, ly_1, lyn_1);                       // row ia
    pq_1 = p_m;                                                       // p of row ia
    release_row(0);                                                   // row ia - 2
  }
  for (int i = ia; i <= ib; i += 2) {
    float r0, d0, g0, w0, y0, yn0;
    // ---- row i (odd): needs d of row i + 1
    form(r0, d0, g0, w0, y0, yn0);                                    // row i + 1; afterwards p_m = p(i+1), lx_c = lx(i+2)
    finish(i, d0, w0, p_m, true);                                     // lxe = lx(i+1) = w0, p_e = p(i+1)
    d_2 = d_1; d_1 = d0; r_1 = r0; pq_2 = pq_1; pq_1 = p_m; diag_1 = g0; lxw_1 = w0; ly_1 = y0; lyn_1 = yn0;
    // ---- row i + 1 (even)
    form(r0, d0, g0, w0, y0, yn0);                                    // row i + 2
    finish(i + 1, d0, w0, p_m, false);
    d_2 = d_1; d_1 = d0; r_1 = r0; pq_2 = pq_1; pq_1 = p_m; diag_1 = g0; lxw_1 = w0; ly_1 = y0; lyn_1 = yn0;
  }
}

// ------------------------------------------------------------------------------------------------
// levels >= 1: the rest of the V-cycle, one CTA per environment (MG.pde:68-77).  Per level the residual
// ping-pongs between the level's `r` and `d` arrays: down writes the smoothed residual to `d`, the
// up pass updates it in place and the strip smoother consumes it, adding its result straight into x.
// Ghost cells of the coarse r and x are never materialised: every reference read of them is either
// overwritten by a setBC before use or multiplied by a boundary coefficient that is 0 on coarse levels.
// ------------------------------------------------------------------------------------------------
// up pass of one coarse level for one env: d = prolongate(coarse.x) incl. its setBC (ghost = adjacent interior,
// MG.pde:139-152), x += d, r -= A d (MG.pde:75-76,94-97).  Warps own rows, lanes own columns; four rows are in
// flight per warp so the L2 round trips overlap.
__device__ __forceinline__ void coarse_up_pass(const DevLevel& L, const DevLevel& C, float* __restrict__ r,
                                               float* __restrict__ x, const float* __restrict__ xc) {
  const int n = L.n, m = L.m, P = L.P, ni = n - 2, mj = m - 2, CP = C.P;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const float* __restrict__ lx = L.lx;
  const float* __restrict__ ly = L.ly;
  constexpr int U = RLFC_UP_ROWS;
  for (int j = 1 + lane; j <= mj; j += 32) {
    const int cj = (j - 1) / 2 + 1, cjm = (max(j - 1, 1) - 1) / 2 + 1, cjp = (min(j + 1, mj) - 1) / 2 + 1;
    for (int i0 = 1 + warp; i0 <= ni; i0 += nw * U) {
      float dc[U], dw[U], de[U], ds[U], dn[U], xo[U], ro[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const int i = min(i0 + u * nw, ni);
        const int ci = (i - 1) / 2 + 1, cim = (max(i - 1, 1) - 1) / 2 + 1, cip = (min(i + 1, ni) - 1) / 2 + 1;
        dc[u] = xc[ci * CP + cj]; dw[u] = xc[cim * CP + cj]; de[u] = xc[cip * CP + cj];
        ds[u] = xc[ci * CP + cjm]; dn[u] = xc[ci * CP + cjp];
        xo[u] = x[IDX(i, j)]; ro[u] = r[IDX(i, j)];
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const int i = i0 + u * nw;
        if (i <= ni) {
          const int k = IDX(i, j);
          x[k] = xo[u] + dc[u];
          const float lw = lx[k], le = lx[k + P], ls = ly[k], ln_ = ly[k + 1];
          const float dg = -(lw + le + ls + ln_);                      // the diagonal is the plain coefficient sum (PoissonMatrix.pde:46-48)
          r[k] = ro[u] - (dc[u] * dg + dw[u] * lw + de[u] * le + ds[u] * ls + dn[u] * ln_);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256, 2)
k_mg_coarse(const __grid_constant__ SolverParams q) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  StripShared* sh = reinterpret_cast<StripShared*>(smem_raw);
  StripMail* mail = reinterpret_cast<StripMail*>(smem_raw + sizeof(StripShared) * q.coarse_strips);
  const int e = blockIdx.x;
  if (!q.sc.active[e]) return;
  const int last = q.nlevels - 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // ---- down: smooth(0) + restrict; warps own coarse rows, lanes own coarse columns ----
  for (int l = 1; l < last; l++) {
    const DevLevel& L = q.lev[l];
    const DevLevel& C = q.lev[l + 1];
    const int nci = C.n - 2, ncj = C.m - 2;
    const size_t eo = (size_t)e * L.stride;
    for (int J = 1 + lane; J <= ncj; J += 32)
#pragma unroll kDownUnroll
      for (int I = 1 + warp; I <= nci; I += nw)
        down_block<false>(L, C, L.r + eo, L.d + eo, L.x + eo, C.r + (size_t)e * C.stride, I, J);
    __syncthreads();
  }
  // ---- coarsest level: smooth(its) only (MG.pde:72-73), x = 0 + d ----
  {
    const DevLevel& L = q.lev[last];
    strip_smooth<1>(L, L.r + (size_t)e * L.stride, L.x + (size_t)e * L.stride, sh, mail);
  }
  // ---- up: prolongate + increment, then smooth(its): x += GS(r)  (MG.pde:73-76) ----
  for (int l = last - 1; l >= 1; l--) {
    const DevLevel& L = q.lev[l];
    const DevLevel& C = q.lev[l + 1];
    const size_t eo = (size_t)e * L.stride;
    float* r = L.d + eo;            // smoothed residual left by the down pass
    float* x = L.x + eo;
    coarse_up_pass(L, C, r, x, C.x + (size_t)e * C.stride);
    __syncthreads();
    strip_smooth<2>(L, r, x, sh, mail);
  }
}

// ------------------------------------------------------------------------------------------------
// level 0, up: d = prolongate(x1) (+setBC), x += d, r -= A d   (MG.pde:75-76)
// ------------------------------------------------------------------------------------------------
// SKEWED: the updated residual goes to the row smoother's skewed array (solver.h rsk) instead of back in place
template <bool SKEWED>
__global__ void __launch_bounds__(256)
k_mg_up0(const __grid_constant__ SolverParams q, float* __restrict__ r_all) {
  const int e = blockIdx.z;
  if (!q.sc.active[e]) return;
  const DevLevel& L0 = q.lev[0];
  const DevLevel& L1 = q.lev[1];
  const int P = L0.P, n = L0.n, m = L0.m;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= n || j >= m) return;
  const float* xc = L1.x + (size_t)e * L1.stride;
  const size_t eo = (size_t)e * L0.stride;
  auto dval = [&](int a, int b) {
    int ci = min(max(a, 1), n - 2), cj = min(max(b, 1), m - 2);
    return xc[((ci - 1) / 2 + 1) * L1.P + ((cj - 1) / 2 + 1)];
  };
  const int k = IDX(i, j);
  const float dc = dval(i, j);
  L0.x[eo + k] += dc;
  if (i >= 1 && j >= 1 && i <= n - 2 && j <= m - 2) {
    float Ad = dc * L0.diag[k] + dval(i - 1, j) * L0.lx[k] + dval(i + 1, j) * L0.lx[k + P] + dval(i, j - 1) * L0.ly[k] +
               dval(i, j + 1) * L0.ly[k + 1];
    if (SKEWED) {
      const int C = L0.rt.C, CP = rows_CP(C);
      const int ln = (j - 1) / C, c = (j - 1) - ln * C;
      q.rsk[(size_t)e * q.rsk_stride + ((size_t)(i + ln) * 32 + ln) * CP + c] = r_all[eo + k] - Ad;
    } else {
      r_all[eo + k] -= Ad;
    }
  }
}

// level 0, up, one thread per COARSE cell (rows smoother path): the four children share the injected value
// xc[I][J]; their outward neighbours take the adjacent coarse cell's value, or -- at the domain edge, where
// d.setBC copies the adjacent interior value (MG.pde:139-152) -- the cell's own.  x += d on the children and on the
// ghost cells they border, r -= A d written to the smoother's skewed array.
// A CTA owns kUpRows fine rows of one environment over the full width (the row smoother's grids are at most 256 columns
// wide).  Its rows of x and r and the coarse x rows around them are contiguous in memory: one thread bulk-copies them
// into shared memory (three cp.async.bulk copies on one mbarrier), so a CTA's loads are in flight at once without
// holding registers.  The new residual overwrites r in shared memory and leaves in a second phase in the skewed order:
// the CTA's part of skewed entry tau (row tau - ln of lane ln, ln in [tau - i0 - kUpRows + 1, tau - i0]) is one
// contiguous range, written by one warp with consecutive stores (the skewed index of a thread's own cells scatters
// 4-byte stores over 24-byte lane blocks).
constexpr int kUpRows = 16;       // fine rows per CTA (even)

static size_t up0_smem(const SolverParams& q) {
  return sizeof(float) * (2 * (size_t)kUpRows * q.P + (size_t)(kUpRows / 2 + 2) * q.lev[1].P) + 16;
}

__global__ void __launch_bounds__(256)
k_mg_up0_blk(const __grid_constant__ SolverParams q, const float* __restrict__ r_all) {
  using namespace rows_detail;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int e = blockIdx.y;
  if (!q.sc.active[e]) return;
  const DevLevel& L0 = q.lev[0];
  const DevLevel& L1 = q.lev[1];
  const int P = L0.P, n = L0.n, m = L0.m, ni = n - 2, mj = m - 2, CPc = L1.P;
  const int nci = L1.n - 2, ncj = L1.m - 2;
  const int i0 = 1 + blockIdx.x * kUpRows, rows = min(kUpRows, ni + 1 - i0);   // fine rows i0 .. i0+rows-1
  const int I0 = (i0 + 1) / 2;                                                  // their first coarse row
  float* s_x = reinterpret_cast<float*>(smem_raw);                              // [rows][P] from row i0
  float* s_r = s_x + kUpRows * P;                                               // [rows][P] from row i0
  float* s_xc = s_r + kUpRows * P;                                              // [rows/2 + 2][CPc] from coarse row I0-1
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(s_xc + (kUpRows / 2 + 2) * CPc);
  const size_t eo = (size_t)e * L0.stride;
  float* __restrict__ x = L0.x + eo;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned fb = (unsigned)(rows * P) * 4u, cb = (unsigned)((rows / 2 + 2) * CPc) * 4u;
    mbar_expect_tx(bar, 2 * fb + cb);
    bulk_g2s(s_x, x + (size_t)i0 * P, fb, bar);
    bulk_g2s(s_r, r_all + eo + (size_t)i0 * P, fb, bar);
    bulk_g2s(s_xc, L1.x + (size_t)e * L1.stride + (size_t)(I0 - 1) * CPc, cb, bar);
  }
  __syncthreads();
  mbar_wait(bar, 0);
  const int C = L0.rt.C, CP = rows_CP(C);
  for (int t = threadIdx.x; t < (rows / 2) * ncj; t += blockDim.x) {
    const int Il = t / ncj, J = t - Il * ncj + 1, I = I0 + Il;
    const float* xc = s_xc + (Il + 1) * CPc;
    const float dc = xc[J];
    const float dWc = (I > 1) ? xc[J - CPc] : dc, dEc = (I < nci) ? xc[J + CPc] : dc;
    const float dSc = (J > 1) ? xc[J - 1] : dc, dNc = (J < ncj) ? xc[J + 1] : dc;
    const int a0 = 2 * Il, ig = i0 + a0, j0 = 2 * J - 1;
    // the 2x2 block's face coefficients, each loaded once: lx on the three rows ig .. ig+2, ly on the three columns
    // j0 .. j0+2; the diagonal is their plain sum (PoissonMatrix.pde:46-48; checked against the host table at create time)
    float lxv[3][2], lyv[2][3];
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
      for (int b = 0; b < 2; b++) lxv[a][b] = L0.lx[IDX(ig + a, j0 + b)];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 3; b++) lyv[a][b] = L0.ly[IDX(ig + a, j0 + b)];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 2; b++) {
        const int i = ig + a, j = j0 + b, ks = IDX(a0 + a, j);
        const float dW = a ? dc : dWc, dE = a ? dEc : dc, dS = b ? dc : dSc, dN = b ? dNc : dc;
        const float dg = -(lxv[a][b] + lxv[a + 1][b] + lyv[a][b] + lyv[a][b + 1]);
        const float Ad = dc * dg + dW * lxv[a][b] + dE * lxv[a + 1][b] + dS * lyv[a][b] + dN * lyv[a][b + 1];
        x[IDX(i, j)] = s_x[ks] + dc;
        s_r[ks] = s_r[ks] - Ad;
      }
    // ghost cells bordering the block (only the blocks on the rim of the level)
    if (I == 1 || I == nci || J == 1 || J == ncj) {
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const int i = ig + a, j = j0 + b;
          const int di = (i == 1) ? -1 : (i == n - 2 ? 1 : 0), dj = (j == 1) ? -1 : (j == m - 2 ? 1 : 0);
          if (di) x[IDX(i + di, j)] += dc;
          if (dj) x[IDX(i, j + dj)] += dc;
          if (di && dj) x[IDX(i + di, j + dj)] += dc;
        }
    }
  }
  __syncthreads();
  // skewed write-out: warp w takes the CTA's entries tau = i0 + t, t = w, w + 8, ...
  float* __restrict__ rsk = q.rsk + (size_t)e * q.rsk_stride;
  const int lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int t = threadIdx.x >> 5; t < rows + 31; t += nw) {
    const int lo = max(0, t - rows + 1) * CP, hi = (min(31, t) + 1) * CP;
    float* __restrict__ ent = rsk + (size_t)(i0 + t) * 32 * CP;
    for (int p = lo + lane; p < hi; p += 32) {
      const int ln = p / CP, c = p - ln * CP, j = ln * C + c + 1;
      if (c < C && j <= mj) ent[p] = s_r[IDX(t - ln, j)];
    }
  }
}

// plain level-0 residual <- skewed residual (the row smoother leaves r - A d there); only environments that
// go on to a further MG iteration need it
__global__ void __launch_bounds__(256)
k_unskew_r(const __grid_constant__ SolverParams q, float* __restrict__ r_all) {
  const int e = blockIdx.z;
  if (!q.sc.active[e]) return;
  const DevLevel& L0 = q.lev[0];
  const int P = L0.P, n = L0.n, m = L0.m;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  if (i < 1 || j < 1 || i > n - 2 || j > m - 2) return;
  const int C = L0.rt.C, CP = rows_CP(C);
  const int ln = (j - 1) / C, c = (j - 1) - ln * C;
  r_all[(size_t)e * L0.stride + IDX(i, j)] = q.rsk[(size_t)e * q.rsk_stride + ((size_t)(i + ln) * 32 + ln) * CP + c];
}

// level 0 smooth(4) complete (MG.pde:79-97) + the MGsolver loop test (MG.pde:32-35), one CTA per env with one
// warp per 32-column strip (smooth_strip.cuh, XMODE 3): d = r*inv, four lexicographic Gauss-Seidel sweeps,
// d.setBC, x += d (p, ghosts included), r -= A d, r.r accumulated in double, then iter++ and the
// `r.r < tol` / `iter == itmx` decision for this environment.
__global__ void __launch_bounds__(256)
k_smooth0(const __grid_constant__ SolverParams q, const float* r_in_all, float* r_out_all, int which) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevLevel& L = q.lev[0];
  const int ns = L.sk.nstrips, n = L.n, m = L.m, P = L.P, ni = n - 2, mj = m - 2;
  StripShared* sh = reinterpret_cast<StripShared*>(smem_raw);
  StripMail* mail = reinterpret_cast<StripMail*>(smem_raw + sizeof(StripShared) * ns);
  float* gbuf = reinterpret_cast<float*>(smem_raw + sizeof(StripShared) * ns + sizeof(StripMail) * (ns + 2));
  __shared__ double wsum[32];
  const int e = blockIdx.x;
  if (!q.sc.active[e]) return;
  float* p = L.x + (size_t)e * L.stride;
  double rr = strip_smooth<3>(L, r_in_all + (size_t)e * L.stride, p, sh, mail, gbuf, r_out_all + (size_t)e * L.stride);
  // ghost cells of x: x.plusEq(d) runs over all cells and d.setBC copied the adjacent interior value (MG.pde:90,95)
  const float *gtop = gbuf, *gbot = gbuf + mj, *gleft = gbuf + 2 * mj, *gright = gbuf + 2 * mj + ni;
  for (int c = threadIdx.x; c < mj; c += blockDim.x) { p[IDX(0, c + 1)] += gtop[c]; p[IDX(n - 1, c + 1)] += gbot[c]; }
  for (int c = threadIdx.x; c < ni; c += blockDim.x) { p[IDX(c + 1, 0)] += gleft[c]; p[IDX(c + 1, m - 1)] += gright[c]; }
  if (threadIdx.x == 0) {
    p[IDX(0, 0)] += gtop[0]; p[IDX(0, m - 1)] += gtop[mj - 1];
    p[IDX(n - 1, 0)] += gbot[0]; p[IDX(n - 1, m - 1)] += gbot[mj - 1];
  }
  // r.r: fixed-order reduction (lanes by shuffle tree, then warps in order)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rr += __shfl_down_sync(0xffffffffu, rr, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = rr;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += wsum[w];
    const int it = ++q.sc.iters[2 * e + which];
    if ((float)s < q.mg_tol || it >= q.mg_max_iters) q.sc.active[e] = 0;
    else atomicExch(q.sc.any_active, 1);
  }
}

// ------------------------------------------------------------------------------------------------
// Row-pipelined variants (smooth_rows.cuh): one warp per sweep, C columns per lane.
// ------------------------------------------------------------------------------------------------
#include "smooth_tiny.cuh"

template <int XMODE>
__device__ __forceinline__ void rows_dispatch(const DevLevel& L, float* r, float* x, unsigned char* smem) {
  switch (L.rt.C) {
    case 1: rows_smooth<1, XMODE>(L, r, x, smem, nullptr); break;
    case 2: rows_smooth<2, XMODE>(L, r, x, smem, nullptr); break;
    case 3: rows_smooth<3, XMODE>(L, r, x, smem, nullptr); break;
    default: rows_smooth<4, XMODE>(L, r, x, smem, nullptr); break;
  }
}

__global__ void __launch_bounds__(kRowsThreads, 2)
k_mg_coarse_rows(const __grid_constant__ SolverParams q, int first) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int e = blockIdx.x;
  if (!q.sc.active[e]) return;
  const int last = q.nlevels - 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#ifdef RLFC_COARSE_TIMING
  long long tk = clock64();
  __shared__ long long tick_log[40];
  __shared__ int tick_n;
  if (threadIdx.x == 0) tick_n = 0;
#define TICK(what, l) do { __syncthreads(); if (threadIdx.x == 0) { long long n_ = clock64(); tick_log[tick_n++] = n_ - tk; tk = n_; } } while (0)
#else
#define TICK(what, l)
#endif
  for (int l = first; l < last; l++) {
    const DevLevel& L = q.lev[l];
    const DevLevel& C = q.lev[l + 1];
    const int nci = C.n - 2, ncj = C.m - 2;
    const size_t eo = (size_t)e * L.stride;
    for (int J = 1 + lane; J <= ncj; J += 32)
#pragma unroll 2
      for (int I = 1 + warp; I <= nci; I += nw)
        down_block<false>(L, C, L.r + eo, L.d + eo, L.x + eo, C.r + (size_t)e * C.stride, I, J);
    __syncthreads();
    TICK("down", l);
  }
  {
    const DevLevel& L = q.lev[last];
    const size_t eo = (size_t)e * L.stride;
    if (L.wave) wave_smooth<1>(L, L.r + eo, L.x + eo, L.d + eo, nullptr, 4);     // L.d is unused on the coarsest level
    else if (q.tiny && tiny_level(L.n - 2, L.m - 2)) tiny_smooth<1>(L, L.r + eo, L.x + eo, smem_raw);
    else rows_dispatch<1>(L, L.r + eo, L.x + eo, smem_raw);
    TICK("smooth", last);
  }
  for (int l = last - 1; l >= first; l--) {
    const DevLevel& L = q.lev[l];
    const DevLevel& C = q.lev[l + 1];
    const size_t eo = (size_t)e * L.stride;
    float* r = L.d + eo;
    float* x = L.x + eo;
    coarse_up_pass(L, C, r, x, C.x + (size_t)e * C.stride);
    __syncthreads();
    TICK("up", l);
    if (L.wave) wave_smooth<2>(L, r, x, L.r + eo, nullptr, 4);   // the level's restricted residual is dead after the down pass
    else if (q.tiny && tiny_level(L.n - 2, L.m - 2)) tiny_smooth<2>(L, r, x, smem_raw);
    else rows_dispatch<2>(L, r, x, smem_raw);
    TICK("smooth", l);
  }
#undef TICK
#ifdef RLFC_COARSE_TIMING
  if (e == 0 && threadIdx.x == 0) {
    printf("coarse ticks:");
    for (int k = 0; k < tick_n; k++) printf(" %lld", tick_log[k]);
    printf("\n");
  }
#endif
}

template <int C>
__global__ void __launch_bounds__(kRows0Threads, 2)
k_smooth0_rows(const __grid_constant__ SolverParams q, int which) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const DevLevel& L = q.lev[0];
  const int n = L.n, m = L.m, P = L.P, ni = n - 2, mj = m - 2;
  float* gbuf = reinterpret_cast<float*>(smem_raw + rows_smem_bytes(C, P, true));
  __shared__ double wsum[32];
  const int e = blockIdx.x;
  if (!q.sc.active[e]) return;
  float* p = L.x + (size_t)e * L.stride;
  double rr = rows_smooth<C, 3>(L, q.rsk + (size_t)e * q.rsk_stride, p, smem_raw, gbuf);
  // ghost cells of x: x.plusEq(d) runs over all cells and d.setBC copied the adjacent interior value (MG.pde:90,95)
  const float *gtop = gbuf, *gbot = gbuf + mj, *gleft = gbuf + 2 * mj, *gright = gbuf + 2 * mj + ni;
  for (int c = threadIdx.x; c < mj; c += blockDim.x) { p[IDX(0, c + 1)] += gtop[c]; p[IDX(n - 1, c + 1)] += gbot[c]; }
  for (int c = threadIdx.x; c < ni; c += blockDim.x) { p[IDX(c + 1, 0)] += gleft[c]; p[IDX(c + 1, m - 1)] += gright[c]; }
  if (threadIdx.x == 0) {
    p[IDX(0, 0)] += gtop[0]; p[IDX(0, m - 1)] += gtop[mj - 1];
    p[IDX(n - 1, 0)] += gbot[0]; p[IDX(n - 1, m - 1)] += gbot[mj - 1];
  }
  // r.r: fixed-order reduction (lanes by shuffle tree, then warps in order)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rr += __shfl_down_sync(0xffffffffu, rr, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = rr;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += wsum[w];
    const int it = ++q.sc.iters[2 * e + which];
    if ((float)s < q.mg_tol || it >= q.mg_max_iters) q.sc.active[e] = 0;
    else atomicExch(q.sc.any_active, 1);
  }
}

// level-0 smooth(4) + increment + r.r + loop test with the wavefront fallback (grids wider than 256 cells)
__global__ void __launch_bounds__(1024)
k_smooth0_wave(const __grid_constant__ SolverParams q, const float* r_in_all, float* r_out_all, int which) {
  const DevLevel& L = q.lev[0];
  __shared__ double wsum[32];
  const int e = blockIdx.x;
  if (!q.sc.active[e]) return;
  const size_t eo = (size_t)e * L.stride;
  double rr = wave_smooth<3>(L, r_in_all + eo, L.x + eo, L.w + eo, r_out_all + eo, 4);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rr += __shfl_down_sync(0xffffffffu, rr, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = rr;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += wsum[w];
    const int it = ++q.sc.iters[2 * e + which];
    if ((float)s < q.mg_tol || it >= q.mg_max_iters) q.sc.active[e] = 0;
    else atomicExch(q.sc.any_active, 1);
  }
}

// ------------------------------------------------------------------------------------------------
// Field.sum (Field.pde:311-318): a serial float accumulation over the interior in i-major order.
// One warp per env: lanes load 32 consecutive values (coalesced), every lane then replays the same
// 32 dependent adds on broadcast values, so the chain is pure FADD latency.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
k_psum(const __grid_constant__ SolverParams q) {
  constexpr int G = 8;                                   // 32-element chunks per group (one row segment each)
  __shared__ __align__(16) float buf[2][G * 32];
  const int e = blockIdx.x, lane = threadIdx.x;
  if (q.sc.frozen[e]) return;
  const int P = q.P, ni = q.n - 2, len = q.m - 2;
  const int cpr = (len + 31) / 32;                       // chunks per row; row tails are padded with +0.f (s + 0.f == s)
  const float* p = q.lev[0].x + (size_t)e * q.stride;
  // group iterator: `cnt` consecutive chunks of row gi starting at chunk gc
  int gi = 1, gc = 0;
  const float* rowp = p + IDX(1, 1) + lane;
  float nxt[G];
  int ncnt;
  auto fetch = [&]() {
    ncnt = (gi <= ni) ? min(G, cpr - gc) : 0;
#pragma unroll
    for (int u = 0; u < G; u++) {
      const int j = (gc + u) * 32 + lane;
      nxt[u] = (u < ncnt && j < len) ? rowp[(gc + u) * 32] : 0.f;
    }
    gc += ncnt;
    if (gc >= cpr) { gc = 0; gi++; rowp += P; }
  };
  fetch();
  float s = 0.f;
  int pb = 0;
  while (ncnt > 0) {
    const int cnt = ncnt;
#pragma unroll
    for (int u = 0; u < G; u++) buf[pb][u * 32 + lane] = nxt[u];
    __syncwarp();
    fetch();                                             // next group's loads are in flight during the chain
    const float4* b4 = reinterpret_cast<const float4*>(buf[pb]);
    for (int c = 0; c < cnt; c++) {
#pragma unroll
      for (int k = 0; k < 8; k++) {                      // every lane replays the same serial chain
        const float4 v = b4[c * 8 + k];
        s += v.x; s += v.y; s += v.z; s += v.w;
      }
    }
    pb ^= 1;
  }
  if (lane == 0) q.sc.psum[e] = s;
}

#include "exact_sum_kernels.cuh"
#include "smooth_chain.cuh"
#include "smooth_chain3.cuh"

// ------------------------------------------------------------------------------------------------
// projection tail (VectorField.pde:136-139): p += -sum/N on all cells; dp = grad p with its setBC
// (dp.x[1][*] = dp.y[*][1] = 0); u += c * (dp * -1) on the interior.  u.setBC follows in k_bc.
// ------------------------------------------------------------------------------------------------
// p must not be shifted in place while neighbouring blocks still read the unshifted values, so the
// velocity correction (k_project_u) and the shift itself (k_shift_p) are separate passes
__global__ void __launch_bounds__(256)
k_project_u(const __grid_constant__ SolverParams q, float* __restrict__ ux_all, float* __restrict__ uy_all) {
  const int P = q.P, n = q.n, m = q.m;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  const int e = blockIdx.z;
  if (i < 1 || j < 1 || i > n - 2 || j > m - 2 || q.sc.frozen[e]) return;
  const size_t eo = (size_t)e * q.stride;
  const float* p = q.lev[0].x + eo;
  const float shift = -1 * q.sc.psum[e] / q.inv_cells;
  const int k = IDX(i, j);
  const float pc = p[k] + shift;
  if (i >= 2) {
    float dpx = pc - (p[k - P] + shift);
    ux_all[eo + k] += q.c_x[k] * (dpx * -1);
  }
  if (j >= 2) {
    float dpy = pc - (p[k - 1] + shift);
    uy_all[eo + k] += q.c_y[k] * (dpy * -1);
  }
}
__global__ void __launch_bounds__(256)
k_shift_p(const __grid_constant__ SolverParams q) {
  const int P = q.P;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  const int e = blockIdx.z;
  if (i >= q.n || j >= q.m || q.sc.frozen[e]) return;
  float* p = q.lev[0].x + (size_t)e * q.stride;
  const float shift = -1 * q.sc.psum[e] / q.inv_cells;
  p[IDX(i, j)] += shift;
}

// projection tail fused (VectorField.pde:136-139): p_out = p_in + shift on all cells (p ping-pongs B -> A, so no
// thread reads a value another thread has already shifted), u += c * (grad(p_in + shift) * -1) on the interior.
// One thread handles four consecutive columns (aligned float4 accesses; the pitch is a multiple of 8 floats).
// HEUN (corrector, BDIM.pde:95-96): away from the lines u.setBC touches the projected velocity goes straight into
// the Heun average  u = (u + us) * 0.5  written to the step-start buffer; inside that zone (heun_zone) the projected
// value is stored as before and k_bc2<.., true> averages after the boundary conditions.
__device__ __forceinline__ bool heun_zone(int i, int j4, int n, int m) {           // j4 = first column of a float4
  return i < 2 || i > n - 3 || j4 < 4 || j4 >= 4 * ((m - 2) / 4);
}

template <bool HEUN>
__global__ void __launch_bounds__(256)
k_project_shift(const __grid_constant__ SolverParams q, const float* __restrict__ pin_all, float* __restrict__ pout_all,
                float* __restrict__ ux_all, float* __restrict__ uy_all, const float* __restrict__ usx_all,
                const float* __restrict__ usy_all, float* __restrict__ uox_all, float* __restrict__ uoy_all) {
  const int P = q.P, n = q.n, m = q.m, nv = P >> 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = blockIdx.y;
  if (idx >= n * nv || q.sc.frozen[e] || slab_skip(blockIdx.x, gridDim.x, q.slab_rank, q.slab_n)) return;
  const int i = idx / nv, j4 = (idx - i * nv) << 2;
  const size_t eo = (size_t)e * q.stride;
  const float shift = -1 * q.sc.psum[e] / q.inv_cells;
  const int k = IDX(i, j4);
  const float4 pv = *reinterpret_cast<const float4*>(pin_all + eo + k);
  const float pc[4] = {pv.x + shift, pv.y + shift, pv.z + shift, pv.w + shift};
  *reinterpret_cast<float4*>(pout_all + eo + k) = make_float4(pc[0], pc[1], pc[2], pc[3]);
  const bool zone = !HEUN || heun_zone(i, j4, n, m);
  if ((i < 1 || i > n - 2 || j4 > m - 2) && zone) return;    // nothing to project here; zone cells are averaged later
  float4 uxv = *reinterpret_cast<const float4*>(ux_all + eo + k);
  float4 uyv = *reinterpret_cast<const float4*>(uy_all + eo + k);
  float uxa[4] = {uxv.x, uxv.y, uxv.z, uxv.w}, uya[4] = {uyv.x, uyv.y, uyv.z, uyv.w};
  if (i >= 1 && i <= n - 2 && j4 <= m - 2) {
    const float4 cxv = *reinterpret_cast<const float4*>(q.c_x + k);
    const float4 cyv = *reinterpret_cast<const float4*>(q.c_y + k);
    const float cxa[4] = {cxv.x, cxv.y, cxv.z, cxv.w}, cya[4] = {cyv.x, cyv.y, cyv.z, cyv.w};
    float pw[4] = {0.f, 0.f, 0.f, 0.f};
    if (i >= 2) {
      const float4 w = *reinterpret_cast<const float4*>(pin_all + eo + k - P);
      pw[0] = w.x + shift; pw[1] = w.y + shift; pw[2] = w.z + shift; pw[3] = w.w + shift;
    }
    const float psm = (j4 >= 1) ? pin_all[eo + k - 1] + shift : 0.f;       // column j4 - 1
#pragma unroll
    for (int c = 0; c < 4; c++) {
      const int j = j4 + c;
      if (j < 1 || j > m - 2) continue;
      if (i >= 2) {
        const float dpx = pc[c] - pw[c];
        uxa[c] += cxa[c] * (dpx * -1);
      }
      if (j >= 2) {
        const float dpy = pc[c] - (c == 0 ? psm : pc[c == 0 ? 0 : c - 1]);
        uya[c] += cya[c] * (dpy * -1);
      }
    }
  }
  if (zone) {
    *reinterpret_cast<float4*>(ux_all + eo + k) = make_float4(uxa[0], uxa[1], uxa[2], uxa[3]);
    *reinterpret_cast<float4*>(uy_all + eo + k) = make_float4(uya[0], uya[1], uya[2], uya[3]);
  } else {                                                  // u = (u + us) * 0.5
    const float4 sx = *reinterpret_cast<const float4*>(usx_all + eo + k);
    const float4 sy = *reinterpret_cast<const float4*>(usy_all + eo + k);
    *reinterpret_cast<float4*>(uox_all + eo + k) =
        make_float4((uxa[0] + sx.x) * 0.5f, (uxa[1] + sx.y) * 0.5f, (uxa[2] + sx.z) * 0.5f, (uxa[3] + sx.w) * 0.5f);
    *reinterpret_cast<float4*>(uoy_all + eo + k) =
        make_float4((uya[0] + sy.x) * 0.5f, (uya[1] + sy.y) * 0.5f, (uya[2] + sy.z) * 0.5f, (uya[3] + sy.w) * 0.5f);
  }
}

// BDIM.update2: u.plusEq(us); u.timesEq(0.5) over all cells (BDIM.pde:95-96)
__global__ void __launch_bounds__(256)
k_heun(const float* __restrict__ ucx, const float* __restrict__ ucy, const float* __restrict__ ubx,
       const float* __restrict__ uby, float* __restrict__ uax, float* __restrict__ uay, int n, int m, int P,
       size_t stride, const int* __restrict__ frozen, int slab_rank, int slab_n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= n || j >= m || frozen[blockIdx.z] || slab_skip(blockIdx.y, gridDim.y, slab_rank, slab_n)) return;
  const size_t k = (size_t)blockIdx.z * stride + IDX(i, j);
  uax[k] = (ucx[k] + ubx[k]) * 0.5f;
  uay[k] = (ucy[k] + uby[k]) * 0.5f;
}

// ------------------------------------------------------------------------------------------------
// readout: pressForce on body 0 (serial edge-order accumulation), probes, time, draw() accumulation
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sample_linear(const float* a, int P, int i, int j, float s, float t) {
  if (s == 0 && t == 0) return a[IDX(i, j)];                                     // Field.pde:184-185
  return s * (t * a[IDX(i + 1, j + 1)] + (1 - t) * a[IDX(i + 1, j)]) + (1 - s) * (t * a[IDX(i, j + 1)] + (1 - t) * a[IDX(i, j)]);
}

__global__ void __launch_bounds__(64)
k_force(const __grid_constant__ SolverParams q, int accumulate) {
  const int e = blockIdx.x, tid = threadIdx.x, P = q.P;
  if (q.sc.frozen[e]) return;
  const float* p = q.lev[0].x + (size_t)e * q.stride;
  __shared__ float sx[64], sy[64];
  if (tid < q.nforce) {
    const ForcePt f = q.force_pts[tid];
    float pdl = sample_linear(p, P, f.i, f.j, f.s, f.t) * f.l;                   // Body.pde:299
    sx[tid] = pdl * f.nx;
    sy[tid] = pdl * f.ny;
  }
  if (tid < q.nprobe) {
    const SamplePt s = q.probe_pts[tid];
    q.sc.probes[(size_t)e * q.nprobe + tid] = sample_linear(p, P, s.i, s.j, s.s, s.t);
  }
  __syncthreads();
  if (tid == 0) {
    float pvx = 0, pvy = 0;
    for (int k = 0; k < q.nforce; k++) { pvx += sx[k]; pvy += sy[k]; }           // Body.pde:300
    const float fx = pvx * -1, fy = pvy * -1;                                     // AFCCylinder.pde:58
    q.sc.force[2 * e] = fx;
    q.sc.force[2 * e + 1] = fy;
    const float t = q.sc.t[e] + q.dt_over_res;                                    // AFCCylinder.pde:56
    q.sc.t[e] = t;
    q.sc.flow_t[e] += q.dt;                                                       // BDIM.update2: t += dt (BDIM.pde:106)
    if (!isfinite(fx) || !isfinite(fy)) q.sc.non_finite[e] = 1;                   // diverged environment (sticky flag)
    if (accumulate && t >= q.episode_time) q.sc.frozen[e] = 1;                    // clientCFD.pde:36: no frame past Time
    if (accumulate && t > q.init_time) {                                          // clientCFD.pde:39-47
      int cl = q.sc.callLearn[e] - 1;
      float Cd = q.sc.Cd[e] + fx, Cl = q.sc.Cl[e] + fy;
      if (cl <= 0) {
        cl = q.substeps;
        Cd = Cd / cl * 2 / q.resolution;
        Cl = Cl / cl * 2 / q.resolution;
        q.sc.obs[2 * e] = Cl;
        q.sc.obs[2 * e + 1] = Cd;
        q.sc.frozen[e] = 1;            // the sketch now blocks in callAction until the agent answers (clientCFD.pde:50)
      }
      q.sc.callLearn[e] = cl;
      q.sc.Cd[e] = Cd;
      q.sc.Cl[e] = Cl;
    }
  }
}

// Start of a call.  mode 0 (single solver steps): xi = act where given, every env runs.  mode 1 (RL step): the reference
// changes xi only when callAction returns, i.e. right after an observation was emitted (clientCFD.pde:44-54): an env
// that has not reached its first callLearn boundary yet (t <= initTime after a reset, or mid-window after an episode
// change with the sketch-global accumulators kept) keeps its xi.  An env past the episode end takes no more steps.
// BDIM.checkCFL (BDIM.pde:217-219) = min(u.CFL(nu), 1), VectorField.CFL (VectorField.pde:225-235): 1/(b + 3 nu) with
// b = max(|ux|+|uy|) over the interior, started from cell [0][0].  A maximum does not depend on the order it is taken in,
// so the reduction is parallel and still exact.  One CTA per environment (a diagnostic / adaptive-dt read-out, not on
// the fixed-dt step path).
__global__ void __launch_bounds__(1024)
k_check_cfl(const __grid_constant__ SolverParams q, const float* __restrict__ ux_all, const float* __restrict__ uy_all,
            float* __restrict__ dt_out) {
  __shared__ float wmax[32];
  const int e = blockIdx.x, P = q.P, ni = q.n - 2, mj = q.m - 2;
  const float* ux = ux_all + (size_t)e * q.stride;
  const float* uy = uy_all + (size_t)e * q.stride;
  float b = fabsf(ux[0]) + fabsf(uy[0]);
  for (int k = threadIdx.x; k < ni * mj; k += blockDim.x) {
    const int i = 1 + k / mj, j = 1 + k - (k / mj) * mj;
    const float c = fabsf(ux[IDX(i, j)]) + fabsf(uy[IDX(i, j)]);
    if (c > b) b = c;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const float v = __shfl_down_sync(0xffffffffu, b, o); if (v > b) b = v; }
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) if (wmax[w] > b) b = wmax[w];
    const float cfl = 1.f / (b + 3.f * q.nu);
    dt_out[e] = cfl < 1.f ? cfl : 1.f;                                      // PApplet.min(u.CFL(nu), 1)
  }
}

__global__ void k_set_actions(const __grid_constant__ SolverParams q, const float* __restrict__ act, int mode) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= q.B) return;
  bool take = act != nullptr, frozen = false;
  if (mode == 1) {
    const float t = q.sc.t[e];
    take = take && t > q.init_time && q.sc.callLearn[e] == q.substeps;
    frozen = t >= q.episode_time;
  }
  if (take) { q.sc.xi[2 * e] = act[2 * e]; q.sc.xi[2 * e + 1] = act[2 * e + 1]; }
  q.sc.frozen[e] = frozen ? 1 : 0;
}

// obs/reward/done of one RL step; reward = server/server.py:61-65 evaluated in double
__global__ void k_emit_obs(const __grid_constant__ SolverParams q, const float* __restrict__ act, float* obs, float* reward,
                           int* done) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= q.B) return;
  const float Cl = q.sc.obs[2 * e], Cd = q.sc.obs[2 * e + 1];
  if (obs) { obs[2 * e] = Cl; obs[2 * e + 1] = Cd; }
  if (reward) {
    double a1 = fabs((double)act[2 * e]), a2 = fabs((double)act[2 * e + 1]);
    double pen = 3.141592653589793 * (1.0 / 8) * 0.0097 * (3.66 * 3.66 * 3.66) * (a1 * a1 * a1 + a2 * a2 * a2);
    reward[e] = (float)(-(double)Cd - pen);
  }
  if (done) done[e] = q.sc.t[e] >= q.episode_time ? 1 : 0;
  if (!q.sc.frozen[e]) atomicAdd(q.sc.n_running, 1);      // still on its way to the next observation
}

// end of one MGsolver iteration inside a CUDA-graph WHILE node: continue while any env is still active
// Slab mode: all devices meet here between dependent kernels.  One arrival counter (device 0's memory) counts every
// device's every barrier; a device has passed its k-th barrier when the counter has reached k * n.
__global__ void k_slab_barrier(SlabBarrier b) {
  __threadfence_system();
  const unsigned ep = *b.epoch + 1u;
  *b.epoch = ep;
  atomicAdd_system(b.count, 1u);
  const unsigned target = ep * b.n;
  unsigned spins = 0;
  while (true) {
    unsigned v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(b.count) : "memory");
    if ((int)(v - target) >= 0) break;
    if (++spins > (1u << 26)) __trap();          // a device that never arrives is a bug, and a trap beats a hung box
    __nanosleep(100);
  }
  __threadfence_system();
}

__global__ void k_loopcond(cudaGraphConditionalHandle h, int* any_active) {
  if (threadIdx.x == 0) {
    const unsigned v = *any_active ? 1u : 0u;
    *any_active = 0;
    cudaGraphSetConditional(h, v);
  }
}

inline dim3 grid2d(int m, int n, int B, dim3 blk) { return dim3((m + blk.x - 1) / blk.x, (n + blk.y - 1) / blk.y, B); }

}  // namespace

// ================================================================================================
// launch wrappers
// ================================================================================================
int launch_advdif(const SolverParams& q, const float* srcx, const float* srcy, const float* u0x, const float* u0y,
                  float* dstx, float* dsty, cudaStream_t st) {
  const int ni = q.n - 2, mj = q.m - 2;
  // rows a warp marches: 48 amortise the 4-row window best; a small batch (one wide domain) needs more warps instead
  const int rows = (long long)q.B * ni * mj < (8ll << 20) ? 16 : kAdvRows;
  dim3 grid((mj + kAdvCols - 1) / kAdvCols, ((ni + rows - 1) / rows + 3) / 4, q.B);
  if (srcx == u0x && srcy == u0y)
    k_advdif<true><<<grid, 128, 0, st>>>(srcx, srcy, u0x, u0y, dstx, dsty, q.n, q.m, q.P, q.stride, q.dt, q.nu, q.sc.frozen, q.slab_rank, q.slab_n, rows);
  else
    k_advdif<false><<<grid, 128, 0, st>>>(srcx, srcy, u0x, u0y, dstx, dsty, q.n, q.m, q.P, q.stride, q.dt, q.nu, q.sc.frozen, q.slab_rank, q.slab_n, rows);
  return 1;
}

static size_t bc2_smem(const SolverParams& q) { return sizeof(float) * (2 * (3 * q.m + 2 * q.n) + q.nband_x + q.nband_y); }

int launch_band_bc(const SolverParams& q, float* ux, float* uy, cudaStream_t st) {
  if (q.fast_bc) k_bc2<true, false><<<q.B, 1024, bc2_smem(q), st>>>(q, ux, uy, nullptr, nullptr, nullptr, nullptr);
  else if (q.nband_x + q.nband_y > 4096) {             // a large band (single wide domain): blend grid-wide first
    k_band_blend<<<dim3((q.nband_x + q.nband_y + 255) / 256, q.B), 256, 0, st>>>(q, ux, uy);
    k_band_bc<true><<<q.B, 1024, sizeof(float) * q.m, st>>>(q, ux, uy);
    return 2;
  } else k_band_bc<false><<<q.B, 1024, sizeof(float) * q.m, st>>>(q, ux, uy);
  return 1;
}

int launch_bc(const SolverParams& q, float* ux, float* uy, cudaStream_t st) {
  if (q.fast_bc) k_bc2<false, false><<<q.B, 1024, bc2_smem(q), st>>>(q, ux, uy, nullptr, nullptr, nullptr, nullptr);
  else k_bc<<<q.B, 512, sizeof(float) * q.m, st>>>(q, ux, uy);
  return 1;
}

int launch_residual(const SolverParams& q, const float* ux, const float* uy, float* r, int which, cudaStream_t st) {
  dim3 blk(32, 8);
  k_residual<<<grid2d(q.m, q.n, q.B, blk), blk, 0, st>>>(q, ux, uy, r, which);
  return 1;
}

int launch_resid_down0(const SolverParams& q, const float* ux, const float* uy, const float* p_in, float* p_out, float* r_out,
                       int which, cudaStream_t st) {
  const DevLevel& L1 = q.lev[1];
  if (q.resid_march) {
    const int ni = q.n - 2, mj = q.m - 2;
    dim3 grid((mj + kRmWarps * kRmCols - 1) / (kRmWarps * kRmCols), (ni + kRmRows - 1) / kRmRows, q.B);
    k_resid_down0_march<<<grid, 32 * (kRmWarps + 1), kRmSmem, st>>>(q, ux, uy, p_in, p_out, r_out, which);
    return 1;
  }
  dim3 blk(kRdJ, kRdI);
  dim3 grid((L1.m - 2 + kRdJ - 1) / kRdJ, (L1.n - 2 + kRdI - 1) / kRdI, q.B);
  k_resid_down0<<<grid, blk, 0, st>>>(q, ux, uy, p_in, p_out, r_out, which);
  return 1;
}

int launch_project_shift(const SolverParams& q, const float* p_in, float* p_out, float* ux, float* uy, cudaStream_t st) {
  const int items = q.n * (q.P >> 2);
  dim3 grid((items + 255) / 256, q.B);
  k_project_shift<false><<<grid, 256, 0, st>>>(q, p_in, p_out, ux, uy, nullptr, nullptr, nullptr, nullptr);
  return 1;
}

int launch_project_shift_heun(const SolverParams& q, const float* p_in, float* p_out, float* ux, float* uy, const float* usx,
                              const float* usy, float* uox, float* uoy, cudaStream_t st) {
  const int items = q.n * (q.P >> 2);
  dim3 grid((items + 255) / 256, q.B);
  k_project_shift<true><<<grid, 256, 0, st>>>(q, p_in, p_out, ux, uy, usx, usy, uox, uoy);
  return 1;
}

int launch_bc_heun(const SolverParams& q, float* ux, float* uy, const float* usx, const float* usy, float* uox, float* uoy,
                   cudaStream_t st) {
  k_bc2<false, true><<<q.B, 1024, bc2_smem(q), st>>>(q, ux, uy, usx, usy, uox, uoy);
  return 1;
}

int launch_slab_barrier(const SlabBarrier& b, cudaStream_t st) {
  k_slab_barrier<<<1, 1, 0, st>>>(b);
  return 1;
}

int launch_loopcond(const SolverParams& q, unsigned long long handle, cudaStream_t st) {
  k_loopcond<<<1, 32, 0, st>>>((cudaGraphConditionalHandle)handle, q.sc.any_active);
  return 1;
}

int launch_mg_down0(const SolverParams& q, const float* r_in, float* r_out, cudaStream_t st) {
  dim3 blk(32, 8);
  const DevLevel& L1 = q.lev[1];
  k_mg_down0<<<grid2d(L1.m - 2, L1.n - 2, q.B, blk), blk, 0, st>>>(q, r_in, r_out);
  return 1;
}

static size_t strip_smem(int nstrips) { return sizeof(StripShared) * nstrips + sizeof(StripMail) * (nstrips + 2); }

static size_t smooth0_smem(const SolverParams& q) {
  return strip_smem(q.lev[0].sk.nstrips) + sizeof(float) * (2 * (q.n - 2) + 2 * (q.m - 2));
}

// opt-in shared-memory sizes; called once per handle, outside any stream capture
static size_t coarse_rows_smem(const SolverParams& q) {
  size_t s = 0;
  for (int l = max(1, q.chain_levels); l < q.nlevels; l++)
    if (!q.lev[l].wave) {
      if (q.tiny && tiny_level(q.lev[l].n - 2, q.lev[l].m - 2)) s = max(s, tiny_smem_bytes(q.lev[l].n - 2));
      else s = max(s, rows_smem_bytes(min(q.lev[l].rt.C, 4), q.lev[l].P, false));
    }
  return s;
}
static size_t smooth0_rows_smem(const SolverParams& q) {
  return rows_smem_bytes(q.lev[0].rt.C, q.P, true) + sizeof(float) * (2 * (q.n - 2) + 2 * (q.m - 2));
}

template <int C>
static cudaError_t set_smooth0_rows_attr(const SolverParams& q) {
  return cudaFuncSetAttribute(k_smooth0_rows<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smooth0_rows_smem(q));
}

int configure_kernels(const SolverParams& q) {
  cudaError_t e1 = cudaSuccess, e2 = cudaSuccess;
  if (!q.use_rows) {
    e1 = cudaFuncSetAttribute(k_mg_coarse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)strip_smem(q.coarse_strips));
    e2 = cudaFuncSetAttribute(k_smooth0, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smooth0_smem(q));
  }
  if (q.fast_bc) {
    if (cudaFuncSetAttribute(k_bc2<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bc2_smem(q)) != cudaSuccess ||
        cudaFuncSetAttribute(k_bc2<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bc2_smem(q)) != cudaSuccess ||
        cudaFuncSetAttribute(k_bc2<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bc2_smem(q)) != cudaSuccess)
      return -1;
  }
  if (cudaFuncSetAttribute(k_xsum_chain_blocks<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXsBlocksSmem) != cudaSuccess ||
      cudaFuncSetAttribute(k_xsum_chain_blocks<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXsBlocksSmem) != cudaSuccess) return -1;
  if (cudaFuncSetAttribute(k_resid_down0_march, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRmSmem) != cudaSuccess) return -1;
  cudaError_t e3 = cudaFuncSetAttribute(k_mg_coarse_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coarse_rows_smem(q));
  if (q.chain_levels > 0 &&
      (cudaFuncSetAttribute(k_chain_sweeps, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kChMaxWpb * sizeof(ChainRing))) != cudaSuccess ||
       cudaFuncSetAttribute(k_chain_sweeps3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Chain3Smem)) != cudaSuccess ||
       cudaFuncSetAttribute(k_chain_sweeps3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Chain3Smem)) != cudaSuccess))
    return -1;
  cudaError_t e4 = cudaSuccess;
  if (!q.lev[0].wave && !q.lev[0].ch.on) switch (q.lev[0].rt.C) {
    case 1: e4 = set_smooth0_rows_attr<1>(q); break;
    case 2: e4 = set_smooth0_rows_attr<2>(q); break;
    case 3: e4 = set_smooth0_rows_attr<3>(q); break;
    case 4: e4 = set_smooth0_rows_attr<4>(q); break;
    case 5: e4 = set_smooth0_rows_attr<5>(q); break;
    case 6: e4 = set_smooth0_rows_attr<6>(q); break;
    case 7: e4 = set_smooth0_rows_attr<7>(q); break;
    default: e4 = set_smooth0_rows_attr<8>(q); break;
  }
  return (e1 == cudaSuccess && e2 == cudaSuccess && e3 == cudaSuccess && e4 == cudaSuccess) ? 0 : -1;
}

// chained strip smoother (smooth_chain.cuh): the pieces of one level, individually launchable (profiling) ...
int launch_chain_sweeps(const SolverParams& q, int l, cudaStream_t st) {
  const ChainLevel& ch = q.lev[l].ch;
  if (q.chain_v == 1) k_chain_sweeps<<<q.B * 4 * ch.nb, 32 * ch.wpb, ch.wpb * sizeof(ChainRing), st>>>(q, l);
  else if (ch.ns_loc > 0) {
    // (slab mode: strips on other devices hand their edge operands over through peer memory: system-scope accesses)
    if (q.slab_n > 1) k_chain_sweeps3<true><<<q.B * 4 * ch.ns_loc, 96, sizeof(Chain3Smem), st>>>(q, l);
    else k_chain_sweeps3<false><<<q.B * 4 * ch.ns_loc, 96, sizeof(Chain3Smem), st>>>(q, l);
  }
  return 1;
}
int launch_chain_incr(const SolverParams& q, int l, float* r_out, int which, cudaStream_t st) {
  const ChainLevel& ch = q.lev[l].ch;
  const int runs = (q.lev[l].n - 2 + 31 + kChIncEntries - 1) / kChIncEntries;
  const dim3 grid((runs + kChIncWarps - 1) / kChIncWarps, ch.NS, q.B);
  if (l == 0) k_chain_incr<true><<<grid, 32 * kChIncWarps, 0, st>>>(q, l, r_out, which);
  else k_chain_incr<false><<<grid, 32 * kChIncWarps, 0, st>>>(q, l, nullptr, 0);
  return 1;
}
int launch_chain_down(const SolverParams& q, int l, cudaStream_t st) {
  dim3 blk(32, 8);
  k_chain_down<<<grid2d(q.lev[l + 1].m - 2, q.lev[l + 1].n - 2, q.B, blk), blk, 0, st>>>(q, l);
  return 1;
}
int launch_chain_up(const SolverParams& q, int l, const float* r, cudaStream_t st) {
  dim3 blk(32, 8);
  if (l == 0) k_chain_up<true><<<grid2d(q.lev[1].m - 2, q.lev[1].n - 2, q.B, blk), blk, 0, st>>>(q, 0, r);
  else k_chain_up<false><<<grid2d(q.lev[l + 1].m - 2, q.lev[l + 1].n - 2, q.B, blk), blk, 0, st>>>(q, l, nullptr);
  return 1;
}
int launch_coarse_cta(const SolverParams& q, cudaStream_t st) {
  k_mg_coarse_rows<<<q.B, kRowsThreads, coarse_rows_smem(q), st>>>(q, max(1, q.chain_levels));
  return 1;
}

int chain_incr_blocks(int ni, int NS) {
  const int runs = (ni + 31 + kChIncEntries - 1) / kChIncEntries;
  return ((runs + kChIncWarps - 1) / kChIncWarps) * NS;
}

// ... and as the composites the step graph captures
int launch_mg_coarse(const SolverParams& q, cudaStream_t st) {
  if (q.use_rows) {
    // wide levels run as grid-wide kernels around the one-CTA-per-environment kernel of the small levels
    int nl = 0;
    const int first = max(1, q.chain_levels);
    for (int l = 1; l < first; l++) nl += launch_chain_down(q, l, st);
    nl += launch_coarse_cta(q, st);
    for (int l = first - 1; l >= 1; l--) {
      nl += launch_chain_up(q, l, nullptr, st);
      nl += launch_chain_sweeps(q, l, st);
      nl += launch_chain_incr(q, l, nullptr, 0, st);
    }
    return nl;
  }
  const size_t smem = strip_smem(q.coarse_strips);
  k_mg_coarse<<<q.B, max(256, 32 * q.coarse_strips), smem, st>>>(q);
  return 1;
}

int launch_mg_up0(const SolverParams& q, float* r, cudaStream_t st) {
  dim3 blk(32, 8);
  if (q.lev[0].ch.on) return launch_chain_up(q, 0, r, st);
  if (q.use_rows && !q.lev[0].wave) k_mg_up0_blk<<<dim3((q.n - 2 + kUpRows - 1) / kUpRows, q.B), 256, up0_smem(q), st>>>(q, r);
  else k_mg_up0<false><<<grid2d(q.m, q.n, q.B, blk), blk, 0, st>>>(q, r);
  return 1;
}

int launch_unskew_r(const SolverParams& q, float* r, cudaStream_t st) {
  if (!q.use_rows || q.lev[0].wave || q.lev[0].ch.on) return 0;   // (the chain increment writes the plain residual itself)
  dim3 blk(32, 8);
  k_unskew_r<<<grid2d(q.m, q.n, q.B, blk), blk, 0, st>>>(q, r);
  return 1;
}

int launch_smooth0(const SolverParams& q, const float* r_in, float* r_out, int which, cudaStream_t st) {
  if (q.lev[0].ch.on) return launch_chain_sweeps(q, 0, st) + launch_chain_incr(q, 0, r_out, which, st);
  if (q.use_rows && q.lev[0].wave) {
    k_smooth0_wave<<<q.B, 1024, 0, st>>>(q, r_in, r_out, which);
    return 1;
  }
  if (q.use_rows) {
    const size_t sm = smooth0_rows_smem(q);
    switch (q.lev[0].rt.C) {
      case 1: k_smooth0_rows<1><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      case 2: k_smooth0_rows<2><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      case 3: k_smooth0_rows<3><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      case 4: k_smooth0_rows<4><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      case 5: k_smooth0_rows<5><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      case 6: k_smooth0_rows<6><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      case 7: k_smooth0_rows<7><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
      default: k_smooth0_rows<8><<<q.B, kRows0Threads, sm, st>>>(q, which); break;
    }
    return 1;
  }
  const int ns = q.lev[0].sk.nstrips;
  const size_t smem = smooth0_smem(q);
  k_smooth0<<<q.B, 32 * ns, smem, st>>>(q, r_in, r_out, which);
  return 1;
}

// Field.sum as segment summaries: the table kernel, then the serial pass (individually launchable for profiling)
int launch_psum_tables(const SolverParams& q, cudaStream_t st) {
  const dim3 grid(q.B, q.xs_nchunks);     // chunk index slow: see the look-back in k_xsum_tables
  if (q.xs_corr) {                        // large domains: two passes, the second with the refined prediction
    k_xsum_tables<1><<<grid, kXsThreads, 0, st>>>(q);
    k_xsum_refine<<<q.B, 1024, 0, st>>>(q);
    if (q.xs_passes >= 3) {               // very large domains: a third pass (PASS 3 = corrected prediction AND new increments)
      k_xsum_tables<3><<<grid, kXsThreads, 0, st>>>(q);
      k_xsum_refine<<<q.B, 1024, 0, st>>>(q);
    }
    k_xsum_tables<2><<<grid, kXsThreads, 0, st>>>(q);
    return q.xs_passes >= 3 ? 5 : 3;
  }
  k_xsum_tables<0><<<grid, kXsThreads, 0, st>>>(q);
  return 1;
}
int launch_psum_pass(const SolverParams& q, cudaStream_t st) {
  if (q.xs_blk) {                       // large domains: runs of records condensed first (in parallel), then crossed
    k_xsum_condense<<<dim3((q.xs_nbatches + 31) / 32, q.B), 32, 0, st>>>(q);
    // (helper warps for rebuilding batches in bulk only where long stretches of them occur: the three-pass sizes)
    if (q.xs_passes >= 3) k_xsum_chain_blocks<true><<<q.B, 32 * kXsBulkWarps, kXsBlocksSmem, st>>>(q);
    else k_xsum_chain_blocks<false><<<q.B, 32, kXsBlocksSmem, st>>>(q);
    return 2;
  }
  k_xsum_chain<false><<<q.B, 32, 0, st>>>(q);
  return 1;
}
int launch_psum(const SolverParams& q, cudaStream_t st) {
  if (!q.xs_recs) {                     // RLFC_PSUM=serial: the plain dependent-add chain, one warp per environment
    k_psum<<<q.B, 32, 0, st>>>(q);
    return 1;
  }
  return launch_psum_tables(q, st) + launch_psum_pass(q, st);
}

int launch_psum_overlapped(const SolverParams& q, cudaStream_t st, cudaStream_t side, cudaEvent_t fork, cudaEvent_t join) {
  if (!q.xs_recs) return launch_psum(q, st);
  cudaEventRecord(fork, st);
  cudaStreamWaitEvent(side, fork, 0);
  const dim3 grid(q.B, q.xs_nchunks);
  k_xsum_tables<0><<<grid, kXsThreads, 0, st>>>(q);
  k_xsum_chain<true><<<q.B, 32, 0, side>>>(q);       // waits for each chunk's record flag (bounded), see the kernel
  cudaEventRecord(join, side);
  cudaStreamWaitEvent(st, join, 0);
  return 2;
}

int launch_project_u(const SolverParams& q, float* ux, float* uy, cudaStream_t st) {
  dim3 blk(32, 8);
  k_project_u<<<grid2d(q.m, q.n, q.B, blk), blk, 0, st>>>(q, ux, uy);
  return 1;
}

int launch_shift_p(const SolverParams& q, cudaStream_t st) {
  dim3 blk(32, 8);
  k_shift_p<<<grid2d(q.m, q.n, q.B, blk), blk, 0, st>>>(q);
  return 1;
}

int launch_heun(const SolverParams& q, const float* ucx, const float* ucy, const float* ubx, const float* uby,
                float* uax, float* uay, cudaStream_t st) {
  dim3 blk(32, 8);
  k_heun<<<grid2d(q.m, q.n, q.B, blk), blk, 0, st>>>(ucx, ucy, ubx, uby, uax, uay, q.n, q.m, q.P, q.stride, q.sc.frozen, q.slab_rank, q.slab_n);
  return 1;
}

int launch_force(const SolverParams& q, int accumulate, cudaStream_t st) {
  k_force<<<q.B, 64, 0, st>>>(q, accumulate);
  return 1;
}

int launch_check_cfl(const SolverParams& q, const float* ux, const float* uy, float* d_dt, cudaStream_t st) {
  k_check_cfl<<<q.B, 1024, 0, st>>>(q, ux, uy, d_dt);
  return 1;
}

int launch_set_actions(const SolverParams& q, const float* d_actions, int mode, cudaStream_t st) {
  k_set_actions<<<(q.B + 127) / 128, 128, 0, st>>>(q, d_actions, mode);
  return 1;
}

int launch_emit_obs(const SolverParams& q, const float* d_actions, float* d_obs, float* d_reward, int* d_done,
                    cudaStream_t st) {
  k_emit_obs<<<(q.B + 127) / 128, 128, 0, st>>>(q, d_actions, d_obs, d_reward, d_done);
  return 1;
}

}  // namespace rlfc
