// geometry_device.cuh -- reset environments into arbitrary parameter sets on the device (rlfc_env_reset_params_device).
// Included at the end of solver_kernels.cu, after param_sets.cuh, whose pair resolution, chunk copy and reset scalars it
// shares.
//
// build_geometry's per-face path (geometry.cpp) restated operation for operation and in the same order: Cylinder with its
// Edge, distance, box_distance and wall_normal, union_kernel, the weight normalisation, mu0, mu1, eval_face, the set_bc of
// del, and band_lists' i-major order.  The host code is float arithmetic with one rounding per operation (compiled without
// contraction, as this file is with --fmad=false), IEEE division, and double sqrt narrowed to float; all of that is exact
// on the device too.  The one remaining part is fsin / fcos = (float)std::sin / cos((double)x): fsin_dev / fcos_dev return
// the host's value for every float with |x| <= 2 pi (DESIGN.md section 3, "Device parameter resets"), which covers every
// argument build_geometry passes them given |theta| <= 2 pi: kPi*d/eps and kPi*d with |d| < eps or |d| < 1, and theta.
// The 40 polygon vertex factors come from the host (circle_vertex_factors).
//
// Two kernels, both grid (.., pairs) like k_reset_sets:
//   k_param_geometry  one CTA per pair.  The winning pair of an environment is validated before anything is written: the
//                     scalar rules, the bodies' convexity, and a pass over every face that evaluates the band predicate
//                     (del, del1 after set_bc, w1, w2) and counts the band without writing.  A refused pair sets
//                     refused[e] and nothing else.  An accepted one writes the slot's ten fields and its band lists (a
//                     ballot scan keeps band_lists' order), then the environment's per-environment scalars.
//   k_reset_params    k_reset_sets' copy of the init state and reset scalars, for the accepted pairs.
// The caller then rebuilds the Poisson hierarchies on the skip mask k_reset_params clears.
#pragma once
#include "solver.h"
#include "snapshot.cuh"
#include "param_sets.cuh"

namespace rlfc {
namespace {

constexpr float kGeoPi = 3.1415927f;     // PConstants.PI (geometry.cpp kPi)
constexpr float kGeoTwoPi = 6.2831855f;  // PConstants.TWO_PI; also the largest |theta| a device reset accepts
constexpr float kGeoEps = 2.0f;          // BDIM.eps (BDIM.pde:35)
constexpr int kGeoVerts = 40;            // EllipseBody.m

// (float)std::sin((double)x) of the host for |x| <= 2 pi.  Host libm narrowed to float is the correctly rounded float over
// that range; a double evaluation narrowed to float can only differ from it where the exact result lies within the
// evaluation's error of a float rounding midpoint.  Of all floats in [0, 2 pi] five have a result within 4 double ulps of
// one (two for sin, three for cos): their host results are tabulated.  Both functions are evaluated on |x| and the
// symmetry applied (the host's sin(-x) == -sin(x) and cos(-x) == cos(x) hold bit for bit).
__device__ __forceinline__ float fsin_dev(float x) {
  const float ax = fabsf(x);
  float r = (float)sin((double)ax);
  const unsigned b = __float_as_uint(ax);
  if (b == 0x3dcf5597u) r = __uint_as_float(0x3dcefaf9u);          // sin(0x1.9eab2ep-4) = 0x1.9df5f2p-4
  else if (b == 0x3ef3830fu) r = __uint_as_float(0x3eea6f45u);     // sin(0x1.e7061ep-2) = 0x1.d4de8ap-2
  return (__float_as_uint(x) >> 31) ? -r : r;
}
__device__ __forceinline__ float fcos_dev(float x) {
  const float ax = fabsf(x);
  float r = (float)cos((double)ax);
  const unsigned b = __float_as_uint(ax);
  if (b == 0x39800000u) r = 1.f;                                   // cos(0x1p-12) = 1
  else if (b == 0x3c107fe6u) r = __uint_as_float(0x3f7ffd74u);     // cos(0x1.20ffccp-7) = 0x1.fffae8p-1
  else if (b == 0x3a544395u) r = __uint_as_float(0x3f7ffffbu);     // cos(0x1.a8872ap-11) = 0x1.fffff6p-1
  return r;
}

__device__ __forceinline__ float gmin2(float a, float b) { return (a < b) ? a : b; }   // PApplet.min
__device__ __forceinline__ float gmax2(float a, float b) { return (a > b) ? a : b; }   // PApplet.max

// OrthoNormal (OrthoNormal.pde:8-28): what the faces need of an Edge
struct GEdge {
  float nx, ny, off, cx, cy;
};
__device__ __forceinline__ GEdge make_edge(float ax, float ay, float bx, float by) {
  GEdge E;
  const float sx = ax - bx, sy = ay - by, sz = 0.f;
  const float l = (float)sqrt((double)(sx * sx + sy * sy + sz * sz));   // PVector.mag
  const float tx = (bx - ax) / l, ty = (by - ay) / l;
  E.nx = -ty;
  E.ny = tx;
  E.off = ax * E.nx + ay * E.ny;
  E.cx = (ax + bx) / 2.f;
  E.cy = (ay + by) / 2.f;
  return E;
}
__device__ __forceinline__ float signed_dist(const GEdge& E, float x, float y) { return x * E.nx + y * E.ny - E.off; }

// CircleBody (Body.pde:386-417)
struct GBody {
  float xc, yc, h;
  GEdge edge[kGeoVerts];
  GEdge box[4];
};

__device__ __forceinline__ float body_distance(const GBody& b, float x, float y) {   // CircleBody.distance
  const float ax = x - b.xc, ay = y - b.yc;
  return (float)sqrt((double)(ax * ax + ay * ay)) - 0.5f * b.h;
}
__device__ __forceinline__ float box_distance(const GBody& b, float x, float y) {
  float dis = -1e10f;
  for (int i = 0; i < 4; i++) dis = gmax2(dis, signed_dist(b.box[i], x, y));
  return dis;
}
__device__ __forceinline__ void wall_normal(const GBody& b, float x, float y, float& ox, float& oy) {
  ox = 0; oy = 0;
  if (box_distance(b, x, y) > 3) return;
  float best = -1e10f;
  for (int i = 0; i < kGeoVerts; i++) {
    const float d2 = signed_dist(b.edge[i], x, y);
    if (d2 > best) { best = d2; ox = b.edge[i].nx; oy = b.edge[i].ny; }
  }
}

__device__ __forceinline__ float union_kernel_dev(float d) {   // BodyUnion.delta0
  if (d <= -1) return 0;
  if (d >= 1) return 1;
  return 0.5f * (1.f + d + fsin_dev(kGeoPi * d) / kGeoPi);
}
__device__ __forceinline__ float mu0_dev(float d, float eps) {   // BDIM.delta0
  if (d <= -eps) return 0;
  if (d >= eps) return 1;
  return 0.5f * (1.f + d / eps + fsin_dev(kGeoPi * d / eps) / kGeoPi);
}
__device__ __forceinline__ float mu1_dev(float d, float eps) {   // BDIM.delta1
  const float ad = (d < 0) ? -d : d;
  if (ad >= eps) return 0;
  return 0.25f * (eps - (d * d) / eps) -
         1 / kGeoTwoPi * (d * fsin_dev(d * kGeoPi / eps) + eps / kGeoPi * (1 + fcos_dev(d * kGeoPi / eps)));
}

// BodyUnion.distance of the three bodies
__device__ __forceinline__ float union_distance(const GBody* body, float x, float y, float dk[3]) {
  float dmin = 1e6f;
  for (int k = 0; k < 3; k++) { dk[k] = body_distance(body[k], x, y); dmin = gmin2(dmin, dk[k]); }
  return dmin;
}
// eval_face up to the wall normal: the normalised union weights w and del / del1 = mu0 / mu1 of the union distance
__device__ __forceinline__ void eval_face_dev(const GBody* body, float x, float y, float w[3], float& del, float& del1) {
  float dk[3];
  const float dist = union_distance(body, x, y, dk);
  float s = 0;
  for (int k = 0; k < 3; k++) { w[k] = union_kernel_dev(-dk[k] / 3.f); s += w[k]; }
  for (int k = 0; k < 3 && s > 0; k++) w[k] /= s;
  del = mu0_dev(dist, kGeoEps);
  del1 = mu1_dev(dist, kGeoEps);
}
// eval_face's BodyUnion.WallNormal
__device__ __forceinline__ void face_normal(const GBody* body, float x, float y, const float w[3], float& nx, float& ny) {
  nx = 0; ny = 0;
  for (int k = 0; k < 3; k++) {
    float ax, ay;
    wall_normal(body[k], x, y, ax, ay);
    nx += ax * w[k];
    ny += ay * w[k];
  }
}

struct ResetParamsArgs {
  ParamLib lib;
  ParamReset pr;
  CircleFactors cf;
  EnvScalars sc;
  float *del_x, *del_y, *w1_x, *w2_x, *ry1_x, *ry2_x, *w1_y, *w2_y, *rx1_y, *rx2_y;   // geometry slots (slot s at s*stride)
  BandFace *band_x, *band_y;                   // slot s at s*cap
  int *env_slot, *env_nbx, *env_nby;
  float *env_nu, *env_dRD;
  unsigned* env_par;                           // [5][B] parameter tuples (nullptr without snapshots or records)
  const float4 *iux, *iuy, *ip;                // the init state (one environment)
  float4 *ux, *uy, *p;                         // the environments' fields (batch base)
  size_t stride, stride4;                      // level-0 per-environment stride in floats / float4
  int nv;                                      // float4 of one field that are copied (n*P/4)
  int n, m, P, nc, mc, resolution, cap, B;
  const int* env;
  const rlfc_env_params* par;
  int npairs, reset_acc, substeps;
  float init_t;
  int* skip;
};

// x-face (i-1/2, j) and y-face (i, j-1/2) of interior cell (i, j): the band predicate of band_lists on the values after
// set_bc, which sets del to 1 and del1 to 0 on row 1 (x) and column 1 (y)
__device__ __forceinline__ bool x_face(const GBody* body, int i, int j, float w[3], float& del, float& del1) {
  eval_face_dev(body, (float)(i - 0.5), (float)j, w, del, del1);
  if (i == 1) { del = 1.f; del1 = 0.f; }
  return del != 1.f || del1 != 0.f || w[1] != 0.f || w[2] != 0.f;
}
__device__ __forceinline__ bool y_face(const GBody* body, int i, int j, float w[3], float& del, float& del1) {
  eval_face_dev(body, (float)i, (float)(j - 0.5), w, del, del1);
  if (j == 1) { del = 1.f; del1 = 0.f; }
  return del != 1.f || del1 != 0.f || w[1] != 0.f || w[2] != 0.f;
}

__device__ __forceinline__ int block_sum(int v, int* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(~0u, v, o);
  if (threadIdx.x == 0) *red = 0;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) atomicAdd(red, v);
  __syncthreads();
  const int s = *red;
  __syncthreads();
  return s;
}

__global__ void __launch_bounds__(kSnapThreads) k_param_geometry(const __grid_constant__ ResetParamsArgs a) {
  __shared__ GBody body[3];
  __shared__ float vx[3][kGeoVerts], vy[3][kGeoVerts];
  __shared__ int wsum[2][kSnapThreads / 32];
  __shared__ int red;
  const int n = a.n, m = a.m, P = a.P, mj = m - 2, cells = (n - 2) * mj;
  const float D = (float)a.resolution;                                         // AFCCylinder.pde:27
  for (int k = blockIdx.y; k < a.npairs; k += gridDim.y) {
    if (!pair_applies(a.env, a.env, k, a.npairs, a.B, a.B, true)) continue;
    const int e = a.env[k];
    const rlfc_env_params q = a.par[k];
    // build_env_geometries' rules, and the range over which fsin_dev / fcos_dev are exact
    bool ok = q.re >= 1 && q.dR > 0 && q.dR <= 1 && q.gR >= 0 && isfinite(q.gR) && isfinite(q.theta) &&
              fabsf(q.theta) <= kGeoTwoPi && isfinite(q.t_step) && q.t_step > 0;
    int nbx = 0, nby = 0;
    if (ok) {
      // the three Cylinders (AFCCylinder.pde:29-32)
      if (threadIdx.x < 3) {
        const int b = threadIdx.x;
        const float r = (D / 2 + q.gR * D + q.dR * D / 2);
        if (b == 0) { body[0].xc = (float)(a.nc / 4); body[0].yc = (float)(a.mc / 2); body[0].h = D; }
        else {
          body[b].xc = a.nc / 4 + r * fcos_dev(q.theta);
          body[b].yc = b == 1 ? a.mc / 2 - r * fsin_dev(q.theta) : a.mc / 2 + r * fsin_dev(q.theta);
          body[b].h = q.dR * D;
        }
      }
      __syncthreads();
      if (threadIdx.x < 3 * kGeoVerts) {
        const int b = threadIdx.x / kGeoVerts, i = threadIdx.x - b * kGeoVerts;
        const float h = body[b].h, aa = 1.f / 1.0f;
        const float dx = 0.5f * h * aa, dy = 0.5f * h;
        vx[b][i] = body[b].xc + dx * a.cf.c[i];
        vy[b][i] = body[b].yc + dy * a.cf.s[i];
      }
      __syncthreads();
      if (threadIdx.x < 3 * kGeoVerts) {
        const int b = threadIdx.x / kGeoVerts, i = threadIdx.x - b * kGeoVerts, k2 = (i + 1) % kGeoVerts;
        body[b].edge[i] = make_edge(vx[b][i], vy[b][i], vx[b][k2], vy[b][k2]);
      } else if (threadIdx.x < 3 * kGeoVerts + 3) {   // bounding box Body.pde:73-87
        const int b = threadIdx.x - 3 * kGeoVerts;
        float lox = body[b].xc, loy = body[b].yc, hix = body[b].xc, hiy = body[b].yc;
        for (int i = 0; i < kGeoVerts; i++) {
          lox = gmin2(lox, vx[b][i]); loy = gmin2(loy, vy[b][i]);
          hix = gmax2(hix, vx[b][i]); hiy = gmax2(hiy, vy[b][i]);
        }
        const float bxs[4] = {lox, lox, hix, hix}, bys[4] = {loy, hiy, hiy, loy};
        for (int i = 0; i < 4; i++) body[b].box[i] = make_edge(bxs[i], bys[i], bxs[(i + 1) % 4], bys[(i + 1) % 4]);
      }
      __syncthreads();
      // Body.end's convexity test (Body.pde:90-96) of every body's 40-gon and box
      int bad = 0;
      constexpr int kPairs = kGeoVerts * kGeoVerts + 16;
      for (int t = threadIdx.x; t < 3 * kPairs; t += blockDim.x) {
        const int b = t / kPairs, u = t - b * kPairs;
        const bool poly = u < kGeoVerts * kGeoVerts;
        const GEdge* E = poly ? body[b].edge : body[b].box;
        const int N = poly ? kGeoVerts : 4, v = poly ? u : u - kGeoVerts * kGeoVerts, i = v / N, j = v - i * N;
        if (signed_dist(E[i], E[j].cx, E[j].cy) > 0.001f) bad = 1;
      }
      ok = !__syncthreads_or(bad);
    }
    if (ok) {
      // the band, counted without writing: no face on the lines next to the boundary, at most `cap` faces per component
      int cx = 0, cy = 0, line = 0;
      for (int t = threadIdx.x; t < cells; t += blockDim.x) {
        const int i = 1 + t / mj, j = 1 + t - (i - 1) * mj;
        float w[3], del, del1;
        const bool bx = x_face(body, i, j, w, del, del1), by = y_face(body, i, j, w, del, del1);
        cx += bx; cy += by;
        if ((bx || by) && (i <= 1 || i >= n - 2 || j <= 1 || j >= m - 2)) line = 1;
      }
      line = __syncthreads_or(line);
      nbx = block_sum(cx, &red);
      nby = block_sum(cy, &red);
      ok = !line && nbx <= a.cap && nby <= a.cap;
    }
    if (threadIdx.x == 0) {
      a.pr.status[e] = ok ? 1 : 2;
      a.pr.refused[e] = ok ? 0 : 1;
    }
    if (!ok) continue;
    // geometry slot e: the interior faces (geometry.cpp build_geometry), the band in band_lists' i-major order
    const size_t so = (size_t)e * a.stride;
    BandFace* bandx = a.band_x + (size_t)e * a.cap;
    BandFace* bandy = a.band_y + (size_t)e * a.cap;
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int offx = 0, offy = 0;
    for (int t0 = 0; t0 < cells; t0 += blockDim.x) {
      const int t = t0 + threadIdx.x;
      bool bx = false, by = false;
      BandFace fx, fy;
      if (t < cells) {
        const int i = 1 + t / mj, j = 1 + t - (i - 1) * mj;
        const size_t kk = so + (size_t)i * P + j;
        float w[3], del, del1;
        {  // x-face (i-1/2, j)
          const float x = (float)(i - 0.5), y = (float)j;
          bx = x_face(body, i, j, w, del, del1);
          a.del_x[kk] = del;
          a.w1_x[kk] = w[1]; a.w2_x[kk] = w[2];
          a.ry1_x[kk] = y - body[1].yc;      // PVector r=(x,y).sub(xc); Body.pde:236-238
          a.ry2_x[kk] = y - body[2].yc;
          if (bx) {
            float nx, ny;
            face_normal(body, x, y, w, nx, ny);
            fx = BandFace{i, j, del, del1, nx, ny};
          }
        }
        {  // y-face (i, j-1/2)
          const float x = (float)i, y = (float)(j - 0.5);
          by = y_face(body, i, j, w, del, del1);
          a.del_y[kk] = del;
          a.w1_y[kk] = w[1]; a.w2_y[kk] = w[2];
          a.rx1_y[kk] = x - body[1].xc;
          a.rx2_y[kk] = x - body[2].xc;
          if (by) {
            float nx, ny;
            face_normal(body, x, y, w, nx, ny);
            fy = BandFace{i, j, del, del1, nx, ny};
          }
        }
      }
      const unsigned mx = __ballot_sync(~0u, bx), my = __ballot_sync(~0u, by);
      if (lane == 0) { wsum[0][wid] = __popc(mx); wsum[1][wid] = __popc(my); }
      __syncthreads();
      int px = offx + __popc(mx & ((1u << lane) - 1)), py = offy + __popc(my & ((1u << lane) - 1));
      for (int v = 0; v < kSnapThreads / 32; v++) {
        if (v < (int)wid) { px += wsum[0][v]; py += wsum[1][v]; }
        offx += wsum[0][v]; offy += wsum[1][v];
      }
      if (bx) bandx[px] = fx;
      if (by) bandy[py] = fy;
      __syncthreads();
    }
    // the ghost ring: set_bc(del_x, btype 1, 1) and set_bc(del_y, btype 2, 1) resolved to the interior face each ghost
    // copies (before row 1 / column 1 are set); the basis fields keep their initial 0
    for (int t = threadIdx.x; t < 2 * m + 2 * (n - 2); t += blockDim.x) {
      int i, j;
      if (t < m) { i = 0; j = t; }
      else if (t < 2 * m) { i = n - 1; j = t - m; }
      else { const int u = t - 2 * m; i = 1 + (u >> 1); j = (u & 1) ? m - 1 : 0; }
      const size_t kk = so + (size_t)i * P + j;
      float dk[3], dx = 1.f, dy = 1.f;
      if (i != 1 && i != n - 1) {
        const int ii = i == 0 ? 1 : i, jj = j == 0 ? 1 : (j == m - 1 ? m - 2 : j);
        dx = mu0_dev(union_distance(body, (float)(ii - 0.5), (float)jj, dk), kGeoEps);
      }
      if (j != 1 && j != m - 1) {
        const int jj = j == 0 ? 1 : j, ii = i == 0 ? 1 : (i == n - 1 ? n - 2 : i);
        dy = mu0_dev(union_distance(body, (float)ii, (float)(jj - 0.5), dk), kGeoEps);
      }
      a.del_x[kk] = dx; a.del_y[kk] = dy;
      a.w1_x[kk] = 0.f; a.w2_x[kk] = 0.f; a.ry1_x[kk] = 0.f; a.ry2_x[kk] = 0.f;
      a.w1_y[kk] = 0.f; a.w2_y[kk] = 0.f; a.rx1_y[kk] = 0.f; a.rx2_y[kk] = 0.f;
    }
    if (threadIdx.x == 0) {
      a.env_slot[e] = e;
      if (a.lib.L) a.lib.env_set[e] = -1;
      a.env_nu[e] = D / q.re;                                                  // AFCCylinder.pde:34
      a.env_dRD[e] = q.dR * D;
      a.env_nbx[e] = nbx;
      a.env_nby[e] = nby;
      a.pr.params[e] = q;
      if (a.env_par) {
        const unsigned bits[5] = {(unsigned)q.re, __float_as_uint(q.dR), __float_as_uint(q.gR), __float_as_uint(q.theta),
                                  __float_as_uint(q.t_step)};
        for (int w = 0; w < 5; w++) a.env_par[(size_t)w * a.B + e] = bits[w];
      }
    }
    __syncthreads();   // (the shared bodies are rebuilt for the CTA's next pair)
  }
}

__global__ void __launch_bounds__(kSnapThreads) k_reset_params(const __grid_constant__ ResetParamsArgs a) {
  const int cpf = (a.nv + kSnapThreads * kSnapVec - 1) / (kSnapThreads * kSnapVec);   // chunks per field
  const int f = blockIdx.x / cpf, c = blockIdx.x - f * cpf;
  for (int k = blockIdx.y; k < a.npairs; k += gridDim.y) {
    if (!pair_applies(a.env, a.env, k, a.npairs, a.B, a.B, true)) continue;
    const int e = a.env[k];
    if (a.pr.status[e] != 1) continue;
    const float4* src = f == 0 ? a.iux : f == 1 ? a.iuy : a.ip;
    float4* dst = (f == 0 ? a.ux : f == 1 ? a.uy : a.p) + (size_t)e * a.stride4;
    copy_chunk(src, dst, c, a.nv);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      reset_scalars(a.sc, e, a.init_t, a.par[k].t_step * a.resolution, a.reset_acc, a.substeps);   // AFCCylinder.pde:20
      a.skip[e] = 0;
    }
  }
}

}  // namespace

int launch_reset_params(const SolverParams& q, const ParamLib& lib, const SnapSlots& snap, const ParamReset& pr,
                        const CircleFactors& cf, int nc, int mc, int cap, const float* init_ux, const float* init_uy,
                        const float* init_p, float init_t, float* ux, float* uy, const int* d_env,
                        const rlfc_env_params* d_par, int n, int reset_accumulators, int* skip, cudaStream_t st) {
  if (n <= 0) return 0;
  ResetParamsArgs a{};
  a.lib = lib;
  a.pr = pr;
  a.cf = cf;
  a.sc = q.sc;
  float** dst[10] = {&a.del_x, &a.del_y, &a.w1_x, &a.w2_x, &a.ry1_x, &a.ry2_x, &a.w1_y, &a.w2_y, &a.rx1_y, &a.rx2_y};
  const float* src[10] = {q.del_x, q.del_y, q.w1_x, q.w2_x, q.ry1_x, q.ry2_x, q.w1_y, q.w2_y, q.rx1_y, q.rx2_y};
  for (int f = 0; f < 10; f++) *dst[f] = const_cast<float*>(src[f]);
  a.band_x = const_cast<BandFace*>(q.band_x);
  a.band_y = const_cast<BandFace*>(q.band_y);
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
  a.stride = q.stride;
  a.stride4 = q.stride / 4;
  a.nv = q.n * q.P / 4;
  a.n = q.n; a.m = q.m; a.P = q.P;
  a.nc = nc; a.mc = mc;
  a.resolution = q.resolution;
  a.cap = cap;
  a.B = q.B;
  a.env = d_env;
  a.par = d_par;
  a.npairs = n;
  a.reset_acc = reset_accumulators;
  a.substeps = q.substeps;
  a.init_t = init_t;
  a.skip = skip;
  const unsigned ny = n < 65535 ? n : 65535;
  k_param_geometry<<<dim3(1, ny), kSnapThreads, 0, st>>>(a);
  const int cpf = (a.nv + kSnapThreads * kSnapVec - 1) / (kSnapThreads * kSnapVec);
  k_reset_params<<<dim3(3 * cpf, ny), kSnapThreads, 0, st>>>(a);
  return 2;
}

}  // namespace rlfc
