// geometry.cpp -- see geometry.h.  Host arithmetic follows Java `float` semantics: one binary32
// rounding per operation (this file must be compiled without FMA contraction), sin/cos/sqrt taken
// in double and narrowed (Processing's PApplet wrappers over java.lang.Math).
#include "geometry.h"

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace rlfc {
namespace {

constexpr float kPi = 3.1415927f;     // PConstants.PI
constexpr float kTwoPi = 6.2831855f;  // PConstants.TWO_PI
constexpr int kCircleVerts = 40;      // EllipseBody.m, Body.pde:384
// MG.divisible's message before its exit() (MG.pde:101-104)
constexpr const char* kMgExitMessage =
    "MultiGrid requires the size in each direction be a large factor of two (2^p) times a small number (N=1..9)";

inline float fsin(float x) { return (float)std::sin((double)x); }
inline float fcos(float x) { return (float)std::cos((double)x); }
inline float fmin2(float a, float b) { return (a < b) ? a : b; }   // PApplet.min
inline float fmax2(float a, float b) { return (a > b) ? a : b; }   // PApplet.max

// ---- OrthoNormal.pde:8-28 -----------------------------------------------------------------
struct Edge {
  float l, nx, ny, tx, ty, off, cx, cy;
  Edge() : l(0), nx(0), ny(0), tx(0), ty(0), off(0), cx(0), cy(0) {}
  Edge(float ax, float ay, float bx, float by) {
    float sx = ax - bx, sy = ay - by, sz = 0.f;
    l = (float)std::sqrt((double)(sx * sx + sy * sy + sz * sz));   // PVector.mag
    tx = (bx - ax) / l;
    ty = (by - ay) / l;
    nx = -ty;
    ny = tx;
    off = ax * nx + ay * ny;
    cx = (ax + bx) / 2.f;
    cy = (ay + by) / 2.f;
  }
  float signed_dist(float x, float y) const { return x * nx + y * ny - off; }
};

// ---- CircleBody (Body.pde:386-417): 40-gon used for normals / force, analytic circle for SDF ----
struct Cylinder {
  float xc, yc, h;
  Edge edge[kCircleVerts];
  Edge box[4];

  Cylinder(float x, float y, float d) : xc(x), yc(y), h(d) {
    float vx[kCircleVerts], vy[kCircleVerts];
    float a = 1.f / 1.0f;
    float dx = 0.5f * h * a, dy = 0.5f * h;
    for (int i = 0; i < kCircleVerts; i++) {
      float th = -kTwoPi * i / ((float)kCircleVerts);
      vx[i] = xc + dx * fcos(th);
      vy[i] = yc + dy * fsin(th);
    }
    for (int i = 0; i < kCircleVerts; i++) {
      int k = (i + 1) % kCircleVerts;
      edge[i] = Edge(vx[i], vy[i], vx[k], vy[k]);
    }
    // bounding box Body.pde:73-87
    float lox = xc, loy = yc, hix = xc, hiy = yc;
    for (int i = 0; i < kCircleVerts; i++) {
      lox = fmin2(lox, vx[i]); loy = fmin2(loy, vy[i]);
      hix = fmax2(hix, vx[i]); hiy = fmax2(hiy, vy[i]);
    }
    const float bxs[4] = {lox, lox, hix, hix}, bys[4] = {loy, hiy, hiy, loy};
    for (int i = 0; i < 4; i++) box[i] = Edge(bxs[i], bys[i], bxs[(i + 1) % 4], bys[(i + 1) % 4]);
  }

  // Body.end's convexity test Body.pde:90-96 for an edge set
  template <int N>
  static bool convex(const Edge (&e)[N]) {
    for (int i = 0; i < N; i++)
      for (int j = 0; j < N; j++)
        if (e[i].signed_dist(e[j].cx, e[j].cy) > 0.001f) return false;
    return true;
  }

  // CircleBody.distance Body.pde:408-410
  float distance(float x, float y) const {
    float ax = x - xc, ay = y - yc;
    return (float)std::sqrt((double)(ax * ax + ay * ay)) - 0.5f * h;
  }
  // Body.distance on the (convex, 4-point) bounding box Body.pde:181-185
  float box_distance(float x, float y) const {
    float dis = -1e10f;
    for (int i = 0; i < 4; i++) dis = fmax2(dis, box[i].signed_dist(x, y));
    return dis;
  }
  // Body.WallNormal Body.pde:215-232 (faceted: normal of the edge with the largest signed distance)
  void wall_normal(float x, float y, float& ox, float& oy) const {
    ox = 0; oy = 0;
    if (box_distance(x, y) > 3) return;
    float best = -1e10f;
    for (int i = 0; i < kCircleVerts; i++) {
      float d2 = edge[i].signed_dist(x, y);
      if (d2 > best) { best = d2; ox = edge[i].nx; oy = edge[i].ny; }
    }
  }
};

// BodyUnion.delta0 BodyUnion.pde:158-166
float union_kernel(float d) {
  if (d <= -1) return 0;
  if (d >= 1) return 1;
  return 0.5f * (1.f + d + fsin(kPi * d) / kPi);
}
// BDIM.delta0 BDIM.pde:199-207
float mu0(float d, float eps) {
  if (d <= -eps) return 0;
  if (d >= eps) return 1;
  return 0.5f * (1.f + d / eps + fsin(kPi * d / eps) / kPi);
}
// BDIM.delta1 BDIM.pde:209-215
float mu1(float d, float eps) {
  float ad = (d < 0) ? -d : d;
  if (ad >= eps) return 0;
  return 0.25f * (eps - (d * d) / eps) - 1 / kTwoPi * (d * fsin(d * kPi / eps) + eps / kPi * (1 + fcos(d * kPi / eps)));
}

struct FacePoint {   // everything BDIM.get_coeffs evaluates at one face location
  float dist, w[3], nx, ny;
};

FacePoint eval_face(const Cylinder* const body[3], float x, float y) {
  FacePoint f;
  // BodyUnion.distance BodyUnion.pde:67-72
  float dmin = 1e6f;
  float dk[3];
  for (int k = 0; k < 3; k++) { dk[k] = body[k]->distance(x, y); dmin = fmin2(dmin, dk[k]); }
  f.dist = dmin;
  // BodyUnion.get_weights BodyUnion.pde:145-156
  float s = 0;
  for (int k = 0; k < 3; k++) { f.w[k] = union_kernel(-dk[k] / 3.f); s += f.w[k]; }
  for (int k = 0; k < 3 && s > 0; k++) f.w[k] /= s;
  // BodyUnion.WallNormal BodyUnion.pde:74-82
  f.nx = 0; f.ny = 0;
  for (int k = 0; k < 3; k++) {
    float ax, ay;
    body[k]->wall_normal(x, y, ax, ay);
    f.nx += ax * f.w[k];
    f.ny += ay * f.w[k];
  }
  return f;
}

// Field.setBC for a non-gradientExit field (Field.pde:209-229) on a plain array
void set_bc(std::vector<float>& a, int n, int m, int btype, float bval) {
  auto at = [&](int i, int j) -> float& { return a[(size_t)i * m + j]; };
  for (int j = 0; j < m; j++) {
    at(0, j) = at(1, j);
    at(n - 1, j) = at(n - 2, j);
    if (btype == 1) { at(1, j) = bval; at(n - 1, j) = bval; }
  }
  for (int i = 0; i < n; i++) {
    at(i, 0) = at(i, 1);
    at(i, m - 1) = at(i, m - 2);
    if (btype == 2) { at(i, 1) = bval; at(i, m - 1) = bval; }
  }
}

// PoissonMatrix ctor PoissonMatrix.pde:38-51
void finish_level(HostLevel& L) {
  const int n = L.n, m = L.m;
  L.diag.assign((size_t)n * m, 0.f);
  L.inv.assign((size_t)n * m, 1.f);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      size_t k = (size_t)i * m + j;
      float sumd = L.lx[k] + L.lx[k + m] + L.ly[k] + L.ly[k + 1];
      L.diag[k] = -sumd;
      if (sumd > 1e-5f) L.inv[k] = -1.f / sumd;
    }
}

// MG.restrict(PoissonMatrix) MG.pde:108-122
HostLevel coarsen(const HostLevel& F) {
  HostLevel C;
  C.n = (F.n - 2) / 2 + 2;
  C.m = (F.m - 2) / 2 + 2;
  C.lx.assign((size_t)C.n * C.m, 0.f);
  C.ly.assign((size_t)C.n * C.m, 0.f);
  for (int i = 1; i < C.n - 1; i++)
    for (int j = 1; j < C.m - 1; j++) {
      int ii = (i - 1) * 2 + 1, jj = (j - 1) * 2 + 1;
      size_t kf = (size_t)ii * F.m + jj;
      C.lx[(size_t)i * C.m + j] = (F.lx[kf] + F.lx[kf + 1]) * 0.5f;
      C.ly[(size_t)i * C.m + j] = (F.ly[kf] + F.ly[kf + F.m]) * 0.5f;
    }
  set_bc(C.lx, C.n, C.m, 1, 0.f);
  set_bc(C.ly, C.n, C.m, 2, 0.f);
  finish_level(C);
  return C;
}

}  // namespace

void circle_vertex_factors(float cos_th[40], float sin_th[40]) {
  for (int i = 0; i < kCircleVerts; i++) {
    const float th = -kTwoPi * i / ((float)kCircleVerts);   // as Cylinder's constructor
    cos_th[i] = fcos(th);
    sin_th[i] = fsin(th);
  }
}

Sample resolve_sample(int n, int m, float x0, float y0, int btype) {
  Sample sp;
  float x = fmin2(fmax2(0.5f, x0), n - 1.5f);
  if (btype == 1) x += 0.5f;
  int i = (int)x; if (i > n - 2) i = n - 2;
  float y = fmin2(fmax2(0.5f, y0), m - 1.5f);
  if (btype == 2) y += 0.5f;
  int j = (int)y; if (j > m - 2) j = m - 2;
  sp.i = i; sp.j = j; sp.s = x - i; sp.t = y - j;
  return sp;
}

int build_geometry(const rlfc_config& cfg, Geometry& g, std::string& err, bool hierarchy) {
  if (cfg.resolution < 2 || cfg.x_lengths < 1 || cfg.y_lengths < 1 || cfg.re <= 0) {
    err = "resolution/x_lengths/y_lengths/re must be positive";
    return RLFC_EINVAL;
  }
  const int nc = cfg.x_lengths * cfg.resolution, mc = cfg.y_lengths * cfg.resolution;   // AFCCylinder.pde:12-13
  const int n = nc + 2, m = mc + 2;                                                     // BDIM.pde:42
  if (nc % 2 != 0 || mc % 2 != 0) {
    // the finest level always restricts (MG.pde:70-72): MG.prolongate (MG.pde:139-152) then builds an even-sized
    // correction and MG.increment (MG.pde:94-97) adds it over the whole odd-sized fine field, past its end.  The coarse
    // levels' MG.divisible (MG.pde:101-104) runs first, inside vCycle: where it would exit(), report that instead.
    err = "level 0 must have an even number of cells in each direction (" + std::to_string(nc) + "x" + std::to_string(mc) +
          "): MG.prolongate / MG.increment cannot correct an odd grid";
    for (int cn = n, cm = m;;) {
      cn = (cn - 2) / 2 + 2; cm = (cm - 2) / 2 + 2;                                     // MG.pde:108-122
      if ((cn - 2) % 2 == 0 && (cm - 2) % 2 == 0 && cn > 4 && cm > 4) continue;
      if (cn > 9 && cm > 9) err = kMgExitMessage;
      break;
    }
    return RLFC_EGRID;
  }
  g.n = n; g.m = m;
  g.resolution = cfg.resolution;
  g.D = (float)cfg.resolution;                                                          // AFCCylinder.pde:27
  g.dR = cfg.dR;
  g.dt = cfg.t_step * cfg.resolution;                                                   // AFCCylinder.pde:20
  g.nu = (float)g.D / cfg.re;                                                           // AFCCylinder.pde:34
  g.eps = 2.0f;                                                                         // BDIM.pde:35
  const float D = g.D;
  // AFCCylinder.pde:29-32
  float r = (D / 2 + cfg.gR * D + cfg.dR * D / 2);
  Cylinder main_cyl((float)(nc / 4), (float)(mc / 2), D);
  Cylinder ctl_lo(nc / 4 + r * fcos(cfg.theta), mc / 2 - r * fsin(cfg.theta), cfg.dR * D);
  Cylinder ctl_hi(nc / 4 + r * fcos(cfg.theta), mc / 2 + r * fsin(cfg.theta), cfg.dR * D);
  const Cylinder* body[3] = {&main_cyl, &ctl_lo, &ctl_hi};
  for (int k = 0; k < 3; k++)
    if (!Cylinder::convex(body[k]->edge) || !Cylinder::convex(body[k]->box)) {
      err = "polygon convexity test failed (Body.pde:90-96); non-convex bodies are not supported";
      return RLFC_EINVAL;
    }

  const size_t N = (size_t)n * m;
  // field initial values follow the BDIM ctor BDIM.pde:57-64: del=1, del1=0, wn=0, ub=0
  g.del_x.assign(N, 1.f); g.del_y.assign(N, 1.f);
  g.del1_x.assign(N, 0.f); g.del1_y.assign(N, 0.f);
  for (auto* v : {&g.wnx_x, &g.wnx_y, &g.wny_x, &g.wny_y, &g.w1_x, &g.w2_x, &g.ry1_x, &g.ry2_x,
                  &g.w1_y, &g.w2_y, &g.rx1_y, &g.rx2_y})
    v->assign(N, 0.f);

  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      const size_t k = (size_t)i * m + j;
      {  // x-face (i-1/2, j)
        const float x = (float)(i - 0.5), y = (float)j;
        FacePoint f = eval_face(body, x, y);
        g.del_x[k] = mu0(f.dist, g.eps);
        g.del1_x[k] = mu1(f.dist, g.eps);
        g.wnx_x[k] = f.nx; g.wny_x[k] = f.ny;
        g.w1_x[k] = f.w[1]; g.w2_x[k] = f.w[2];
        g.ry1_x[k] = y - ctl_lo.yc;      // PVector r=(x,y).sub(xc); Body.pde:236-238
        g.ry2_x[k] = y - ctl_hi.yc;
      }
      {  // y-face (i, j-1/2)
        const float x = (float)i, y = (float)(j - 0.5);
        FacePoint f = eval_face(body, x, y);
        g.del_y[k] = mu0(f.dist, g.eps);
        g.del1_y[k] = mu1(f.dist, g.eps);
        g.wnx_y[k] = f.nx; g.wny_y[k] = f.ny;
        g.w1_y[k] = f.w[1]; g.w2_y[k] = f.w[2];
        g.rx1_y[k] = x - ctl_lo.xc;
        g.rx2_y[k] = x - ctl_hi.xc;
      }
    }
  set_bc(g.del_x, n, m, 1, 1.f); set_bc(g.del_y, n, m, 2, 1.f);     // BDIM.pde:183
  set_bc(g.del1_x, n, m, 1, 0.f); set_bc(g.del1_y, n, m, 2, 0.f);   // BDIM.pde:195

  // c = del * (rhoi * dt) with rhoi == 1 everywhere (BDIM.pde:59-61,81)
  g.c_x.resize(N); g.c_y.resize(N);
  for (size_t k = 0; k < N; k++) {
    g.c_x[k] = g.del_x[k] * (1.f * g.dt);
    g.c_y[k] = g.del_y[k] * (1.f * g.dt);
  }

  // multigrid hierarchy (MG.pde:68-77,99-122): the finest level always restricts; a coarse level
  // recurses only while divisible
  g.levels.clear();
  if (hierarchy) {
  {
    HostLevel L0;
    L0.n = n; L0.m = m; L0.lx = g.c_x; L0.ly = g.c_y;
    finish_level(L0);
    g.levels.push_back(std::move(L0));
  }
  for (;;) {
    const HostLevel& F = g.levels.back();
    bool divisible = (F.n - 2) % 2 == 0 && (F.m - 2) % 2 == 0 && F.n > 4 && F.m > 4;
    if (g.levels.size() == 1) {
      if ((F.n - 2) < 2 || (F.m - 2) < 2) { err = "grid too small for multigrid"; return RLFC_EGRID; }
    } else if (!divisible) {
      if (F.n > 9 && F.m > 9) {
        err = kMgExitMessage;
        return RLFC_EGRID;   // MG.pde:101-104 would exit()
      }
      break;
    }
    g.levels.push_back(coarsen(F));
  }
  }

  // MG.tol MG.pde:49-50: inner product of a field of 1e-4f with itself (float products, double sum)
  {
    double s = 0;
    const float prod = 1e-4f * 1e-4f;
    for (int i = 1; i < n - 1; i++)
      for (int j = 1; j < m - 1; j++) s += prod;
    g.mg_tol = (float)s;
  }

  // Body.pressForce sample table for body 0 (Body.pde:296-303)
  g.force_edges.clear();
  for (int e = 0; e < kCircleVerts; e++) {
    const Edge& o = main_cyl.edge[e];
    ForceEdge fe;
    fe.at = resolve_sample(n, m, o.cx, o.cy, 0);
    fe.l = o.l; fe.nx = o.nx; fe.ny = o.ny;
    g.force_edges.push_back(fe);
  }
  // SaveScalar probes SaveScalar.pde:28-41,61-72
  g.probes.clear();
  {
    const float res = (float)cfg.resolution;
    const float nf = (float)cfg.x_lengths * res, mf = (float)cfg.y_lengths * res;
    const float cx = nf / 4, cy = mf / 2;
    for (int i = 0; i < RLFC_NUM_PROBES; i++) {
      float xp = fcos((float)i / RLFC_NUM_PROBES * kPi * 2) * res / 2 + cx;
      float yp = fsin((float)i / RLFC_NUM_PROBES * kPi * 2) * res / 2 + cy;
      g.probes.push_back(resolve_sample(n, m, xp, yp, 0));
    }
  }
  return RLFC_OK;
}

// ---- checkpoints -------------------------------------------------------------------------------

int read_checkpoint(const std::string& path, int n, int m, float& t, float& dt, std::vector<float>& ux,
                    std::vector<float>& uy, std::vector<float>& p, std::string& err) {
  FILE* f = std::fopen(path.c_str(), "rb");
  if (!f) { err = "cannot open " + path; return RLFC_EIO; }
  const size_t N = (size_t)n * m;
  ux.resize(N); uy.resize(N); p.resize(N);
  char magic[8];
  size_t got = std::fread(magic, 1, 8, f);
  if (got == 8 && !std::memcmp(magic, "RLFCBDIM", 8)) {
    int32_t hdr[2]; float th[2];
    bool ok = std::fread(hdr, 4, 2, f) == 2 && std::fread(th, 4, 2, f) == 2;
    if (ok && (hdr[0] != n || hdr[1] != m)) {
      std::fclose(f);
      err = "checkpoint grid " + std::to_string(hdr[0]) + "x" + std::to_string(hdr[1]) + " does not match " +
            std::to_string(n) + "x" + std::to_string(m);
      return RLFC_EIO;
    }
    ok = ok && std::fread(ux.data(), 4, N, f) == N && std::fread(uy.data(), 4, N, f) == N &&
         std::fread(p.data(), 4, N, f) == N;
    std::fclose(f);
    if (!ok) { err = "truncated binary checkpoint " + path; return RLFC_EIO; }
    t = th[0]; dt = th[1];
    return RLFC_OK;
  }
  // text form: line 0 t, line 1 dt, then "ux, uy, p" per cell, i-major (BDIM.pde:226-251)
  std::rewind(f);
  char line[512];
  auto next = [&]() { return std::fgets(line, sizeof line, f) != nullptr; };
  if (!next()) { std::fclose(f); err = "empty checkpoint " + path; return RLFC_EIO; }
  t = std::strtof(line, nullptr);
  if (!next()) { std::fclose(f); err = "truncated checkpoint " + path; return RLFC_EIO; }
  dt = std::strtof(line, nullptr);
  for (size_t k = 0; k < N; k++) {
    if (!next()) { std::fclose(f); err = "checkpoint " + path + " has too few lines for the grid"; return RLFC_EIO; }
    char* q = line; char* end;
    float v[3];
    for (int c = 0; c < 3; c++) {
      v[c] = std::strtof(q, &end);
      if (end == q) { std::fclose(f); err = "malformed line in " + path; return RLFC_EIO; }
      q = end;
      while (*q == ',' || *q == ' ') q++;
    }
    // BDIM.write puts exactly three numbers on a line: anything behind them means another format
    while (*q == '\r' || *q == '\n' || *q == ' ' || *q == '\t') q++;
    if (*q) { std::fclose(f); err = "trailing data on a line of " + path; return RLFC_EIO; }
    ux[k] = v[0]; uy[k] = v[1]; p[k] = v[2];
  }
  // ... and exactly n*m cell lines: a checkpoint of a larger grid would otherwise be accepted with its rows reinterpreted
  while (next()) {
    const char* q = line;
    while (*q == '\r' || *q == '\n' || *q == ' ' || *q == '\t') q++;
    if (*q) {
      std::fclose(f);
      err = "checkpoint " + path + " has more lines than the " + std::to_string(n) + "x" + std::to_string(m) + " grid";
      return RLFC_EIO;
    }
  }
  std::fclose(f);
  return RLFC_OK;
}

namespace {
// java.lang.Float.toString: shortest decimal that round-trips; plain notation for
// 1e-3 <= |x| < 1e7 (at least one fractional digit), otherwise d.dddE[-]n.
std::string java_float(float v) {
  if (v != v) return "NaN";
  if (v == 0) return std::signbit(v) ? "-0.0" : "0.0";
  if (std::isinf(v)) return v > 0 ? "Infinity" : "-Infinity";
  char buf[64];
  int prec = 1;
  for (; prec <= 9; prec++) {
    std::snprintf(buf, sizeof buf, "%.*e", prec - 1, (double)v);
    if (std::strtof(buf, nullptr) == v) break;
  }
  // buf = [-]d.ddde[+-]xx
  std::string s(buf);
  size_t epos = s.find('e');
  int ex = std::atoi(s.c_str() + epos + 1);
  std::string mant = s.substr(0, epos);
  bool neg = mant[0] == '-';
  if (neg) mant.erase(0, 1);
  std::string digits;
  for (char ch : mant) if (ch != '.') digits.push_back(ch);
  std::string out;
  float av = v < 0 ? -v : v;
  if (av >= 1e-3f && av < 1e7f) {
    if (ex >= 0) {
      std::string ip = digits.substr(0, std::min((size_t)ex + 1, digits.size()));
      while ((int)ip.size() < ex + 1) ip.push_back('0');
      std::string fp = (int)digits.size() > ex + 1 ? digits.substr(ex + 1) : "0";
      out = ip + "." + fp;
    } else {
      out = "0." + std::string(-ex - 1, '0') + digits;
    }
  } else {
    std::string fp = digits.size() > 1 ? digits.substr(1) : "0";
    out = digits.substr(0, 1) + "." + fp + "E" + std::to_string(ex);
  }
  return neg ? "-" + out : out;
}
}  // namespace

std::string format_float_java(float v) { return java_float(v); }

int write_bdim_text(const std::string& path, int n, int m, float t, float dt, const float* ux, const float* uy,
                    const float* p, std::string& err) {
  FILE* f = std::fopen(path.c_str(), "w");
  if (!f) { err = "cannot create " + path; return RLFC_EIO; }
  std::fprintf(f, "%s\n%s\n", java_float(t).c_str(), java_float(dt).c_str());
  for (size_t k = 0; k < (size_t)n * m; k++)
    std::fprintf(f, "%s, %s, %s\n", java_float(ux[k]).c_str(), java_float(uy[k]).c_str(), java_float(p[k]).c_str());
  if (std::fclose(f) != 0) { err = "write failed for " + path; return RLFC_EIO; }
  return RLFC_OK;
}

}  // namespace rlfc
