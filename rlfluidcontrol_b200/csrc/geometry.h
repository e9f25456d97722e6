// geometry.h -- host-side, once-per-handle precompute of everything that is constant for an
// AFCCylinder environment's life: BDIM kernel moments, wall normals, body-velocity basis, the
// Poisson coefficient hierarchy of the multigrid solver, and the pressure sample tables.
//
// Reference behaviour being reproduced (clientLilypad/): BDIM.get_coeffs BDIM.pde:132-196,
// BodyUnion.pde:67-92,145-166, Body.pde:215-240,386-417, OrthoNormal.pde:8-28,
// PoissonMatrix.pde:38-51, MG.pde:99-122, Body.pressForce Body.pde:296-303, Field.linear
// Field.pde:175-190, SaveScalar.pde:61-72.  The reference recomputes all of this every solver step
// whenever an action is non-zero (BDIM.pde:127); none of it depends on the action except the body
// velocity ub, which is linear in the two rotation increments and is evaluated on the device from
// the basis stored here.
#pragma once
#include <string>
#include <vector>

#include "../../include/rlfc.h"

namespace rlfc {

// One multigrid level in reference layout (n x m, i-major, ghosts included).
struct HostLevel {
  int n = 0, m = 0;
  std::vector<float> lx, ly, inv, diag;
};

// Bilinear sample point of Field.linear, pre-resolved to a cell and two fractions.
struct Sample {
  int i, j;
  float s, t;
};

// Field.linear's index/fraction part (Field.pde:175-190) for a field of the given btype (0 = p, 1 = u.x, 2 = u.y): the
// point clamped to [0.5, n-1.5] x [0.5, m-1.5], shifted by +0.5 in x (btype 1) or y (btype 2), truncated and capped at n-2 / m-2
Sample resolve_sample(int n, int m, float x0, float y0, int btype);

struct ForceEdge {    // one polygon edge of body 0: OrthoNormal {l, nx, ny, cen}
  Sample at;
  float l, nx, ny;
};

struct Geometry {
  int n = 0, m = 0;                 // array dims incl. ghost ring
  float dt = 0, nu = 0, D = 0, dR = 0, eps = 2.0f;
  int resolution = 0;
  // level-0 face fields, reference layout
  std::vector<float> del_x, del_y, del1_x, del1_y, wnx_x, wnx_y, wny_x, wny_y, c_x, c_y;
  // body-velocity basis: ub.x = (0 + ((0 - ry1*dphi1)/dt)*w1) + ((0 - ry2*dphi2)/dt)*w2 at x-faces,
  //                      ub.y = (0 + ((0 + rx1*dphi1)/dt)*w1) + ((0 + rx2*dphi2)/dt)*w2 at y-faces
  std::vector<float> w1_x, w2_x, ry1_x, ry2_x, w1_y, w2_y, rx1_y, rx2_y;
  std::vector<HostLevel> levels;    // levels[0] built from c = del*dt
  std::vector<ForceEdge> force_edges;   // 40 edges of the main cylinder
  std::vector<Sample> probes;           // 32 surface probes
  float mg_tol = 0;                 // MG.tol at level 0 (MG.pde:49-50)
};

// Builds the geometry for a configuration.  Returns 0 or an RLFC_E* code (err gets a message).  hierarchy = false leaves
// `levels` empty (and skips the grid checks that come with it): the per-environment geometries, whose hierarchy the device
// builds.
int build_geometry(const rlfc_config& cfg, Geometry& g, std::string& err, bool hierarchy = true);

// The factors cos(th_i), sin(th_i) of the 40 polygon vertex angles th_i = -TWO_PI*i/40 of every body, as build_geometry
// takes them (the device geometry builder, geometry_device.cuh, reads this table instead of evaluating them).
void circle_vertex_factors(float cos_th[40], float sin_th[40]);

// Checkpoint IO (BDIM.write / BDIM.resume text format BDIM.pde:226-251, and the .bdimb binary form).
int read_checkpoint(const std::string& path, int n, int m, float& t, float& dt,
                    std::vector<float>& ux, std::vector<float>& uy, std::vector<float>& p, std::string& err);
// java.lang.Float.toString(v): the text form the reference writes into checkpoints, traces and RPC payloads
std::string format_float_java(float v);
int write_bdim_text(const std::string& path, int n, int m, float t, float dt,
                    const float* ux, const float* uy, const float* p, std::string& err);

}  // namespace rlfc
