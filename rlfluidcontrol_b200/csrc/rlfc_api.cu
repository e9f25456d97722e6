// rlfc_api.cu -- the C ABI of include/rlfc.h: handle lifetime, host orchestration of one solver step
// (AFCCylinder.update2, AFCCylinder.pde:45-61) and of one RL step (clientCFD.draw, clientCFD.pde:35-55).
// There is no CPU fallback anywhere in this file: every numerical operation is a CUDA kernel of
// solver_kernels.cu; the host only sequences launches and moves the caller's buffers.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rlfc.h"
#include "geometry.h"
#include "solver.h"
#include "smooth_rows.cuh"
#include "vmm.h"

using namespace rlfc;

namespace {
thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t _e = (call);                                                                           \
    if (_e != cudaSuccess)                                                                             \
      return fail(RLFC_ECUDA, std::string(#call) + ": " + cudaGetErrorString(_e));                     \
  } while (0)

inline int round_up(int v, int a) { return (v + a - 1) / a * a; }
}  // namespace

struct rlfc_env {
  rlfc_config cfg{};
  std::string init_path;
  Geometry geo;
  SolverParams sp{};
  // per-environment constructor arguments (rlfc_config.env_params): env_mode = the handle was created with them
  bool env_mode = false;
  std::vector<rlfc_env_params> params;     // [B]
  std::vector<float> dt0;                  // [B] t_step*resolution: sc.dt after a reset, the fixed dt without adaptive_dt
  std::vector<float> h_nu, h_dRD;          // [B] host copies of sp.env_nu, sp.env_dRD
  std::vector<int> h_nbx, h_nby;           // [B] host copies of sp.env_nband_x / y
  int* d_skip = nullptr;                   // [B] mask of launch_poisson_rebuild* outside a step (1 = keep)
  SnapSlots snap{};                        // rlfc_config.n_snapshots slots (snap.S = 0: none)
  int *snap_env = nullptr, *snap_slot = nullptr;   // [max(B, S)] the pairs of a host snapshot / restore call
  SensorSet sens{};                        // rlfc_config.sensors of the whole batch (sens.n = 0: none)
  std::vector<rlfc_sensor> sensor_table;   // rlfc_config.sensors as given (what a record's sensor table holds)
  FlowStats fs{};                          // rlfc_config.stats_every of the whole batch (fs.every = 0: none)
  // state records (records.cuh): nothing is allocated before the first record call (rec.refused = nullptr until then)
  RecordBufs rec{};
  std::vector<void*> rec_bufs;             // rec's growing scratch, its id buffer and the host calls' staging buffer
  size_t rec_pairs = 0, rec_partials = 0, rec_id_cap = 0, rec_stage_bytes = 0;
  int* rec_ids = nullptr;                  // [rec_pairs] the ids of a host export / import call
  unsigned char* rec_stage = nullptr;      // the records of a host export / import call
  // parameter library (rlfc_config.param_sets; lib.L = 0: none)
  ParamLib lib{};
  std::vector<rlfc_env_params> lib_params; // [L] the sets as given
  std::vector<LibSet> h_lib;               // [L] host copy of lib.sets
  std::vector<int> h_env_set;              // [B] host copy of lib.env_set as of the last sync_env_sets
  int *set_env = nullptr, *set_ids = nullptr;   // [B] the pairs of a host rlfc_env_reset_sets call
  // device parameter resets (rlfc_env_reset_params_device; per-environment handles)
  ParamReset pr{};
  CircleFactors circle{};                  // the 40 polygon vertex factors the device builder reads
  bool par_pending = false;                // a device parameter reset was enqueued since the last sync_env_sets
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::vector<void*> allocs;               // every cudaMalloc, freed in destroy
  // velocity buffers (see solver.h)
  float *uAx = nullptr, *uAy = nullptr, *uBx = nullptr, *uBy = nullptr, *uCx = nullptr, *uCy = nullptr;
  // initial state in pitched device layout (one env) for fast batched reset
  float *init_ux = nullptr, *init_uy = nullptr, *init_p = nullptr;
  float* pB = nullptr;                       // second pressure buffer (solver.h: k_resid_down0 / k_project_shift)
  float init_t = 0, init_dt = 0;
  // staging
  float *d_actions = nullptr, *d_obs = nullptr, *d_reward = nullptr;
  int* d_done = nullptr;
  float *h_actions = nullptr, *h_obs = nullptr, *h_reward = nullptr, *h_force = nullptr, *h_probes = nullptr;
  int *h_done = nullptr, *h_any = nullptr;
  long long launches = 0;
  long long mg_iter_launch_rounds = 0;
  unsigned long long* chain_tickets = nullptr;   // [views][kMaxLevels] (smooth_chain.cuh)
  // Environment groups: the batch is split into contiguous groups, each advanced by its own stream (and its own
  // CUDA graphs), so the latency-bound per-env kernels of one group overlap the bandwidth-bound kernels of another.
  struct Group {
    int e0 = 0, B = 0;
    SolverParams sp{};                       // view of the batch arrays restricted to [e0, e0 + B); lev[0].x = pressure buffer A
    SolverParams spB{};                      // same view with lev[0].x = pressure buffer B (p ping-pongs A -> B -> A per half step)
    SensorSet sens{};                        // the view's sensors (out at e0 * n)
    FlowStats fs{};                          // the view's flow statistics (at environment e0)
    float *uAx = nullptr, *uAy = nullptr, *uBx = nullptr, *uBy = nullptr, *uCx = nullptr, *uCy = nullptr;
    cudaStream_t st = nullptr;               // group 0 runs on the handle's stream
    cudaEvent_t done = nullptr;
    cudaGraphExec_t step_graph[2] = {nullptr, nullptr};   // [accumulate]
    long long graph_launches = 0;            // kernel nodes of one replay outside the MG loops' WHILE bodies
  };
  std::vector<Group> groups;
  Group whole;                               // the entire batch on the handle's stream (eager / profiled path; slab mode:
                                             // the whole domain as device 0 sees it alone)
  // Slab mode (cfg.n_devices > 1, BASELINE config 5): one domain advanced by several devices over one shared address
  // range (vmm.h); every device runs the same kernel sequence on its row blocks / strips, a barrier between kernels
  struct SlabDev {
    int device = 0;
    cudaStream_t st = nullptr;
    SolverParams sp{}, spB{};                // this device's view (slab_rank, its strips, its ticket counters); B: lev[0].x = pressure buffer B
    SlabBarrier bar{};
    void* local[2] = {nullptr, nullptr};     // cudaMalloc'd on this device: ticket counters, barrier epoch
  };
  std::vector<SlabDev> slab;
  VmmPool vmm;
  bool home_only = false;                    // dmalloc: keep the next allocations on device 0 (data only it touches)
  long long slab_barriers = 0;
  cudaStream_t aux_stream = nullptr;         // used to capture the bodies of the conditional nodes
  cudaEvent_t fork_ev = nullptr;
  bool use_graph = true;
  // optional per-kernel CUDA-event timing (rlfc_env_set_profiling)
  bool profiling = false;
  struct ProfRec { int id; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> event_pool;
  struct ProfAgg { std::string name; double ms = 0; long long count = 0; double floats_per_cell = 0; };
  std::vector<ProfAgg> prof;

  int prof_id(const char* name, double floats_per_cell) {
    for (size_t k = 0; k < prof.size(); k++) if (prof[k].name == name) return (int)k;
    prof.push_back({name, 0.0, 0, floats_per_cell});
    return (int)prof.size() - 1;
  }
  cudaEvent_t get_event() {
    if (!event_pool.empty()) { cudaEvent_t e = event_pool.back(); event_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
  // run one kernel launch, optionally bracketed by events on the handle's stream
  template <typename F>
  void run(const char* name, double floats_per_cell, F&& launch, cudaStream_t st = nullptr) {
    if (!profiling) { launches += launch(); return; }
    if (!st) st = stream;
    ProfRec r{prof_id(name, floats_per_cell), get_event(), get_event()};
    cudaEventRecord(r.e0, st);
    launches += launch();
    cudaEventRecord(r.e1, st);
    prof_recs.push_back(r);
  }
  void prof_collect() {
    if (prof_recs.empty()) return;
    cudaStreamSynchronize(stream);
    for (auto& G : groups) if (G.st) cudaStreamSynchronize(G.st);
    for (auto& r : prof_recs) {
      float ms = 0;
      cudaEventElapsedTime(&ms, r.e0, r.e1);
      prof[r.id].ms += ms; prof[r.id].count++;
      event_pool.push_back(r.e0); event_pool.push_back(r.e1);
    }
    prof_recs.clear();
  }

  template <typename T>
  int dmalloc(T** p, size_t count, bool zero = true) {
    void* q = nullptr;
    cudaError_t e;
    if (cfg.n_devices > 1) {                 // slab mode: visible to every device at this address, striped over them
      std::string err;
      int rc = vmm.alloc(&q, std::max<size_t>(count, 1) * sizeof(T), !home_only, 0, err);
      if (rc) return fail(rc, err);
    } else {
      e = cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T));
      if (e != cudaSuccess) return fail(RLFC_ENOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
      allocs.push_back(q);
    }
    if (zero) {
      e = cudaMemsetAsync(q, 0, std::max<size_t>(count, 1) * sizeof(T), stream);
      if (e != cudaSuccess) return fail(RLFC_ECUDA, std::string("cudaMemset: ") + cudaGetErrorString(e));
    }
    *p = (T*)q;
    return RLFC_OK;
  }
};

namespace {

// reference layout (n x m) -> pitched (n x P), padding zeroed
std::vector<float> to_pitched(const float* a, int n, int m, int P) {
  std::vector<float> out((size_t)n * P, 0.f);
  for (int i = 0; i < n; i++) std::memcpy(&out[(size_t)i * P], &a[(size_t)i * m], sizeof(float) * m);
  return out;
}

int upload_static(rlfc_env* E, const std::vector<float>& host, int n, int m, int P, const float** dst) {
  float* d = nullptr;
  int rc = E->dmalloc(&d, (size_t)n * P, false);
  if (rc) return rc;
  std::vector<float> pit = to_pitched(host.data(), n, m, P);
  CU(cudaMemcpyAsync(d, pit.data(), pit.size() * sizeof(float), cudaMemcpyHostToDevice, E->stream));
  CU(cudaStreamSynchronize(E->stream));   // `pit` dies at scope exit
  *dst = d;
  return RLFC_OK;
}

template <typename T>
int upload_vec(rlfc_env* E, const std::vector<T>& host, const T** dst) {
  T* d = nullptr;
  int rc = E->dmalloc(&d, host.size(), false);
  if (rc) return rc;
  if (!host.empty()) {
    CU(cudaMemcpyAsync(d, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice, E->stream));
    CU(cudaStreamSynchronize(E->stream));
  }
  *dst = d;
  return RLFC_OK;
}

// copy one pitched field into env slot(s)
int broadcast_field(rlfc_env* E, float* batch, const float* one, const int* ids, int nids) {
  const SolverParams& sp = E->sp;
  const size_t bytes = (size_t)sp.n * sp.P * sizeof(float);
  for (int k = 0; k < nids; k++) {
    int e = ids ? ids[k] : k;
    CU(cudaMemcpyAsync(batch + (size_t)e * sp.stride, one, bytes, cudaMemcpyDeviceToDevice, E->stream));
  }
  return RLFC_OK;
}

// ---- per-environment geometry (rlfc_config.env_params) ----

rlfc_env_params params_of(const rlfc_config& c) { return rlfc_env_params{c.re, c.dR, c.gR, c.theta, c.t_step}; }

bool same_params(const rlfc_env_params& a, const rlfc_env_params& b) {
  return a.re == b.re && !std::memcmp(&a.dR, &b.dR, 4) && !std::memcmp(&a.gR, &b.gR, 4) && !std::memcmp(&a.theta, &b.theta, 4) &&
         !std::memcmp(&a.t_step, &b.t_step, 4);
}

// body band: faces where the BDIM blend is not the identity (del != 1, del1 != 0, or a control cylinder's velocity kernel
// is non-zero)
void band_lists(const Geometry& g, std::vector<BandFace>& bx, std::vector<BandFace>& by) {
  bx.clear(); by.clear();
  for (int i = 1; i < g.n - 1; i++)
    for (int j = 1; j < g.m - 1; j++) {
      size_t k = (size_t)i * g.m + j;
      if (g.del_x[k] != 1.f || g.del1_x[k] != 0.f || g.w1_x[k] != 0.f || g.w2_x[k] != 0.f)
        bx.push_back({i, j, g.del_x[k], g.del1_x[k], g.wnx_x[k], g.wny_x[k]});
      if (g.del_y[k] != 1.f || g.del1_y[k] != 0.f || g.w1_y[k] != 0.f || g.w2_y[k] != 0.f)
        by.push_back({i, j, g.del_y[k], g.del1_y[k], g.wnx_y[k], g.wny_y[k]});
    }
}

// Band faces per component that one geometry slot holds.  Every band face lies within 3 cells of a body's surface (mu0 /
// mu1 have half-width eps = 2, the union weights behind w1 / w2 vanish from distance 3 on), so inside one of the three
// bodies' bounding boxes grown by 4 cells; the largest body has diameter D (dR <= 1), and a square of side D + 8 holds at
// most (D + 9)^2 faces of one component.  With this capacity a new parameter set never needs more room.
int band_capacity(const rlfc_config& c) {
  const long long side = c.resolution + 9, cap = 3 * side * side;
  const long long faces = (long long)c.x_lengths * c.resolution * c.y_lengths * c.resolution;
  return (int)std::min(cap, faces);
}

struct EnvGeometry {
  Geometry g;
  std::vector<BandFace> bx, by;
};

// Validates the parameter sets p[0 .. n-1] for the grid of `cfg` and builds their geometries (without the hierarchy, which
// the device builds): equal sets once, on a few threads.  set_of[k] = the entry of `out` that p[k] uses.  Touches no device.
// Messages name the entry as table[k].
int build_env_geometries(const rlfc_config& cfg, const rlfc_env_params* p, int n, std::vector<EnvGeometry>& out,
                         std::vector<int>& set_of, std::string& err, const char* table = "env_params") {
  std::vector<int> uniq;                   // index into p of the first occurrence of each distinct set
  set_of.assign(n, 0);
  for (int k = 0; k < n; k++) {
    const rlfc_env_params& q = p[k];
    const std::string at = std::string(table) + "[" + std::to_string(k) + "]: ";
    if (q.re < 1) { err = at + "re must be >= 1"; return RLFC_EINVAL; }
    if (!(q.dR > 0 && q.dR <= 1)) { err = at + "dR must be in (0, 1]"; return RLFC_EINVAL; }
    if (!(q.gR >= 0) || !std::isfinite(q.gR)) { err = at + "gR must be finite and >= 0"; return RLFC_EINVAL; }
    if (!std::isfinite(q.theta)) { err = at + "theta must be finite"; return RLFC_EINVAL; }
    if (!std::isfinite(q.t_step) || !(q.t_step > 0)) { err = at + "t_step must be finite and > 0"; return RLFC_EINVAL; }
    size_t u = 0;
    while (u < uniq.size() && !same_params(p[uniq[u]], q)) u++;
    if (u == uniq.size()) uniq.push_back(k);
    set_of[k] = (int)u;
  }
  out.clear();
  out.resize(uniq.size());
  std::vector<int> rc(uniq.size(), RLFC_OK);
  std::vector<std::string> msg(uniq.size());
  const int cap = band_capacity(cfg);
  auto build = [&](size_t u) {
    rlfc_config c = cfg;
    const rlfc_env_params& q = p[uniq[u]];
    c.re = q.re; c.dR = q.dR; c.gR = q.gR; c.theta = q.theta; c.t_step = q.t_step; c.env_params = nullptr;
    EnvGeometry& G = out[u];
    if ((rc[u] = build_geometry(c, G.g, msg[u], false))) return;
    band_lists(G.g, G.bx, G.by);
    // the two-phase setBC kernel (k_bc2) reads rows 1, n-2 and columns 1, m-2 before it blends the band
    for (const auto* v : {&G.bx, &G.by})
      for (const BandFace& f : *v)
        if (f.i <= 1 || f.i >= G.g.n - 2 || f.j <= 1 || f.j >= G.g.m - 2) {
          rc[u] = RLFC_EINVAL;
          msg[u] = "the body band reaches the lines next to the domain boundary (face " + std::to_string(f.i) + ", " +
                   std::to_string(f.j) + ")";
          return;
        }
    if ((int)G.bx.size() > cap || (int)G.by.size() > cap) {
      rc[u] = RLFC_EINVAL;
      msg[u] = "body band larger than the slot capacity of " + std::to_string(cap) + " faces";
    }
  };
  const int nth = (int)std::min<size_t>(uniq.size(), std::max(1u, std::min(8u, std::thread::hardware_concurrency())));
  std::vector<std::thread> th;
  for (int t = 1; t < nth; t++)
    th.emplace_back([&, t] { for (size_t u = t; u < uniq.size(); u += nth) build(u); });
  for (size_t u = 0; u < uniq.size(); u += std::max(nth, 1)) build(u);
  for (auto& x : th) x.join();
  for (size_t u = 0; u < uniq.size(); u++)
    if (rc[u]) {
      err = std::string(table) + "[" + std::to_string(uniq[u]) + "]: " + msg[u];
      return RLFC_EINVAL;
    }
  return RLFC_OK;
}

// a geometry into geometry slot `slot` (del, the body-velocity basis, the band lists)
int upload_slot_geometry(rlfc_env* E, int slot, const EnvGeometry& G) {
  SolverParams& sp = E->sp;
  const Geometry& g = G.g;
  const std::vector<float>* src[10] = {&g.del_x, &g.del_y, &g.w1_x, &g.w2_x, &g.ry1_x, &g.ry2_x, &g.w1_y, &g.w2_y, &g.rx1_y, &g.rx2_y};
  const float* dst[10] = {sp.del_x, sp.del_y, sp.w1_x, sp.w2_x, sp.ry1_x, sp.ry2_x, sp.w1_y, sp.w2_y, sp.rx1_y, sp.rx2_y};
  for (int f = 0; f < 10; f++)
    CU(cudaMemcpy2DAsync(const_cast<float*>(dst[f]) + (size_t)slot * sp.stride, sp.P * sizeof(float), src[f]->data(),
                         g.m * sizeof(float), g.m * sizeof(float), g.n, cudaMemcpyHostToDevice, E->stream));
  if (!G.bx.empty())
    CU(cudaMemcpyAsync(const_cast<BandFace*>(sp.band_x) + (size_t)slot * sp.nband_x, G.bx.data(), G.bx.size() * sizeof(BandFace),
                       cudaMemcpyHostToDevice, E->stream));
  if (!G.by.empty())
    CU(cudaMemcpyAsync(const_cast<BandFace*>(sp.band_y) + (size_t)slot * sp.nband_y, G.by.data(), G.by.size() * sizeof(BandFace),
                       cudaMemcpyHostToDevice, E->stream));
  return RLFC_OK;
}

// environment e's parameters: its geometry into slot e and the host copies of its scalars; the caller uploads the
// per-environment arrays and rebuilds the hierarchy
int upload_env_geometry(rlfc_env* E, int e, const rlfc_env_params& p, const EnvGeometry& G) {
  const Geometry& g = G.g;
  int rc = upload_slot_geometry(E, e, G);
  if (rc) return rc;
  E->params[e] = p;
  E->dt0[e] = g.dt;
  E->h_nu[e] = g.nu;
  E->h_dRD[e] = g.dR * g.D;
  E->h_nbx[e] = (int)G.bx.size();
  E->h_nby[e] = (int)G.by.size();
  return RLFC_OK;
}

// the host copies of the per-environment scalars -> sp.env_*
int upload_env_scalars(rlfc_env* E) {
  SolverParams& sp = E->sp;
  const size_t B = E->params.size();
  CU(cudaMemcpyAsync(const_cast<float*>(sp.env_nu), E->h_nu.data(), B * sizeof(float), cudaMemcpyHostToDevice, E->stream));
  CU(cudaMemcpyAsync(const_cast<float*>(sp.env_dRD), E->h_dRD.data(), B * sizeof(float), cudaMemcpyHostToDevice, E->stream));
  CU(cudaMemcpyAsync(const_cast<int*>(sp.env_nband_x), E->h_nbx.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  CU(cudaMemcpyAsync(const_cast<int*>(sp.env_nband_y), E->h_nby.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  if (E->pr.params)
    CU(cudaMemcpyAsync(E->pr.params, E->params.data(), B * sizeof(rlfc_env_params), cudaMemcpyHostToDevice, E->stream));
  if (E->lib.L) {   // (env_slot is written at create otherwise; with a library the device changes it too)
    std::vector<int> slot(B);
    for (int e = 0; e < (int)B; e++) slot[e] = E->h_env_set[e] < 0 ? e : E->h_lib[E->h_env_set[e]].slot;
    CU(cudaMemcpyAsync(const_cast<int*>(sp.env_slot), slot.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream));
    CU(cudaMemcpyAsync(E->lib.env_set, E->h_env_set.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  }
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

// ---- parameter library (rlfc_config.param_sets) ----

// The host copies of what an environment holds (params, dt0, h_nu, h_dRD, h_nbx, h_nby) go stale once the device switches
// it to a library set or builds it a new set (rlfc_env_reset_params_device).  Host entry points that read them call this
// first: it synchronises the handle's stream, reads lib.env_set back and refreshes the copies of the environments that
// hold a library set; after a device parameter reset it also reads back the set and band counts each environment holds on
// its own slot.  (Otherwise an environment on its own slot got its copies from rlfc_env_reset_params, which put it there.)
// Without a library and without a device parameter reset since the last call it does nothing.
int sync_env_sets(rlfc_env* E) {
  if (!E->lib.L && !E->par_pending) return RLFC_OK;
  const int B = E->sp.B;
  std::vector<rlfc_env_params> own(E->par_pending ? B : 0);
  std::vector<int> nbx(own.size()), nby(own.size());
  if (E->lib.L) CU(cudaMemcpyAsync(E->h_env_set.data(), E->lib.env_set, B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  if (E->par_pending) {
    CU(cudaMemcpyAsync(own.data(), E->pr.params, B * sizeof(rlfc_env_params), cudaMemcpyDeviceToHost, E->stream));
    CU(cudaMemcpyAsync(nbx.data(), E->sp.env_nband_x, B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
    CU(cudaMemcpyAsync(nby.data(), E->sp.env_nband_y, B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  }
  CU(cudaStreamSynchronize(E->stream));
  for (int e = 0; e < B; e++) {
    const int s = E->lib.L ? E->h_env_set[e] : -1;
    if (s >= 0) {
      const LibSet& L = E->h_lib[s];
      E->params[e] = E->lib_params[s];
      E->dt0[e] = L.dt0;
      E->h_nu[e] = L.nu; E->h_dRD[e] = L.dRD;
      E->h_nbx[e] = L.nbx; E->h_nby[e] = L.nby;
    } else if (E->par_pending) {   // what build_geometry makes of the set (geometry.cpp)
      const rlfc_env_params& p = own[e];
      const float D = (float)E->cfg.resolution;
      E->params[e] = p;
      E->dt0[e] = p.t_step * E->cfg.resolution;
      E->h_nu[e] = D / p.re; E->h_dRD[e] = p.dR * D;
      E->h_nbx[e] = nbx[e]; E->h_nby[e] = nby[e];
    }
  }
  E->par_pending = false;
  return RLFC_OK;
}

// environment e's geometry slot per the host copies (after sync_env_sets)
int slot_of(const rlfc_env* E, int e) {
  if (!E->env_mode) return 0;
  return E->lib.L && E->h_env_set[e] >= 0 ? E->h_lib[E->h_env_set[e]].slot : e;
}

// the one reset path of both variants: n pairs in device memory, enqueued on the handle's stream, then the Poisson
// hierarchies of the environments reset, from their new del and dt (fixed and adaptive dt alike)
int reset_sets_enqueue(rlfc_env* E, const int* d_env, const int* d_set, int n, int reset_accumulators) {
  if (n <= 0) return RLFC_OK;
  SolverParams& sp = E->whole.sp;
  CU(cudaMemsetAsync(E->d_skip, 1, sp.B * sizeof(int), E->stream));   // nonzero = keep; the reset clears
  E->run("k_reset_sets", 0, [&] {
    return launch_reset_sets(sp, E->lib, E->snap, E->init_ux, E->init_uy, E->init_p, E->init_t, E->uAx, E->uAy, d_env, d_set, n,
                             reset_accumulators, E->d_skip, E->stream);
  });
  E->run("k_poisson_rebuild0", 0, [&] { return launch_poisson_rebuild0(sp, E->d_skip, E->stream); });
  E->run("k_poisson_rebuild_coarse", 0, [&] { return launch_poisson_rebuild_coarse(sp, E->d_skip, E->stream); });
  CU(cudaGetLastError());
  return RLFC_OK;
}

int reset_sets_check_handle(rlfc_env* E, int n, bool have_ptrs) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->lib.L) return fail(RLFC_EINVAL, "the handle has no parameter library (rlfc_config.n_param_sets = 0)");
  if (n < 0) return fail(RLFC_EINVAL, "bad pair count");
  if (n > 0 && !have_ptrs) return fail(RLFC_EINVAL, "null argument");
  return RLFC_OK;
}

// ---- snapshot slots (rlfc_config.n_snapshots) ----

// the bits of a parameter tuple as a slot header stores them (words 1 .. 5)
void param_bits(const rlfc_env_params& p, unsigned out[5]) {
  std::memcpy(&out[0], &p.re, 4); std::memcpy(&out[1], &p.dR, 4); std::memcpy(&out[2], &p.gR, 4);
  std::memcpy(&out[3], &p.theta, 4); std::memcpy(&out[4], &p.t_step, 4);
}

// E->params -> snap.env_par (what a restore compares a slot's header with, and what a record's header holds)
int upload_snapshot_params(rlfc_env* E) {
  if (!E->snap.env_par) return RLFC_OK;
  const int B = (int)E->params.size();
  std::vector<unsigned> bits((size_t)5 * B);
  for (int e = 0; e < B; e++) {
    unsigned b[5];
    param_bits(E->params[e], b);
    for (int w = 0; w < 5; w++) bits[(size_t)w * B + e] = b[w];
  }
  CU(cudaMemcpyAsync(E->snap.env_par, bits.data(), bits.size() * sizeof(unsigned), cudaMemcpyHostToDevice, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

// the one copy path of both variants: n pairs in device memory, enqueued on the handle's stream; an adaptive-dt restore
// then rebuilds the Poisson hierarchy of the environments it restored from their restored dt
int snapshot_enqueue(rlfc_env* E, const int* d_env, const int* d_slot, int n, int restore, int keep) {
  if (n <= 0) return RLFC_OK;
  SolverParams& sp = E->whole.sp;
  const bool rebuild = restore && sp.adaptive;
  if (rebuild) CU(cudaMemsetAsync(E->d_skip, 1, sp.B * sizeof(int), E->stream));   // nonzero = keep; the copy clears
  E->run("k_snapshot_copy", 0, [&] {
    return launch_snapshot_copy(sp, E->snap, E->sens, E->uAx, E->uAy, d_env, d_slot, n, restore, keep, rebuild ? E->d_skip : nullptr,
                                E->stream);
  });
  if (rebuild) {
    E->run("k_poisson_rebuild0", 0, [&] { return launch_poisson_rebuild0(sp, E->d_skip, E->stream); });
    E->run("k_poisson_rebuild_coarse", 0, [&] { return launch_poisson_rebuild_coarse(sp, E->d_skip, E->stream); });
  }
  CU(cudaGetLastError());
  return RLFC_OK;
}

int snapshot_check_handle(rlfc_env* E, int n, bool have_ptrs) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->snap.S) return fail(RLFC_EINVAL, "the handle has no snapshot slots (rlfc_config.n_snapshots = 0)");
  if (n < 0) return fail(RLFC_EINVAL, "bad pair count");
  if (n > 0 && !have_ptrs) return fail(RLFC_EINVAL, "null argument");
  return RLFC_OK;
}

// the host variants: validated all or nothing, then the device path, synchronous on return
int snapshot_host(rlfc_env* E, const int* env_ids, const int* slots, int n, int restore, int keep) {
  int rc = snapshot_check_handle(E, n, env_ids && slots);
  if (rc) return rc;
  const int B = E->sp.B, S = E->snap.S;
  std::vector<char> seen(restore ? B : S, 0);
  for (int k = 0; k < n; k++) {
    if (env_ids[k] < 0 || env_ids[k] >= B) return fail(RLFC_EINVAL, "env id " + std::to_string(env_ids[k]) + " out of range");
    if (slots[k] < 0 || slots[k] >= S) return fail(RLFC_EINVAL, "slot " + std::to_string(slots[k]) + " out of range");
    const int dst = restore ? env_ids[k] : slots[k];
    if (seen[dst]++) return fail(RLFC_EINVAL, std::string(restore ? "env id " : "slot ") + std::to_string(dst) + " listed twice");
  }
  CU(cudaSetDevice(E->device));
  if (restore && n > 0 && (rc = sync_env_sets(E))) return rc;   // (params[e]: the set the destination holds now)
  if (restore && n > 0) {
    // device snapshots write slots the host never sees: read the headers back
    std::vector<unsigned> hdr((size_t)kSnapHdr * S);
    CU(cudaMemcpyAsync(hdr.data(), E->snap.hdr, hdr.size() * sizeof(unsigned), cudaMemcpyDeviceToHost, E->stream));
    CU(cudaStreamSynchronize(E->stream));
    for (int k = 0; k < n; k++) {
      const int e = env_ids[k], s = slots[k];
      if (!hdr[s]) return fail(RLFC_EINVAL, "slot " + std::to_string(s) + " has never been written");
      unsigned b[5];
      param_bits(E->params[e], b);
      for (int w = 0; w < 5; w++)
        if (hdr[(size_t)(1 + w) * S + s] != b[w])
          return fail(RLFC_EINVAL, "slot " + std::to_string(s) + " holds a state of another parameter set than env " + std::to_string(e));
    }
  }
  if (n > 0) {
    CU(cudaMemcpyAsync(E->snap_env, env_ids, n * sizeof(int), cudaMemcpyHostToDevice, E->stream));
    CU(cudaMemcpyAsync(E->snap_slot, slots, n * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  }
  if ((rc = snapshot_enqueue(E, E->snap_env, E->snap_slot, n, restore, keep))) return rc;
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

// ---- state records (rlfc.h "State records"; records.cuh) ----

const char* record_check_name(int v) {
  switch (v) {
    case kRecMagic: return "magic (not a state record)";
    case kRecVersion: return "version (not RLFC_RECORD_VERSION)";
    case kRecLength: return "length (does not match its header, or not the size of the call's records)";
    case kRecGrid: return "grid (resolution, x_lengths, y_lengths, n, m or probes differ from the handle's)";
    case kRecChecksum: return "checksum (the record is corrupted)";
    case kRecTuple: return "parameter tuple (differs from the destination's)";
    case kRecDt: return "dt (not the destination's fixed dt, or not a finite dt > 0)";
    default: return "?";
  }
}

int records_check_handle(rlfc_env* E, int n, bool have_ptrs) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->slab.empty()) return fail(RLFC_EINVAL, "state records are not available in slab mode (n_devices > 1)");
  if (n < 0) return fail(RLFC_EINVAL, "bad pair count");
  if (n > 0 && !have_ptrs) return fail(RLFC_EINVAL, "null argument");
  return RLFC_OK;
}

// a device buffer of at least `need` T (contents kept only when it does not grow; zeroed when it does)
template <typename T>
int rec_grow(rlfc_env* E, T** p, size_t& cap, size_t need) {
  if (need <= cap) return RLFC_OK;
  if (*p) {   // (cudaFree waits for the device: no enqueued launch still reads the old buffer)
    E->rec_bufs.erase(std::find(E->rec_bufs.begin(), E->rec_bufs.end(), (void*)*p));
    CU(cudaFree(*p));
    *p = nullptr;
    cap = 0;
  }
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, need * sizeof(T));
  if (e != cudaSuccess) return fail(RLFC_ENOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  E->rec_bufs.push_back(q);
  CU(cudaMemsetAsync(q, 0, need * sizeof(T), E->stream));
  *p = (T*)q;
  cap = need;
  return RLFC_OK;
}

// what a record call of n pairs of `bytes`-long records needs: on the first call the parameter tuples (snap.env_par, kept
// current by every later device reset), the refusal flags and the sensor table; the per-pair scratch
int records_prepare(rlfc_env* E, int n, size_t bytes) {
  int rc;
  if (!E->rec.refused) {
    const int B = E->sp.B;
    if (!E->snap.env_par) {
      if ((rc = sync_env_sets(E))) return rc;
      if ((rc = E->dmalloc(&E->snap.env_par, (size_t)5 * B))) return rc;
      if ((rc = upload_snapshot_params(E))) return rc;
    }
    if ((rc = E->dmalloc(&E->rec.refused, B))) return rc;
    if (!E->sensor_table.empty()) {
      const rlfc_sensor* t = nullptr;
      if ((rc = upload_vec(E, E->sensor_table, &t))) return rc;
      E->rec.sensors = t;
    }
    E->rec.env_par = E->snap.env_par;
    E->rec.grid[0] = E->cfg.resolution; E->rec.grid[1] = E->cfg.x_lengths; E->rec.grid[2] = E->cfg.y_lengths;
  }
  size_t cap = E->rec_pairs;
  if ((rc = rec_grow(E, &E->rec.ticket, cap, (size_t)n))) return rc;
  cap = E->rec_pairs;
  if ((rc = rec_grow(E, &E->rec.hcode, cap, (size_t)n))) return rc;
  cap = E->rec_pairs;
  if ((rc = rec_grow(E, &E->rec.verdict, cap, (size_t)n))) return rc;
  E->rec_pairs = std::max(E->rec_pairs, (size_t)n);
  return rec_grow(E, &E->rec.partial, E->rec_partials, (size_t)n * record_chunks(E->sp.n, E->sp.m, bytes));
}

size_t own_record_bytes(const rlfc_env* E) { return record_bytes(E->sp.n, E->sp.m, E->sens.n); }

int record_export_enqueue(rlfc_env* E, const int* d_ids, int n, void* d_buf) {
  if (n <= 0) return RLFC_OK;
  int rc = records_prepare(E, n, own_record_bytes(E));
  if (rc) return rc;
  SolverParams& sp = E->whole.sp;
  E->run("k_export", 0, [&] { return launch_record_export(sp, E->sens, E->rec, E->uAx, E->uAy, d_ids, n, d_buf, E->stream); });
  CU(cudaGetLastError());
  return RLFC_OK;
}

// the check pass (verdicts only); the host variant reads the verdicts before it applies
int record_check_enqueue(rlfc_env* E, const int* d_ids, int n, const void* d_buf, size_t bytes) {
  int rc = records_prepare(E, n, bytes);
  if (rc) return rc;
  SolverParams& sp = E->whole.sp;
  E->run("k_import_check", 0, [&] {
    return launch_record_import(sp, E->sens, E->rec, E->uAx, E->uAy, d_ids, n, d_buf, bytes, 1, 0, nullptr, E->stream);
  });
  CU(cudaGetLastError());
  return RLFC_OK;
}

// the apply pass; in adaptive mode then the Poisson hierarchy of exactly the environments imported (restore's skip mask)
int record_apply_enqueue(rlfc_env* E, const int* d_ids, int n, const void* d_buf, size_t bytes, int keep) {
  SolverParams& sp = E->whole.sp;
  const bool rebuild = sp.adaptive;
  if (rebuild) CU(cudaMemsetAsync(E->d_skip, 1, sp.B * sizeof(int), E->stream));   // nonzero = keep; the import clears
  E->run("k_import", 0, [&] {
    return launch_record_import(sp, E->sens, E->rec, E->uAx, E->uAy, d_ids, n, d_buf, bytes, 0, keep,
                                rebuild ? E->d_skip : nullptr, E->stream);
  });
  if (rebuild) {
    E->run("k_poisson_rebuild0", 0, [&] { return launch_poisson_rebuild0(sp, E->d_skip, E->stream); });
    E->run("k_poisson_rebuild_coarse", 0, [&] { return launch_poisson_rebuild_coarse(sp, E->d_skip, E->stream); });
  }
  CU(cudaGetLastError());
  return RLFC_OK;
}

// host ids: in range and (import) no destination twice
int record_host_ids(rlfc_env* E, const int* ids, int n, bool import) {
  const int B = E->sp.B;
  std::vector<char> seen(B, 0);
  for (int k = 0; k < n; k++) {
    if (ids[k] < 0 || ids[k] >= B) return fail(RLFC_EINVAL, "env id " + std::to_string(ids[k]) + " out of range");
    if (import && seen[ids[k]]++) return fail(RLFC_EINVAL, "env id " + std::to_string(ids[k]) + " listed twice");
  }
  return RLFC_OK;
}

int record_stage(rlfc_env* E, const int* ids, int n, size_t bytes) {
  int rc = rec_grow(E, &E->rec_ids, E->rec_id_cap, (size_t)n);
  if (rc) return rc;
  if ((rc = rec_grow(E, &E->rec_stage, E->rec_stage_bytes, (size_t)n * bytes))) return rc;
  CU(cudaMemcpyAsync(E->rec_ids, ids, n * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  return RLFC_OK;
}

// ---- one solver step (AFCCylinder.update2, AFCCylinder.pde:45-61), written once for every path ----
// solver_step lists the kernels of one step in launch order and hands each to a sink, which launches it eagerly (EagerSink:
// RLFC_NO_GRAPH, rlfc_env_set_profiling), captures it into a group's step graph (CaptureSink) or launches it on every device
// of a slab-mode handle (SlabSink).  The floats-per-interior-cell figures are each kernel's ALGORITHMIC traffic per env
// (SURVEY 8d convention: per-env arrays only, one read per input and one write per output).
using Group = rlfc_env::Group;
using SlabDev = rlfc_env::SlabDev;

enum View : bool { kA = false, kB = true };      // the view a kernel takes: pressure buffer A (sp) or B (spB) at lev[0].x
enum Place : bool { kEach = false, kSolo = true };   // slab mode: every device on its own rows / strips, or device 0 alone
struct StepKernel {
  const char* name;         // profile name (rlfc_env_get_profile)
  double fpc;               // floats per interior cell
  View view;
  Place place;
};

enum { kDown, kUp, kSweeps, kIncr };
// profile name of one kernel of a chained level l; the levels from 4 on share one name
const char* chain_name(int piece, int l) {
  static const char* const nm[4][5] = {
      {"k_chain_down_L0", "k_chain_down_L1", "k_chain_down_L2", "k_chain_down_L3", "k_chain_down_L4+"},
      {"k_chain_up_L0", "k_chain_up_L1", "k_chain_up_L2", "k_chain_up_L3", "k_chain_up_L4+"},
      {"k_chain_sweeps_L0", "k_chain_sweeps_L1", "k_chain_sweeps_L2", "k_chain_sweeps_L3", "k_chain_sweeps_L4+"},
      {"k_chain_incr_L0", "k_chain_incr_L1", "k_chain_incr_L2", "k_chain_incr_L3", "k_chain_incr_L4+"}};
  return nm[piece][std::min(l, 4)];
}

// One MG-projected half step on velocity buffer U (BDIM.updateUP tail + VectorField.project); which = 1: the corrector.
// Level-0 residual flow of one MG iteration: down0 reads r and writes the smoothed residual to the `d` buffer, up0 updates
// it in place, smooth0 consumes it and writes the new residual back to r.
template <class Sink>
int project(Sink& S, const Group& G, float* Ux, float* Uy, int which) {
  const SolverParams& sp = G.sp;
  float* r = sp.lev[0].r;
  float* rs = sp.lev[0].d;
  float* pA = sp.lev[0].x;
  float* pB = G.spB.lev[0].x;
  const int nch = sp.chain_levels;   // levels 0 .. nch-1 chained (grid-wide kernels); the one-CTA kernel takes the rest
  // below level 0's restriction: the chained levels' restrictions, the coarse levels, the chained levels' corrections and
  // smooth(4) top down; then level 0's
  auto vcycle = [&] {
    for (int l = 1; l < nch; l++) {
      S.run({chain_name(kDown, l), 0, kB, kEach}, [&](auto& v, auto st) { return launch_chain_down(v, l, st); });
      S.sync();
    }
    S.run({nch ? "k_mg_coarse_cta" : "k_mg_coarse", 0.5, kB, kSolo}, [&](auto& v, auto st) { return launch_coarse_cta(v, st); });
    S.sync();
    for (int l = nch - 1; l >= 0; l--) {
      S.run({chain_name(kUp, l), l ? 0 : 4.25, kB, kEach}, [&](auto& v, auto st) { return launch_chain_up(v, l, l ? nullptr : rs, st); });
      S.sync();
      S.run({chain_name(kSweeps, l), l ? 0 : 3.0, kB, kEach}, [&](auto& v, auto st) { return launch_chain_sweeps(v, l, st); });
      S.sync();
      S.run({chain_name(kIncr, l), l ? 0 : 4.0, kB, kEach},
            [&](auto& v, auto st) { return launch_chain_incr(v, l, l ? nullptr : r, l ? 0 : which, st); });
      S.sync();
    }
    if (!nch) {
      S.run({"k_mg_up0", 4.25, kB, kEach}, [&](auto& v, auto st) { return launch_mg_up0(v, rs, st); });
      S.run({"k_smooth0", 4, kB, kEach}, [&](auto& v, auto st) { return launch_smooth0(v, rs, r, which, st); });
    }
  };
  int rc = S.mg_loop(
      [&] {   // the first iteration (MG.pde:32-35 is a do-while in effect: iter < itmx holds on entry)
        S.run({"k_resid_down0", 5.25, kA, kEach},
              [&](auto& v, auto st) { return launch_resid_down0(v, Ux, Uy, pA, pB, rs, which, st); });
        S.sync();
        vcycle();
      },
      [&] {   // a further iteration (the row smoother has left the residual skewed)
        if (!nch && !sp.lev[0].wave) S.run({"k_unskew_r", 2, kB, kEach}, [&](auto& v, auto st) { return launch_unskew_r(v, r, st); });
        S.run({"k_mg_down0", 4.25, kB, kEach}, [&](auto& v, auto st) { return launch_mg_down0(v, r, rs, st); });
        S.sync();
        vcycle();
      });
  if (rc) return rc;
  // Field.sum (a serial float chain over the whole field): segment summaries (tables, then the serial pass), or the plain chain
  if (sp.xs_recs) {
    S.run({"k_xsum_tables", 1, kB, kSolo}, [&](auto& v, auto st) { return launch_psum_tables(v, st); });
    S.run({"k_xsum_pass", 0, kB, kSolo}, [&](auto& v, auto st) { return launch_psum_pass(v, st); });
  } else {
    S.run({"k_psum", 1, kB, kSolo}, [&](auto& v, auto st) { return launch_psum(v, st); });
  }
  S.sync();
  if (which == 1 && sp.fast_bc) {
    // corrector: Heun average fused into the projection and the boundary-condition kernels (BDIM.pde:95-96)
    S.run({"k_project_shift_heun", 8, kA, kEach},
          [&](auto& v, auto st) { return launch_project_shift_heun(v, pB, pA, Ux, Uy, G.uBx, G.uBy, G.uAx, G.uAy, st); });
    S.sync();
    S.run({"k_bc_heun", 0, kA, kSolo}, [&](auto& v, auto st) { return launch_bc_heun(v, Ux, Uy, G.uBx, G.uBy, G.uAx, G.uAy, st); });
  } else {
    S.run({"k_project_shift", 6, kA, kEach}, [&](auto& v, auto st) { return launch_project_shift(v, pB, pA, Ux, Uy, st); });
    S.sync();
    S.run({"k_bc", 0, kA, kSolo}, [&](auto& v, auto st) { return launch_bc(v, Ux, Uy, st); });
  }
  S.sync();
  return RLFC_OK;
}

// AFCCylinder.update2 for view G.  Sink: run(StepKernel, launch(view, stream) -> launches), sync() (slab mode: a barrier
// of all devices between dependent kernels; the other sinks ignore it) and mg_loop(first iteration, further iteration).
template <class Sink>
int solver_step(Sink& S, const Group& G, int accumulate) {
  const SolverParams& sp = G.sp;
  int rc;
  S.sync();   // (slab mode: whatever device 0 enqueued since the last step -- actions, resets, field uploads -- is visible to all)
  if (sp.adaptive) {
    // AFCCylinder.update (AFCCylinder.pde:63-84): dt = flow.checkCFL(), then the Poisson hierarchy of c = del*dt, on the
    // device (dt never goes to the host).  (Slab mode has neither adaptive dt nor sensors.)
    S.run({"k_check_cfl", 2, kA, kSolo}, [&](auto& v, auto st) { return launch_step_cfl(v, G.uAx, G.uAy, st); });
    S.run({"k_poisson_rebuild0", 0, kA, kSolo}, [&](auto& v, auto st) { return launch_poisson_rebuild0(v, v.sc.frozen, st); });
    S.run({"k_poisson_rebuild_coarse", 0, kA, kSolo},
          [&](auto& v, auto st) { return launch_poisson_rebuild_coarse(v, v.sc.frozen, st); });
  }
  // which = 0, predictor BDIM.update(): u0 = u (buffer A), F = AdvDif(u) -> B, updateUP
  // which = 1, corrector BDIM.update2(): us = u (B), F = AdvDif(u; + u0) -> C, updateUP, u = (u + us)/2 -> A
  for (int which = 0; which < 2; which++) {
    float* sx = which ? G.uBx : G.uAx;
    float* sy = which ? G.uBy : G.uAy;
    float* dx = which ? G.uCx : G.uBx;
    float* dy = which ? G.uCy : G.uBy;
    S.run({"k_advdif", 5, kA, kEach}, [&](auto& v, auto st) { return launch_advdif(v, sx, sy, G.uAx, G.uAy, dx, dy, st); });
    S.sync();
    S.run({"k_band_bc", 0, kA, kSolo}, [&](auto& v, auto st) { return launch_band_bc(v, dx, dy, st); });
    S.sync();
    if ((rc = project(S, G, dx, dy, which))) return rc;
  }
  if (!sp.fast_bc) {
    S.run({"k_heun", 6, kA, kEach}, [&](auto& v, auto st) { return launch_heun(v, G.uCx, G.uCy, G.uBx, G.uBy, G.uAx, G.uAy, st); });
    S.sync();
  }
  // (before k_force, which freezes an environment at the end of its window: this step's sample is its observation)
  if (G.sens.n > 0) S.run({"k_sensors", 0, kA, kSolo}, [&](auto& v, auto st) { return launch_sensors(v, G.sens, G.uAx, G.uAy, st); });
  if (G.fs.every > 0) {
    // a sampled step reads 3 floats and reads and writes 7 doubles on every cell of the n x m layout: 124 B per cell
    const double fpc = 31.0 * sp.n * sp.m / ((double)(sp.n - 2) * (sp.m - 2));
    S.run({"k_flow_stats", fpc, kA, kSolo}, [&](auto& v, auto st) { return launch_flow_stats(v, G.fs, G.uAx, G.uAy, st); });
  }
  S.run({"k_force", 0, kA, kSolo}, [&](auto& v, auto st) { return launch_force(v, accumulate, st); });
  S.sync();
  return RLFC_OK;
}

// the MG loop driven from the host (eager and slab paths): the data-dependent loop exit (MG.pde:34) costs one 4-byte
// readback of any_active per iteration, on device 0's stream `st`
template <class First, class Body>
int polled_mg_loop(rlfc_env* E, const SolverParams& sp, cudaStream_t st, First& first, Body& body) {
  for (int it = 0; it < sp.mg_max_iters; it++) {
    cudaSetDevice(E->device);   // (slab mode: the iteration's kernels leave another device current)
    CU(cudaMemsetAsync(sp.sc.any_active, 0, sizeof(int), st));
    if (it == 0) first();
    else body();
    E->mg_iter_launch_rounds++;
    cudaSetDevice(E->device);
    CU(cudaMemcpyAsync(E->h_any, sp.sc.any_active, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (!*E->h_any) break;
  }
  return RLFC_OK;
}

// eager path: every kernel launched on its own on the view's stream, event-timed when profiling
struct EagerSink {
  rlfc_env* E;
  const Group& G;
  template <class F>
  void run(const StepKernel& k, F&& launch) {
    E->run(k.name, k.fpc, [&] { return launch(k.view == kB ? G.spB : G.sp, G.st); }, G.st);
  }
  void sync() {}
  template <class First, class Body>
  int mg_loop(First&& first, Body&& body) { return polled_mg_loop(E, G.sp, G.st, first, body); }
};

// graph path: one CUDA graph per group = one solver step; each MGsolver loop is a WHILE conditional node whose body is one
// further iteration and whose condition is written on the device (k_loopcond), so no host round trip remains
struct CaptureSink {
  rlfc_env* E;
  const Group& G;
  cudaStream_t st;          // the stream being captured: the group's, or aux_stream while a WHILE body is recorded
  long long launches = 0;   // kernel nodes outside the WHILE bodies (Group::graph_launches)
  template <class F>
  void run(const StepKernel& k, F&& launch) {
    launches += launch(k.view == kB ? G.spB : G.sp, st);
  }
  void sync() {}
  template <class First, class Body>
  int mg_loop(First&& first, Body&& body) {
    first();
    cudaStreamCaptureStatus status;
    cudaGraph_t graph;
    const cudaGraphNode_t* deps;
    size_t ndeps;
    CU(cudaStreamGetCaptureInfo(st, &status, nullptr, &graph, &deps, &ndeps));
    cudaGraphConditionalHandle handle;
    CU(cudaGraphConditionalHandleCreate(&handle, graph, 0, cudaGraphCondAssignDefault));
    // the condition is written by a kernel ahead of the node and again at the end of every body pass
    auto loopcond = [&] { return launch_loopcond(G.spB, (unsigned long long)handle, st); };
    launches += loopcond();
    CU(cudaStreamGetCaptureInfo(st, &status, nullptr, &graph, &deps, &ndeps));
    cudaGraphNodeParams np{};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = handle;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t cond;
    CU(cudaGraphAddNode(&cond, graph, deps, ndeps, &np));
    CU(cudaStreamBeginCaptureToGraph(E->aux_stream, np.conditional.phGraph_out[0], nullptr, nullptr, 0,
                                     cudaStreamCaptureModeThreadLocal));
    const cudaStream_t outer = st;
    const long long outer_launches = launches;
    st = E->aux_stream;
    body();
    loopcond();
    st = outer;
    launches = outer_launches;
    CU(cudaStreamEndCapture(E->aux_stream, nullptr));
    CU(cudaStreamUpdateCaptureDependencies(st, &cond, 1, cudaStreamSetCaptureDependencies));
    return RLFC_OK;
  }
};

int build_step_graph(rlfc_env* E, Group& G, int accumulate) {
  CaptureSink S{E, G, G.st};
  CU(cudaStreamBeginCapture(G.st, cudaStreamCaptureModeThreadLocal));
  const int rc = solver_step(S, G, accumulate);
  cudaGraph_t graph = nullptr;
  cudaError_t ce = cudaStreamEndCapture(G.st, &graph);
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (ce != cudaSuccess) return fail(RLFC_ECUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
  ce = cudaGraphInstantiate(&G.step_graph[accumulate], graph, 0);
  cudaGraphDestroy(graph);
  if (ce != cudaSuccess) return fail(RLFC_ECUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce));
  G.graph_launches = S.launches;
  return RLFC_OK;
}

// Slab mode: one solver step of ONE domain on several devices, eager launches.  Grid-wide kernels are launched with their
// full grid on every device (blocks of other devices' rows / strips exit at once); kernels that are one CTA per environment
// (setBC, the coarsest levels, Field.sum, the force read-out) run on device 0; a barrier separates dependent kernels.  Halo
// operands and the few remote results travel as ordinary loads and stores through the shared address range; the
// Gauss-Seidel sweeps cross device boundaries strip to strip through the tagged edge arrays (smooth_chain3.cuh).
struct SlabSink {
  rlfc_env* E;
  // launch(D) on every device D, event-timed on device 0 when profiling
  template <class F>
  void each(const char* name, double fpc, F&& launch) {
    for (size_t d = 0; d < E->slab.size(); d++) {
      SlabDev& D = E->slab[d];
      cudaSetDevice(D.device);
      if (d == 0) E->run(name, fpc, [&] { return launch(D); }, D.st);
      else E->launches += launch(D);
    }
  }
  template <class F>
  void run(const StepKernel& k, F&& launch) {
    if (k.place == kEach) {
      each(k.name, k.fpc, [&](SlabDev& D) { return launch(k.view == kB ? D.spB : D.sp, D.st); });
      return;
    }
    const Group& W = E->whole;   // the whole domain as device 0 sees it alone (W.st = device 0's stream)
    cudaSetDevice(E->device);
    E->run(k.name, k.fpc, [&] { return launch(k.view == kB ? W.spB : W.sp, W.st); }, W.st);
  }
  void sync() {
    each("k_slab_barrier", 0, [](SlabDev& D) { return launch_slab_barrier(D.bar, D.st); });
    E->slab_barriers++;
  }
  template <class First, class Body>
  int mg_loop(First&& first, Body&& body) { return polled_mg_loop(E, E->whole.sp, E->whole.st, first, body); }
};

// fork the group streams off the handle's stream / join them back
int fork_groups(rlfc_env* E) {
  if (E->groups.size() <= 1) return RLFC_OK;
  CU(cudaEventRecord(E->fork_ev, E->stream));
  for (size_t g = 1; g < E->groups.size(); g++) CU(cudaStreamWaitEvent(E->groups[g].st, E->fork_ev, 0));
  return RLFC_OK;
}
int join_groups(rlfc_env* E) {
  for (size_t g = 1; g < E->groups.size(); g++) {
    CU(cudaEventRecord(E->groups[g].done, E->groups[g].st));
    CU(cudaStreamWaitEvent(E->stream, E->groups[g].done, 0));
  }
  return RLFC_OK;
}

// `nsteps` solver steps (AFCCylinder.update2) for the whole batch
int solver_steps(rlfc_env* E, int nsteps, int accumulate) {
  int rc;
  if (!E->slab.empty()) {
    SlabSink S{E};
    for (int s = 0; s < nsteps; s++) {
      if ((rc = solver_step(S, E->whole, accumulate))) return rc;
      cudaSetDevice(E->device);
      CU(cudaGetLastError());
    }
    return RLFC_OK;
  }
  if (!E->use_graph || E->profiling) {
    EagerSink S{E, E->whole};
    for (int s = 0; s < nsteps; s++) {
      if ((rc = solver_step(S, E->whole, accumulate))) return rc;
      CU(cudaGetLastError());
    }
    return RLFC_OK;
  }
  if ((rc = fork_groups(E))) return rc;
  for (auto& G : E->groups) {
    if (!G.step_graph[accumulate] && (rc = build_step_graph(E, G, accumulate))) return rc;
    for (int s = 0; s < nsteps; s++) {
      CU(cudaGraphLaunch(G.step_graph[accumulate], G.st));
      E->launches += G.graph_launches;   // lower bound: one MG iteration per solve
    }
  }
  if ((rc = join_groups(E))) return rc;
  CU(cudaGetLastError());
  return RLFC_OK;
}

// G = the view of environments [e0, e0 + n) of the batch arrays (E->sp): sp, spB (lev[0].x = pressure buffer B), sensors
// and velocity buffers.  `row` selects the view's own ticket counters, launch tags and any_active word.
void make_view(const rlfc_env* E, int e0, int n, int row, Group& G) {
  const SolverParams& sp = E->sp;
  G.e0 = e0; G.B = n;
  G.sp = sp;
  SolverParams& v = G.sp;
  v.B = n;
  for (int l = 0; l < v.nlevels; l++) {
    const size_t o = (size_t)e0 * v.lev[l].stride;
    v.lev[l].r += o; v.lev[l].x += o; v.lev[l].d += o;
    if (v.lev[l].w) v.lev[l].w += o;
    if (v.per_env) {
      v.lev[l].lx += o; v.lev[l].ly += o; v.lev[l].inv += o; v.lev[l].diag += o;
      if (v.lev[l].rt.T) { v.lev[l].rt.T += (size_t)e0 * v.lev[l].rt.entries * v.lev[l].rt.K * 32; v.lev[l].rt.copies = n; }
    }
  }
  if (v.per_env) {
    v.c_x = v.lev[0].lx; v.c_y = v.lev[0].ly; v.sc.dt += e0;
    v.env_slot += e0; v.env_nu += e0; v.env_dRD += e0; v.env_nband_x += e0; v.env_nband_y += e0;
  }
  for (int l = 0; l < v.chain_levels; l++) {
    ChainLevel& ch = v.lev[l].ch;
    ch.rsk += (size_t)e0 * ch.sk_stride;
    for (int gsw = 0; gsw < 5; gsw++) ch.dsk[gsw] += (size_t)e0 * ch.sk_stride;
    ch.edge += (size_t)e0 * ch.NS * ch.TE;
    ch.ticket = E->chain_tickets + (size_t)row * kMaxLevels + l;
    ch.tag_hi = (unsigned)(row + 1) << 26;
  }
  if (v.chain_levels > 0) { v.rr_chain += (size_t)e0 * v.rr_chain_n; v.rr_count += e0; }
  v.band_tmp += (size_t)e0 * (v.nband_x + v.nband_y);
  v.rsk += (size_t)e0 * v.rsk_stride;
  v.sc.flow_t += e0;
  v.sc.xi += 2 * e0; v.sc.t += e0; v.sc.force += 2 * e0; v.sc.probes += (size_t)e0 * RLFC_NUM_PROBES;
  v.sc.callLearn += e0; v.sc.Cd += e0; v.sc.Cl += e0; v.sc.obs += 2 * e0; v.sc.active += e0; v.sc.iters += 2 * e0;
  v.sc.frozen += e0; v.sc.non_finite += e0;
  v.sc.psum += e0; v.sc.any_active += row;
  if (v.xs_recs) {
    v.xs_ctot += (size_t)e0 * v.xs_nchunks;
    v.xs_cflag += (size_t)e0 * v.xs_nchunks; v.xs_epoch += e0;
    v.xs_recs += (size_t)e0 * v.xs_nbatches * 192;
    if (v.xs_blk) {
      v.xs_blk += (size_t)e0 * ((v.xs_nbatches + 31) / 32) * 256;
      if (v.xs_corr) { v.xs_pred += (size_t)e0 * v.xs_nbatches; v.xs_inc += (size_t)e0 * v.xs_nbatches; v.xs_corr += (size_t)e0 * v.xs_nbatches; }
    }
  }
  v.xs_stats += 8 * e0;
  G.spB = v;
  G.spB.lev[0].x = E->pB + (size_t)e0 * sp.stride;
  G.sens = E->sens;
  if (G.sens.out) G.sens.out += (size_t)e0 * G.sens.n;
  G.fs = E->fs;
  if (G.fs.every > 0) {
    G.fs.sums += (size_t)e0 * kNumStats * sp.stride;
    G.fs.count += e0; G.fs.step += e0; G.fs.ticket += e0;
  }
  const size_t o = (size_t)e0 * sp.stride;
  G.uAx = E->uAx + o; G.uAy = E->uAy + o; G.uBx = E->uBx + o; G.uBy = E->uBy + o; G.uCx = E->uCx + o; G.uCy = E->uCy + o;
}

int load_initial_state(rlfc_env* E) {
  const Geometry& g = E->geo;
  const SolverParams& sp = E->sp;
  const size_t N = (size_t)g.n * g.m;
  std::vector<float> ux, uy, p;
  if (!E->init_path.empty()) {
    std::string err;
    int rc = read_checkpoint(E->init_path, g.n, g.m, E->init_t, E->init_dt, ux, uy, p, err);
    if (rc) return fail(rc, err);
  } else {
    // BDIM ctor BDIM.pde:51-54: u = (1, 0) on all cells, p = 0
    ux.assign(N, 1.f); uy.assign(N, 0.f); p.assign(N, 0.f);
    E->init_t = 0; E->init_dt = g.dt;
  }
  const float* src[3] = {ux.data(), uy.data(), p.data()};
  float* dst[3] = {E->init_ux, E->init_uy, E->init_p};
  for (int c = 0; c < 3; c++) {
    std::vector<float> pit = to_pitched(src[c], g.n, g.m, sp.P);
    CU(cudaMemcpyAsync(dst[c], pit.data(), pit.size() * sizeof(float), cudaMemcpyHostToDevice, E->stream));
    CU(cudaStreamSynchronize(E->stream));
  }
  return RLFC_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

void rlfc_default_config(rlfc_config* c) {
  if (!c) return;
  std::memset(c, 0, sizeof(*c));
  c->resolution = 24; c->x_lengths = 16; c->y_lengths = 8; c->re = 500;       // clientCFD.pde:14,94
  c->dR = .125f; c->gR = .2f; c->theta = 3.1415927f / 3; c->t_step = .0075f;   // clientCFD.pde:9,95-96
  c->action_scale = 5.f;                                                       // clientCFD.pde:53-54
  c->substeps = 16; c->init_time = 1.f; c->episode_time = 50.f;                // clientCFD.pde:5-6,12
  c->n_envs = 1; c->device = -1; c->exact = 1; c->mg_max_iters = 20; c->n_groups = 0; c->n_devices = 1;
  c->init_bdim_path = nullptr; c->stream = nullptr;
}

const char* rlfc_last_error(void) { return g_err.c_str(); }
const char* rlfc_version(void) { return "rlfc-b200 0.1 (sm_100a, exact fp32)"; }

void rlfc_env_destroy(rlfc_env* E) {
  if (!E) return;
  cudaSetDevice(E->device);
  if (E->stream) cudaStreamSynchronize(E->stream);
  E->prof_collect();
  for (cudaEvent_t ev : E->event_pool) cudaEventDestroy(ev);
  for (size_t g = 0; g < E->groups.size(); g++) {
    auto& G = E->groups[g];
    for (int a = 0; a < 2; a++) if (G.step_graph[a]) cudaGraphExecDestroy(G.step_graph[a]);
    if (G.done) cudaEventDestroy(G.done);
    if (g > 0 && G.st) { cudaStreamSynchronize(G.st); cudaStreamDestroy(G.st); }
  }
  for (size_t d = 0; d < E->slab.size(); d++) {
    auto& D = E->slab[d];
    cudaSetDevice(D.device);
    if (D.st) cudaStreamSynchronize(D.st);
    if (d > 0 && D.st) cudaStreamDestroy(D.st);
    for (void* q : D.local) if (q) cudaFree(q);
  }
  cudaSetDevice(E->device);
  if (E->aux_stream) cudaStreamDestroy(E->aux_stream);
  if (E->fork_ev) cudaEventDestroy(E->fork_ev);
  for (void* p : E->allocs) cudaFree(p);
  for (void* p : E->rec_bufs) cudaFree(p);
  for (void* p : {(void*)E->h_actions, (void*)E->h_obs, (void*)E->h_reward, (void*)E->h_force, (void*)E->h_probes,
                  (void*)E->h_done, (void*)E->h_any})
    if (p) cudaFreeHost(p);
  if (E->own_stream && E->stream) cudaStreamDestroy(E->stream);
  delete E;
}

int rlfc_env_create(const rlfc_config* cfg, rlfc_env** out) {
  if (!cfg || !out) return fail(RLFC_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->n_envs < 1) return fail(RLFC_EINVAL, "n_envs must be >= 1");
  if (!cfg->exact) return fail(RLFC_EINVAL, "only exact mode is implemented");
  if ((long long)cfg->resolution * cfg->x_lengths * cfg->resolution * cfg->y_lengths >= (1ll << 31))
    return fail(RLFC_EINVAL, "grid too large (the kernels index cells with 32 bits)");
  if (cfg->substeps < 1 || cfg->mg_max_iters < 1) return fail(RLFC_EINVAL, "substeps and mg_max_iters must be >= 1");
  if (cfg->adaptive_dt != 0 && cfg->adaptive_dt != 1) return fail(RLFC_EINVAL, "adaptive_dt must be 0 or 1");
  if (cfg->adaptive_dt && cfg->n_devices > 1) return fail(RLFC_EINVAL, "adaptive_dt is not available in slab mode (n_devices > 1)");
  if (cfg->n_snapshots < 0) return fail(RLFC_EINVAL, "n_snapshots must be >= 0");
  if (cfg->n_snapshots > 0 && cfg->n_devices > 1)
    return fail(RLFC_EINVAL, "n_snapshots is not available in slab mode (n_devices > 1)");
  if (cfg->n_sensors < 0) return fail(RLFC_EINVAL, "n_sensors must be >= 0");
  if (cfg->n_sensors > 0) {
    if (!cfg->sensors) return fail(RLFC_EINVAL, "sensors is NULL with n_sensors > 0");
    if (cfg->n_devices > 1) return fail(RLFC_EINVAL, "n_sensors is not available in slab mode (n_devices > 1)");
    for (int k = 0; k < cfg->n_sensors; k++) {
      const rlfc_sensor& s = cfg->sensors[k];
      if (s.field < RLFC_SENSOR_P || s.field > RLFC_SENSOR_UY)
        return fail(RLFC_EINVAL, "sensors[" + std::to_string(k) + "]: field must be 0 (p), 1 (u.x) or 2 (u.y)");
      if (!std::isfinite(s.x) || !std::isfinite(s.y))
        return fail(RLFC_EINVAL, "sensors[" + std::to_string(k) + "]: coordinates must be finite");
    }
  }
  if (cfg->stats_every < 0) return fail(RLFC_EINVAL, "stats_every must be >= 0");
  if (cfg->stats_every > 0 && cfg->n_devices > 1)
    return fail(RLFC_EINVAL, "stats_every is not available in slab mode (n_devices > 1)");
  // per-environment parameters: every set validated and its geometry built before any device call
  std::vector<EnvGeometry> env_geo;
  std::vector<int> env_set;
  if (cfg->env_params) {
    if (cfg->n_devices > 1) return fail(RLFC_EINVAL, "env_params is not available in slab mode (n_devices > 1)");
    std::string err;
    if (build_env_geometries(*cfg, cfg->env_params, cfg->n_envs, env_geo, env_set, err)) return fail(RLFC_EINVAL, err);
  }
  // parameter library: the same, for its entries
  std::vector<EnvGeometry> lib_geo;
  std::vector<int> lib_set;
  if (cfg->n_param_sets < 0) return fail(RLFC_EINVAL, "n_param_sets must be >= 0");
  if (cfg->n_param_sets > 0) {
    if (!cfg->param_sets) return fail(RLFC_EINVAL, "param_sets is NULL with n_param_sets > 0");
    if (cfg->n_devices > 1) return fail(RLFC_EINVAL, "param_sets is not available in slab mode (n_devices > 1)");
    std::string err;
    if (build_env_geometries(*cfg, cfg->param_sets, cfg->n_param_sets, lib_geo, lib_set, err, "param_sets"))
      return fail(RLFC_EINVAL, err);
    if (!cfg->env_params) {   // every environment on the scalar config's set, in its own slot (as env_params would give)
      const rlfc_env_params p0 = params_of(*cfg);
      std::vector<rlfc_env_params> own(cfg->n_envs, p0);
      if (build_env_geometries(*cfg, own.data(), cfg->n_envs, env_geo, env_set, err)) return fail(RLFC_EINVAL, err);
    }
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(RLFC_ENODEV, "no CUDA device available (rlfc has no CPU fallback)");
  rlfc_env* E = new rlfc_env();
  E->cfg = *cfg;
  if (cfg->init_bdim_path) E->init_path = cfg->init_bdim_path;
  E->cfg.init_bdim_path = nullptr;
  E->env_mode = cfg->env_params != nullptr || cfg->n_param_sets > 0;
  E->cfg.env_params = nullptr;              // (copied into E->params below)
  E->cfg.param_sets = nullptr;              // (copied into E->lib_params below)
  if (cfg->n_sensors > 0 && cfg->sensors) E->sensor_table.assign(cfg->sensors, cfg->sensors + cfg->n_sensors);
  E->cfg.sensors = nullptr;                 // (resolved into E->sens below)
  int rc = RLFC_OK;
  auto bail = [&](int code) { rlfc_env_destroy(E); return code; };

  if (cfg->device >= 0) {
    if (cfg->device >= ndev) { delete E; return fail(RLFC_ENODEV, "device ordinal out of range"); }
    E->device = cfg->device;
  } else if (cudaGetDevice(&E->device) != cudaSuccess) {
    delete E;
    return fail(RLFC_ENODEV, "cudaGetDevice failed");
  }
  if (cudaSetDevice(E->device) != cudaSuccess) { delete E; return fail(RLFC_ENODEV, "cudaSetDevice failed"); }
  if (E->cfg.n_devices < 1) E->cfg.n_devices = 1;
  if (E->cfg.n_devices > 1) {
    // slab mode: ONE domain on devices device .. device + n_devices - 1 (BASELINE config 5)
    if (cfg->n_envs != 1) { delete E; return fail(RLFC_EINVAL, "slab mode (n_devices > 1) advances one environment"); }
    if (E->device + E->cfg.n_devices > ndev) { delete E; return fail(RLFC_ENODEV, "n_devices exceeds the devices present"); }
    if (cfg->stream) { delete E; return fail(RLFC_EINVAL, "slab mode creates its own streams"); }
    std::vector<int> devs;
    for (int d = 0; d < E->cfg.n_devices; d++) devs.push_back(E->device + d);
    std::string err;
    int vrc = E->vmm.init(devs, err);
    if (vrc) { delete E; return fail(vrc, err); }
    cudaSetDevice(E->device);
  }
  if (cfg->stream) {
    E->stream = (cudaStream_t)cfg->stream;
  } else {
    if (cudaStreamCreateWithFlags(&E->stream, cudaStreamNonBlocking) != cudaSuccess) {
      delete E;
      return fail(RLFC_ECUDA, "cudaStreamCreate failed");
    }
    E->own_stream = true;
  }

  {
    std::string err;
    rc = build_geometry(E->cfg, E->geo, err);
    if (rc) { g_err = err; return bail(rc); }
  }
  const Geometry& g = E->geo;
  SolverParams& sp = E->sp;
  const int B = cfg->n_envs;
  sp.B = B;
  sp.n = g.n; sp.m = g.m; sp.P = round_up(g.m, 8);
  sp.stride = (size_t)round_up(sp.n * sp.P, 32);
  sp.dt = g.dt; sp.nu = g.nu;
  sp.dRD = g.dR * g.D;
  sp.dt_over_res = g.dt / g.resolution;
  sp.action_scale = cfg->action_scale;
  sp.inv_cells = (float)((g.n - 2) * (g.m - 2));
  sp.mg_tol = g.mg_tol;
  const bool force_wave = std::getenv("RLFC_SMOOTHER") && std::string(std::getenv("RLFC_SMOOTHER")) == "wave";
  // RLFC_SMOOTHER=chain: the chained strip smoother (smooth_chain.cuh) on every level but the coarsest (tests); by default it
  // takes the levels that are too wide for the row pipeline
  const bool force_chain = std::getenv("RLFC_SMOOTHER") && std::string(std::getenv("RLFC_SMOOTHER")) == "chain";
  const bool slab = E->cfg.n_devices > 1;   // slab mode: level 0 always runs the chained smoother (its sweeps span devices)
  const bool adaptive = cfg->adaptive_dt == 1;
  const bool env_mode = E->env_mode;
  const bool per_env = adaptive || env_mode;   // per-environment dt, hierarchy and geometry slots
  sp.adaptive = adaptive ? 1 : 0;
  sp.per_env = per_env ? 1 : 0;
  int chain_min_cols = 33;            // RLFC_CHAIN_MIN_COLS: coarse levels at least this wide follow a chained level 0 (levels of
                                      // at most 32 columns are faster in the one-CTA kernel's single-warp smoother: 521 -> 528 steps/s)
  if (const char* ev = std::getenv("RLFC_CHAIN_MIN_COLS")) chain_min_cols = std::max(1, std::atoi(ev));
  sp.nlevels = (int)g.levels.size();
  sp.resolution = cfg->resolution; sp.substeps = cfg->substeps; sp.mg_max_iters = cfg->mg_max_iters;
  sp.init_time = cfg->init_time; sp.episode_time = cfg->episode_time;
  if (sp.nlevels > kMaxLevels) return bail(fail(RLFC_EGRID, "too many multigrid levels"));
  if (sp.nlevels < 2) return bail(fail(RLFC_EGRID, "grid has no coarse level"));

#define TRY(x) do { rc = (x); if (rc) return bail(rc); } while (0)
  // static level-0 fields
  if (!per_env) {
    TRY(upload_static(E, g.c_x, g.n, g.m, sp.P, &sp.c_x));
    TRY(upload_static(E, g.c_y, g.n, g.m, sp.P, &sp.c_y));
  }
  // geometry slots: one per environment, then one per distinct library set
  const int nslots = B + (int)lib_geo.size();
  if (env_mode) {
    // one geometry slot per environment: del and the body-velocity basis at e * stride (filled by upload_env_geometry)
    const float** slot[10] = {&sp.del_x, &sp.del_y, &sp.w1_x, &sp.w2_x, &sp.ry1_x, &sp.ry2_x, &sp.w1_y, &sp.w2_y, &sp.rx1_y, &sp.rx2_y};
    for (const float** f : slot) {
      float* d = nullptr;
      TRY(E->dmalloc(&d, sp.stride * nslots));
      *f = d;
    }
  } else {
  TRY(upload_static(E, g.w1_x, g.n, g.m, sp.P, &sp.w1_x));
  TRY(upload_static(E, g.w2_x, g.n, g.m, sp.P, &sp.w2_x));
  TRY(upload_static(E, g.ry1_x, g.n, g.m, sp.P, &sp.ry1_x));
  TRY(upload_static(E, g.ry2_x, g.n, g.m, sp.P, &sp.ry2_x));
  TRY(upload_static(E, g.w1_y, g.n, g.m, sp.P, &sp.w1_y));
  TRY(upload_static(E, g.w2_y, g.n, g.m, sp.P, &sp.w2_y));
  TRY(upload_static(E, g.rx1_y, g.n, g.m, sp.P, &sp.rx1_y));
  TRY(upload_static(E, g.rx2_y, g.n, g.m, sp.P, &sp.rx2_y));
  }
  // multigrid hierarchy
  for (int l = 0; l < sp.nlevels; l++) {
    const HostLevel& H = g.levels[l];
    DevLevel& L = sp.lev[l];
    L.n = H.n; L.m = H.m; L.P = round_up(H.m, 8);
    L.stride = (size_t)round_up(L.n * L.P, 32);
    if (per_env) {
      // one copy per environment at the level's stride, rebuilt on the device from each environment's dt
      float* a[4] = {nullptr, nullptr, nullptr, nullptr};
      for (int k = 0; k < 4; k++) TRY(E->dmalloc(&a[k], L.stride * B));
      L.lx = a[0]; L.ly = a[1]; L.inv = a[2]; L.diag = a[3];
    } else {
      TRY(upload_static(E, H.lx, H.n, H.m, L.P, &L.lx));
      TRY(upload_static(E, H.ly, H.n, H.m, L.P, &L.ly));
      TRY(upload_static(E, H.inv, H.n, H.m, L.P, &L.inv));
      TRY(upload_static(E, H.diag, H.n, H.m, L.P, &L.diag));
    }
    {  // pre-skewed coefficient table for the row-pipelined smoother (layout: solver.h RowTab)
      const int ni = H.n - 2, mj = H.m - 2;
      const int C = (mj + 31) / 32, K = (3 * C + 1 + 3) / 4, nl = (mj + C - 1) / C;
      const int front = 10 /*kTabFront*/, entries = rows_table_entries(ni, nl);
      // levels too wide for the row pipeline (more than 8 columns per lane on level 0, 4 on coarse levels) are smoothed by
      // the wavefront fallback (smooth_wave.cuh); RLFC_SMOOTHER=wave forces it everywhere (tests)
      L.wave = (C > (l == 0 ? 8 : 4)) || force_wave;
      L.ch = ChainLevel{};
      // levels the row pipeline could take, but which are faster chained when one domain has the GPU to itself
      const bool prefer_chain = sp.chain_levels > 0 && l >= 1 && mj >= chain_min_cols;
      if (!force_wave && l < sp.nlevels - 1 && (force_chain || L.wave || prefer_chain || (slab && l == 0)) && sp.chain_levels == l) {
        // chained strip smoother: static coefficient table in the strip-skewed layout (solver.h ChainLevel)
        ChainLevel& ch = L.ch;
        ch.on = 1; ch.NS = (mj + 31) / 32; ch.T = round_up(ni + 33, 32) + 32;   // (>= ni + 34; whole batches of up to 32 steps stay inside a strip)
        ch.s0 = 0; ch.ns_loc = ch.NS;
        ch.sk_stride = (size_t)ch.NS * ch.T * 32;
        std::vector<float4> ct(ch.sk_stride, make_float4(0.f, 0.f, 0.f, 0.f));
        for (int s = 0; s < ch.NS; s++)
          for (int t = 0; t < ch.T; t++)
            for (int ln = 0; ln < 32; ln++) {
              const int i = t - ln, j = 32 * s + ln + 1;
              if (j > mj || i < 0 || i > ni) continue;
              float4 v = make_float4(H.lx[(size_t)(i + 1) * H.m + j], 0.f, 0.f, 0.f);   // row 0 only feeds lxW of row 1
              if (i >= 1) {
                const size_t k = (size_t)i * H.m + j;
                v.y = H.ly[k]; v.z = H.ly[k + 1]; v.w = -H.inv[k];
                if (H.diag[k] != -(H.lx[k] + H.lx[k + H.m] + H.ly[k] + H.ly[k + 1]))
                  return bail(fail(RLFC_EGRID, "PoissonMatrix diagonal is not the plain coefficient sum"));
              }
              ct[((size_t)s * ch.T + t) * 32 + ln] = v;
            }
        TRY(upload_vec(E, ct, &ch.ct));
        TRY(E->dmalloc(&ch.rsk, ch.sk_stride * B));
        for (int gsw = 0; gsw < 5; gsw++) TRY(E->dmalloc(&ch.dsk[gsw], ch.sk_stride * B));
        ch.TE = ch.T + 72;               // smooth_chain3.cuh: consumer steps 0 .. T-1 behind kC2EdgePad, producer indices up to T + 62
        ch.edge_arr = (size_t)B * ch.NS * ch.TE;
        TRY(E->dmalloc(&ch.edge, ch.edge_arr * 10 + 64));
        L.wave = 0;
        sp.chain_levels = l + 1;
      }
      L.rt.C = C; L.rt.K = K; L.rt.entries = 0; L.rt.copies = 1; L.rt.T = nullptr;
      if (per_env && !L.wave && !L.ch.on) {
        // one table per environment (k_poisson_rebuild*); a view of the batch sets `copies` to its B, so the smoother's
        // CTA e (= environment e of the view) reads table e
        float4* T = nullptr;
        TRY(E->dmalloc(&T, (size_t)entries * K * 32 * B));
        L.rt.entries = entries; L.rt.copies = B; L.rt.T = T;
      } else if (!L.wave && !L.ch.on) {
      std::vector<float4> T((size_t)entries * K * 32, make_float4(0.f, 0.f, 0.f, 0.f));
      std::vector<float> f(4 * K);
      for (int e = 0; e < entries; e++)
        for (int ln = 0; ln < 32; ln++) {
          const int row = (e - front) - ln, j0 = C * ln + 1;
          std::fill(f.begin(), f.end(), 0.f);
          for (int c = 0; c < C; c++) {
            const int j = j0 + c;
            if (row >= 1 && row <= ni + 1 && j <= mj) f[2 * C + 1 + c] = H.lx[(size_t)row * H.m + j];
            if (row >= 1 && row <= ni && j <= mj) {
              f[C + 1 + c] = -H.inv[(size_t)row * H.m + j];
              // the smoother recomputes the diagonal as PoissonMatrix does (PoissonMatrix.pde:46-48); it must agree
              const size_t k = (size_t)row * H.m + j;
              if (H.diag[k] != -(H.lx[k] + H.lx[k + H.m] + H.ly[k] + H.ly[k + 1]))
                return bail(fail(RLFC_EGRID, "PoissonMatrix diagonal is not the plain coefficient sum"));
            }
          }
          for (int c = 0; c <= C; c++) {
            const int j = j0 + c;
            if (row >= 1 && row <= ni && j <= mj + 1) f[c] = H.ly[(size_t)row * H.m + j];
          }
          for (int k = 0; k < K; k++)
            T[((size_t)e * K + k) * 32 + ln] = make_float4(f[4 * k], f[4 * k + 1], f[4 * k + 2], f[4 * k + 3]);
        }
      // the table is shared by every environment and all CTAs walk it in near lockstep, so each 128-byte line is
      // requested by ~148 SMs at once from the ONE L2 slice that owns it; kTabCopies copies at different addresses
      // spread that burst over several slices (CTA e reads copy e % kTabCopies)
      const int copies = 8;
      std::vector<float4> Trep;
      Trep.reserve(T.size() * copies);
      for (int c = 0; c < copies; c++) Trep.insert(Trep.end(), T.begin(), T.end());
      L.rt.C = C; L.rt.K = K; L.rt.entries = entries; L.rt.copies = copies;
      TRY(upload_vec(E, Trep, &L.rt.T));
      }
    }
    TRY(E->dmalloc(&L.r, L.stride * B));
    TRY(E->dmalloc(&L.x, L.stride * B));
    TRY(E->dmalloc(&L.d, L.stride * B));
    L.r2 = nullptr;
    L.w = nullptr;
    if (l == 0 && L.wave) TRY(E->dmalloc(&L.w, L.stride * B));
  }
  if (per_env) {
    // the per-environment hierarchy exists for the row-pipeline and single-warp smoothers only
    const std::string what = adaptive ? "adaptive_dt" : cfg->env_params ? "env_params" : "param_sets";
    if (sp.chain_levels > 0)
      return bail(fail(RLFC_EINVAL, what + " is not available with the chained strip smoother (a level too wide for the "
                                           "row pipeline, or RLFC_SMOOTHER=chain)"));
    for (int l = 0; l < sp.nlevels; l++)
      if (sp.lev[l].wave)
        return bail(fail(RLFC_EINVAL, what + " is not available with the wavefront smoother (RLFC_SMOOTHER=wave, or a "
                                             "coarsest level wider than the row pipeline)"));
    if (!env_mode) {   // one geometry slot, shared by every environment
      TRY(upload_static(E, g.del_x, g.n, g.m, sp.P, &sp.del_x));
      TRY(upload_static(E, g.del_y, g.n, g.m, sp.P, &sp.del_y));
    }
    sp.c_x = sp.lev[0].lx; sp.c_y = sp.lev[0].ly;   // c = del*(1*dt) is level 0's lower (geometry.cpp)
  }
  {
    std::vector<BandFace> bx, by;
    band_lists(g, bx, by);
    sp.nband_x = (int)bx.size(); sp.nband_y = (int)by.size();
    if (env_mode) sp.nband_x = sp.nband_y = band_capacity(E->cfg);   // every slot's lists at this capacity
    // the two-phase setBC kernel fetches rows 1, n-2 and columns 1, m-2 before the band is blended: no band face may
    // sit on them, and the shared-memory image of the lines (+ the blended band) must fit one CTA.  The kernel strides over
    // longer lines too, but ONE CTA blending the band of a 2048x1024 domain is slower than the grid-wide k_band_blend + the
    // literal kernels (measured: 122 vs 52 us), so large grids keep those.
    sp.fast_bc = (g.n <= 1024 && g.m <= 1024 &&
                  sizeof(float) * (2 * (3 * (size_t)g.m + 2 * (size_t)g.n) + bx.size() + by.size()) <= 200 * 1024) ? 1 : 0;
    // (per-environment sets are validated to keep the band off those lines; the scalar config's band is not used then)
    if (!env_mode)
      for (const auto* v : {&bx, &by})
        for (const BandFace& f : *v)
          if (f.i <= 1 || f.i >= g.n - 2 || f.j <= 1 || f.j >= g.m - 2) sp.fast_bc = 0;
    if (env_mode)
      sp.fast_bc = (g.n <= 1024 && g.m <= 1024 &&
                    sizeof(float) * (2 * (3 * (size_t)g.m + 2 * (size_t)g.n) + (size_t)sp.nband_x + sp.nband_y) <= 200 * 1024) ? 1 : 0;
    if (const char* ev = std::getenv("RLFC_FAST_BC")) sp.fast_bc = sp.fast_bc && std::atoi(ev) != 0;
    if (env_mode) {
      BandFace* d = nullptr;
      TRY(E->dmalloc(&d, (size_t)sp.nband_x * nslots)); sp.band_x = d;
      TRY(E->dmalloc(&d, (size_t)sp.nband_y * nslots)); sp.band_y = d;
    } else {
      TRY(upload_vec(E, bx, &sp.band_x));
      TRY(upload_vec(E, by, &sp.band_y));
    }
    TRY(E->dmalloc(&sp.band_tmp, (size_t)B * (sp.nband_x + sp.nband_y)));
  }
  // per-environment parameters: the scalar config's for every environment unless env_params gives them
  E->params.assign(B, params_of(E->cfg));
  E->dt0.assign(B, g.dt);
  E->h_nu.assign(B, g.nu); E->h_dRD.assign(B, g.dR * g.D);
  E->h_nbx.assign(B, sp.nband_x); E->h_nby.assign(B, sp.nband_y);
  if (per_env) {
    std::vector<int> slot(B, 0);
    if (env_mode) {
      for (int e = 0; e < B; e++) {
        slot[e] = e;
        TRY(upload_env_geometry(E, e, cfg->env_params ? cfg->env_params[e] : params_of(E->cfg), env_geo[env_set[e]]));
      }
      // the library: set s in slot B + (its first equal set's index among the distinct ones)
      for (size_t u = 0; u < lib_geo.size(); u++) TRY(upload_slot_geometry(E, B + (int)u, lib_geo[u]));
      if (cudaStreamSynchronize(E->stream) != cudaSuccess) return bail(fail(RLFC_ECUDA, "geometry upload failed"));
      E->lib_params.assign(cfg->param_sets, cfg->param_sets + cfg->n_param_sets);
      for (int k = 0; k < cfg->n_param_sets; k++) {
        const EnvGeometry& G = lib_geo[lib_set[k]];
        LibSet L{};
        L.slot = B + lib_set[k];
        L.nbx = (int)G.bx.size(); L.nby = (int)G.by.size();
        L.nu = G.g.nu; L.dRD = G.g.dR * G.g.D; L.dt0 = G.g.dt;
        param_bits(cfg->param_sets[k], L.bits);
        E->h_lib.push_back(L);
      }
      env_geo.clear();
      lib_geo.clear();
    }
    if (!E->h_lib.empty()) {
      E->lib.L = (int)E->h_lib.size();
      TRY(upload_vec(E, E->h_lib, &E->lib.sets));
      TRY(E->dmalloc(&E->lib.env_set, B, false));
      TRY(E->dmalloc(&E->set_env, B)); TRY(E->dmalloc(&E->set_ids, B));
      E->h_env_set.assign(B, -1);
      if (cudaMemcpyAsync(E->lib.env_set, E->h_env_set.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream) != cudaSuccess)
        return bail(fail(RLFC_ECUDA, "library table upload failed"));
    }
    int* d = nullptr;
    TRY(E->dmalloc(&d, B)); sp.env_slot = d;
    TRY(E->dmalloc(&d, B)); sp.env_nband_x = d;
    TRY(E->dmalloc(&d, B)); sp.env_nband_y = d;
    TRY(E->dmalloc(&E->d_skip, B));
    float* f = nullptr;
    TRY(E->dmalloc(&f, B)); sp.env_nu = f;
    TRY(E->dmalloc(&f, B)); sp.env_dRD = f;
    if (env_mode) {   // rlfc_env_reset_params_device
      TRY(E->dmalloc(&E->pr.params, B)); TRY(E->dmalloc(&E->pr.status, B)); TRY(E->dmalloc(&E->pr.refused, B));
      circle_vertex_factors(E->circle.c, E->circle.s);
    }
    if (cudaMemcpyAsync(d = const_cast<int*>(sp.env_slot), slot.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream) != cudaSuccess)
      return bail(fail(RLFC_ECUDA, "slot table upload failed"));
    TRY(upload_env_scalars(E));
  }
  {
    std::vector<ForcePt> fp;
    for (const ForceEdge& fe : g.force_edges) fp.push_back({fe.at.i, fe.at.j, fe.at.s, fe.at.t, fe.l, fe.nx, fe.ny});
    std::vector<SamplePt> pp;
    for (const Sample& s : g.probes) pp.push_back({s.i, s.j, s.s, s.t});
    sp.nforce = (int)fp.size(); sp.nprobe = (int)pp.size();
    if (sp.nforce > 64 || sp.nprobe > 64) return bail(fail(RLFC_EINVAL, "too many force/probe points"));
    TRY(upload_vec(E, fp, &sp.force_pts));
    TRY(upload_vec(E, pp, &sp.probe_pts));
    // sensors: resolved once to their cell and fractions (Field.linear with the field's btype = the sensor's field code)
    std::vector<SensorPt> sv;
    for (int k = 0; k < cfg->n_sensors; k++) {
      const rlfc_sensor& s = cfg->sensors[k];
      const Sample a = resolve_sample(g.n, g.m, s.x, s.y, s.field);
      sv.push_back({a.i, a.j, a.s, a.t, s.field});
    }
    E->sens.n = (int)sv.size();
    if (E->sens.n > 0) {
      TRY(upload_vec(E, sv, &E->sens.pts));
      TRY(E->dmalloc(&E->sens.out, (size_t)B * E->sens.n));
    }
  }
  // per-env fields
  const size_t S = sp.stride * B;
  TRY(E->dmalloc(&E->uAx, S)); TRY(E->dmalloc(&E->uAy, S));
  TRY(E->dmalloc(&E->uBx, S)); TRY(E->dmalloc(&E->uBy, S));
  TRY(E->dmalloc(&E->uCx, S)); TRY(E->dmalloc(&E->uCy, S));
  TRY(E->dmalloc(&E->init_ux, sp.stride)); TRY(E->dmalloc(&E->init_uy, sp.stride)); TRY(E->dmalloc(&E->init_p, sp.stride));
  if (cfg->stats_every > 0) {   // flow statistics (solver.h FlowStats), all zero: no samples yet
    FlowStats& f = E->fs;
    f.every = cfg->stats_every;
    TRY(E->dmalloc(&f.sums, (size_t)kNumStats * sp.stride * B));
    TRY(E->dmalloc(&f.count, B)); TRY(E->dmalloc(&f.step, B)); TRY(E->dmalloc(&f.ticket, B));
  }
  // per-env scalars
  sp.rr_blocks = 0;
  sp.tiny = 1;
  if (const char* ev = std::getenv("RLFC_TINY")) sp.tiny = std::atoi(ev) != 0;
  sp.resid_march = 1;
  if (const char* ev = std::getenv("RLFC_RESID")) sp.resid_march = std::strcmp(ev, "tile") != 0;
  // (the kernel pairs level-0 rows / columns for the restriction, which build_geometry's even level 0 guarantees; a batch of
  // fewer than ~8 Mi cells does not give the marching kernel enough warps -- one 2048x1024 domain: 38 vs 31 us)
  if ((long long)B * (g.n - 2) * (g.m - 2) < (8ll << 20)) sp.resid_march = 0;
  if (const char* ev = std::getenv("RLFC_RESID")) if (std::strcmp(ev, "march") == 0) sp.resid_march = 1;
  // slab mode keeps the tile kernel: the marching kernel bulk-copies its rows (cp.async.bulk), which here would read
  // other devices' memory through the shared address range, a combination that has not been run on several devices
  if (slab) sp.resid_march = 0;
  int n_groups = cfg->n_groups;
  if (const char* ev = std::getenv("RLFC_GROUPS")) n_groups = std::atoi(ev);
  // (measured, 256 default-grid envs, final round-2 kernels: 1 group 7 120, 2 groups 7 333-7 364, 3 groups 7 230, 4 groups 7 242
  // env-steps/s device-resident, end-to-end figures within 1 % of each other.  Batches larger than one wave of the
  // one-CTA-per-environment kernels keep 4 groups.)
  // 512 envs: 2 groups 8 230, 4 groups 8 078 env-steps/s; larger batches were only measured with 4 groups.
  if (n_groups <= 0) n_groups = B > 512 ? 4 : (B >= 128 ? 2 : 1);
  n_groups = std::min(n_groups, B);
  if (slab) n_groups = 1;
  if (const char* ev = std::getenv("RLFC_NO_GRAPH")) E->use_graph = std::atoi(ev) == 0;
  TRY(E->dmalloc(&sp.sc.flow_t, B));
  TRY(E->dmalloc(&sp.sc.xi, 2 * B)); TRY(E->dmalloc(&sp.sc.t, B)); TRY(E->dmalloc(&sp.sc.force, 2 * B));
  TRY(E->dmalloc(&sp.sc.probes, (size_t)B * RLFC_NUM_PROBES));
  TRY(E->dmalloc(&sp.sc.callLearn, B)); TRY(E->dmalloc(&sp.sc.Cd, B)); TRY(E->dmalloc(&sp.sc.Cl, B));
  TRY(E->dmalloc(&sp.sc.obs, 2 * B)); TRY(E->dmalloc(&sp.sc.active, B)); TRY(E->dmalloc(&sp.sc.iters, 2 * B));
  TRY(E->dmalloc(&sp.sc.frozen, B)); TRY(E->dmalloc(&sp.sc.non_finite, B)); TRY(E->dmalloc(&sp.sc.n_running, 1));
  sp.sc.rr_part = nullptr;
  TRY(E->dmalloc(&sp.sc.psum, B));
  TRY(E->dmalloc(&sp.sc.dt, B));
  if (cfg->n_snapshots > 0) {
    // snapshot slots (solver.h SnapSlots); the zeroed headers mark every slot unwritten
    SnapSlots& s = E->snap;
    s.S = cfg->n_snapshots;
    TRY(E->dmalloc(&s.ux, sp.stride * s.S)); TRY(E->dmalloc(&s.uy, sp.stride * s.S)); TRY(E->dmalloc(&s.p, sp.stride * s.S));
    TRY(E->dmalloc(&s.rec, (size_t)kSnapWords * s.S)); TRY(E->dmalloc(&s.hdr, (size_t)kSnapHdr * s.S));
    if (E->sens.n > 0) TRY(E->dmalloc(&s.sens, (size_t)E->sens.n * s.S));
    TRY(E->dmalloc(&s.env_par, (size_t)5 * B)); TRY(E->dmalloc(&s.refused, B));
    TRY(E->dmalloc(&E->snap_env, std::max(B, s.S))); TRY(E->dmalloc(&E->snap_slot, std::max(B, s.S)));
    TRY(upload_snapshot_params(E));
  }
  {
    // Field.sum: segment summaries (exact_sum.cuh) or the plain dependent-add chain (k_psum).  The chain costs
    // 6 cycles per cell of pure latency whatever the batch size and next to no issue slots; the summaries cost
    // throughput proportional to batch x cells and a short serial pass.  Measured on B200 (default grid): summaries
    // +2.5 % step throughput at 256 envs, -8 % at 512.  Both costs are proportional to the cells per environment (chain: ~3 ns
    // per cell of latency; summaries: ~8 ps per cell and environment of throughput), so the choice depends on the batch size
    // alone: summaries up to 320 environments, whatever the grid (one 8192x4096 domain: 88 ms per solve as a chain).
    // RLFC_PSUM=serial | parallel overrides.
    const char* ev = std::getenv("RLFC_PSUM");
    const long long N = (long long)(g.n - 2) * (g.m - 2);
    sp.xs_nseg = (int)((N + 31) / 32);
    sp.xs_nchunks = (sp.xs_nseg + 255) / 256;
    sp.xs_nbatches = (sp.xs_nseg + 31) / 32;
    sp.xs_ctot = nullptr; sp.xs_recs = nullptr;
    // (the prediction of a zero-mean field's running sum misses the accumulator's binade more often the longer the sum: a second
    // refinement of the prediction pays from about 8 Mi cells on, profiles/r02_field_sum_large.md)
    sp.xs_passes = sp.xs_nbatches >= 8192 ? 3 : 2;
    if (const char* ev3 = std::getenv("RLFC_XS_PASSES")) sp.xs_passes = std::atoi(ev3) >= 3 ? 3 : 2;
    if (const char* ev2 = std::getenv("RLFC_XS_REDO")) sp.xs_flags |= std::strcmp(ev2, "serial") == 0 ? 1 : 0;
    const bool xs_refine = !(std::getenv("RLFC_XS_REFINE") && std::atoi(std::getenv("RLFC_XS_REFINE")) == 0);
    TRY(E->dmalloc(&sp.xs_stats, (size_t)8 * B));
    bool summaries = B <= 320 || slab;
    E->home_only = true;                            // Field.sum runs on device 0 only
    if (ev && std::strcmp(ev, "serial") == 0) summaries = false;
    if (ev && std::strcmp(ev, "parallel") == 0) summaries = true;
    if (summaries) {
      TRY(E->dmalloc(&sp.xs_ctot, (size_t)sp.xs_nchunks * B));
      TRY(E->dmalloc(&sp.xs_cflag, (size_t)sp.xs_nchunks * B));
      TRY(E->dmalloc(&sp.xs_epoch, (size_t)B));
      TRY(E->dmalloc(&sp.xs_recs, (size_t)sp.xs_nbatches * 192 * B));
      sp.xs_blk = nullptr;
      if (sp.xs_nbatches >= 256) {
        TRY(E->dmalloc(&sp.xs_blk, (size_t)((sp.xs_nbatches + 31) / 32) * 256 * B));
        if (xs_refine) {
        TRY(E->dmalloc(&sp.xs_pred, (size_t)sp.xs_nbatches * B));
        TRY(E->dmalloc(&sp.xs_inc, (size_t)sp.xs_nbatches * B));
        TRY(E->dmalloc(&sp.xs_corr, (size_t)sp.xs_nbatches * B));
        }
      }
    }
    E->home_only = false;
  }
  TRY(E->dmalloc(&sp.sc.any_active, n_groups + 1));   // one word per view of the batch: the groups and the whole batch
  if (sp.chain_levels > 0) {
    sp.rr_chain_n = chain_incr_blocks(g.n - 2, sp.lev[0].ch.NS);
    TRY(E->dmalloc(&sp.rr_chain, (size_t)sp.rr_chain_n * B));
    TRY(E->dmalloc(&sp.rr_count, (size_t)B));
    // ticket counters: one per (view of the batch, level); views = the groups and the whole batch
    TRY(E->dmalloc(&E->chain_tickets, (size_t)(n_groups + 1) * kMaxLevels));
  }
  TRY(E->dmalloc(&E->d_actions, 2 * B)); TRY(E->dmalloc(&E->d_obs, 2 * B)); TRY(E->dmalloc(&E->d_reward, B));
  TRY(E->dmalloc(&E->d_done, B));
  TRY(E->dmalloc(&E->pB, S));
  {
    const int C0 = sp.lev[0].rt.C, mj0 = g.m - 2;
    sp.rsk_stride = (sp.lev[0].wave || sp.lev[0].ch.on) ? 32 : (size_t)round_up((int)rows_skew_floats(C0, g.n - 2, (mj0 + C0 - 1) / C0), 32);
    TRY(E->dmalloc(&sp.rsk, sp.rsk_stride * B));
  }
#undef TRY
  auto hostalloc = [&](void** p, size_t bytes) { return cudaMallocHost(p, bytes) == cudaSuccess; };
  if (!hostalloc((void**)&E->h_actions, 2 * B * sizeof(float)) || !hostalloc((void**)&E->h_obs, 2 * B * sizeof(float)) ||
      !hostalloc((void**)&E->h_reward, B * sizeof(float)) || !hostalloc((void**)&E->h_force, 2 * B * sizeof(float)) ||
      !hostalloc((void**)&E->h_probes, (size_t)B * RLFC_NUM_PROBES * sizeof(float)) ||
      !hostalloc((void**)&E->h_done, B * sizeof(int)) || !hostalloc((void**)&E->h_any, sizeof(int)))
    return bail(fail(RLFC_ENOMEM, "cudaMallocHost failed"));

  // views of the batch: the environment groups (contiguous, each on its own stream; group 0 on the handle's), then the
  // whole batch on the handle's stream
  if ((rc = configure_kernels(sp))) return bail(fail(RLFC_ECUDA, "kernel attribute configuration failed"));
  E->groups.resize(n_groups);
  for (int g = 0; g < n_groups; g++) {
    Group& G = E->groups[g];
    const int e0 = (int)((long long)B * g / n_groups), e1 = (int)((long long)B * (g + 1) / n_groups);
    make_view(E, e0, e1 - e0, g, G);
    if (g == 0) G.st = E->stream;
    else if (cudaStreamCreateWithFlags(&G.st, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(RLFC_ECUDA, "cudaStreamCreate failed"));
    if (cudaEventCreateWithFlags(&G.done, cudaEventDisableTiming) != cudaSuccess) return bail(fail(RLFC_ECUDA, "cudaEventCreate failed"));
  }
  make_view(E, 0, B, n_groups, E->whole);
  E->whole.st = E->stream;
  if (sp.chain_levels > 0) {
    // every counter starts at one full launch's worth of tickets, so that launch serials (the tags) start at 1 and
    // never equal the 0 the arrays are initialised with
    std::vector<unsigned long long> init((size_t)(n_groups + 1) * kMaxLevels, 0ull);
    for (int gv = 0; gv <= n_groups; gv++)
      for (int l = 0; l < sp.chain_levels; l++) {
        const int Bv = gv < n_groups ? E->groups[gv].B : B;
        init[(size_t)gv * kMaxLevels + l] = (unsigned long long)Bv * 4ull * (unsigned)sp.lev[l].ch.ns_loc;
      }
    if (cudaMemcpyAsync(E->chain_tickets, init.data(), init.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, E->stream) != cudaSuccess ||
        cudaStreamSynchronize(E->stream) != cudaSuccess)
      return bail(fail(RLFC_ECUDA, "ticket initialisation failed"));
  }
  if (slab) {
    // per-device views: the same arrays (one address range), each device its row blocks / strips, its own streams,
    // ticket counters and barrier epoch in its own memory
    if (!sp.lev[0].ch.on) return bail(fail(RLFC_EGRID, "slab mode needs the chained smoother on level 0"));
    const int nd = E->cfg.n_devices;
    unsigned* bar_count = nullptr;
    E->home_only = true;
    if ((rc = E->dmalloc(&bar_count, 1))) return bail(rc);
    E->home_only = false;
    if (cudaStreamSynchronize(E->stream) != cudaSuccess) return bail(fail(RLFC_ECUDA, "initialisation failed"));
    E->slab.resize(nd);
    for (int d = 0; d < nd; d++) {
      rlfc_env::SlabDev& D = E->slab[d];
      D.device = E->device + d;
      if (cudaSetDevice(D.device) != cudaSuccess) return bail(fail(RLFC_ENODEV, "cudaSetDevice failed"));
      if (d == 0) D.st = E->stream;
      else if (cudaStreamCreateWithFlags(&D.st, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(RLFC_ECUDA, "cudaStreamCreate failed"));
      if (d > 0 && configure_kernels(sp)) return bail(fail(RLFC_ECUDA, "kernel attribute configuration failed"));
      unsigned long long* tickets = nullptr;
      unsigned* epoch = nullptr;
      if (cudaMalloc(&tickets, sizeof(unsigned long long) * kMaxLevels) != cudaSuccess || cudaMalloc(&epoch, sizeof(unsigned)) != cudaSuccess)
        return bail(fail(RLFC_ENOMEM, "cudaMalloc failed"));
      D.local[0] = tickets; D.local[1] = epoch;
      D.sp = E->whole.sp;
      D.sp.slab_n = nd; D.sp.slab_rank = d;
      std::vector<unsigned long long> init(kMaxLevels, 0ull);
      for (int l = 0; l < sp.chain_levels; l++) {
        ChainLevel& ch = D.sp.lev[l].ch;
        ch.s0 = (int)((long long)ch.NS * d / nd);
        ch.ns_loc = (int)((long long)ch.NS * (d + 1) / nd) - ch.s0;
        ch.ticket = tickets + l;
        ch.tag_hi = 1u << 26;                                  // the same launch tags on every device
        init[l] = (unsigned long long)B * 4ull * (unsigned)std::max(ch.ns_loc, 1);
      }
      if (cudaMemcpy(tickets, init.data(), sizeof(unsigned long long) * kMaxLevels, cudaMemcpyHostToDevice) != cudaSuccess ||
          cudaMemset(epoch, 0, sizeof(unsigned)) != cudaSuccess)
        return bail(fail(RLFC_ECUDA, "slab initialisation failed"));
      D.spB = D.sp;
      D.spB.lev[0].x = E->pB;
      D.bar.count = bar_count; D.bar.epoch = epoch; D.bar.n = (unsigned)nd;
    }
    cudaSetDevice(E->device);
  }
  if (cudaStreamCreateWithFlags(&E->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&E->fork_ev, cudaEventDisableTiming) != cudaSuccess)
    return bail(fail(RLFC_ECUDA, "stream/event creation failed"));

  if ((rc = load_initial_state(E))) return bail(rc);
  if ((rc = rlfc_env_reset(E, nullptr, B, 1))) return bail(rc);
  if (per_env) {   // the hierarchy of the initial dt (d_skip: all zero)
    E->launches += launch_poisson_rebuild0(E->whole.sp, E->d_skip, E->stream);
    E->launches += launch_poisson_rebuild_coarse(E->whole.sp, E->d_skip, E->stream);
    if (cudaGetLastError() != cudaSuccess) return bail(fail(RLFC_ECUDA, "initial Poisson hierarchy build failed"));
  }
  if (cudaStreamSynchronize(E->stream) != cudaSuccess) return bail(fail(RLFC_ECUDA, "initialisation failed"));
  *out = E;
  return RLFC_OK;
}

int rlfc_env_reset(rlfc_env* E, const int* env_ids, int n, int reset_accumulators) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  SolverParams& sp = E->sp;
  if (!env_ids) n = sp.B;
  if (n < 0 || n > sp.B) return fail(RLFC_EINVAL, "bad env count");
  for (int k = 0; env_ids && k < n; k++)
    if (env_ids[k] < 0 || env_ids[k] >= sp.B) return fail(RLFC_EINVAL, "env id out of range");
  CU(cudaSetDevice(E->device));
  int rc;
  if ((rc = sync_env_sets(E))) return rc;   // (dt0: the set each environment holds now)
  if ((rc = broadcast_field(E, E->uAx, E->init_ux, env_ids, n))) return rc;
  if ((rc = broadcast_field(E, E->uAy, E->init_uy, env_ids, n))) return rc;
  if ((rc = broadcast_field(E, sp.lev[0].x, E->init_p, env_ids, n))) return rc;
  const int one16 = E->cfg.substeps;      // callLearn starts at the sketch's constant (clientCFD.pde:12), here `substeps`
  for (int k = 0; k < n; k++) {
    int e = env_ids ? env_ids[k] : k;
    CU(cudaMemsetAsync(sp.sc.xi + 2 * e, 0, 2 * sizeof(float), E->stream));
    CU(cudaMemsetAsync(sp.sc.t + e, 0, sizeof(float), E->stream));
    CU(cudaMemcpyAsync(sp.sc.flow_t + e, &E->init_t, sizeof(float), cudaMemcpyHostToDevice, E->stream));   // BDIM.resume: t = stuff[0]
    CU(cudaMemsetAsync(sp.sc.force + 2 * e, 0, 2 * sizeof(float), E->stream));
    CU(cudaMemsetAsync(sp.sc.frozen + e, 0, sizeof(int), E->stream));
    CU(cudaMemsetAsync(sp.sc.non_finite + e, 0, sizeof(int), E->stream));
    CU(cudaMemcpyAsync(sp.sc.dt + e, &E->dt0[e], sizeof(float), cudaMemcpyHostToDevice, E->stream));   // t_step*resolution
    if (reset_accumulators) {
      CU(cudaMemcpyAsync(sp.sc.callLearn + e, &one16, sizeof(int), cudaMemcpyHostToDevice, E->stream));
      CU(cudaMemsetAsync(sp.sc.Cd + e, 0, sizeof(float), E->stream));
      CU(cudaMemsetAsync(sp.sc.Cl + e, 0, sizeof(float), E->stream));
      CU(cudaMemsetAsync(sp.sc.obs + 2 * e, 0, 2 * sizeof(float), E->stream));
    }
  }
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_reset_params(rlfc_env* E, const int* env_ids, int n, const rlfc_env_params* params, int reset_accumulators) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->env_mode) return fail(RLFC_EINVAL, "rlfc_env_reset_params needs a handle created with env_params or param_sets");
  const int B = E->sp.B;
  if (n < 0 || n > B) return fail(RLFC_EINVAL, "bad env count");
  if (n > 0 && (!env_ids || !params)) return fail(RLFC_EINVAL, "null argument");
  std::vector<char> listed(B, 0);
  for (int k = 0; k < n; k++) {
    if (env_ids[k] < 0 || env_ids[k] >= B) return fail(RLFC_EINVAL, "env id out of range");
    if (listed[env_ids[k]]++) return fail(RLFC_EINVAL, "env id " + std::to_string(env_ids[k]) + " listed twice");
  }
  // all or nothing: every set validated and every geometry built before the device changes
  std::vector<EnvGeometry> geo;
  std::vector<int> set;
  {
    std::string err;
    if (build_env_geometries(E->cfg, params, n, geo, set, err)) return fail(RLFC_EINVAL, err);
  }
  CU(cudaSetDevice(E->device));
  int rc;
  if ((rc = sync_env_sets(E))) return rc;   // (the others' host copies, which upload_env_scalars writes back)
  for (int k = 0; k < n; k++) {
    if ((rc = upload_env_geometry(E, env_ids[k], params[k], geo[set[k]]))) return rc;
    if (E->lib.L) E->h_env_set[env_ids[k]] = -1;   // back on its own slot
  }
  if ((rc = upload_env_scalars(E))) return rc;
  if ((rc = upload_snapshot_params(E))) return rc;
  if ((rc = rlfc_env_reset(E, env_ids, n, reset_accumulators))) return rc;   // (sc.dt = the new t_step*resolution)
  // the new hierarchies, of the listed environments only
  std::vector<int> skip(B);
  for (int e = 0; e < B; e++) skip[e] = listed[e] ? 0 : 1;
  CU(cudaMemcpyAsync(E->d_skip, skip.data(), B * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  E->launches += launch_poisson_rebuild0(E->whole.sp, E->d_skip, E->stream);
  E->launches += launch_poisson_rebuild_coarse(E->whole.sp, E->d_skip, E->stream);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_get_params(rlfc_env* E, rlfc_env_params* params) {
  if (!E || !params) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  int rc = sync_env_sets(E);
  if (rc) return rc;
  std::copy(E->params.begin(), E->params.end(), params);
  return RLFC_OK;
}

// one round of an RL step: `substeps` solver steps with the draw() accumulation, then the observation read-out
static int step_round(rlfc_env* E, const float* d_actions, float* d_obs, float* d_reward, int* d_done) {
  SolverParams& sp = E->sp;
  int rc = solver_steps(E, sp.substeps, 1);
  if (rc) return rc;
  CU(cudaMemsetAsync(sp.sc.n_running, 0, sizeof(int), E->stream));
  E->launches += launch_emit_obs(sp, d_actions, d_obs, d_reward, d_done, E->stream);
  CU(cudaGetLastError());
  return RLFC_OK;
}

int rlfc_env_step_device(rlfc_env* E, const float* d_actions, float* d_obs, float* d_reward, int* d_done) {
  if (!E || !d_actions) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  E->launches += launch_set_actions(E->sp, d_actions, 1, E->stream);
  return step_round(E, d_actions, d_obs, d_reward, d_done);
}

int rlfc_env_step(rlfc_env* E, const float* actions, float* obs, float* reward, int* done) {
  if (!E || !actions || !obs) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  const SolverParams& sp = E->sp;
  const int B = sp.B;
  std::memcpy(E->h_actions, actions, 2 * B * sizeof(float));
  CU(cudaMemcpyAsync(E->d_actions, E->h_actions, 2 * B * sizeof(float), cudaMemcpyHostToDevice, E->stream));
  E->launches += launch_set_actions(sp, E->d_actions, 1, E->stream);
  // Every environment advances to ITS next observation (clientCFD.pde:39-50).  Environments at a callLearn boundary need
  // exactly `substeps` solver steps -- one round; an environment fresh from a reset first runs uncontrolled until
  // t > init_time and then through its first accumulation window, over several rounds, while the others stay frozen.
  // (adaptive mode: the bound follows the smallest dt any environment has taken in the rounds so far)
  // (per-environment mode: the smallest t_step*resolution to start with)
  const float init_time = sp.init_time > 0 ? sp.init_time : 0;
  if (E->par_pending) {   // (dt0 after a device parameter reset)
    int rc = sync_env_sets(E);
    if (rc) return rc;
  }
  float dt_min = sp.dt;
  if (sp.per_env) dt_min = *std::min_element(E->dt0.begin(), E->dt0.end());
  for (const LibSet& L : E->h_lib) dt_min = std::min(dt_min, L.dt0);   // (a bound over own and library sets: no sync)
  int max_rounds = sp.per_env ? 3 + (int)(init_time / (dt_min / sp.resolution)) / sp.substeps
                              : 3 + (int)(init_time / sp.dt_over_res) / sp.substeps;
  std::vector<float> h_dt(sp.adaptive ? B : 0);
  for (int round = 0;; round++) {
    int rc = step_round(E, E->d_actions, E->d_obs, E->d_reward, E->d_done);
    if (rc) return rc;
    CU(cudaMemcpyAsync(E->h_any, sp.sc.n_running, sizeof(int), cudaMemcpyDeviceToHost, E->stream));
    CU(cudaMemcpyAsync(E->h_obs, E->d_obs, 2 * B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
    if (reward) CU(cudaMemcpyAsync(E->h_reward, E->d_reward, B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
    if (done) CU(cudaMemcpyAsync(E->h_done, E->d_done, B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
    if (sp.adaptive) CU(cudaMemcpyAsync(h_dt.data(), sp.sc.dt, B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
    CU(cudaStreamSynchronize(E->stream));
    if (*E->h_any == 0) break;
    if (sp.adaptive) {
      for (float d : h_dt) if (d > 0 && d < dt_min) dt_min = d;
      max_rounds = 3 + (int)(init_time / (dt_min / sp.resolution)) / sp.substeps;
    }
    if (round >= max_rounds) return fail(RLFC_ENOTCONV, "an environment did not reach its next observation");
  }
  std::memcpy(obs, E->h_obs, 2 * B * sizeof(float));
  if (reward) std::memcpy(reward, E->h_reward, B * sizeof(float));
  if (done) std::memcpy(done, E->h_done, B * sizeof(int));
  return RLFC_OK;
}

int rlfc_env_substep_device(rlfc_env* E, const float* d_actions) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  CU(cudaSetDevice(E->device));
  E->launches += launch_set_actions(E->sp, d_actions, 0, E->stream);
  return solver_steps(E, 1, 0);
}

int rlfc_env_substep(rlfc_env* E, const float* actions, float* force, float* probes) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  CU(cudaSetDevice(E->device));
  SolverParams& sp = E->sp;
  const int B = sp.B;
  if (actions) {
    std::memcpy(E->h_actions, actions, 2 * B * sizeof(float));
    CU(cudaMemcpyAsync(E->d_actions, E->h_actions, 2 * B * sizeof(float), cudaMemcpyHostToDevice, E->stream));
  }
  E->launches += launch_set_actions(sp, actions ? E->d_actions : nullptr, 0, E->stream);
  int rc = solver_steps(E, 1, 0);
  if (rc) return rc;
  if (force) CU(cudaMemcpyAsync(E->h_force, sp.sc.force, 2 * B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  if (probes)
    CU(cudaMemcpyAsync(E->h_probes, sp.sc.probes, (size_t)B * RLFC_NUM_PROBES * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  if (force) std::memcpy(force, E->h_force, 2 * B * sizeof(float));
  if (probes) std::memcpy(probes, E->h_probes, (size_t)B * RLFC_NUM_PROBES * sizeof(float));
  return RLFC_OK;
}

static int copy_field_out(rlfc_env* E, const float* dev, int e, float* out) {
  const SolverParams& sp = E->sp;
  CU(cudaMemcpy2DAsync(out, sp.m * sizeof(float), dev + (size_t)e * sp.stride, sp.P * sizeof(float), sp.m * sizeof(float),
                       sp.n, cudaMemcpyDeviceToHost, E->stream));
  return RLFC_OK;
}
static int copy_field_in(rlfc_env* E, float* dev, int e, const float* in) {
  const SolverParams& sp = E->sp;
  CU(cudaMemcpy2DAsync(dev + (size_t)e * sp.stride, sp.P * sizeof(float), in, sp.m * sizeof(float), sp.m * sizeof(float),
                       sp.n, cudaMemcpyHostToDevice, E->stream));
  return RLFC_OK;
}

int rlfc_env_get_fields(rlfc_env* E, int e, float* ux, float* uy, float* p) {
  if (!E || e < 0 || e >= E->sp.B) return fail(RLFC_EINVAL, "bad handle or env index");
  CU(cudaSetDevice(E->device));
  int rc;
  if (ux && (rc = copy_field_out(E, E->uAx, e, ux))) return rc;
  if (uy && (rc = copy_field_out(E, E->uAy, e, uy))) return rc;
  if (p && (rc = copy_field_out(E, E->sp.lev[0].x, e, p))) return rc;
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_set_fields(rlfc_env* E, int e, const float* ux, const float* uy, const float* p) {
  if (!E || e < 0 || e >= E->sp.B) return fail(RLFC_EINVAL, "bad handle or env index");
  CU(cudaSetDevice(E->device));
  int rc;
  if (ux && (rc = copy_field_in(E, E->uAx, e, ux))) return rc;
  if (uy && (rc = copy_field_in(E, E->uAy, e, uy))) return rc;
  if (p && (rc = copy_field_in(E, E->sp.lev[0].x, e, p))) return rc;
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_save_bdim(rlfc_env* E, int e, const char* path) {
  if (!E || !path || e < 0 || e >= E->sp.B) return fail(RLFC_EINVAL, "bad argument");
  const size_t N = (size_t)E->sp.n * E->sp.m;
  std::vector<float> ux(N), uy(N), p(N);
  int rc = rlfc_env_get_fields(E, e, ux.data(), uy.data(), p.data());
  if (rc) return rc;
  // BDIM.t counts grid-unit time: set by resume, += dt per solver step (AFCCylinder.t advances by dt/resolution instead)
  float flow_t = 0, dt = E->sp.dt;
  CU(cudaMemcpyAsync(&flow_t, E->sp.sc.flow_t + e, sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  if (E->sp.per_env) CU(cudaMemcpyAsync(&dt, E->sp.sc.dt + e, sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  std::string err;
  rc = write_bdim_text(path, E->sp.n, E->sp.m, flow_t, dt, ux.data(), uy.data(), p.data(), err);
  return rc ? fail(rc, err) : RLFC_OK;
}

int rlfc_env_load_bdim(rlfc_env* E, int e, const char* path) {
  if (!E || !path || e < 0 || e >= E->sp.B) return fail(RLFC_EINVAL, "bad argument");
  std::vector<float> ux, uy, p;
  float t, dt;
  std::string err;
  int rc = read_checkpoint(path, E->sp.n, E->sp.m, t, dt, ux, uy, p, err);
  if (rc) return fail(rc, err);
  if (E->sp.adaptive) {
    // adaptive mode: any positive dt; it becomes the environment's current dt
    if (!(dt > 0) || !std::isfinite(dt)) return fail(RLFC_EIO, "checkpoint dt " + std::to_string(dt) + " is not a positive number");
  } else {
    CU(cudaSetDevice(E->device));
    if ((rc = sync_env_sets(E))) return rc;
    const float fixed = E->dt0[e];   // the environment's t_step*resolution (the handle's without env_params)
    if (dt != fixed && !(std::fabs(dt - fixed) <= 1e-6f * fixed))
      return fail(RLFC_EIO, "checkpoint dt " + std::to_string(dt) + " does not match the environment's " + std::to_string(fixed));
  }
  CU(cudaSetDevice(E->device));
  if (E->sp.adaptive) CU(cudaMemcpyAsync(E->sp.sc.dt + e, &dt, sizeof(float), cudaMemcpyHostToDevice, E->stream));
  CU(cudaMemcpyAsync(E->sp.sc.flow_t + e, &t, sizeof(float), cudaMemcpyHostToDevice, E->stream));   // BDIM.resume: t = stuff[0]
  CU(cudaStreamSynchronize(E->stream));
  return rlfc_env_set_fields(E, e, ux.data(), uy.data(), p.data());
}

int rlfc_env_dims(const rlfc_env* E, int* n, int* m, int* n_envs) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (n) *n = E->sp.n;
  if (m) *m = E->sp.m;
  if (n_envs) *n_envs = E->sp.B;
  return RLFC_OK;
}

int rlfc_env_get_time(rlfc_env* E, float* t) {
  if (!E || !t) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(t, E->sp.sc.t, E->sp.B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_running(rlfc_env* E, int* n_running) {
  if (!E || !n_running) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(E->h_any, E->sp.sc.n_running, sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  *n_running = *E->h_any;
  return RLFC_OK;
}

int rlfc_env_get_flags(rlfc_env* E, int* flags) {
  if (!E || !flags) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  std::vector<int> refused(E->snap.S ? E->sp.B : 0), par_refused(E->pr.refused ? E->sp.B : 0),
      rec_refused(E->rec.refused ? E->sp.B : 0);
  CU(cudaMemcpyAsync(E->h_done, E->sp.sc.non_finite, E->sp.B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  if (E->snap.S) CU(cudaMemcpyAsync(refused.data(), E->snap.refused, E->sp.B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  if (E->pr.refused)
    CU(cudaMemcpyAsync(par_refused.data(), E->pr.refused, E->sp.B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  if (E->rec.refused)
    CU(cudaMemcpyAsync(rec_refused.data(), E->rec.refused, E->sp.B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  for (int e = 0; e < E->sp.B; e++)
    flags[e] = (E->h_done[e] ? 1 : 0) | (E->snap.S && refused[e] ? 2 : 0) | (E->pr.refused && par_refused[e] ? 4 : 0) |
               (E->rec.refused && rec_refused[e] ? 8 : 0);
  return RLFC_OK;
}

int rlfc_env_snapshot(rlfc_env* E, const int* env_ids, const int* slots, int n) {
  return snapshot_host(E, env_ids, slots, n, 0, 0);
}

int rlfc_env_restore(rlfc_env* E, const int* env_ids, const int* slots, int n, int keep_accumulators) {
  return snapshot_host(E, env_ids, slots, n, 1, keep_accumulators != 0);
}

int rlfc_env_snapshot_device(rlfc_env* E, const int* d_env_ids, const int* d_slots, int n) {
  int rc = snapshot_check_handle(E, n, d_env_ids && d_slots);
  if (rc) return rc;
  CU(cudaSetDevice(E->device));
  return snapshot_enqueue(E, d_env_ids, d_slots, n, 0, 0);
}

int rlfc_env_restore_device(rlfc_env* E, const int* d_env_ids, const int* d_slots, int n, int keep_accumulators) {
  int rc = snapshot_check_handle(E, n, d_env_ids && d_slots);
  if (rc) return rc;
  CU(cudaSetDevice(E->device));
  return snapshot_enqueue(E, d_env_ids, d_slots, n, 1, keep_accumulators != 0);
}

int rlfc_env_reset_sets(rlfc_env* E, const int* env_ids, const int* sets, int n, int reset_accumulators) {
  int rc = reset_sets_check_handle(E, n, env_ids && sets);
  if (rc) return rc;
  const int B = E->sp.B;
  if (n > B) return fail(RLFC_EINVAL, "bad pair count");
  std::vector<char> seen(B, 0);
  for (int k = 0; k < n; k++) {
    if (env_ids[k] < 0 || env_ids[k] >= B) return fail(RLFC_EINVAL, "env id " + std::to_string(env_ids[k]) + " out of range");
    if (sets[k] < 0 || sets[k] >= E->lib.L) return fail(RLFC_EINVAL, "set " + std::to_string(sets[k]) + " out of range");
    if (seen[env_ids[k]]++) return fail(RLFC_EINVAL, "env id " + std::to_string(env_ids[k]) + " listed twice");
  }
  CU(cudaSetDevice(E->device));
  if (n > 0) {
    CU(cudaMemcpyAsync(E->set_env, env_ids, n * sizeof(int), cudaMemcpyHostToDevice, E->stream));
    CU(cudaMemcpyAsync(E->set_ids, sets, n * sizeof(int), cudaMemcpyHostToDevice, E->stream));
  }
  if ((rc = reset_sets_enqueue(E, E->set_env, E->set_ids, n, reset_accumulators != 0))) return rc;
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_reset_sets_device(rlfc_env* E, const int* d_env_ids, const int* d_sets, int n, int reset_accumulators) {
  int rc = reset_sets_check_handle(E, n, d_env_ids && d_sets);
  if (rc) return rc;
  CU(cudaSetDevice(E->device));
  return reset_sets_enqueue(E, d_env_ids, d_sets, n, reset_accumulators != 0);
}

int rlfc_env_reset_params_device(rlfc_env* E, const int* d_env_ids, const rlfc_env_params* d_params, int n,
                                 int reset_accumulators) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->env_mode)
    return fail(RLFC_EINVAL, "rlfc_env_reset_params_device needs a handle created with env_params or param_sets");
  if (n < 0) return fail(RLFC_EINVAL, "bad pair count");
  if (n > 0 && (!d_env_ids || !d_params)) return fail(RLFC_EINVAL, "null argument");
  if (n == 0) return RLFC_OK;
  CU(cudaSetDevice(E->device));
  SolverParams& sp = E->whole.sp;
  CU(cudaMemsetAsync(E->d_skip, 1, sp.B * sizeof(int), E->stream));   // nonzero = keep; the reset clears
  E->run("k_param_geometry+k_reset_params", 0, [&] {
    return launch_reset_params(sp, E->lib, E->snap, E->pr, E->circle, E->cfg.x_lengths * E->cfg.resolution,
                               E->cfg.y_lengths * E->cfg.resolution, sp.nband_x, E->init_ux, E->init_uy, E->init_p, E->init_t,
                               E->uAx, E->uAy, d_env_ids, d_params, n, reset_accumulators != 0, E->d_skip, E->stream);
  });
  E->run("k_poisson_rebuild0", 0, [&] { return launch_poisson_rebuild0(sp, E->d_skip, E->stream); });
  E->run("k_poisson_rebuild_coarse", 0, [&] { return launch_poisson_rebuild_coarse(sp, E->d_skip, E->stream); });
  CU(cudaGetLastError());
  E->par_pending = true;
  return RLFC_OK;
}

int rlfc_record_bytes(const rlfc_config* cfg, size_t* bytes) {
  if (!cfg || !bytes) return fail(RLFC_EINVAL, "null argument");
  if (cfg->resolution < 1 || cfg->x_lengths < 1 || cfg->y_lengths < 1) return fail(RLFC_EINVAL, "the grid must be positive");
  if (cfg->n_sensors < 0) return fail(RLFC_EINVAL, "n_sensors must be >= 0");
  *bytes = record_bytes(cfg->x_lengths * cfg->resolution + 2, cfg->y_lengths * cfg->resolution + 2, cfg->n_sensors);
  return RLFC_OK;
}

unsigned long long rlfc_record_checksum(const void* record, size_t bytes) {
  const unsigned char* r = static_cast<const unsigned char*>(record);
  unsigned long long sum = 0;
  for (size_t w = 4; w < bytes / 4; w++) {
    unsigned x;
    std::memcpy(&x, r + 4 * w, 4);
    sum += record_mix(w, x);
  }
  return sum;
}

int rlfc_env_export(rlfc_env* E, const int* env_ids, int n, void* host_buf) {
  int rc = records_check_handle(E, n, env_ids && host_buf);
  if (rc || n == 0) return rc;
  if ((rc = record_host_ids(E, env_ids, n, false))) return rc;
  CU(cudaSetDevice(E->device));
  const size_t bytes = own_record_bytes(E);
  if ((rc = records_prepare(E, n, bytes)) || (rc = record_stage(E, env_ids, n, bytes))) return rc;
  if ((rc = record_export_enqueue(E, E->rec_ids, n, E->rec_stage))) return rc;
  CU(cudaMemcpyAsync(host_buf, E->rec_stage, (size_t)n * bytes, cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_import(rlfc_env* E, const int* env_ids, int n, const void* host_buf, int keep_accumulators) {
  int rc = records_check_handle(E, n, env_ids && host_buf);
  if (rc || n == 0) return rc;
  if ((rc = record_host_ids(E, env_ids, n, true))) return rc;
  // record 0's header gives the size of every record of the call: checked here before any of them is read
  unsigned w[RLFC_RECORD_HEADER_BYTES / 4];
  std::memcpy(w, host_buf, sizeof(w));
  const unsigned long long len = w[6] | (unsigned long long)w[7] << 32;
  int v = kRecApply;
  if (std::memcmp(w, "RLFCSTAT", 8)) v = kRecMagic;
  else if (w[4] != RLFC_RECORD_VERSION) v = kRecVersion;
  else if (w[11] > 0xffffu || w[12] > 0xffffu || len != record_bytes((int)w[11], (int)w[12], 0) + 16ull * w[19]) v = kRecLength;
  else if ((int)w[8] != E->cfg.resolution || (int)w[9] != E->cfg.x_lengths || (int)w[10] != E->cfg.y_lengths ||
           (int)w[11] != E->sp.n || (int)w[12] != E->sp.m || (int)w[18] != E->sp.nprobe) v = kRecGrid;
  if (v) return fail(RLFC_EINVAL, std::string("record 0: ") + record_check_name(v));
  CU(cudaSetDevice(E->device));
  if ((rc = records_prepare(E, n, len)) || (rc = record_stage(E, env_ids, n, len))) return rc;
  CU(cudaMemcpyAsync(E->rec_stage, host_buf, (size_t)n * len, cudaMemcpyHostToDevice, E->stream));
  if ((rc = record_check_enqueue(E, E->rec_ids, n, E->rec_stage, len))) return rc;
  std::vector<int> verdict(n);
  CU(cudaMemcpyAsync(verdict.data(), E->rec.verdict, n * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  for (int k = 0; k < n; k++)
    if (verdict[k])
      return fail(RLFC_EINVAL, "record " + std::to_string(k) + " (env id " + std::to_string(env_ids[k]) + "): " +
                                   record_check_name(verdict[k]));
  if ((rc = record_apply_enqueue(E, E->rec_ids, n, E->rec_stage, len, keep_accumulators != 0))) return rc;
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_export_device(rlfc_env* E, const int* d_env_ids, int n, void* d_buf) {
  int rc = records_check_handle(E, n, d_env_ids && d_buf);
  if (rc) return rc;
  if (reinterpret_cast<uintptr_t>(d_buf) % 16) return fail(RLFC_EINVAL, "the record buffer must be 16-byte aligned");
  CU(cudaSetDevice(E->device));
  return record_export_enqueue(E, d_env_ids, n, d_buf);
}

int rlfc_env_import_device(rlfc_env* E, const int* d_env_ids, int n, const void* d_buf, size_t record_bytes_,
                           int keep_accumulators) {
  int rc = records_check_handle(E, n, d_env_ids && d_buf);
  if (rc) return rc;
  if (reinterpret_cast<uintptr_t>(d_buf) % 16) return fail(RLFC_EINVAL, "the record buffer must be 16-byte aligned");
  const size_t base = record_bytes(E->sp.n, E->sp.m, 0);
  if (record_bytes_ < base || (record_bytes_ - base) % 16 || (record_bytes_ - base) / 16 > (1u << 24))
    return fail(RLFC_EINVAL, "record_bytes " + std::to_string(record_bytes_) + " is not the size of a record of the handle's grid");
  if (n == 0) return RLFC_OK;
  CU(cudaSetDevice(E->device));
  if ((rc = record_check_enqueue(E, d_env_ids, n, d_buf, record_bytes_))) return rc;
  return record_apply_enqueue(E, d_env_ids, n, d_buf, record_bytes_, keep_accumulators != 0);
}

int rlfc_env_get_stats(rlfc_env* E, int e, long long* count, double* sums) {
  if (!E || !count) return fail(RLFC_EINVAL, "null argument");
  if (!E->fs.every) return fail(RLFC_EINVAL, "the handle has no flow statistics (rlfc_config.stats_every = 0)");
  const SolverParams& sp = E->sp;
  if (e < 0 || e >= sp.B) return fail(RLFC_EINVAL, "env id " + std::to_string(e) + " out of range");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(count, E->fs.count + e, sizeof(long long), cudaMemcpyDeviceToHost, E->stream));
  for (int s = 0; sums && s < kNumStats; s++)
    CU(cudaMemcpy2DAsync(sums + (size_t)s * sp.n * sp.m, sp.m * sizeof(double), E->fs.sums + ((size_t)e * kNumStats + s) * sp.stride,
                         sp.P * sizeof(double), sp.m * sizeof(double), sp.n, cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_stats_reset(rlfc_env* E, const int* env_ids, int n) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->fs.every) return fail(RLFC_EINVAL, "the handle has no flow statistics (rlfc_config.stats_every = 0)");
  const int B = E->sp.B;
  if (!env_ids) n = B;
  if (n < 0) return fail(RLFC_EINVAL, "bad env count");
  for (int k = 0; env_ids && k < n; k++)
    if (env_ids[k] < 0 || env_ids[k] >= B) return fail(RLFC_EINVAL, "env id " + std::to_string(env_ids[k]) + " out of range");
  CU(cudaSetDevice(E->device));
  const FlowStats& f = E->fs;
  const size_t per_env = (size_t)kNumStats * E->sp.stride;
  if (!env_ids) {
    CU(cudaMemsetAsync(f.sums, 0, per_env * B * sizeof(double), E->stream));
    CU(cudaMemsetAsync(f.count, 0, B * sizeof(long long), E->stream));
    CU(cudaMemsetAsync(f.step, 0, B * sizeof(int), E->stream));
  }
  for (int k = 0; env_ids && k < n; k++) {
    const int e = env_ids[k];
    CU(cudaMemsetAsync(f.sums + e * per_env, 0, per_env * sizeof(double), E->stream));
    CU(cudaMemsetAsync(f.count + e, 0, sizeof(long long), E->stream));
    CU(cudaMemsetAsync(f.step + e, 0, sizeof(int), E->stream));
  }
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_stats_reset_device(rlfc_env* E, const int* d_env_ids, int n) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (!E->fs.every) return fail(RLFC_EINVAL, "the handle has no flow statistics (rlfc_config.stats_every = 0)");
  if (n < 0) return fail(RLFC_EINVAL, "bad env count");
  if (n > 0 && !d_env_ids) return fail(RLFC_EINVAL, "null argument");
  if (n == 0) return RLFC_OK;
  CU(cudaSetDevice(E->device));
  E->run("k_stats_reset", 0, [&] { return launch_stats_reset(E->sp, E->fs, d_env_ids, n, E->stream); });
  CU(cudaGetLastError());
  return RLFC_OK;
}

int rlfc_env_get_sensors(rlfc_env* E, float* out) {
  if (!E || !out) return fail(RLFC_EINVAL, "null argument");
  if (!E->sens.n) return fail(RLFC_EINVAL, "the handle has no sensors (rlfc_config.n_sensors = 0)");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(out, E->sens.out, (size_t)E->sp.B * E->sens.n * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_get_sensors_device(rlfc_env* E, float* d_out) {
  if (!E || !d_out) return fail(RLFC_EINVAL, "null argument");
  if (!E->sens.n) return fail(RLFC_EINVAL, "the handle has no sensors (rlfc_config.n_sensors = 0)");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(d_out, E->sens.out, (size_t)E->sp.B * E->sens.n * sizeof(float), cudaMemcpyDeviceToDevice, E->stream));
  return RLFC_OK;
}

int rlfc_env_check_cfl(rlfc_env* E, float* dt) {
  if (!E || !dt) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  E->launches += launch_check_cfl(E->sp, E->uAx, E->uAy, E->d_reward, E->stream);      // (d_reward: a [B] float scratch)
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(E->h_reward, E->d_reward, E->sp.B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  std::memcpy(dt, E->h_reward, E->sp.B * sizeof(float));
  return RLFC_OK;
}

int rlfc_env_get_dt(rlfc_env* E, float* dt) {
  if (!E || !dt) return fail(RLFC_EINVAL, "null argument");
  if (!E->sp.per_env) {
    for (int e = 0; e < E->sp.B; e++) dt[e] = E->sp.dt;
    return RLFC_OK;
  }
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(dt, E->sp.sc.dt, E->sp.B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_get_mg_iters(rlfc_env* E, int* iters) {
  if (!E || !iters) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(iters, E->sp.sc.iters, 2 * E->sp.B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_field_sum(rlfc_env* E, float* sums) {
  if (!E || !sums) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  E->launches += launch_set_actions(E->sp, nullptr, 0, E->stream);      // (no environment is frozen for this evaluation)
  E->launches += launch_psum(E->whole.sp, E->stream);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(sums, E->sp.sc.psum, E->sp.B * sizeof(float), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_field_sum_stats(rlfc_env* E, int* stats) {
  if (!E || !stats) return fail(RLFC_EINVAL, "null argument");
  CU(cudaSetDevice(E->device));
  CU(cudaMemcpyAsync(stats, E->sp.xs_stats, (size_t)8 * E->sp.B * sizeof(int), cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_env_num_levels(const rlfc_env* E) { return E ? E->sp.nlevels : RLFC_EINVAL; }

static int static_lookup(const Geometry& g, const char* name, int level, float* out, int* n, int* m) {
  if (level < 0 || level >= (int)g.levels.size()) return fail(RLFC_EINVAL, "level out of range");
  const std::vector<float>* src = nullptr;
  const HostLevel& H = g.levels[level];
  std::string nm(name);
  if (nm == "lower.x") src = &H.lx;
  else if (nm == "lower.y") src = &H.ly;
  else if (nm == "inv") src = &H.inv;
  else if (nm == "diag") src = &H.diag;
  else if (level == 0) {
    if (nm == "del.x") src = &g.del_x; else if (nm == "del.y") src = &g.del_y;
    else if (nm == "del1.x") src = &g.del1_x; else if (nm == "del1.y") src = &g.del1_y;
    else if (nm == "wnx.x") src = &g.wnx_x; else if (nm == "wnx.y") src = &g.wnx_y;
    else if (nm == "wny.x") src = &g.wny_x; else if (nm == "wny.y") src = &g.wny_y;
    else if (nm == "c.x") src = &g.c_x; else if (nm == "c.y") src = &g.c_y;
    else if (nm == "w1.x") src = &g.w1_x; else if (nm == "w2.x") src = &g.w2_x;
    else if (nm == "w1.y") src = &g.w1_y; else if (nm == "w2.y") src = &g.w2_y;
    else if (nm == "ry1.x") src = &g.ry1_x; else if (nm == "ry2.x") src = &g.ry2_x;
    else if (nm == "rx1.y") src = &g.rx1_y; else if (nm == "rx2.y") src = &g.rx2_y;
  }
  if (!src) return fail(RLFC_EINVAL, "unknown static field " + nm);
  if (n) *n = H.n;
  if (m) *m = H.m;
  if (out) std::memcpy(out, src->data(), src->size() * sizeof(float));
  return RLFC_OK;
}

int rlfc_env_get_static(rlfc_env* E, const char* name, int level, float* out, int* n, int* m) {
  if (!E || !name) return fail(RLFC_EINVAL, "null argument");
  return static_lookup(E->geo, name, level, out, n, m);
}

int rlfc_env_get_coeffs(rlfc_env* E, int e, const char* name, int level, float* out, int* n, int* m) {
  if (!E || !name) return fail(RLFC_EINVAL, "null argument");
  if (e < 0 || e >= E->sp.B) return fail(RLFC_EINVAL, "env index out of range");
  if (level < 0 || level >= E->sp.nlevels) return fail(RLFC_EINVAL, "level out of range");
  const std::string nm(name);
  const bool c0 = level == 0 && (nm == "c.x" || nm == "c.y" || nm == "del.x" || nm == "del.y");
  if (!c0 && nm != "lower.x" && nm != "lower.y" && nm != "inv" && nm != "diag")
    return fail(RLFC_EINVAL, "unknown Poisson coefficient field " + nm);
  if (!E->sp.per_env) return static_lookup(E->geo, name, level, out, n, m);
  const DevLevel& L = E->sp.lev[level];
  if (n) *n = L.n;
  if (m) *m = L.m;
  if (!out) return RLFC_OK;
  const float* src = (nm == "lower.x" || nm == "c.x") ? L.lx : (nm == "lower.y" || nm == "c.y") ? L.ly : nm == "inv" ? L.inv : L.diag;
  size_t off = (size_t)e * L.stride;
  CU(cudaSetDevice(E->device));
  if (nm == "del.x" || nm == "del.y") {   // the environment's geometry slot
    int rc = sync_env_sets(E);
    if (rc) return rc;
    src = nm == "del.x" ? E->sp.del_x : E->sp.del_y;
    off = (size_t)slot_of(E, e) * E->sp.stride;
  }
  CU(cudaMemcpy2DAsync(out, L.m * sizeof(float), src + off, L.P * sizeof(float), L.m * sizeof(float), L.n,
                       cudaMemcpyDeviceToHost, E->stream));
  CU(cudaStreamSynchronize(E->stream));
  return RLFC_OK;
}

int rlfc_geometry_static(const rlfc_config* cfg, const char* name, int level, float* out, int* n, int* m, int* nlevels) {
  if (!cfg || !name) return fail(RLFC_EINVAL, "null argument");
  Geometry g;
  std::string err;
  int rc = build_geometry(*cfg, g, err);
  if (rc) return fail(rc, err);
  if (nlevels) *nlevels = (int)g.levels.size();
  return static_lookup(g, name, level, out, n, m);
}

int rlfc_env_set_profiling(rlfc_env* E, int on) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  E->prof_collect();
  E->profiling = on != 0;
  if (on) for (auto& a : E->prof) { a.ms = 0; a.count = 0; }
  return RLFC_OK;
}

int rlfc_env_get_profile(rlfc_env* E, int idx, char* name, int name_cap, double* ms_total, long long* launches,
                         double* algorithmic_bytes_per_launch) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  E->prof_collect();
  if (idx < 0 || idx >= (int)E->prof.size()) return 1;   // end of list
  const auto& a = E->prof[idx];
  if (name && name_cap > 0) { std::strncpy(name, a.name.c_str(), name_cap - 1); name[name_cap - 1] = 0; }
  if (ms_total) *ms_total = a.ms;
  if (launches) *launches = a.count;
  if (algorithmic_bytes_per_launch)
    *algorithmic_bytes_per_launch = 4.0 * a.floats_per_cell * (double)(E->sp.n - 2) * (E->sp.m - 2) * E->sp.B;
  return RLFC_OK;
}

int rlfc_format_float_java(float v, char* buf, int cap) {
  if (!buf || cap <= 0) return RLFC_EINVAL;
  const std::string s = format_float_java(v);
  std::strncpy(buf, s.c_str(), cap - 1);
  buf[cap - 1] = 0;
  return (int)s.size();
}

void* rlfc_env_stream(rlfc_env* E) { return E ? (void*)E->stream : nullptr; }
int rlfc_env_slab_info(const rlfc_env* E, int* n_devices, long long* barriers, long long* bytes_shared) {
  if (!E) return fail(RLFC_EINVAL, "null handle");
  if (n_devices) *n_devices = E->slab.empty() ? 1 : (int)E->slab.size();
  if (barriers) *barriers = E->slab_barriers;
  if (bytes_shared) *bytes_shared = (long long)E->vmm.bytes_mapped();
  return RLFC_OK;
}

long long rlfc_env_launch_count(const rlfc_env* E) { return E ? E->launches : 0; }

double rlfc_env_model_bytes_per_solver_step(const rlfc_env* E) {
  if (!E) return 0;
  // SURVEY 8d: 4 B * N_int * (28 + 13*(kP + kC)) with on-chip coarse levels; use k = 1 + 1 here, the
  // caller scales with the measured iteration counts
  const double nint = (double)(E->sp.n - 2) * (E->sp.m - 2);
  return 4.0 * nint * (28 + 13 * 2);
}

}  // extern "C"
