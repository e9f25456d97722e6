// solver.h -- device data layout and kernel launch interface of the batched BDIM solver.
//
// Layout in HBM (all fp32):
//   * every per-environment field is an (n x P) pitched array (i = x outer, j = y contiguous, ghost
//     ring included, P = m rounded up to 8 floats so rows are 32 B-sector aligned), and the batch is
//     struct-of-arrays: field[e] = base + e * stride, stride = n*P rounded up to 32 floats;
//   * static geometry / coefficient fields are stored once (shared by the whole batch, L2-resident).
// Velocity lives in three rotating buffers A (step-start u, doubles as u0), B (predictor result,
// doubles as `us`), C (corrector result); see BDIM.pde:79-107 for the data flow reproduced.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "../../include/rlfc.h"

namespace rlfc {

constexpr int kMaxLevels = 16;

// Pre-skewed static coefficient table of one level for the row-pipelined smoother (smooth_rows.cuh):
// entry tau (stored at index tau + kTabFront) holds, for lane l, the coefficients of row tau - l of the
// lane's C columns j0 = C*l+1 .. C*l+C as the float stream [ly[row][j0+c] (C+1) | -inv[row][j0+c] (C) |
// lx[row][j0+c] (C)], packed into K = ceil((3C+1)/4) float4 vectors that are
// lane-contiguous: vector k of lane l of entry e sits at T[(e*K + k)*32 + l].
struct RowTab {
  const float4* T;
  int C, K, entries, copies;   // `copies` identical tables back to back (L2-slice load spreading)
};

#define IDX(i, j) ((i) * P + (j))

// Chained strip smoother (smooth_chain.cuh): per level, the columns are cut into strips of 32 (lane L of strip s owns
// column j = 32 s + L + 1) and every array the sweeps touch is stored STRIP-SKEWED: element (s, tau, L) at
// (s*T + tau)*32 + L holds the cell (i = tau - L, j), so that the cells a warp works on in one step form one
// contiguous 128-byte line.  Entries 0 .. T-1 with T = ni + 34; elements outside the interior are zero.
struct ChainLevel {
  int on;                   // 1 = this level is smoothed by the chained strip smoother
  int NS, T;                // strips, entries per strip
  size_t sk_stride;         // elements per environment of a skewed array = NS*T*32
  const float4* ct;         // static coefficients {lx[i+1][j], ly[i][j], ly[i][j+1], -inv[i][j]}   [NS][T][32]
  float* rsk;               // [B] residual entering smooth(4)                                     (4 B / element)
  uint2* dsk[5];            // [B] iterate after sweep g = 0..4 as {value bits, launch tag}         (8 B / element)
  unsigned long long* ticket;   // [1] CTA tickets of this level's sweep launches (role order = start order)
  unsigned tag_hi;          // high bits of the launch tag (unique per ticket counter)
  // smooth_chain3.cuh: compact copies of every strip's lane-31 (S edge) and lane-0 (N edge) results, indexed by the
  // CONSUMER's step (+ kC2EdgePad), array (2 g + which) of sweep g at edge + (2 g + which) * edge_arr, [B][NS][TE]
  uint2* edge;
  size_t edge_arr;
  int TE;
  int s0, ns_loc;           // strips s0 .. s0 + ns_loc - 1 are swept by this device (slab mode; otherwise 0, NS)
};

struct DevLevel {
  RowTab rt;
  int n, m, P;              // dims incl. ghosts, pitch
  size_t stride;            // per-env stride (floats) of r/x/d at this level
  const float *lx, *ly, *inv, *diag;   // static, pitched
  float *r, *r2, *x, *d;    // per-env batch arrays (level 0: x = p; r2 = ping-pong residual)
  float *w;                 // level 0, wavefront smoother only: scratch for the Gauss-Seidel iterate
  int wave;                 // 1 = this level is smoothed by the wavefront fallback (smooth_wave.cuh)
  ChainLevel ch;            // chained strip smoother (wide levels; smooth_chain.cuh)
};

struct BandFace {           // a face where the BDIM blend differs from the identity
  int i, j;
  float del, del1, wnx, wny;
};

struct SamplePt { int i, j; float s, t; };
struct SensorPt { int i, j; float s, t; int field; };   // a sample point of field 0 = p, 1 = u.x, 2 = u.y (rlfc_sensor)
struct ForcePt { int i, j; float s, t, l, nx, ny; };

// Per-env scalar state (struct of arrays on the device)
struct EnvScalars {
  float *xi;        // [B][2] current action (xi1, xi2)
  float *t;         // [B]    AFCCylinder.t
  float *flow_t;    // [B]    BDIM.t: grid-unit time, += dt per solver step (BDIM.pde:106), set from the checkpoint
  float *force;     // [B][2] last raw force (-pressForce)
  float *probes;    // [B][32]
  int   *callLearn; // [B]    draw() accumulators (clientCFD.pde:11-13)
  float *Cd, *Cl;   // [B]
  float *obs;       // [B][2] last produced (Cl, Cd)
  int   *frozen;    // [B]    env takes no part in the solver steps of this call: it has emitted its observation and waits
                    //        for the next action (clientCFD.pde:44-54), or its episode is over (clientCFD.pde:36)
  int   *non_finite;// [B]    sticky: a non-finite force was produced (diverged environment)
  int   *n_running; // [1]    environments not frozen, counted by k_emit_obs
  int   *active;    // [B]    MG: env still iterating
  int   *iters;     // [B][2] MG iterations of the last predictor/corrector solve
  double *rr_part;  // [B][rr_blocks] partial sums of r.r
  float *psum;      // [B]    serial interior sum of p
  int   *any_active;// [1]
  float *dt;        // [B]    adaptive mode: dt of the env's current / last solver step (k_check_cfl<true> writes it)
};

// Slab mode (BASELINE config 5): one domain advanced by several devices that share every array through one virtual
// address range (vmm.h).  A device owns a contiguous range of a kernel's row blocks (plain arrays) or strips (skewed
// arrays); kernels are launched with their full grid on every device and blocks outside the device's range exit.
struct SlabBarrier {
  unsigned* count;          // [1] arrivals of all devices, all barriers (memory of device 0, mapped everywhere)
  unsigned* epoch;          // [1] this device's barrier count (its own memory)
  unsigned n;               // devices
};

struct SolverParams {
  int slab_n, slab_rank;    // devices sharing the domain (0/1 = not in slab mode), this device's index
  int B;                    // environments in the batch
  int n, m, P;              // level-0 dims
  size_t stride;            // level-0 per-env stride
  float dt, nu, dRD;        // dRD = dR*D (AFCCylinder.pde:48)
  float dt_over_res;        // dt/resolution (AFCCylinder.pde:56)
  float action_scale;       // 5
  float inv_cells;          // (float)((n-2)*(m-2))
  float mg_tol;
  int   nlevels;
  int   chain_levels;       // levels 0 .. chain_levels-1 run as grid-wide kernels with the chained strip smoother; the
                            // one-CTA-per-env coarse kernel starts at level max(chain_levels, 1)
  double *rr_chain;         // [B][rr_chain_n] per-CTA partial sums of r.r of the level-0 chain increment
  unsigned *rr_count;       // [B] CTAs of the increment kernel that have delivered their partial sum
  int   rr_chain_n;
  int   tiny;               // 1 = levels of at most 32 columns are smoothed by one warp in registers (smooth_tiny.cuh; RLFC_TINY=0: row pipeline)
  int   resid_march;        // 1 = k_resid_down0_march (default), 0 = the shared-memory tile version (RLFC_RESID=tile)
  int   fast_bc;            // 1 = two-phase setBC kernels (no band face on the lines setBC reads; grid fits one CTA)
  int   resolution, substeps, mg_max_iters;
  float init_time, episode_time;
  DevLevel lev[kMaxLevels];
  // static level-0 fields
  const float *c_x, *c_y;
  const float *w1_x, *w2_x, *ry1_x, *ry2_x, *w1_y, *w2_y, *rx1_y, *rx2_y;
  const BandFace *band_x, *band_y;
  int nband_x, nband_y;
  float *band_tmp;          // [B][nband_x + nband_y]
  float *rsk;               // [B][rsk_stride] level-0 residual in the smoother's skewed layout (smooth_rows.cuh)
  size_t rsk_stride;
  const ForcePt *force_pts; int nforce;
  const SamplePt *probe_pts; int nprobe;
  int rr_blocks;            // number of per-env partial sums written by the increment kernel
  // Field.sum as segment summaries (exact_sum.cuh); xs_recs == nullptr selects the plain serial chain (k_psum)
  double *xs_ctot;          // [B][xs_nchunks] chunk totals, valid when xs_cflag == xs_epoch + 1
  unsigned *xs_cflag;       // [B][xs_nchunks]
  unsigned *xs_epoch;       // [B] passes completed
  unsigned *xs_recs;        // [B][xs_nbatches][192] batch records (32 summaries condensed)
  unsigned *xs_blk;         // [B][ceil(xs_nbatches/32)][8][32] blocks of 32 records condensed (large domains; else nullptr)
  double *xs_pred, *xs_inc, *xs_corr;   // [B][xs_nbatches] large domains: first-pass prediction at every batch start, the batches'
                            // float increments, and the correction the second table pass adds (k_xsum_refine)
  int xs_nseg, xs_nchunks, xs_nbatches;
  int xs_passes;            // table passes of a large domain's Field.sum: 2, or 3 from 8 Mi cells on (RLFC_XS_PASSES)
  int xs_flags;             // cross-check switches: bit 0 = redo batches as plain additions (RLFC_XS_REDO=serial)
  int *xs_stats;            // [B][8] counters of the last serial pass (rlfc_env_field_sum_stats)
  EnvScalars sc;
  // (appended last, so the fields above keep their offsets in the kernels' parameter space)
  int   adaptive;           // 1 = every solver step opens with k_check_cfl<true> and the hierarchy rebuild (adaptive dt)
                            // per_env (below) = per-environment dt (sc.dt) and Poisson hierarchy: every level's lx, ly, inv,
                            // diag hold one copy per environment at the level's `stride` (like r, x, d), c_x / c_y are level
                            // 0's lx / ly, and each row-pipeline level's RowTab holds one table per environment (rt.copies = the
                            // view's B, so the row smoother's `blockIdx.x % copies` pick selects environment blockIdx.x's table)
  const float *del_x, *del_y;   // per_env: level-0 BDIM del of every geometry slot (pitched, slot s at s * stride), c = del*(1*dt)
  // per_env = 1 (adaptive mode, or per-environment parameters, rlfc_config.env_params): the kernels run their
  // per-environment instances (ADT), which read sc.dt[e], the per-environment hierarchy above and the arrays below.  An
  // environment's geometry lives in its SLOT: del_x/del_y and the body-velocity basis w1_x .. rx2_y at env_slot[e] *
  // stride, its band lists at band_x + env_slot[e] * nband_x and band_y + env_slot[e] * nband_y (nband_x / nband_y are
  // then the per-slot capacities; band_tmp keeps its [B][nband_x + nband_y] layout).  `adaptive` alone says whether a
  // step opens with the CFL and rebuild kernels.
  int   per_env;
  const int   *env_slot;    // [B] geometry slot of each environment (adaptive mode without env_params: all 0)
  const float *env_nu;      // [B] D/Re
  const float *env_dRD;     // [B] dR*D
  const int   *env_nband_x, *env_nband_y;   // [B] band faces of each environment (<= nband_x / nband_y)
};

// Flow sensors (rlfc_config.sensors) of a view of the batch; n = 0: none, nothing is launched for them.  Kept out of
// SolverParams: growing that struct by even 8 bytes changes the register allocation of k_resid_down0<true> (-Xptxas -v).
struct SensorSet {
  const SensorPt* pts;      // [n] resolved sample points
  int n;
  float* out;               // [B][n] the sample of each environment's last solver step (k_sensors)
};

// Flow statistics (rlfc_config.stats_every; flow_stats.cuh) of a view of the batch, pointers at the view's environment e0;
// every = 0: none, nothing is allocated or launched for them.  Kept out of SolverParams for the reason SensorSet is.
constexpr int kNumStats = RLFC_NUM_STATS;
struct FlowStats {
  int every;                // a sample after every `every`-th solver step an environment takes part in
  double* sums;             // [B][kNumStats][stride] the running sums in the level-0 pitched layout, sum s of e at (e*7 + s)*stride
  long long* count;         // [B] samples taken
  int* step;                // [B] solver steps taken part in since the last sample (or the last statistics reset)
  unsigned* ticket;         // [B] CTAs of the running launch that have read `step` (zero between launches)
};

// Snapshot slots (rlfc_config.n_snapshots; snapshot.cuh).  Slot s holds one environment's state: u.x, u.y (step-start
// buffer A) and p (lev[0].x) at s * stride in the level-0 pitched layout, the scalar record rec[w * S + s] (word w of
// snap_word in snapshot.cuh) and the header hdr[w * S + s]: w = 0 written (0 = never), w = 1 .. 5 the bits of the
// (re, dR, gR, theta, t_step) tuple of the environment it was taken from.  With sensors, slot s also holds the
// environment's n sensor values at sens + s * n (SensorSet).
constexpr int kSnapWords = 48;
constexpr int kSnapHdr = 6;
struct SnapSlots {
  int S;                    // slots (0 = none allocated)
  float *ux, *uy, *p;       // [S] fields at s * stride
  unsigned *rec;            // [kSnapWords][S]
  float *sens;              // [S][n] sensors (nullptr without sensors)
  unsigned *hdr;            // [kSnapHdr][S]
  unsigned *env_par;        // [5][B] each environment's parameter tuple (bits), what a restore compares the header with
  int *refused;             // [B] 1 = the last restore into the environment was skipped (rlfc_env_get_flags bit 1)
};

// State records (rlfc.h "State records"; records.cuh).  Allocated by the first record call of a handle, kept out of
// SolverParams for the reason SensorSet is.
struct RecordBufs {
  const unsigned *env_par;  // [5][B] each environment's parameter tuple (bits): SnapSlots::env_par
  const rlfc_sensor *sensors;   // [n_sensors] the sensor table as given at create (nullptr without sensors)
  int *refused;             // [B] 1 = the last device import aimed at the environment was refused (rlfc_env_get_flags bit 3)
  unsigned long long *partial;  // [pairs][chunks] partial checksums
  unsigned *ticket;         // [pairs] CTAs of a pair done (zero between launches)
  int *hcode, *verdict;     // [pairs] header verdict, final verdict (RecordCheck, kRecSkip)
  int grid[3];              // resolution, x_lengths, y_lengths
};
// The checks of an import, in the order they are made; the verdict of a pair is the first that fails (0: apply)
enum RecordCheck { kRecSkip = -1, kRecApply = 0, kRecMagic, kRecVersion, kRecLength, kRecGrid, kRecChecksum, kRecTuple, kRecDt };
// the checksum term of word value x at word index w of a record: MurmurHash3's 64-bit finalizer of (w << 32 | x), a
// bijection, so that changing any one word changes the sum mod 2^64
__host__ __device__ inline unsigned long long record_mix(unsigned long long w, unsigned x) {
  unsigned long long h = w << 32 | x;
  h ^= h >> 33;
  h *= 0xff51afd7ed558ccdull;
  h ^= h >> 33;
  h *= 0xc4ceb9fe1a85ec53ull;
  h ^= h >> 33;
  return h;
}
// bytes of a record of an n x m grid (incl. ghosts) with K sensors
__host__ __device__ inline size_t record_bytes(int n, int m, int K) {
  return RLFC_RECORD_HEADER_BYTES + 4 * kSnapWords + 16 * (size_t)K + 12 * (size_t)n * m;
}

// Parameter library (rlfc_config.param_sets; param_sets.cuh).  Set s's geometry lives in geometry slot sets[s].slot >= B
// (equal sets share one); the rest of what an environment of set s holds per environment is in its LibSet.  Kept out of
// SolverParams for the reason SensorSet is.
struct LibSet {
  int slot;                 // geometry slot: del_x .. rx2_y at slot * stride, band lists at slot * nband_x / nband_y
  int nbx, nby;             // band faces (env_nband_x / env_nband_y)
  float nu, dRD, dt0;       // D/Re, dR*D, t_step*resolution
  unsigned bits[5];         // the (re, dR, gR, theta, t_step) tuple's bits (SnapSlots::env_par)
};
struct ParamLib {
  int L;                    // sets (0 = no library: nothing allocated)
  const LibSet* sets;       // [L]
  int* env_set;             // [B] the set each environment holds, -1 = its own slot (env_params / rlfc_env_reset_params)
};

// Device parameter resets (rlfc_env_reset_params_device; geometry_device.cuh) of a per-environment handle.  Kept out of
// SolverParams for the reason SensorSet is.
struct ParamReset {
  rlfc_env_params* params;  // [B] the set each environment holds on its own slot (what the host copies are refreshed from)
  int* status;              // [B] outcome for the winning pair of the last call: 1 = applied, 2 = refused
  int* refused;             // [B] 1 = the last device parameter reset aimed at the environment was refused (flags bit 2)
};
// The factors of the 40 polygon vertex angles (geometry.h circle_vertex_factors), passed by value.
struct CircleFactors {
  float c[40], s[40];
};

#ifdef __CUDACC__
// true = block `blk` of `nblk` (a kernel's row-block or strip index) belongs to another device
__device__ __forceinline__ bool slab_skip(unsigned blk, unsigned nblk, int rank, int n) {
  if (n <= 1) return false;
  const unsigned lo = (unsigned)((unsigned long long)nblk * (unsigned)rank / (unsigned)n);
  const unsigned hi = (unsigned)((unsigned long long)nblk * (unsigned)(rank + 1) / (unsigned)n);
  return blk < lo || blk >= hi;
}
#endif

// every device of a slab-mode handle waits here for all the others (between dependent kernels)
int launch_slab_barrier(const SlabBarrier& b, cudaStream_t st);

// opt-in shared-memory attributes of the strip kernels; call once per handle before the first launch / capture
int configure_kernels(const SolverParams& P);
// CTAs of the level-0 chain increment kernel per environment (= per-env partial sums of r.r it writes)
int chain_incr_blocks(int ni, int NS);

// ---- launch wrappers (solver_kernels.cu).  All enqueue on `st`; return number of launches. ----
int launch_advdif(const SolverParams& P, const float* srcx, const float* srcy, const float* u0x, const float* u0y,
                  float* dstx, float* dsty, cudaStream_t st);
int launch_band_bc(const SolverParams& P, float* ux, float* uy, cudaStream_t st);
// first MG iteration fused: residual + level-0 smooth(0)/increment/restriction; p_in -> p_out (different buffers)
int launch_resid_down0(const SolverParams& P, const float* ux, const float* uy, const float* p_in, float* p_out, float* r_out,
                       int which, cudaStream_t st);
// projection tail fused: p_out = p_in + shift (different buffers), u -= c * grad(p_in + shift)
int launch_project_shift(const SolverParams& P, const float* p_in, float* p_out, float* ux, float* uy, cudaStream_t st);
// corrector (P.fast_bc only): projection + Heun average u_out = (u + us)/2 away from the boundary lines, then u.setBC and
// the Heun average on the remaining zone
int launch_project_shift_heun(const SolverParams& P, const float* p_in, float* p_out, float* ux, float* uy, const float* usx,
                              const float* usy, float* uox, float* uoy, cudaStream_t st);
int launch_bc_heun(const SolverParams& P, float* ux, float* uy, const float* usx, const float* usy, float* uox, float* uoy,
                   cudaStream_t st);
// one MG iteration (V-cycle + smooth(4)) on active envs = down0, the chained levels' down passes, the one-CTA coarse kernel
// (levels max(1, chain_levels) ..), the chained levels' up / sweeps / incr top down, then level 0's up0 and smooth0 unless
// level 0 is chained; r_in/r_out are the level-0 ping-pong residual buffers
int launch_mg_down0(const SolverParams& P, const float* r_in, float* r_out, cudaStream_t st);
int launch_chain_down(const SolverParams& P, int level, cudaStream_t st);
int launch_coarse_cta(const SolverParams& P, cudaStream_t st);
int launch_chain_up(const SolverParams& P, int level, const float* r, cudaStream_t st);
int launch_chain_sweeps(const SolverParams& P, int level, cudaStream_t st);
int launch_chain_incr(const SolverParams& P, int level, float* r_out, int which, cudaStream_t st);
// level 0 row-smoothed or wavefront-smoothed (not chained)
int launch_mg_up0(const SolverParams& P, float* r, cudaStream_t st);
// rows smoother only: plain level-0 residual <- skewed residual (needed before a further MG iteration's down0)
int launch_unskew_r(const SolverParams& P, float* r, cudaStream_t st);
int launch_smooth0(const SolverParams& P, const float* r_in, float* r_out, int which, cudaStream_t st);
// last node of the MG iteration body inside a CUDA-graph WHILE node: cond = any env still active
int launch_loopcond(const SolverParams& P, unsigned long long cond_handle, cudaStream_t st);
int launch_psum(const SolverParams& P, cudaStream_t st);
int launch_psum_tables(const SolverParams& P, cudaStream_t st);   // (the two kernels of launch_psum, segment-summary mode)
int launch_psum_pass(const SolverParams& P, cudaStream_t st);
int launch_bc(const SolverParams& P, float* ux, float* uy, cudaStream_t st);
int launch_heun(const SolverParams& P, const float* ucx, const float* ucy, const float* ubx, const float* uby,
                float* uax, float* uay, cudaStream_t st);
// force + probes + time advance; accumulate != 0 applies the clientCFD.draw() accumulation
int launch_force(const SolverParams& P, int accumulate, cudaStream_t st);
// flow sensors: s.out[e][k] = Field.linear of sensor k's field (u.x = ux, u.y = uy, p = P.lev[0].x) for every environment
// not frozen.  A step runs it after the corrector's last kernel and before launch_force, which may freeze the environment
int launch_sensors(const SolverParams& P, const SensorSet& s, const float* ux, const float* uy, cudaStream_t st);
// flow statistics: every environment not frozen advances its step counter, and on every f.every-th step adds u.x = ux, u.y = uy,
// p = P.lev[0].x to its sums (rlfc.h "Flow statistics").  A step runs it right after launch_sensors, for the same reason
int launch_flow_stats(const SolverParams& P, const FlowStats& f, const float* ux, const float* uy, cudaStream_t st);
// zero the sums, count and step counter of environments d_ids[0 .. n-1] (device array; ids out of range are skipped)
int launch_stats_reset(const SolverParams& P, const FlowStats& f, const int* d_ids, int n, cudaStream_t st);
// BDIM.checkCFL of every environment's current velocity: d_dt[B] = min(1/(max(|ux|+|uy|) + 3 nu), 1)
int launch_check_cfl(const SolverParams& P, const float* ux, const float* uy, float* d_dt, cudaStream_t st);
// adaptive mode, start of a solver step: sc.dt[e] = BDIM.checkCFL of u for every environment not frozen (frozen ones keep theirs)
int launch_step_cfl(const SolverParams& P, const float* ux, const float* uy, cudaStream_t st);
// adaptive mode: every level's lx, ly, inv, diag and row tables of the environments not frozen, from c = del*(1*dt[e])
// (geometry.cpp finish_level / coarsen restated); level 0 grid-wide, then the coarse levels one CTA per environment
// `skip` [B] (the view's environments): 1 = leave this environment's hierarchy as it is (the step passes sc.frozen)
int launch_poisson_rebuild0(const SolverParams& P, const int* skip, cudaStream_t st);
int launch_poisson_rebuild_coarse(const SolverParams& P, const int* skip, cudaStream_t st);
// mode 0 (single solver steps): xi = actions (NULL keeps xi), every env runs.  mode 1 (RL step): an env takes its
// action only where the reference would have asked for one (t > init_time and at a callLearn boundary); envs whose
// episode is over (t >= episode_time) are frozen for the call
int launch_set_actions(const SolverParams& P, const float* d_actions, int mode, cudaStream_t st);
int launch_emit_obs(const SolverParams& P, const float* d_actions, float* d_obs, float* d_reward, int* d_done,
                    cudaStream_t st);
// Snapshot copy of n (environment, slot) pairs, device arrays d_env[n], d_slot[n]: restore = 0 copies environment
// d_env[k]'s state (u.x = ux, u.y = uy, p = P.lev[0].x, P.sc) to slot d_slot[k], restore = 1 slot d_slot[k] to
// environment d_env[k].  A pair with an entry out of range is skipped; of pairs with the same destination the last wins;
// a restore from an unwritten slot or a slot of another parameter tuple is skipped and sets refused[e] (else clears it).
// keep_accumulators = 1: a restore leaves callLearn, Cd, Cl and obs as they are.  skip != nullptr: a restore writes
// skip[e] = 0 for every environment it restored (the mask of a following launch_poisson_rebuild*).  The environments' sensors
// `sens` move with the state (sens.n = 0: none).
int launch_snapshot_copy(const SolverParams& P, const SnapSlots& s, const SensorSet& sens, float* ux, float* uy, const int* d_env,
                         const int* d_slot, int n, int restore, int keep_accumulators, int* skip, cudaStream_t st);
// Parameter-library reset of n (environment, set) pairs, device arrays d_env[n], d_set[n] (P: the whole batch, per_env):
// environment d_env[k] takes library set d_set[k] (env_slot, env_set, env_nu, env_dRD, env_nband_x/y, sc.dt = dt0, and
// with snapshots snap.env_par), the init fields init_ux / init_uy / init_p (one environment, pitched) into ux, uy and
// P.lev[0].x, and the reset scalars of rlfc_env_reset (flow_t = init_t; reset_accumulators: callLearn = substeps, Cd = Cl =
// obs = 0).  Pairs out of range are skipped, of pairs with the same environment the last wins, and skip[e] = 0 is written
// for every environment reset (the mask of the following launch_poisson_rebuild*).
int launch_reset_sets(const SolverParams& P, const ParamLib& lib, const SnapSlots& snap, const float* init_ux,
                      const float* init_uy, const float* init_p, float init_t, float* ux, float* uy, const int* d_env,
                      const int* d_set, int n, int reset_accumulators, int* skip, cudaStream_t st);
// Device parameter reset of n (environment, parameter set) pairs, device arrays d_env[n], d_par[n] (P: the whole batch,
// per_env; two launches): the winning pair of each environment (pairs out of range are skipped, the last in-range pair per
// environment wins) is validated as build_env_geometries validates a set, plus |theta| <= 2 pi.  An applied pair builds the
// set's geometry into the environment's own slot (del, the body-velocity basis, the band lists, as build_geometry and
// band_lists make them), points the environment at it (env_slot, lib.env_set = -1, env_nu, env_dRD, env_nband_x/y,
// pr.params, snap.env_par) and does what launch_reset_sets does with dt = t_step*resolution; a refused pair changes
// nothing but pr.refused[e] = 1.  cap = the slots' band capacity (nband_x == nband_y).
int launch_reset_params(const SolverParams& P, const ParamLib& lib, const SnapSlots& snap, const ParamReset& pr,
                        const CircleFactors& cf, int nc, int mc, int cap, const float* init_ux, const float* init_uy,
                        const float* init_p, float init_t, float* ux, float* uy, const int* d_env,
                        const rlfc_env_params* d_par, int n, int reset_accumulators, int* skip, cudaStream_t st);

// State records (records.cuh): record_chunks = the partial checksums per pair a launch of bytes-long records needs.
// Export writes record k (record_bytes(P.n, P.m, sens.n) bytes at rec + k * that) of environment d_ids[k], a record with a
// zero header for an id out of range.  Import with check = 1 writes rb.verdict (the winning pair of each destination is
// checked, the others skipped) and nothing else; check = 0 then applies the pairs whose verdict is 0, writes rb.refused of
// every winning pair and skip[e] = 0 of those applied.
int record_chunks(int n, int m, size_t bytes);
int launch_record_export(const SolverParams& P, const SensorSet& sens, const RecordBufs& rb, float* ux, float* uy,
                         const int* d_ids, int n, void* rec, cudaStream_t st);
int launch_record_import(const SolverParams& P, const SensorSet& sens, const RecordBufs& rb, float* ux, float* uy,
                         const int* d_ids, int n, const void* rec, size_t bytes, int check, int keep_accumulators, int* skip,
                         cudaStream_t st);

}  // namespace rlfc
