/*
 * rlfc.h -- C ABI of rlfluidcontrol_b200: batched Lilypad AFCCylinder environments on B200 (sm_100a).
 *
 * This is the drop-in boundary for the CFD environment step of LiuYangMage/RLFluidControl.  The
 * reference has no FFI layer; the path sits behind a Java object boundary, and each entry point
 * below names the reference interface it replaces (paths relative to clientLilypad/):
 *
 *   rlfc_env_create      <- new AFCCylinder(resolution,Re,dR,gR,theta,xi1,xi2,tStep,xLengths,yLengths,
 *                           zoom,isResume)              AFCCylinder.pde:11-42, clientCFD.pde:93-102
 *                           (+ BDIM ctor BDIM.pde:41-71, BDIM.resume BDIM.pde:239-251)
 *   rlfc_env_reset       <- setUpNewSim(): a fresh AFCCylinder resumed from saved/init/init.bdim
 *                           clientCFD.pde:93-102
 *   rlfc_env_substep     <- AFCCylinder.update2() + test.force + SaveScalar.addData03 probes
 *                           AFCCylinder.pde:45-61, SaveScalar.pde:61-72
 *   rlfc_env_step        <- `substeps` frames of clientCFD.draw(): update2(), force accumulation,
 *                           (Cl,Cd) observation, xi/xi_m update         clientCFD.pde:35-55
 *                           reward = server/server.py:61-65 (_reward_func) of the unchanged peer
 *   rlfc_env_get_fields  <- BDIM.write layout (u.x, u.y, p; i-major, ghosts included) BDIM.pde:226-237
 *   rlfc_env_set_fields  <- BDIM.resume                                  BDIM.pde:239-251
 *   rlfc_env_save_bdim / rlfc_env_load_bdim <- BDIM.write / BDIM.resume text checkpoint format
 *
 * Conventions: every call returns 0 on success or a negative RLFC_E* code and never aborts;
 * rlfc_last_error() gives a thread-local message.  One host thread per handle (no locking).
 * Host-pointer calls are synchronous on return.  *_device calls take device pointers, enqueue on
 * the handle's stream and return without synchronising.  Field import/export always uses the
 * reference layout a[i][j] (i = x outer, j = y contiguous, ghost ring included: (n+2) x (m+2))
 * regardless of the internal pitched device layout.  There is NO CPU fallback: if no CUDA device is
 * usable rlfc_env_create fails with RLFC_ENODEV.
 */
#ifndef RLFC_H
#define RLFC_H

#ifdef __cplusplus
extern "C" {
#endif

#define RLFC_OK        0
#define RLFC_EINVAL   -1   /* bad argument / configuration                                   */
#define RLFC_ENODEV   -2   /* no usable CUDA device (there is no CPU fallback)               */
#define RLFC_ECUDA    -3   /* CUDA runtime error (message in rlfc_last_error)                */
#define RLFC_EIO      -4   /* checkpoint file could not be read / written / parsed           */
#define RLFC_ENOMEM   -5
#define RLFC_EGRID    -6   /* a grid the reference's multigrid cannot run: level 0 (x_lengths*resolution by
                              y_lengths*resolution cells) must be even in both directions, because MG.prolongate
                              and MG.increment (MG.pde:94-97,139-152) would write past the coarse correction, and a
                              coarse level that is not divisible must have a side <= 9 (incl. ghosts), because
                              MG.divisible (MG.pde:99-106) would exit()                                          */
#define RLFC_ENOTCONV -7   /* reserved                                                       */

#define RLFC_NUM_PROBES 32 /* SaveScalar numTheta, clientCFD.pde:102                         */

typedef struct rlfc_env rlfc_env;   /* opaque; owns all device + pinned-host memory */

/* The per-environment arguments of the AFCCylinder constructor (AFCCylinder.pde:11-42).  resolution, x_lengths and
   y_lengths fix the grid and stay handle-wide.  Valid sets: re >= 1, 0 < dR <= 1, gR >= 0, theta finite, t_step finite
   and > 0, convex bodies (Body.pde:90-96), and no body-band face on rows 0, 1, n-2, n-1 or columns 0, 1, m-2, m-1. */
typedef struct {
  int   re;
  float dR, gR, theta, t_step;
} rlfc_env_params;

/* A flow sensor: the value of one field at one point, sampled on the device after every solver step (rlfc_env_get_sensors).
   (x, y) are grid coordinates as Body and SaveScalar use them: one unit is one cell, the main cylinder's centre is at
   (x_lengths*resolution/4, y_lengths*resolution/2).  The value is the reference's Field.linear(x, y) (Field.pde:175-190) of
   that field with the field's own btype: the point is clamped to [0.5, n-1.5] x [0.5, m-1.5], then shifted by +0.5 in x
   for u.x and in y for u.y, and interpolated bilinearly.  A p sensor at a SaveScalar point equals that probe bit for bit. */
#define RLFC_SENSOR_P   0   /* pressure p (btype 0)                                                  */
#define RLFC_SENSOR_UX  1   /* velocity u.x (btype 1)                                                */
#define RLFC_SENSOR_UY  2   /* velocity u.y (btype 2)                                                */
typedef struct {
  int   field;          /* RLFC_SENSOR_P, _UX or _UY                                                */
  float x, y;
} rlfc_sensor;

typedef struct {
  /* defaults (rlfc_default_config) reproduce clientCFD.pde:5-14,94-96 and AFCCylinder.pde:4-7 */
  int   resolution;     /* 24   cells per main-cylinder diameter                     */
  int   x_lengths;      /* 16   domain length in diameters  -> n = 384 cells         */
  int   y_lengths;      /* 8                                -> m = 192 cells         */
  int   re;             /* 500  Reynolds number, nu = D/Re                           */
  float dR;             /* .125 control-cylinder diameter / D                        */
  float gR;             /* .2   gap / D                                              */
  float theta;          /* PI/3 control-cylinder position angle                      */
  float t_step;         /* .0075 non-dimensional time step; dt = t_step*resolution   */
  float action_scale;   /* 5    xi_m = action_scale * xi  (clientCFD.pde:53-54)      */
  int   substeps;       /* 16   solver steps per RL step (callLearn, clientCFD.pde:12) */
  float init_time;      /* 1    no accumulation/actions while t <= init_time         */
  float episode_time;   /* 50   done when t >= episode_time                          */
  int   n_envs;         /* number of independent environments batched on this device */
  int   device;         /* CUDA device ordinal; -1 = current device                  */
  int   exact;          /* 1 = bit-faithful mode (only mode implemented)             */
  int   mg_max_iters;   /* 20   MGsolver itmx (VectorField.pde:135)                  */
  const char *init_bdim_path; /* NULL = uniform flow u=(1,0), p=0; else a .bdim text
                                 checkpoint (BDIM.write format) or a .bdimb binary one */
  void *stream;         /* cudaStream_t to run on; NULL = the library creates its own */
  int   n_groups;       /* env groups advanced concurrently on separate streams; 0 = auto    */
  int   n_devices;      /* 1 (default) = the handle lives on `device`.  > 1 = SLAB MODE (n_envs must be 1): ONE domain
                           advanced by devices device .. device + n_devices - 1 of this process, which share every
                           field through one address range (CUDA virtual memory management + peer access over
                           NVLink): rows / strips are distributed, halo operands are ordinary peer loads, the
                           lexicographic Gauss-Seidel sweeps cross devices strip to strip, results are bit-identical
                           to the single-device run (BASELINE config 5; DESIGN.md 5)                         */
  int   adaptive_dt;    /* 0 (default) = every solver step is AFCCylinder.update2 with the fixed dt = t_step*resolution.
                           1 = every solver step of every entry point is AFCCylinder.update() (AFCCylinder.pde:63-84):
                           each environment taking part in the step first sets dt[e] = min(CFL(u[e], nu), 1)
                           (BDIM.checkCFL) and then runs the update2 statements with it.  The Poisson hierarchy
                           (c = del*dt and every coarse level) is rebuilt per environment on the device before each step.
                           Not available in slab mode or with the chained / wavefront smoothers (RLFC_EINVAL).       */
  const rlfc_env_params *env_params;
                        /* NULL (default) = every environment uses re, dR, gR, theta, t_step above.  Else n_envs entries:
                           PER-ENVIRONMENT MODE, environment e is new AFCCylinder(resolution, env_params[e]..., x_lengths,
                           y_lengths) with its own Reynolds number, control cylinders, fixed dt = t_step*resolution and
                           Poisson hierarchy.  Combines with adaptive_dt 0 and 1; has the same restrictions as adaptive_dt
                           (RLFC_EINVAL in slab mode and with the chained / wavefront smoothers).  The entries are copied
                           and validated before any device call; an invalid one fails with RLFC_EINVAL.                */
  int   n_snapshots;    /* 0 (default) = no snapshot slots: nothing is allocated or launched for them.  > 0 = that many
                           device slots, each holding one environment's complete state (rlfc_env_snapshot below; about
                           0.93 MB per slot at the default grid).  RLFC_EINVAL if < 0, or > 0 in slab mode.             */
  int   n_sensors;      /* 0 (default) = no sensors: nothing is allocated or launched for them.  > 0 = the number of entries
                           of `sensors`, sampled in every environment (rlfc_env_get_sensors below).  The set is handle-wide
                           and fixed at create.  RLFC_EINVAL if < 0, or > 0 in slab mode.                               */
  const rlfc_sensor *sensors;
                        /* n_sensors entries, copied and validated before any device call: RLFC_EINVAL for NULL with
                           n_sensors > 0, a field outside RLFC_SENSOR_P .. RLFC_SENSOR_UY or a non-finite coordinate.     */
  int   n_param_sets;   /* 0 (default) = no parameter library: nothing is allocated or launched for it.  > 0 = the number of
                           entries of `param_sets`, a library of constructor arguments that rlfc_env_reset_sets(_device)
                           switches environments to on the device.  Puts the handle in per-environment mode: without
                           env_params it is a handle created with env_params = n_envs copies of the scalar config's set.
                           About 3.25 MB of device memory per distinct set at the default grid.                        */
  const rlfc_env_params *param_sets;
                        /* n_param_sets entries, copied, validated (as env_params) and their geometries built at create,
                           before any device call.  RLFC_EINVAL for n_param_sets < 0, NULL with n_param_sets > 0, an
                           invalid entry (the message names param_sets[k]), slab mode, or a grid with chained or wavefront
                           levels.                                                                                     */
} rlfc_config;

void rlfc_default_config(rlfc_config *cfg);

int  rlfc_env_create(const rlfc_config *cfg, rlfc_env **out);
void rlfc_env_destroy(rlfc_env *env);

/* Reload the initial state into the listed environments (NULL = all): u, p from the init
   checkpoint (or uniform flow), t = 0, xi = 0, dt = t_step*resolution.  The draw()-loop accumulators (callLearn, Cd, Cl)
   are sketch globals in the reference and survive setUpNewSim (clientCFD.pde:11-13); pass
   reset_accumulators != 0 to also restore them to (16, 0, 0). */
int  rlfc_env_reset(rlfc_env *env, const int *env_ids, int n, int reset_accumulators);

/* setUpNewSim with new constructor arguments (clientCFD.pde:93-102), per-environment handles only (else RLFC_EINVAL):
   environment env_ids[k] takes params[k], its geometry and Poisson hierarchy, and then exactly what rlfc_env_reset does.
   Every set is validated and every geometry built before anything on the device changes: if one set is invalid
   (RLFC_EINVAL) no environment changes.  The environments not listed are untouched. */
int  rlfc_env_reset_params(rlfc_env *env, const int *env_ids, int n, const rlfc_env_params *params,
                           int reset_accumulators);
/* params[n_envs]: each environment's constructor arguments (the scalar config's for every environment of a handle
   created without env_params), as the environments hold them now, including sets switched by rlfc_env_reset_sets_device. */
int  rlfc_env_get_params(rlfc_env *env, rlfc_env_params *params);

/* setUpNewSim into the parameter library (rlfc_config.param_sets), handles with a library only.  Environment env_ids[k]
   becomes what rlfc_env_reset_params({env_ids[k]}, {param_sets[sets[k]]}, reset_accumulators) makes it -- the set's
   geometry, nu, dR*D, dt = t_step*resolution and Poisson hierarchy, u and p from the init state, t = 0, xi = 0, BDIM.t from
   the checkpoint, force = 0, the frozen and non-finite flags cleared, with reset_accumulators callLearn = substeps and
   Cd = Cl = obs = 0 -- bit for bit, without building anything on the host.  Sensors, probes, MG iteration counts and flags
   bit 1 stay as they are (as with rlfc_env_reset).  A later rlfc_env_reset keeps the set; rlfc_env_reset_params puts the
   environment back on its own geometry slot.
   HOST arrays, synchronous on return, all or nothing: RLFC_EINVAL (and nothing changes) for a handle without a library, an
   id or set out of range, or an environment listed twice. */
int  rlfc_env_reset_sets(rlfc_env *env, const int *env_ids, const int *sets, int n, int reset_accumulators);
/* Same with DEVICE int arrays of length n, asynchronous on the handle's stream.  Defined for every input: a pair with an
   entry out of range is skipped (a negative set is the way to skip one, e.g. sets = where(done, draw, -1)); of pairs with
   the same environment the last in-range pair wins. */
int  rlfc_env_reset_sets_device(rlfc_env *env, const int *d_env_ids, const int *d_sets, int n, int reset_accumulators);

/* One RL step for every environment, with the cadence of clientCFD.draw() (clientCFD.pde:35-55).  All pointers are
   HOST memory.
     actions [n_envs][2] in [-1,1]
     obs     [n_envs][2] = (Cl, Cd) exactly as clientCFD.pde:44-47 forms them (incl. the carry-over)
     reward  [n_envs]    = -Cd - pi/8*0.0097*3.66^3*sum|a|^3 (server.py:61-65), may be NULL
     done    [n_envs]    = t >= episode_time, may be NULL
   Every environment advances to ITS next observation and then waits (the sketch blocks in callAction until the agent
   answers, clientCFD.pde:50):
     * an environment that emitted an observation at the end of the previous call (t > init_time, callLearn back at
       `substeps`) takes actions[e] as its new xi (xi_m = action_scale*xi) and runs exactly `substeps` solver steps --
       the reference changes xi only at a callLearn boundary, so each observation covers `substeps` steps under ONE action;
     * an environment that has not reached its first callLearn boundary yet -- fresh from rlfc_env_reset with
       t <= init_time, or mid-window after an episode change with the sketch-global accumulators kept -- IGNORES
       actions[e] (the reference has not asked for an action yet: xi stays what it is, 0 after a reset) and runs,
       uncontrolled, until t > init_time and then through its first accumulation window (defaults: 133 + 16 solver
       steps).  The first call after a reset therefore returns the reference's first observation; pass zeros as its
       action (the reward formula uses what is passed).  While such an environment catches up the others stay put;
     * an environment whose episode is over (t >= episode_time, clientCFD.pde:36) takes no more solver steps: done[e]
       stays 1 and obs[e] is the last observation until the caller resets it.
   With init_time < 0 every environment is at a boundary right after a reset and every call is `substeps` steps. */
int  rlfc_env_step(rlfc_env *env, const float *actions, float *obs, float *reward, int *done);

/* Same, DEVICE pointers, asynchronous on the handle's stream (no host copies, no sync).  Runs ONE round of `substeps`
   solver steps with the same per-environment rules; an environment that is still short of its first observation after
   the round (see above) simply continues in the next call -- rlfc_env_running() tells.  For batches whose environments
   are all at a callLearn boundary (the steady state) it is identical to rlfc_env_step. */
int  rlfc_env_step_device(rlfc_env *env, const float *d_actions, float *d_obs, float *d_reward, int *d_done);

/* Number of environments that had NOT emitted their observation when the last RL-step round ended (0 in the steady
   state).  Synchronises the handle's stream. */
int  rlfc_env_running(rlfc_env *env, int *n_running);

/* Per-environment health flags, flags[n_envs]: bit 0 = a non-finite force was produced since the last reset (the
   environment has diverged; SURVEY section 5 failure detection).  Bit 1 = the last restore aimed at the environment was
   skipped because its slot was never written or holds a state of another parameter set (rlfc_env_restore_device; a restore
   that applies clears it).  Synchronises the handle's stream. */
int  rlfc_env_get_flags(rlfc_env *env, int *flags);

/* Snapshots of complete environment states in the handle's rlfc_config.n_snapshots device slots (ALE cloneState /
   restoreState for the batch).  A state is everything the next solver or RL step reads and the read-outs return: u, p
   (the MG initial guess), xi, t, BDIM.t, dt, force, probes, callLearn, Cd, Cl, the last observation, the frozen and
   non-finite flags, the MG iteration counts and the parameter set.  After rlfc_env_snapshot(e -> s) and
   rlfc_env_restore(s -> e'), e' continues bit-identically to what e did from the snapshot, through every entry point.
   A state moves only between environments with bitwise equal (re, dR, gR, theta, t_step); in adaptive mode a restore
   rebuilds the destination's Poisson hierarchy from the restored dt.
     rlfc_env_snapshot: environment env_ids[k] -> slot slots[k];  rlfc_env_restore: slot slots[k] -> environment env_ids[k].
     keep_accumulators != 0: the destination keeps its own callLearn, Cd, Cl and obs (sketch globals that survive
       setUpNewSim); 0 takes the snapshot's.  With S0 taken right after rlfc_env_reset(all, reset_accumulators = 1),
       rlfc_env_restore(e, S0, k) is rlfc_env_reset({e}, reset_accumulators = !k) for every step that follows.
   HOST arrays, synchronous on return, all or nothing: RLFC_EINVAL (and nothing changes) for a handle without slots, an id
   or slot out of range, a destination listed twice, a restore from a slot never written or of another parameter set. */
int  rlfc_env_snapshot(rlfc_env *env, const int *env_ids, const int *slots, int n);
int  rlfc_env_restore(rlfc_env *env, const int *env_ids, const int *slots, int n, int keep_accumulators);
/* Same with DEVICE int arrays of length n, asynchronous on the handle's stream (the host never sees the ids).  Defined for
   every input: a pair with an entry out of range is skipped (a negative entry is the way to skip one, e.g.
   slots = where(done, S0, -1)); of pairs with the same destination the last in-range pair wins; a restore from a slot never
   written or of another parameter set is skipped and sets flags bit 1 of the destination. */
int  rlfc_env_snapshot_device(rlfc_env *env, const int *d_env_ids, const int *d_slots, int n);
int  rlfc_env_restore_device(rlfc_env *env, const int *d_env_ids, const int *d_slots, int n, int keep_accumulators);

/* The sensors (rlfc_config.sensors) of every environment, out[n_envs][n_sensors].  Each environment's sensors hold the
   sample of its most recent solver step, taken from the state the next step starts from -- the u and p rlfc_env_get_fields
   returns -- so right after any call sensor == Field.linear of rlfc_env_get_fields(e).  An environment that takes no part
   in a solver step keeps its values: after rlfc_env_step an environment holds the sample of the step that completed its
   observation window (its sensor observation), one whose episode is over keeps its last one.  rlfc_env_reset and
   rlfc_env_reset_params leave sensors alone (the next step overwrites them); snapshots carry them with the state.
   HOST memory, synchronises the handle's stream.  RLFC_EINVAL for a handle created without sensors. */
int  rlfc_env_get_sensors(rlfc_env *env, float *out);
/* Same into DEVICE memory: one device-to-device copy on the handle's stream, no sync.  Enqueued after
   rlfc_env_step_device, it gives a GPU-resident policy its observation without the host. */
int  rlfc_env_get_sensors_device(rlfc_env *env, float *d_out);

/* One solver step (AFCCylinder.update2) without the draw() accumulation.  HOST pointers.
     actions [n_envs][2] (NULL = keep current xi); force [n_envs][2] raw (fx, fy) = -pressForce;
     probes  [n_envs][32] surface pressure samples or NULL.                                     */
int  rlfc_env_substep(rlfc_env *env, const float *actions, float *force, float *probes);

/* Same solver step, asynchronous on the handle's stream: d_actions is a DEVICE pointer ([n_envs][2]) or NULL (keep xi);
   nothing is copied back (force and probes stay on the device: rlfc_env_substep(env, NULL, ...) style read-outs or
   rlfc_env_get_fields synchronise later). */
int  rlfc_env_substep_device(rlfc_env *env, const float *d_actions);

/* Field export/import for one environment, reference layout (n+2)*(m+2) floats each; NULL skips. */
int  rlfc_env_get_fields(rlfc_env *env, int e, float *ux, float *uy, float *p);
int  rlfc_env_set_fields(rlfc_env *env, int e, const float *ux, const float *uy, const float *p);

/* Field.sum() of every environment's pressure field (Field.pde:311-318: serial float accumulation over the
   interior, i-major): sums[n_envs].  Runs the same device path the projection uses (VectorField.pde:136). */
int  rlfc_env_field_sum(rlfc_env *env, float *sums);
/* Counters of the last Field.sum evaluation of every environment (the projection's or rlfc_env_field_sum's),
   stats[n_envs][8]: [0] batches (32 segment summaries) crossed by their condensed record, [1] batches walked
   summary by summary, [2] record entries applied, [3] segments redone as 32 float additions; [4..7] reserved.
   All zero with RLFC_PSUM=serial. */
int  rlfc_env_field_sum_stats(rlfc_env *env, int *stats);

/* Text checkpoint of one environment in the BDIM.write format (readable by BDIM.resume).  Line 1 holds the dt: the
   handle's fixed dt, or in adaptive or per-environment mode the environment's own.  Loading requires the environment's
   fixed dt in fixed mode and accepts any positive dt in adaptive mode, where it becomes the environment's current dt. */
int  rlfc_env_save_bdim(rlfc_env *env, int e, const char *path);
int  rlfc_env_load_bdim(rlfc_env *env, int e, const char *path);

/* BDIM.checkCFL (BDIM.pde:217-219, VectorField.CFL VectorField.pde:225-235) of every environment's current velocity:
   dt[n_envs] = min(1 / (max_interior(|ux| + |uy|) + 3 nu[e]), 1), the time step the reference's adaptive variant
   AFCCylinder.update() (AFCCylinder.pde:63-84) would take next.  A handle created with adaptive_dt = 1 takes exactly
   that dt in its next solver step; with adaptive_dt = 0 the steps run the fixed dt of AFCCylinder.update2 (what
   clientCFD.pde calls). */
int  rlfc_env_check_cfl(rlfc_env *env, float *dt);
/* dt[n_envs]: the time step (grid units) of each environment's last solver step.  Fixed mode: t_step*resolution (the
   environment's own t_step in per-environment mode).  Adaptive mode: the CFL step the environment took last;
   t_step*resolution after create / reset, the checkpoint's dt after rlfc_env_load_bdim.  Synchronises the handle's stream. */
int  rlfc_env_get_dt(rlfc_env *env, float *dt);
/* Environment e's Poisson coefficients as its last solver step used them, reference layout at the given MG level:
   "lower.x", "lower.y", "inv", "diag" (any level), "c.x", "c.y", "del.x", "del.y" (level 0 only).  Fixed mode without
   env_params: the same fields as rlfc_env_get_static.  Adaptive or per-environment mode: the environment's own hierarchy,
   built on the device from c = del[e]*dt[e]. */
int  rlfc_env_get_coeffs(rlfc_env *env, int e, const char *name, int level, float *out, int *n, int *m);

/* Introspection. */
int  rlfc_env_dims(const rlfc_env *env, int *n_with_ghosts, int *m_with_ghosts, int *n_envs);
int  rlfc_env_get_time(rlfc_env *env, float *t /*[n_envs]*/);
/* MG iterations used by the last predictor / corrector solve of each env: iters[n_envs][2]. */
int  rlfc_env_get_mg_iters(rlfc_env *env, int *iters);
/* Static geometry/coefficient fields by name, reference layout at the given MG level:
   "del.x","del.y","del1.x","del1.y","wnx.x","wnx.y","wny.x","wny.y","c.x","c.y" (level 0 only),
   "lower.x","lower.y","inv","diag" (any level).  Used by the parity tests. */
int  rlfc_env_get_static(rlfc_env *env, const char *name, int level, float *out, int *n, int *m);
int  rlfc_env_num_levels(const rlfc_env *env);
/* Same lookup without a device: builds the host-side geometry for `cfg` and returns one static
   field (also "w1.x","w2.x","ry1.x","ry2.x","w1.y","w2.y","rx1.y","rx2.y": the body-velocity basis).
   Needs no GPU; used by the CPU-side tests of the host logic. */
int  rlfc_geometry_static(const rlfc_config *cfg, const char *name, int level, float *out,
                          int *n, int *m, int *nlevels);
/* Per-kernel device timing with CUDA events on the handle's stream.  While profiling is on every
   kernel launch is bracketed by an event pair; rlfc_env_get_profile(idx) returns the idx-th kernel's
   name, accumulated milliseconds, launch count and its ALGORITHMIC bytes per launch (per-env arrays
   only, one read per input / one write per output, whole batch); it returns 1 past the last entry. */
int  rlfc_env_set_profiling(rlfc_env *env, int on);
int  rlfc_env_get_profile(rlfc_env *env, int idx, char *name, int name_cap, double *ms_total,
                          long long *launches, double *algorithmic_bytes_per_launch);
/* The stream the handle enqueues on (cudaStream_t), for event timing by the caller. */
void *rlfc_env_stream(rlfc_env *env);
/* Slab mode (rlfc_config.n_devices > 1): the devices sharing the domain, the device-wide barriers executed so far (one
   between any two dependent kernels: the exchange count), and the bytes of the shared address range.  n_devices = 1,
   0, 0 for an ordinary handle. */
int  rlfc_env_slab_info(const rlfc_env *env, int *n_devices, long long *barriers, long long *bytes_shared);
/* Number of kernel launches (incl. those inside replayed CUDA graphs) issued so far. */
long long rlfc_env_launch_count(const rlfc_env *env);
/* Algorithmic bytes moved per solver step per env (SURVEY section 8d model) given the MG iteration
   counts of the last step; used by bench.py for the roofline line. */
double rlfc_env_model_bytes_per_solver_step(const rlfc_env *env);

/* java.lang.Float.toString(v) (what String.valueOf(float) / ""+float give in the reference: checkpoint lines,
   SaveScalar traces, the "<Cl>_<Cd>" RPC payload, clientCFD.pde:119).  Returns the length. */
int  rlfc_format_float_java(float v, char *buf, int cap);

const char *rlfc_last_error(void);
const char *rlfc_version(void);

#ifdef __cplusplus
}
#endif
#endif
