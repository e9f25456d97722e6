/*
 * lilypad_oracle.h -- CPU restatement of the Lilypad AFCCylinder environment step.
 *
 * TEST INFRASTRUCTURE ONLY.  This is the correctness oracle and the CPU baseline
 * for rlfluidcontrol_b200.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may build, link, import or execute it.  The product
 * (rlfluidcontrol_b200/, include/rlfc.h, librlfc.so) never calls into this file.
 *
 * PARITY UNPINNED: the reference (Processing/Java, /root/reference/clientLilypad)
 * ships no tests and no golden outputs for this path, and no JVM exists in the
 * build image, so this restatement cannot be diffed against the Java itself.  It is
 * pinned only by (i) the three docstring known-answers (Body.pde:27, MG.pde:13-25,
 * PoissonMatrix.pde:17-31), (ii) the invariants of the shipped input fixture
 * saved/init/init.bdim, (iii) drift-check values from an independent survey probe
 * (SURVEY.md section 8c).  Residual risks: java.lang.Math.sin/cos vs glibc (geometry
 * set-up only), Float.parseFloat vs strtof.
 *
 * All arithmetic is IEEE binary32 with no FMA contraction (build with
 * -ffp-contract=off), exactly as Java `float`; sin/cos/sqrt are evaluated in double
 * and narrowed, as Processing's PApplet wrappers do.
 */
#ifndef LILYPAD_ORACLE_H
#define LILYPAD_ORACLE_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- Field.pde:24-58 : scalar field float[n][m] (i-major, j contiguous) + ghost ring ---- */
typedef struct {
  int n, m, btype, gradientExit;
  float bval;
  float *a;
} ora_field;

typedef struct { ora_field x, y; } ora_vfield;          /* VectorField.pde:22-39 */

/* OrthoNormal.pde:3-18 */
typedef struct { float l, nx, ny, tx, ty, off, t1, t2, cenx, ceny; } ora_ortho;

/* Body.pde:40-100 (+ EllipseBody/CircleBody :382-417); box is the 4-point bounding Body */
typedef struct ora_body {
  int n;                  /* number of vertices */
  int north;              /* number of segments */
  float *cx, *cy;         /* coords */
  ora_ortho *orth;
  float xcx, xcy;         /* xc */
  float dxcx, dxcy, phi, dphi;
  float area, I0, mass;
  int convex;
  int is_circle;          /* CircleBody overrides distance() and rotate() */
  float h;                /* EllipseBody.h (diameter for CircleBody) */
  struct ora_body *box;
} ora_body;

/* PoissonMatrix.pde:32-51 */
typedef struct { int n, m; ora_vfield lower; ora_field diagonal, inv; } ora_poisson;

typedef struct ora_env ora_env;

/* ---------------- field algebra (Field.pde / VectorField.pde) ---------------- */
ora_field  ora_field_new(int n, int m, int btype, float bval);            /* Field.pde:30-37 */
ora_field  ora_field_copy(const ora_field *b);                            /* Field.pde:51-58 */
void       ora_field_free(ora_field *f);
void       ora_field_setBC(ora_field *f);                                 /* Field.pde:209-234 */
float      ora_field_linear(const ora_field *f, float x0, float y0);      /* Field.pde:175-190 */
float      ora_field_inner(const ora_field *a, const ora_field *b);       /* Field.pde:302-310 */
float      ora_field_sum(const ora_field *a);                             /* Field.pde:311-318 */
float      ora_field_Linf(const ora_field *a);                            /* Field.pde:340-347 */
ora_vfield ora_vfield_new(int n, int m, float xval, float yval);          /* VectorField.pde:27-32 */
ora_vfield ora_vfield_copy(const ora_vfield *b);
void       ora_vfield_free(ora_vfield *v);
void       ora_vfield_setBC(ora_vfield *v);                               /* VectorField.pde:41-44 */
void       ora_vfield_AdvDif(ora_vfield *F, const ora_vfield *u0, float dt, float nu); /* :170-179 */
ora_field  ora_vfield_divergence(const ora_vfield *u);                    /* :56-65 */
ora_vfield ora_field_gradient(const ora_field *p);                        /* Field.pde:71-81 */
/* VectorField.project (VectorField.pde:130-143); returns MG iterations used */
int        ora_vfield_project(ora_vfield *u, const ora_vfield *coeffs, ora_field *p, int literal,
                              const void *cached_hierarchy);

/* ---------------- PoissonMatrix / MG ---------------- */
ora_poisson ora_poisson_new(const ora_vfield *lower);                     /* PoissonMatrix.pde:38-51 */
void        ora_poisson_free(ora_poisson *A);
ora_field   ora_poisson_times(const ora_poisson *A, const ora_field *x);  /* :53-64 */
/* MGsolver(itmx, A, x, b) MG.pde:30-38.  x is updated in place.  Returns iterations.
   If hier!=NULL it is an array of pre-restricted matrices hier[0]=A, hier[1]=restrict(A)...
   (numerically identical to rebuilding them every V-cycle as MG.pde:70 does). */
int         ora_mg_solve(float itmx, const ora_poisson *A, ora_field *x, const ora_field *b,
                         const ora_poisson *hier, int nhier, float *rr_out, float *tol_out);
ora_poisson ora_mg_restrict_matrix(const ora_poisson *A);                 /* MG.pde:108-122 */
ora_field   ora_mg_restrict_field(const ora_field *a);                    /* MG.pde:124-137 */
ora_field   ora_mg_prolongate(const ora_field *a);                        /* MG.pde:139-152 */

/* ---------------- bodies ---------------- */
ora_body *ora_body_new(float x, float y);                                 /* Body.pde:57-60 */
void      ora_body_add(ora_body *b, float x, float y);                    /* :62-64 */
void      ora_body_end(ora_body *b);                                      /* :66-100 */
ora_body *ora_circle_new(float x, float y, float d);                      /* :386-406 */
void      ora_body_free(ora_body *b);
float     ora_body_distance(const ora_body *b, float x, float y);         /* :174-192 / :408-410 */
void      ora_body_wallnormal(const ora_body *b, float x, float y, float *nx, float *ny); /* :215-232 */
float     ora_body_velocity(const ora_body *b, int d, float dt, float x, float y);        /* :234-240 */
void      ora_body_pressForce(const ora_body *b, const ora_field *p, float *fx, float *fy); /* :296-303 */
float     ora_bdim_delta0(float d, float eps);                            /* BDIM.pde:199-207 */
float     ora_bdim_delta1(float d, float eps);                            /* BDIM.pde:209-215 */
float     ora_union_delta0(float d);                                      /* BodyUnion.pde:158-166 */

/* ---------------- the environment: AFCCylinder + BDIM + clientCFD accumulation ---------------- */
typedef struct {
  int resolution, xLengths, yLengths, Re;
  float dR, gR, theta, tStep;
  int literal;     /* 1: rebuild coefficients/matrices exactly where the reference does
                      (BDIM.pde:127, VectorField.pde:135, MG.pde:70); 0: cache them (same numbers) */
} ora_config;

ora_config ora_default_config(void);                                      /* clientCFD.pde:9,14,94-96 */
/* AFCCylinder.pde:11-42 (no resume).  NULL for a grid the reference cannot run: an odd level 0 (MG.prolongate /
   MG.increment, MG.pde:94-97,139-152, would write past the coarse correction) or a non-divisible coarse level with
   both sides > 9 (MG.divisible, MG.pde:101-104, would exit()). */
ora_env *ora_env_new(const ora_config *cfg);
void     ora_env_free(ora_env *e);
int      ora_env_n(const ora_env *e);   /* array dims incl. ghosts */
int      ora_env_m(const ora_env *e);
/* BDIM.resume (BDIM.pde:239-251) from arrays already parsed; arrays are n*m, i-major */
void     ora_env_set_state(ora_env *e, const float *ux, const float *uy, const float *p);
void     ora_env_get_state(const ora_env *e, float *ux, float *uy, float *p);
void     ora_env_set_xi(ora_env *e, float xi1, float xi2);                /* clientCFD.pde:51-54 */
void     ora_env_update2(ora_env *e);                                     /* AFCCylinder.pde:45-61 */
float    ora_env_t(const ora_env *e);
float    ora_vfield_CFL(const ora_vfield *u, float nu);                   /* VectorField.pde:225-235 */
float    ora_env_check_cfl(const ora_env *e);                             /* BDIM.pde:217-219 */
void     ora_env_update_adaptive(ora_env *e);                             /* AFCCylinder.pde:63-84 (one NT pass) */
float    ora_env_dt(const ora_env *e);
void     ora_env_force(const ora_env *e, float *fx, float *fy);
void     ora_env_probes(const ora_env *e, int numTheta, float *out);      /* SaveScalar.pde:61-72 */
int      ora_env_last_mg_iters(const ora_env *e, int which /*0 predictor, 1 corrector*/);
/* static coefficient views (pointers into the env; n*m floats each) */
const float *ora_env_coeff(const ora_env *e, const char *name);
/* One RL step as clientCFD.draw() drives it (clientCFD.pde:35-55): `substeps` solver steps with the
   force accumulation quirk Q1 (Cd, Cl and callLearn persist; not zeroed).  The observation
   (Cl, Cd) is written to obs[0], obs[1].  This helper assumes t > initTime already. */
typedef struct { int callLearn; float Cd, Cl; } ora_driver;
ora_driver ora_driver_new(void);
/* Advance one solver step and apply the draw() accumulation; returns 1 when an observation was
   produced on this step (callAction would be invoked), else 0. */
int      ora_driver_step(ora_driver *d, ora_env *e, float initTime, float *Cl, float *Cd);

/* ---------------- checkpoint IO ---------------- */
/* Parse a Lilypad text checkpoint (BDIM.write format, BDIM.pde:226-237). Returns 0 on success. */
int ora_read_bdim_text(const char *path, int n, int m, float *t, float *dt,
                       float *ux, float *uy, float *p);
/* Raw little-endian binary form used for the committed fixture (tests/golden/init_state.bdimb):
   "RLFCBDIM", int32 n, int32 m, float t, float dt, ux[n*m], uy[n*m], p[n*m]. */
int ora_write_bdimb(const char *path, int n, int m, float t, float dt,
                    const float *ux, const float *uy, const float *p);
int ora_read_bdimb(const char *path, int *n, int *m, float *t, float *dt,
                   float **ux, float **uy, float **p);

#ifdef __cplusplus
}
#endif
#endif
