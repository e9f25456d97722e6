/*
 * lilypad_oracle.c -- literal single-threaded C99 restatement of the Lilypad AFCCylinder
 * environment step of LiuYangMage/RLFluidControl (clientLilypad/*.pde).
 *
 * TEST INFRASTRUCTURE ONLY (see lilypad_oracle.h).  PARITY UNPINNED (no reference goldens,
 * no JVM in the image) -- pinned by docstring known-answers + fixture invariants only.
 *
 * Every function cites the reference file:line it follows.  Java semantics kept:
 *   - all `float`, one rounding per operation, no FMA (compile with -ffp-contract=off);
 *   - Processing turns unsuffixed literals into float (0.5 -> 0.5f, 1e-5 -> 1e-5f);
 *   - PApplet.sin/cos/sqrt/mag = java.lang.Math in double, narrowed to float;
 *   - PApplet.min/max(float,float) are the ternaries (a<b)?a:b / (a>b)?a:b;
 *   - int division truncates toward zero; (int)x truncates.
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared (see oracle/Makefile).
 */
#include "lilypad_oracle.h"

#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define PI_F 3.1415927f      /* processing.core.PConstants.PI = (float)Math.PI */
#define TWO_PI_F 6.2831855f  /* PConstants.TWO_PI */

static inline float pmin(float a, float b) { return (a < b) ? a : b; }   /* PApplet.min */
static inline float pmax(float a, float b) { return (a > b) ? a : b; }   /* PApplet.max */
static inline float psin(float x) { return (float)sin((double)x); }      /* PApplet.sin */
static inline float pcos(float x) { return (float)cos((double)x); }      /* PApplet.cos */
static inline float pmag(float a, float b) { return (float)sqrt((double)(a * a + b * b)); } /* PApplet.mag */
static inline float pabs(float a) { return (a < 0) ? -a : a; }           /* PApplet.abs */

#define AT(f, i, j) ((f)->a[(size_t)(i) * (f)->m + (j)])

/* ============================ Field ============================ */

/* Field.pde:30-37 */
ora_field ora_field_new(int n, int m, int btype, float bval) {
  ora_field f;
  f.n = n; f.m = m; f.btype = btype; f.bval = bval; f.gradientExit = 0;
  f.a = (float *)malloc(sizeof(float) * (size_t)n * m);
  for (size_t k = 0; k < (size_t)n * m; k++) f.a[k] = bval;
  return f;
}

/* Field.pde:51-58 -- copies btype and bval but NOT gradientExit */
ora_field ora_field_copy(const ora_field *b) {
  ora_field f;
  f.n = b->n; f.m = b->m; f.btype = b->btype; f.bval = b->bval; f.gradientExit = 0;
  f.a = (float *)malloc(sizeof(float) * (size_t)b->n * b->m);
  memcpy(f.a, b->a, sizeof(float) * (size_t)b->n * b->m);
  return f;
}

void ora_field_free(ora_field *f) { free(f->a); f->a = NULL; }

/* Field.eq(Field) Field.pde:326-331 -- values only */
static void field_eq(ora_field *dst, const ora_field *src) {
  memcpy(dst->a, src->a, sizeof(float) * (size_t)dst->n * dst->m);
}

/* Field.pde:209-234, statement order kept */
void ora_field_setBC(ora_field *f) {
  const int n = f->n, m = f->m;
  float s = 0;
  for (int j = 0; j < m; j++) {
    AT(f, 0, j) = AT(f, 1, j);
    AT(f, n - 1, j) = AT(f, n - 2, j);
    if (f->btype == 1) {
      if (f->gradientExit) {
        AT(f, 1, j) = f->bval;
        if (j > 0 && j < m - 1) s += AT(f, n - 1, j);
      } else {
        AT(f, 1, j) = f->bval;
        AT(f, n - 1, j) = f->bval;
      }
    }
  }
  for (int i = 0; i < n; i++) {
    AT(f, i, 0) = AT(f, i, 1);
    AT(f, i, m - 1) = AT(f, i, m - 2);
    if (f->btype == 2) {
      AT(f, i, 1) = f->bval;
      AT(f, i, m - 1) = f->bval;
    }
  }
  if (f->gradientExit) {
    s /= (float)(m - 2);
    for (int j = 1; j < m - 1; j++) AT(f, n - 1, j) += f->bval - s;
  }
}

/* Field.pde:175-190 */
float ora_field_linear(const ora_field *f, float x0, float y0) {
  const int n = f->n, m = f->m;
  float x = pmin(pmax(0.5f, x0), n - 1.5f);
  if (f->btype == 1 || f->btype == 3) x += 0.5f;
  int i = (int)x; if (i > n - 2) i = n - 2;
  float s = x - i;
  float y = pmin(pmax(0.5f, y0), m - 1.5f);
  if (f->btype == 2 || f->btype == 3) y += 0.5f;
  int j = (int)y; if (j > m - 2) j = m - 2;
  float t = y - j;
  if (s == 0 && t == 0) {
    return AT(f, i, j);
  } else {
    return s * (t * AT(f, i + 1, j + 1) + (1 - t) * AT(f, i + 1, j)) +
           (1 - s) * (t * AT(f, i, j + 1) + (1 - t) * AT(f, i, j));
  }
}

/* Field.pde:302-310 -- float product, double accumulator, interior only */
float ora_field_inner(const ora_field *a, const ora_field *b) {
  double s = 0;
  for (int i = 1; i < a->n - 1; i++)
    for (int j = 1; j < a->m - 1; j++) {
      float prod = AT(a, i, j) * AT(b, i, j);
      s += prod;
    }
  return (float)s;
}

/* Field.pde:311-318 -- serial float accumulator, i-major order */
float ora_field_sum(const ora_field *a) {
  float s = 0;
  for (int i = 1; i < a->n - 1; i++)
    for (int j = 1; j < a->m - 1; j++) s += AT(a, i, j);
  return s;
}

/* Field.pde:340-347 */
float ora_field_Linf(const ora_field *a) {
  float mx = 0;
  for (size_t k = 0; k < (size_t)a->n * a->m; k++) mx = pmax(mx, pabs(a->a[k]));
  return mx;
}

/* ============================ VectorField ============================ */

/* VectorField.pde:27-32 */
ora_vfield ora_vfield_new(int n, int m, float xval, float yval) {
  ora_vfield v;
  v.x = ora_field_new(n, m, 1, xval);
  v.y = ora_field_new(n, m, 2, yval);
  return v;
}
/* VectorField.pde:33-39 */
ora_vfield ora_vfield_copy(const ora_vfield *b) {
  ora_vfield v;
  v.x = ora_field_copy(&b->x);
  v.y = ora_field_copy(&b->y);
  return v;
}
void ora_vfield_free(ora_vfield *v) { ora_field_free(&v->x); ora_field_free(&v->y); }
void ora_vfield_setBC(ora_vfield *v) { ora_field_setBC(&v->x); ora_field_setBC(&v->y); }

/* VectorField.pde:221 */
static inline float med(float a, float b, float c) { return pmax(pmin(a, b), pmin(pmax(a, b), c)); }

/* VectorField.pde:202-219; CF=1./6., S=10. (VectorField.pde:25) */
static float bho(const ora_field *b, int n, int m, int i, int j, int d1, int d2, float uf) {
  const float CF = 1.f / 6.f, S = 10.f;
  float bf = 0.5f * (AT(b, i + d1, j + d2) + AT(b, i, j));
  if (d1 * uf < 0) { i += d1; d1 = -d1; }
  if (d2 * uf < 0) { j += d2; d2 = -d2; }
  if (i > n - 2 || i < 2 || j > m - 2 || j < 2) return bf;
  float bc = AT(b, i, j);
  float bd = AT(b, i + d1, j + d2);
  float bu = AT(b, i - d1, j - d2);
  bf -= CF * (bd - 2 * bc + bu);
  float b1 = bu + S * (bc - bu);
  return med(bf, bc, med(bc, bd, b1));
}

/* VectorField.pde:181-196 */
static float advection(const ora_vfield *v, const ora_field *b, int i, int j) {
  const ora_field *x = &v->x, *y = &v->y;
  const int n = x->n, m = x->m;
  float uo, ue, vs, vn;
  if (b->btype == 1) {
    uo = 0.5f * (AT(x, i - 1, j) + AT(x, i, j));
    ue = 0.5f * (AT(x, i + 1, j) + AT(x, i, j));
    vs = 0.5f * (AT(y, i, j) + AT(y, i - 1, j));
    vn = 0.5f * (AT(y, i, j + 1) + AT(y, i - 1, j + 1));
  } else {
    uo = 0.5f * (AT(x, i, j - 1) + AT(x, i, j));
    ue = 0.5f * (AT(x, i + 1, j - 1) + AT(x, i + 1, j));
    vs = 0.5f * (AT(y, i, j - 1) + AT(y, i, j));
    vn = 0.5f * (AT(y, i, j) + AT(y, i, j + 1));
  }
  return ((uo * bho(b, n, m, i, j, -1, 0, uo) - ue * bho(b, n, m, i, j, 1, 0, ue)) +
          (vs * bho(b, n, m, i, j, 0, -1, vs) - vn * bho(b, n, m, i, j, 0, 1, vn)));
}

/* VectorField.pde:198-200 */
static inline float diffusion(const ora_field *b, int i, int j) {
  return AT(b, i + 1, j) + AT(b, i, j + 1) - 4 * AT(b, i, j) + AT(b, i - 1, j) + AT(b, i, j - 1);
}

/* VectorField.pde:170-179.  v starts as a copy of this (ghosts keep this's values); the stencils
   read the un-updated `this`; result assigned back with eq(). */
void ora_vfield_AdvDif(ora_vfield *F, const ora_vfield *u0, float dt, float nu) {
  const int n = F->x.n, m = F->x.m;
  ora_vfield v = ora_vfield_copy(F);
  for (int j = 1; j < m - 1; j++) {
    for (int i = 1; i < n - 1; i++) {
      AT(&v.x, i, j) = (advection(F, &F->x, i, j) + nu * diffusion(&F->x, i, j)) * dt + AT(&u0->x, i, j);
      AT(&v.y, i, j) = (advection(F, &F->y, i, j) + nu * diffusion(&F->y, i, j)) * dt + AT(&u0->y, i, j);
    }
  }
  field_eq(&F->x, &v.x);
  field_eq(&F->y, &v.y);
  ora_vfield_free(&v);
}

/* VectorField.pde:56-65 */
ora_field ora_vfield_divergence(const ora_vfield *u) {
  const int n = u->x.n, m = u->x.m;
  ora_field d = ora_field_new(n, m, 0, 0);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++)
      AT(&d, i, j) = AT(&u->x, i + 1, j) - AT(&u->x, i, j) + AT(&u->y, i, j + 1) - AT(&u->y, i, j);
  return d;
}

/* VectorField.pde:46-54: g = 0.5*(wnx*(d/dx) + wny*(d/dy)), interior only, ghosts 0 */
static ora_vfield vfield_normalGrad(const ora_vfield *du, const ora_vfield *wnx, const ora_vfield *wny) {
  const int n = du->x.n, m = du->x.m;
  ora_vfield g = ora_vfield_new(n, m, 0, 0);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&g.x, i, j) = 0.5f * (AT(&wnx->x, i, j) * (AT(&du->x, i + 1, j) - AT(&du->x, i - 1, j)) +
                               AT(&wny->x, i, j) * (AT(&du->x, i, j + 1) - AT(&du->x, i, j - 1)));
      AT(&g.y, i, j) = 0.5f * (AT(&wnx->y, i, j) * (AT(&du->y, i + 1, j) - AT(&du->y, i - 1, j)) +
                               AT(&wny->y, i, j) * (AT(&du->y, i, j + 1) - AT(&du->y, i, j - 1)));
    }
  return g;
}

/* Field.pde:71-81 */
ora_vfield ora_field_gradient(const ora_field *p) {
  const int n = p->n, m = p->m;
  ora_vfield g = ora_vfield_new(n, m, 0, 0);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&g.x, i, j) = AT(p, i, j) - AT(p, i - 1, j);
      AT(&g.y, i, j) = AT(p, i, j) - AT(p, i, j - 1);
    }
  ora_vfield_setBC(&g);
  return g;
}

/* ============================ PoissonMatrix ============================ */

/* PoissonMatrix.pde:38-51 */
ora_poisson ora_poisson_new(const ora_vfield *lower) {
  ora_poisson A;
  const int n = lower->x.n, m = lower->x.m;
  A.n = n; A.m = m;
  A.lower = ora_vfield_copy(lower);
  A.diagonal = ora_field_new(n, m, 0, 0);
  A.inv = ora_field_new(n, m, 0, 1);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      float sumd = AT(&lower->x, i, j) + AT(&lower->x, i + 1, j) + AT(&lower->y, i, j) + AT(&lower->y, i, j + 1);
      AT(&A.diagonal, i, j) = -sumd;
      if (sumd > 1e-5f) AT(&A.inv, i, j) = -1.f / sumd;
    }
  return A;
}

void ora_poisson_free(ora_poisson *A) {
  ora_vfield_free(&A->lower);
  ora_field_free(&A->diagonal);
  ora_field_free(&A->inv);
}

/* PoissonMatrix.pde:53-64 */
ora_field ora_poisson_times(const ora_poisson *A, const ora_field *x) {
  const int n = A->n, m = A->m;
  ora_field ab = ora_field_new(n, m, 0, 0);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++)
      AT(&ab, i, j) = AT(x, i, j) * AT(&A->diagonal, i, j) + AT(x, i - 1, j) * AT(&A->lower.x, i, j) +
                      AT(x, i + 1, j) * AT(&A->lower.x, i + 1, j) + AT(x, i, j - 1) * AT(&A->lower.y, i, j) +
                      AT(x, i, j + 1) * AT(&A->lower.y, i, j + 1);
  return ab;
}

/* ============================ MG ============================ */

typedef struct {
  const ora_poisson *A;
  ora_field r, x, d;
  int has_d;
  int iter, level;
  float tol;
  const ora_poisson *hier; /* cached hierarchy or NULL (literal: rebuild as MG.pde:70) */
  int nhier;
} mg_t;

/* MG.pde:108-122 */
ora_poisson ora_mg_restrict_matrix(const ora_poisson *A) {
  int n = (A->lower.x.n - 2) / 2 + 2;
  int m = (A->lower.x.m - 2) / 2 + 2;
  ora_vfield lower = ora_vfield_new(n, m, 0, 0);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      int ii = (i - 1) * 2 + 1;
      int jj = (j - 1) * 2 + 1;
      AT(&lower.x, i, j) = (AT(&A->lower.x, ii, jj) + AT(&A->lower.x, ii, jj + 1)) * 0.5f;
      AT(&lower.y, i, j) = (AT(&A->lower.y, ii, jj) + AT(&A->lower.y, ii + 1, jj)) * 0.5f;
    }
  ora_vfield_setBC(&lower);
  ora_poisson c = ora_poisson_new(&lower);
  ora_vfield_free(&lower);
  return c;
}

/* MG.pde:124-137 */
ora_field ora_mg_restrict_field(const ora_field *a) {
  int n = (a->n - 2) / 2 + 2;
  int m = (a->m - 2) / 2 + 2;
  ora_field b = ora_field_new(n, m, 0, 0);
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      int ii = (i - 1) * 2 + 1;
      int jj = (j - 1) * 2 + 1;
      AT(&b, i, j) = AT(a, ii, jj) + AT(a, ii, jj + 1) + AT(a, ii + 1, jj) + AT(a, ii + 1, jj + 1);
    }
  ora_field_setBC(&b);
  return b;
}

/* MG.pde:139-152 (Java int division truncates toward zero: (0-1)/2 == 0) */
ora_field ora_mg_prolongate(const ora_field *a) {
  int n = (a->n - 2) * 2 + 2;
  int m = (a->m - 2) * 2 + 2;
  ora_field b = ora_field_new(n, m, 0, 0);
  for (int i = 0; i < n; i++)
    for (int j = 0; j < m; j++) {
      int ii = (i - 1) / 2 + 1;
      int jj = (j - 1) / 2 + 1;
      AT(&b, i, j) = AT(a, ii, jj);
    }
  ora_field_setBC(&b);
  return b;
}

/* MG.pde:94-97: x.plusEq(d) and r.minusEq(A.times(d)) over ALL cells */
static void mg_increment(mg_t *g) {
  const size_t N = (size_t)g->x.n * g->x.m;
  for (size_t k = 0; k < N; k++) g->x.a[k] += g->d.a[k];
  ora_field Ad = ora_poisson_times(g->A, &g->d);
  for (size_t k = 0; k < N; k++) g->r.a[k] -= Ad.a[k];
  ora_field_free(&Ad);
}

/* MG.pde:79-92: in-place lexicographic Gauss-Seidel, i outer, j inner */
static void mg_smooth(mg_t *g, int itmx) {
  const ora_poisson *A = g->A;
  const int n = g->r.n, m = g->r.m;
  if (g->has_d) ora_field_free(&g->d);
  g->d = ora_field_copy(&g->r);           /* r.times(A.inv): Field c=new Field(this); c*=inv, all cells */
  g->has_d = 1;
  for (size_t k = 0; k < (size_t)n * m; k++) g->d.a[k] *= A->inv.a[k];
  for (int it = 0; it < itmx; it++)
    for (int i = 1; i < n - 1; i++)
      for (int j = 1; j < m - 1; j++)
        AT(&g->d, i, j) = -(AT(&g->d, i - 1, j) * AT(&A->lower.x, i, j) + AT(&g->d, i + 1, j) * AT(&A->lower.x, i + 1, j) +
                            AT(&g->d, i, j - 1) * AT(&A->lower.y, i, j) + AT(&g->d, i, j + 1) * AT(&A->lower.y, i, j + 1) -
                            AT(&g->r, i, j)) * AT(&A->inv, i, j);
  ora_field_setBC(&g->d);
  mg_increment(g);
}

/* MG.pde:99-106 */
static int mg_divisible(const mg_t *g) {
  int flag = (g->x.n - 2) % 2 == 0 && (g->x.m - 2) % 2 == 0 && g->x.n > 4 && g->x.m > 4;
  if (!flag && g->x.n > 9 && g->x.m > 9) {
    fprintf(stderr, "MultiGrid requires the size in each direction be a large factor of two (2^p) times a small number (N=1..9).\n");
    exit(1);
  }
  return flag;
}

/* MG.pde:68-77 */
static void mg_vcycle(mg_t *g) {
  const int its = 4;
  mg_smooth(g, 0);
  mg_t c;
  ora_poisson built;
  int own = 0;
  if (g->hier && g->level + 1 < g->nhier) {
    c.A = &g->hier[g->level + 1];
  } else {
    built = ora_mg_restrict_matrix(g->A);
    c.A = &built;
    own = 1;
  }
  c.r = ora_mg_restrict_field(&g->r);
  c.x = ora_field_new(c.r.n, c.r.m, 0, 0);
  c.has_d = 0;
  c.level = g->level + 1;
  c.iter = g->iter;
  c.hier = g->hier; c.nhier = g->nhier;
  if (mg_divisible(&c)) mg_vcycle(&c);
  mg_smooth(&c, its);
  if (g->has_d) ora_field_free(&g->d);
  g->d = ora_mg_prolongate(&c.x);
  g->has_d = 1;
  mg_increment(g);
  ora_field_free(&c.r); ora_field_free(&c.x);
  if (c.has_d) ora_field_free(&c.d);
  if (own) ora_poisson_free(&built);
}

/* MGsolver MG.pde:30-38 + MG ctor :46-52 + update :61-66 */
int ora_mg_solve(float itmx, const ora_poisson *A, ora_field *x, const ora_field *b,
                 const ora_poisson *hier, int nhier, float *rr_out, float *tol_out) {
  mg_t g;
  g.A = A; g.x = *x; g.has_d = 0; g.iter = 0; g.level = 0; g.hier = hier; g.nhier = nhier;
  ora_field tolf = ora_field_new(x->n, x->m, 0, 1e-4f);
  g.tol = ora_field_inner(&tolf, &tolf);
  ora_field_free(&tolf);
  /* r = A.residual(b,x) = b.minus(A.times(x)) over all cells (PoissonMatrix.pde:66-68) */
  g.r = ora_field_copy(b);
  {
    ora_field Ax = ora_poisson_times(A, x);
    for (size_t k = 0; k < (size_t)x->n * x->m; k++) g.r.a[k] -= Ax.a[k];
    ora_field_free(&Ax);
  }
  float rr = 0;
  while (g.iter < itmx) {
    g.iter++;
    mg_vcycle(&g);
    mg_smooth(&g, 4);
    rr = ora_field_inner(&g.r, &g.r);
    if (rr < g.tol) break;
  }
  if (rr_out) *rr_out = rr;
  if (tol_out) *tol_out = g.tol;
  ora_field_free(&g.r);
  if (g.has_d) ora_field_free(&g.d);
  *x = g.x;   /* same storage: updated in place */
  return g.iter;
}

/* VectorField.project VectorField.pde:130-143 */
int ora_vfield_project(ora_vfield *u, const ora_vfield *coeffs, ora_field *p, int literal,
                       const void *cached_hierarchy) {
  const int n = u->x.n, m = u->x.m;
  const size_t N = (size_t)n * m;
  ora_field s = ora_vfield_divergence(u);
  int iters;
  if (literal || !cached_hierarchy) {
    ora_poisson A = ora_poisson_new(coeffs);
    iters = ora_mg_solve(20, &A, p, &s, NULL, 0, NULL, NULL);
    ora_poisson_free(&A);
  } else {
    const ora_poisson *h = (const ora_poisson *)cached_hierarchy;
    int nh = 0;
    while (h[nh].n != 0) nh++;
    iters = ora_mg_solve(20, &h[0], p, &s, h, nh, NULL, NULL);
  }
  ora_field_free(&s);
  /* p.plusEq(-1*p.sum()/(float)((n-2)*(m-2))) over all cells */
  float shift = -1 * ora_field_sum(p) / (float)((n - 2) * (m - 2));
  for (size_t k = 0; k < N; k++) p->a[k] += shift;
  ora_vfield dp = ora_field_gradient(p);
  /* x.plusEq(coeffs.x.times(dp.x.times(-1))) over all cells */
  for (size_t k = 0; k < N; k++) u->x.a[k] += coeffs->x.a[k] * (dp.x.a[k] * -1);
  for (size_t k = 0; k < N; k++) u->y.a[k] += coeffs->y.a[k] * (dp.y.a[k] * -1);
  ora_vfield_free(&dp);
  ora_vfield_setBC(u);
  return iters;
}

/* ============================ OrthoNormal / Body ============================ */

/* OrthoNormal.pde:8-18; PVector.mag() = (float)Math.sqrt(x*x+y*y+z*z) with z=0 */
static ora_ortho ortho_new(float x1x, float x1y, float x2x, float x2y) {
  ora_ortho o;
  float sx = x1x - x2x, sy = x1y - x2y, sz = 0.f;
  o.l = (float)sqrt((double)(sx * sx + sy * sy + sz * sz));
  o.tx = (x2x - x1x) / o.l;
  o.ty = (x2y - x1y) / o.l;
  o.t1 = x1x * o.tx + x1y * o.ty;
  o.t2 = x2x * o.tx + x2y * o.ty;
  o.nx = -o.ty; o.ny = o.tx;
  o.off = x1x * o.nx + x1y * o.ny;
  o.cenx = (x1x + x2x) / 2.f;
  o.ceny = (x1y + x2y) / 2.f;
  return o;
}

/* OrthoNormal.pde:20-28 */
static float ortho_distance(const ora_ortho *o, float x, float y, int projected) {
  float d = x * o->nx + y * o->ny - o->off;
  if (projected) return d;
  float d1 = x * o->tx + y * o->ty - o->t1;
  float d2 = x * o->tx + y * o->ty - o->t2;
  return pabs(d) + pmax(0, -d1) + pmax(0, d2);
}

/* Body.pde:57-60 */
ora_body *ora_body_new(float x, float y) {
  ora_body *b = (ora_body *)calloc(1, sizeof(ora_body));
  b->xcx = x; b->xcy = y;
  b->mass = 1; b->I0 = 1;
  return b;
}

/* Body.pde:62-64 */
void ora_body_add(ora_body *b, float x, float y) {
  b->cx = (float *)realloc(b->cx, sizeof(float) * (b->n + 1));
  b->cy = (float *)realloc(b->cy, sizeof(float) * (b->n + 1));
  b->cx[b->n] = x; b->cy[b->n] = y;
  b->n++;
}

/* Body.pde:66-121 (end(true): getOrth, getArea, bounding box, convexity) */
void ora_body_end(ora_body *b) {
  const int n = b->n;
  b->north = n;
  b->orth = (ora_ortho *)malloc(sizeof(ora_ortho) * n);
  for (int i = 0; i < n; i++) {                       /* getOrth :102-108 */
    int k = (i + 1) % n;
    b->orth[i] = ortho_new(b->cx[i], b->cy[i], b->cx[k], b->cy[k]);
  }
  {                                                   /* getArea :109-121 */
    float s = 0, t = 0;
    for (int i = 0; i < n; i++) {
      int k = (i + 1) % n;
      float x1 = b->cx[i] - b->xcx, x2 = b->cx[k] - b->xcx, y1 = b->cy[i] - b->xcy, y2 = b->cy[k] - b->xcy;
      float da = x1 * y2 - x2 * y1;
      s -= da;
      t -= (x1 * x1 + x1 * x2 + x2 * x2 + y1 * y1 + y1 * y2 + y2 * y2) * da;
    }
    b->area = 0.5f * s;
    b->I0 = t / 12.f;
    b->mass = b->area;
  }
  if (n > 4) {                                        /* bounding box :73-87 */
    float mnx = b->xcx, mny = b->xcy, mxx = b->xcx, mxy = b->xcy;
    for (int i = 0; i < n; i++) {
      mnx = pmin(mnx, b->cx[i]); mny = pmin(mny, b->cy[i]);
      mxx = pmax(mxx, b->cx[i]); mxy = pmax(mxy, b->cy[i]);
    }
    b->box = ora_body_new(b->xcx, b->xcy);
    ora_body_add(b->box, mnx, mny);
    ora_body_add(b->box, mnx, mxy);
    ora_body_add(b->box, mxx, mxy);
    ora_body_add(b->box, mxx, mny);
    ora_body_end(b->box);
  }
  b->convex = 1;                                      /* convexity :90-96 */
  for (int i = 0; i < b->north && b->convex; i++)
    for (int j = 0; j < b->north; j++)
      if (ortho_distance(&b->orth[i], b->orth[j].cenx, b->orth[j].ceny, 1) > 0.001f) { b->convex = 0; break; }
}

/* EllipseBody ctor Body.pde:386-398 with _a = 1.0 (CircleBody ctor :404-406) */
ora_body *ora_circle_new(float x, float y, float d) {
  ora_body *b = ora_body_new(x, y);
  const int m = 40;
  b->h = d;
  float a = 1.f / 1.0f;
  float dx = 0.5f * b->h * a, dy = 0.5f * b->h;
  for (int i = 0; i < m; i++) {
    float theta = -TWO_PI_F * i / ((float)m);
    ora_body_add(b, b->xcx + dx * pcos(theta), b->xcy + dy * psin(theta));
  }
  ora_body_end(b);
  b->is_circle = 1;
  return b;
}

void ora_body_free(ora_body *b) {
  if (!b) return;
  if (b->box) ora_body_free(b->box);
  free(b->cx); free(b->cy); free(b->orth); free(b);
}

/* Body.wn Body.pde:199-213 */
static int body_wn(const ora_body *b, float x, float y) {
  int wn = 0;
  for (int i = 0; i < b->n - 1; i++) {
    float yi = b->cy[i], yi1 = b->cy[i + 1];
    const ora_ortho *o = &b->orth[i];
    if (yi <= y) { if (yi1 > y && ortho_distance(o, x, y, 1) > 0) wn++; }
    else         { if (yi1 <= y && ortho_distance(o, x, y, 1) < 0) wn--; }
  }
  return wn;
}

/* Body.distance Body.pde:174-192; CircleBody.distance :408-410 */
float ora_body_distance(const ora_body *b, float x, float y) {
  if (b->is_circle) return pmag(x - b->xcx, y - b->xcy) - 0.5f * b->h;
  float dis;
  if (b->n > 4) {
    dis = ora_body_distance(b->box, x, y);
    if (dis > 3) return dis;
  }
  if (b->convex) {
    dis = -1e10f;
    for (int i = 0; i < b->north; i++) dis = pmax(dis, ortho_distance(&b->orth[i], x, y, 1));
    return dis;
  } else {
    dis = 1e10f;
    for (int i = 0; i < b->north; i++) dis = pmin(dis, ortho_distance(&b->orth[i], x, y, 0));
    return (body_wn(b, x, y) == 0) ? dis : -dis;
  }
}

/* Body.WallNormal Body.pde:215-232 (CircleBody does not override it: faceted normal) */
void ora_body_wallnormal(const ora_body *b, float x, float y, float *nx, float *ny) {
  *nx = 0; *ny = 0;
  float dis = -1e10f, dis2;
  if (b->n > 4) {
    if (ora_body_distance(b->box, x, y) > 3) return;   /* box is a plain Body: Body.distance */
  }
  for (int i = 0; i < b->north; i++) {
    dis2 = ortho_distance(&b->orth[i], x, y, 1);
    if (dis2 > dis) { dis = dis2; *nx = b->orth[i].nx; *ny = b->orth[i].ny; }
  }
}

/* Body.velocity Body.pde:234-240 */
float ora_body_velocity(const ora_body *b, int d, float dt, float x, float y) {
  float rx = x - b->xcx, ry = y - b->xcy;
  if (d == 1) return (b->dxcx - ry * b->dphi) / dt;
  else        return (b->dxcy + rx * b->dphi) / dt;
}

/* Body.pressForce Body.pde:296-303 */
void ora_body_pressForce(const ora_body *b, const ora_field *p, float *fx, float *fy) {
  float pvx = 0, pvy = 0;
  for (int i = 0; i < b->north; i++) {
    const ora_ortho *o = &b->orth[i];
    float pdl = ora_field_linear(p, o->cenx, o->ceny) * o->l;
    pvx += pdl * o->nx;
    pvy += pdl * o->ny;
  }
  *fx = pvx; *fy = pvy;
}

/* BDIM.delta0 BDIM.pde:199-207 */
float ora_bdim_delta0(float d, float eps) {
  if (d <= -eps) return 0;
  else if (d >= eps) return 1;
  else return 0.5f * (1.f + d / eps + psin(PI_F * d / eps) / PI_F);
}

/* BDIM.delta1 BDIM.pde:209-215 */
float ora_bdim_delta1(float d, float eps) {
  if (pabs(d) >= eps) return 0;
  else return 0.25f * (eps - (d * d) / eps) -
              1 / TWO_PI_F * (d * psin(d * PI_F / eps) + eps / PI_F * (1 + pcos(d * PI_F / eps)));
}

/* BodyUnion.delta0 BodyUnion.pde:158-166 */
float ora_union_delta0(float d) {
  if (d <= -1) return 0;
  else if (d >= 1) return 1;
  else return 0.5f * (1.f + d + psin(PI_F * d) / PI_F);
}

/* ============================ BodyUnion of the three cylinders ============================ */

#define NB 3
typedef struct { ora_body *b[NB]; } ora_union;

/* BodyUnion.get_weights BodyUnion.pde:145-156 */
static void union_weights(const ora_union *U, float x, float y, float *w) {
  float s = 0;
  for (int i = 0; i < NB; i++) {
    float d = ora_body_distance(U->b[i], x, y);
    w[i] = ora_union_delta0(-d / 3.f);
    s += w[i];
  }
  for (int i = 0; i < NB && s > 0; i++) w[i] /= s;
}
/* BodyUnion.distance BodyUnion.pde:67-72 */
static float union_distance(const ora_union *U, float x, float y) {
  float d = 1e6f;
  for (int i = 0; i < NB; i++) d = pmin(d, ora_body_distance(U->b[i], x, y));
  return d;
}
/* BodyUnion.WallNormal BodyUnion.pde:74-82 */
static void union_wallnormal(const ora_union *U, float x, float y, float *mx, float *my) {
  float w[NB];
  union_weights(U, x, y, w);
  *mx = 0; *my = 0;
  for (int i = 0; i < NB; i++) {
    float nx, ny;
    ora_body_wallnormal(U->b[i], x, y, &nx, &ny);
    *mx += nx * w[i];
    *my += ny * w[i];
  }
}
/* BodyUnion.velocity BodyUnion.pde:84-92 */
static float union_velocity(const ora_union *U, int d, float dt, float x, float y) {
  float w[NB];
  union_weights(U, x, y, w);
  float v = 0;
  for (int i = 0; i < NB; i++) {
    float u = ora_body_velocity(U->b[i], d, dt, x, y);
    v += u * w[i];
  }
  return v;
}
/* BodyUnion.unsteady BodyUnion.pde:116-122 / Body.unsteady Body.pde:242 */
static int union_unsteady(const ora_union *U) {
  int uns = 0;
  for (int i = 0; i < NB; i++) {
    const ora_body *b = U->b[i];
    float mag = (float)sqrt((double)(b->dxcx * b->dxcx + b->dxcy * b->dxcy + 0.f * 0.f));
    uns = uns | ((mag != 0) | (b->dphi != 0));
  }
  return uns;
}

/* ============================ BDIM + AFCCylinder ============================ */

struct ora_env {
  ora_config cfg;
  /* AFCCylinder fields AFCCylinder.pde:2-9 */
  int n_cells, m_cells;     /* AFCCylinder.n, m (no ghosts) */
  float dt, t, D, xi1, xi2, xi1_m, xi2_m, dphi1, dphi2;
  float forcex, forcey;
  ora_union body;
  /* BDIM fields BDIM.pde:33-39 */
  int n, m;                 /* with ghosts */
  float flow_t, flow_dt, nu, eps;
  ora_vfield u, del, del1, c, u0, ub, wnx, wny, distance, rhoi;
  ora_field p;
  ora_poisson *hier;        /* cached hierarchy, terminated by n==0 (only when !literal) */
  int mg_iters[2];
};

ora_config ora_default_config(void) {
  ora_config c;
  c.resolution = 24; c.xLengths = 16; c.yLengths = 8; c.Re = 500;   /* clientCFD.pde:14,94 */
  c.dR = .125f; c.gR = .2f; c.theta = PI_F / 3; c.tStep = .0075f;   /* clientCFD.pde:9,95-96 */
  c.literal = 1;
  return c;
}

/* BDIM.get_coeffs BDIM.pde:132-196 */
static void bdim_get_coeffs(ora_env *e) {
  const int n = e->n, m = e->m;
  const ora_union *U = &e->body;
  /* get_dist :165-172 */
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&e->distance.x, i, j) = union_distance(U, (float)(i - 0.5), j);
      AT(&e->distance.y, i, j) = union_distance(U, i, (float)(j - 0.5));
    }
  /* get_del :174-184 */
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&e->del.x, i, j) = ora_bdim_delta0(AT(&e->distance.x, i, j), e->eps);
      AT(&e->del.y, i, j) = ora_bdim_delta0(AT(&e->distance.y, i, j), e->eps);
    }
  ora_vfield_setBC(&e->del);
  /* get_del1 :186-196 */
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&e->del1.x, i, j) = ora_bdim_delta1(AT(&e->distance.x, i, j), e->eps);
      AT(&e->del1.y, i, j) = ora_bdim_delta1(AT(&e->distance.y, i, j), e->eps);
    }
  ora_vfield_setBC(&e->del1);
  /* get_ub :140-149 */
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&e->ub.x, i, j) = union_velocity(U, 1, e->flow_dt, (float)(i - 0.5), j);
      AT(&e->ub.y, i, j) = union_velocity(U, 2, e->flow_dt, i, (float)(j - 0.5));
    }
  /* get_wn :151-163 */
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      float wx, wy;
      union_wallnormal(U, (float)(i - 0.5), j, &wx, &wy);
      AT(&e->wnx.x, i, j) = wx; AT(&e->wny.x, i, j) = wy;
      union_wallnormal(U, i, (float)(j - 0.5), &wx, &wy);
      AT(&e->wnx.y, i, j) = wx; AT(&e->wny.y, i, j) = wy;
    }
}

/* only the action-dependent part of get_coeffs (get_ub), used when !literal */
static void bdim_get_ub_only(ora_env *e) {
  const int n = e->n, m = e->m;
  for (int i = 1; i < n - 1; i++)
    for (int j = 1; j < m - 1; j++) {
      AT(&e->ub.x, i, j) = union_velocity(&e->body, 1, e->flow_dt, (float)(i - 0.5), j);
      AT(&e->ub.y, i, j) = union_velocity(&e->body, 2, e->flow_dt, i, (float)(j - 0.5));
    }
}

static void build_hierarchy(ora_env *e) {
  /* c = del*dt is constant for the env's life (SURVEY 9.2); cache PoissonMatrix(c) and its restrictions */
  ora_poisson tmp[32];
  int nl = 0;
  tmp[nl++] = ora_poisson_new(&e->c);
  for (;;) {
    const ora_poisson *A = &tmp[nl - 1];
    /* a level is restricted further when it is the finest, or when it is divisible (MG.pde:70-72,99-106) */
    int divisible = (A->n - 2) % 2 == 0 && (A->m - 2) % 2 == 0 && A->n > 4 && A->m > 4;
    if (nl > 1 && !divisible) break;
    tmp[nl] = ora_mg_restrict_matrix(A);
    nl++;
  }
  e->hier = (ora_poisson *)calloc(nl + 1, sizeof(ora_poisson));
  memcpy(e->hier, tmp, sizeof(ora_poisson) * nl);
  e->hier[nl].n = 0;
}

/* Grids the reference cannot run, decided from the level sizes alone (n, m incl. ghosts):
   - an odd level 0: MG.prolongate (MG.pde:139-152) builds an even-sized correction from the coarse level and
     MG.increment (MG.pde:94-97) adds it over the whole fine field, past the correction's end;
   - a coarse level that is not divisible while both sides are > 9: MG.divisible (MG.pde:101-104) calls exit(). */
static int grid_runnable(int n, int m) {
  if ((n - 2) % 2 != 0 || (m - 2) % 2 != 0) return 0;
  for (;;) {
    n = (n - 2) / 2 + 2;                          /* MG.restrict MG.pde:108-122 */
    m = (m - 2) / 2 + 2;
    int divisible = (n - 2) % 2 == 0 && (m - 2) % 2 == 0 && n > 4 && m > 4;
    if (divisible) continue;
    return !(n > 9 && m > 9);
  }
}

/* AFCCylinder ctor AFCCylinder.pde:11-42 + BDIM ctor BDIM.pde:41-71 (without resume) */
ora_env *ora_env_new(const ora_config *cfg) {
  if (!grid_runnable(cfg->xLengths * cfg->resolution + 2, cfg->yLengths * cfg->resolution + 2)) return NULL;
  ora_env *e = (ora_env *)calloc(1, sizeof(ora_env));
  e->cfg = *cfg;
  const int resolution = cfg->resolution;
  e->n_cells = cfg->xLengths * resolution;
  e->m_cells = cfg->yLengths * resolution;
  e->xi1 = 0; e->xi2 = 0;
  e->dt = cfg->tStep * resolution;
  e->xi1_m = 5 * e->xi1; e->xi2_m = 5 * e->xi2;
  float theta_m = cfg->theta;
  e->D = resolution;
  float D = e->D, dR = cfg->dR, gR = cfg->gR;
  float r = (D / 2 + gR * D + dR * D / 2);
  int nn = e->n_cells, mm = e->m_cells;
  e->body.b[0] = ora_circle_new(nn / 4, mm / 2, D);
  e->body.b[1] = ora_circle_new(nn / 4 + r * pcos(theta_m), mm / 2 - r * psin(theta_m), dR * D);
  e->body.b[2] = ora_circle_new(nn / 4 + r * pcos(theta_m), mm / 2 + r * psin(theta_m), dR * D);
  /* BDIM(n,m,dt,body,(float)D/Re,QUICK) */
  const int n = nn + 2, m = mm + 2;
  e->n = n; e->m = m;
  e->flow_t = 0; e->flow_dt = e->dt; e->nu = (float)D / cfg->Re; e->eps = 2.0f;
  e->u = ora_vfield_new(n, m, 1, 0);
  if (e->u.x.bval != 0) e->u.x.gradientExit = 1;
  e->u0 = ora_vfield_new(n, m, 0, 0);
  e->p = ora_field_new(n, m, 0, 0);
  e->ub = ora_vfield_new(n, m, 0, 0);
  e->distance = ora_vfield_new(n, m, 10, 10);
  e->del = ora_vfield_new(n, m, 1, 1);
  e->del1 = ora_vfield_new(n, m, 0, 0);
  e->rhoi = ora_vfield_copy(&e->del);
  e->c = ora_vfield_copy(&e->del);
  e->wnx = ora_vfield_new(n, m, 0, 0);
  e->wny = ora_vfield_new(n, m, 0, 0);
  bdim_get_coeffs(e);
  if (!cfg->literal) {
    /* c.eq(del.times(rhoi.times(dt))) BDIM.pde:81 evaluated once */
    for (size_t k = 0; k < (size_t)n * m; k++) {
      e->c.x.a[k] = e->del.x.a[k] * (e->rhoi.x.a[k] * e->flow_dt);
      e->c.y.a[k] = e->del.y.a[k] * (e->rhoi.y.a[k] * e->flow_dt);
    }
    build_hierarchy(e);
  }
  return e;
}

void ora_env_free(ora_env *e) {
  if (!e) return;
  for (int i = 0; i < NB; i++) ora_body_free(e->body.b[i]);
  ora_vfield *vs[] = {&e->u, &e->del, &e->del1, &e->c, &e->u0, &e->ub, &e->wnx, &e->wny, &e->distance, &e->rhoi};
  for (size_t k = 0; k < sizeof(vs) / sizeof(vs[0]); k++) ora_vfield_free(vs[k]);
  ora_field_free(&e->p);
  if (e->hier) {
    for (int l = 0; e->hier[l].n != 0; l++) ora_poisson_free(&e->hier[l]);
    free(e->hier);
  }
  free(e);
}

int ora_env_n(const ora_env *e) { return e->n; }
int ora_env_m(const ora_env *e) { return e->m; }
float ora_env_t(const ora_env *e) { return e->t; }
void ora_env_force(const ora_env *e, float *fx, float *fy) { *fx = e->forcex; *fy = e->forcey; }
int ora_env_last_mg_iters(const ora_env *e, int which) { return e->mg_iters[which & 1]; }

/* BDIM.resume BDIM.pde:239-251: overwrite u.x, u.y, p on all cells (ghosts included) */
void ora_env_set_state(ora_env *e, const float *ux, const float *uy, const float *p) {
  size_t N = (size_t)e->n * e->m;
  memcpy(e->u.x.a, ux, N * sizeof(float));
  memcpy(e->u.y.a, uy, N * sizeof(float));
  memcpy(e->p.a, p, N * sizeof(float));
}
void ora_env_get_state(const ora_env *e, float *ux, float *uy, float *p) {
  size_t N = (size_t)e->n * e->m;
  if (ux) memcpy(ux, e->u.x.a, N * sizeof(float));
  if (uy) memcpy(uy, e->u.y.a, N * sizeof(float));
  if (p) memcpy(p, e->p.a, N * sizeof(float));
}

/* clientCFD.pde:51-54 */
void ora_env_set_xi(ora_env *e, float xi1, float xi2) {
  e->xi1 = xi1; e->xi2 = xi2;
  e->xi1_m = 5 * e->xi1; e->xi2_m = 5 * e->xi2;
}

const float *ora_env_coeff(const ora_env *e, const char *name) {
  struct { const char *nm; const float *p; } tab[] = {
    {"del.x", e->del.x.a}, {"del.y", e->del.y.a}, {"del1.x", e->del1.x.a}, {"del1.y", e->del1.y.a},
    {"ub.x", e->ub.x.a}, {"ub.y", e->ub.y.a}, {"wnx.x", e->wnx.x.a}, {"wnx.y", e->wnx.y.a},
    {"wny.x", e->wny.x.a}, {"wny.y", e->wny.y.a}, {"dist.x", e->distance.x.a}, {"dist.y", e->distance.y.a},
    {"c.x", e->c.x.a}, {"c.y", e->c.y.a}, {"u0.x", e->u0.x.a}, {"u0.y", e->u0.y.a}};
  for (size_t k = 0; k < sizeof(tab) / sizeof(tab[0]); k++)
    if (!strcmp(tab[k].nm, name)) return tab[k].p;
  return NULL;
}

/* BDIM.updateUP BDIM.pde:109-124 (g = 0 so R.plusEq(g*dt) adds +0: omitted only for -0 inputs,
   which cannot change any later value; kept anyway for literalness) */
static int bdim_updateUP(ora_env *e, ora_vfield *R, int which) {
  const int n = e->n, m = e->m;
  const size_t N = (size_t)n * m;
  /* du = R.minus(ub) (all cells): the 2-argument overload evaluates it before the body runs (:124) */
  ora_vfield du = ora_vfield_copy(R);
  for (size_t k = 0; k < N; k++) { du.x.a[k] -= e->ub.x.a[k]; du.y.a[k] -= e->ub.y.a[k]; }
  for (size_t k = 0; k < N; k++) { R->x.a[k] += 0.f * e->flow_dt; R->y.a[k] += 0.f * e->flow_dt; }
  /* u.eq(del.times(R).minus(ub.times(del.plus(-1)))) all cells */
  for (size_t k = 0; k < N; k++) {
    e->u.x.a[k] = e->del.x.a[k] * R->x.a[k] - e->ub.x.a[k] * (e->del.x.a[k] + (-1));
    e->u.y.a[k] = e->del.y.a[k] * R->y.a[k] - e->ub.y.a[k] * (e->del.y.a[k] + (-1));
  }
  /* if(mu1) u.plusEq(del1.times(du.normalGrad(wnx,wny))) all cells (normalGrad ghosts are 0) */
  ora_vfield g = vfield_normalGrad(&du, &e->wnx, &e->wny);
  for (size_t k = 0; k < N; k++) {
    e->u.x.a[k] += e->del1.x.a[k] * g.x.a[k];
    e->u.y.a[k] += e->del1.y.a[k] * g.y.a[k];
  }
  ora_vfield_free(&g);
  ora_vfield_free(&du);
  ora_vfield_setBC(&e->u);
  int it = ora_vfield_project(&e->u, &e->c, &e->p, e->cfg.literal, e->hier);
  e->mg_iters[which] = it;
  return it;
}

/* BDIM.update(Body) BDIM.pde:126-129 + update() :79-87 */
static void bdim_update(ora_env *e) {
  const size_t N = (size_t)e->n * e->m;
  if (union_unsteady(&e->body)) {
    if (e->cfg.literal) bdim_get_coeffs(e); else bdim_get_ub_only(e);
  } else {
    for (size_t k = 0; k < N; k++) { e->ub.x.a[k] = 0.f; e->ub.y.a[k] = 0.f; }
  }
  if (e->cfg.literal)
    for (size_t k = 0; k < N; k++) {
      e->c.x.a[k] = e->del.x.a[k] * (e->rhoi.x.a[k] * e->flow_dt);
      e->c.y.a[k] = e->del.y.a[k] * (e->rhoi.y.a[k] * e->flow_dt);
    }
  field_eq(&e->u0.x, &e->u.x); field_eq(&e->u0.y, &e->u.y);
  ora_vfield F = ora_vfield_copy(&e->u);
  ora_vfield_AdvDif(&F, &e->u0, e->flow_dt, e->nu);
  bdim_updateUP(e, &F, 0);
  ora_vfield_free(&F);
}

/* BDIM.update2() BDIM.pde:89-107 (QUICK branch, adaptive=false) */
static void bdim_update2(ora_env *e) {
  const size_t N = (size_t)e->n * e->m;
  ora_vfield us = ora_vfield_copy(&e->u), F = ora_vfield_copy(&e->u);
  ora_vfield_AdvDif(&F, &e->u0, e->flow_dt, e->nu);
  bdim_updateUP(e, &F, 1);
  for (size_t k = 0; k < N; k++) { e->u.x.a[k] += us.x.a[k]; e->u.y.a[k] += us.y.a[k]; }
  for (size_t k = 0; k < N; k++) { e->u.x.a[k] *= 0.5f; e->u.y.a[k] *= 0.5f; }
  e->flow_t += e->flow_dt;
  ora_vfield_free(&us); ora_vfield_free(&F);
}

/* AFCCylinder.update2 AFCCylinder.pde:45-61 */
void ora_env_update2(ora_env *e) {
  const float dR = e->cfg.dR, D = e->D;
  e->flow_dt = e->dt;
  e->dphi1 = (2 * e->xi1_m * e->dt) / (dR * D);
  e->dphi2 = (2 * e->xi2_m * e->dt) / (dR * D);
  /* CircleBody.rotate Body.pde:412-415: stores dphi, accumulates phi; polygon is NOT rotated */
  e->body.b[1]->dphi = e->dphi1; e->body.b[1]->phi += e->dphi1;
  e->body.b[2]->dphi = e->dphi2; e->body.b[2]->phi += e->dphi2;
  bdim_update(e);
  bdim_update2(e);
  e->t += e->dt / e->cfg.resolution;
  float fx, fy;
  ora_body_pressForce(e->body.b[0], &e->p, &fx, &fy);
  e->forcex = fx * -1; e->forcey = fy * -1;     /* PVector.mult(-1) */
}

/* VectorField.CFL VectorField.pde:225-235 (Processing float literals: 1./(b+3.*nu) is float arithmetic) */
float ora_vfield_CFL(const ora_vfield *u, float nu) {
  float b = pabs(AT(&u->x, 0, 0)) + pabs(AT(&u->y, 0, 0));
  for (int i = 1; i < u->x.n - 1; i++)
    for (int j = 1; j < u->x.m - 1; j++) {
      float c = pabs(AT(&u->x, i, j)) + pabs(AT(&u->y, i, j));
      if (c > b) b = c;
    }
  return 1.f / (b + 3.f * nu);
}

/* BDIM.checkCFL BDIM.pde:217-219 */
float ora_env_check_cfl(const ora_env *e) { return pmin(ora_vfield_CFL(&e->u, e->nu), 1.f); }

/* One pass of the NT loop of AFCCylinder.update() AFCCylinder.pde:63-84 (QUICK: dt = flow.checkCFL() before every
   step).  dt changes from step to step, so c = del*rhoi*dt and the whole Poisson hierarchy change with it: the step runs
   in the literal mode (everything rebuilt where the reference rebuilds it) whatever the env was created with. */
void ora_env_update_adaptive(ora_env *e) {
  const int lit = e->cfg.literal;
  e->cfg.literal = 1;
  e->dt = ora_env_check_cfl(e);
  ora_env_update2(e);               /* from `flow.dt = dt` on the two methods are the same statements */
  e->cfg.literal = lit;
}

float ora_env_dt(const ora_env *e) { return e->dt; }

/* SaveScalar.addData03 SaveScalar.pde:61-72 with the ctor's centX=n/4, centY=m/2 (:36-40) */
void ora_env_probes(const ora_env *e, int numTheta, float *out) {
  float res = (float)e->cfg.resolution;
  float D = res;
  float nf = (float)e->cfg.xLengths * res, mf = (float)e->cfg.yLengths * res;
  float centX = nf / 4, centY = mf / 2;
  for (int i = 0; i < numTheta; i++) {
    float xPre = pcos((float)i / numTheta * PI_F * 2) * D / 2 + centX;
    float yPre = psin((float)i / numTheta * PI_F * 2) * D / 2 + centY;
    out[i] = ora_field_linear(&e->p, xPre, yPre);
  }
}

/* clientCFD.pde:11-13 */
ora_driver ora_driver_new(void) { ora_driver d; d.callLearn = 16; d.Cd = 0; d.Cl = 0; return d; }

/* clientCFD.draw clientCFD.pde:35-55 (the solver-step + accumulation part) */
int ora_driver_step(ora_driver *d, ora_env *e, float initTime, float *Cl, float *Cd) {
  ora_env_update2(e);
  int produced = 0;
  if (e->t > initTime) {
    d->callLearn--;
    d->Cd += e->forcex;
    d->Cl += e->forcey;
    if (d->callLearn <= 0) {
      d->callLearn = 16;
      d->Cd = d->Cd / d->callLearn * 2 / e->cfg.resolution;
      d->Cl = d->Cl / d->callLearn * 2 / e->cfg.resolution;
      *Cl = d->Cl; *Cd = d->Cd;
      produced = 1;
    }
  }
  return produced;
}

/* ============================ checkpoint IO ============================ */

/* BDIM.resume BDIM.pde:239-251: line0 t, line1 dt, then "ux, uy, p" per cell, i-major */
int ora_read_bdim_text(const char *path, int n, int m, float *t, float *dt, float *ux, float *uy, float *p) {
  FILE *f = fopen(path, "r");
  if (!f) return -1;
  char line[256];
  if (!fgets(line, sizeof line, f)) { fclose(f); return -2; }
  *t = strtof(line, NULL);
  if (!fgets(line, sizeof line, f)) { fclose(f); return -2; }
  *dt = strtof(line, NULL);
  for (size_t k = 0; k < (size_t)n * m; k++) {
    if (!fgets(line, sizeof line, f)) { fclose(f); return -3; }
    char *q = line, *end;
    ux[k] = strtof(q, &end); if (end == q) { fclose(f); return -4; }
    q = end; while (*q == ',' || *q == ' ') q++;
    uy[k] = strtof(q, &end); if (end == q) { fclose(f); return -4; }
    q = end; while (*q == ',' || *q == ' ') q++;
    p[k] = strtof(q, &end); if (end == q) { fclose(f); return -4; }
  }
  fclose(f);
  return 0;
}

int ora_write_bdimb(const char *path, int n, int m, float t, float dt, const float *ux, const float *uy, const float *p) {
  FILE *f = fopen(path, "wb");
  if (!f) return -1;
  int32_t hdr[2] = {n, m};
  float th[2] = {t, dt};
  size_t N = (size_t)n * m;
  int ok = fwrite("RLFCBDIM", 1, 8, f) == 8 && fwrite(hdr, 4, 2, f) == 2 && fwrite(th, 4, 2, f) == 2 &&
           fwrite(ux, 4, N, f) == N && fwrite(uy, 4, N, f) == N && fwrite(p, 4, N, f) == N;
  fclose(f);
  return ok ? 0 : -2;
}

int ora_read_bdimb(const char *path, int *n, int *m, float *t, float *dt, float **ux, float **uy, float **p) {
  FILE *f = fopen(path, "rb");
  if (!f) return -1;
  char magic[8]; int32_t hdr[2]; float th[2];
  if (fread(magic, 1, 8, f) != 8 || memcmp(magic, "RLFCBDIM", 8) || fread(hdr, 4, 2, f) != 2 || fread(th, 4, 2, f) != 2) {
    fclose(f); return -2;
  }
  size_t N = (size_t)hdr[0] * hdr[1];
  *n = hdr[0]; *m = hdr[1]; *t = th[0]; *dt = th[1];
  *ux = (float *)malloc(4 * N); *uy = (float *)malloc(4 * N); *p = (float *)malloc(4 * N);
  int ok = fread(*ux, 4, N, f) == N && fread(*uy, 4, N, f) == N && fread(*p, 4, N, f) == N;
  fclose(f);
  return ok ? 0 : -3;
}
