/*
 * oracle_cli.c -- command-line front end of the CPU oracle (TEST INFRASTRUCTURE / CPU BASELINE).
 *
 *   oracle_cli convert <in.bdim text> <out.bdimb> <n> <m>
 *       parse a Lilypad text checkpoint (BDIM.pde:226-251 format) into the raw binary fixture form
 *   oracle_cli run <state.bdimb|uniform> <env_steps> [literal=1] [trace.txt]
 *       BASELINE config 1: default AFCCylinder grid, state from the fixture, fixed action sequence
 *       a_k = (0.8 sin(2 pi k/25), -0.8 sin(2 pi k/25 + 1)), 16 solver steps per env step, with the
 *       clientCFD.draw() accumulation.  Prints one JSON line with env-steps/s (single thread).
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "lilypad_oracle.h"

static double now_s(void) {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

int main(int argc, char **argv) {
  if (argc >= 6 && !strcmp(argv[1], "convert")) {
    int n = atoi(argv[4]), m = atoi(argv[5]);
    size_t N = (size_t)n * m;
    float *ux = malloc(4 * N), *uy = malloc(4 * N), *p = malloc(4 * N), t, dt;
    int rc = ora_read_bdim_text(argv[2], n, m, &t, &dt, ux, uy, p);
    if (rc) { fprintf(stderr, "read failed: %d\n", rc); return 1; }
    rc = ora_write_bdimb(argv[3], n, m, t, dt, ux, uy, p);
    if (rc) { fprintf(stderr, "write failed: %d\n", rc); return 1; }
    printf("converted %s: n=%d m=%d t=%.9g dt=%.9g\n", argv[2], n, m, t, dt);
    return 0;
  }
  if (argc >= 4 && !strcmp(argv[1], "run")) {
    int env_steps = atoi(argv[3]);
    ora_config cfg = ora_default_config();
    if (argc >= 5) cfg.literal = atoi(argv[4]);
    FILE *trace = argc >= 6 ? fopen(argv[5], "w") : NULL;
    ora_env *e = ora_env_new(&cfg);
    if (!e) { fprintf(stderr, "the reference cannot run this grid\n"); return 1; }
    if (strcmp(argv[2], "uniform")) {
      int n, m; float t, dt, *ux, *uy, *p;
      int rc = ora_read_bdimb(argv[2], &n, &m, &t, &dt, &ux, &uy, &p);
      if (rc || n != ora_env_n(e) || m != ora_env_m(e)) { fprintf(stderr, "bad state file (%d)\n", rc); return 1; }
      ora_env_set_state(e, ux, uy, p);
      free(ux); free(uy); free(p);
    }
    ora_driver d = ora_driver_new();
    d.callLearn = 16;
    int k = 0;
    double t0 = now_s();
    long solver_steps = 0;
    float Cl = 0, Cd = 0;
    while (k < env_steps) {
      /* initTime = -1: accumulate from the first step (the timing/parity workload has no warm-up gap) */
      int produced = ora_driver_step(&d, e, -1.0f, &Cl, &Cd);
      solver_steps++;
      if (trace) {
        float fx, fy; ora_env_force(e, &fx, &fy);
        fprintf(trace, "%ld %.9g %.9g\n", solver_steps, fx, fy);
      }
      if (produced) {
        float a1 = (float)(0.8 * sin(2.0 * M_PI * k / 25.0));
        float a2 = (float)(-0.8 * sin(2.0 * M_PI * k / 25.0 + 1.0));
        ora_env_set_xi(e, a1, a2);
        k++;
      }
    }
    double el = now_s() - t0;
    if (trace) fclose(trace);
    printf("{\"env_steps\": %d, \"solver_steps\": %ld, \"seconds\": %.6f, \"env_steps_per_s\": %.6f, "
           "\"literal\": %d, \"last_Cl\": %.9g, \"last_Cd\": %.9g}\n",
           env_steps, solver_steps, el, env_steps / el, cfg.literal, Cl, Cd);
    ora_env_free(e);
    return 0;
  }
  fprintf(stderr, "usage: oracle_cli convert <in.bdim> <out.bdimb> <n> <m> | run <state.bdimb|uniform> <env_steps> [literal] [trace]\n");
  return 2;
}
