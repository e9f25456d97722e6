/* Prints the layout of rlfc_config as a C compiler lays it out from include/rlfc.h: "sizeof <bytes>", then one
   "<field> <offset>" line per field (test_flow_stats_host.py compares it with the ctypes mirror, env.Config). */
#include <stddef.h>
#include <stdio.h>

#include "rlfc.h"

#define F(x) printf(#x " %zu\n", offsetof(rlfc_config, x))

int main(void) {
  printf("sizeof %zu\n", sizeof(rlfc_config));
  F(resolution); F(x_lengths); F(y_lengths); F(re); F(dR); F(gR); F(theta); F(t_step); F(action_scale); F(substeps);
  F(init_time); F(episode_time); F(n_envs); F(device); F(exact); F(mg_max_iters); F(init_bdim_path); F(stream);
  F(n_groups); F(n_devices); F(adaptive_dt); F(env_params); F(n_snapshots); F(n_sensors); F(sensors); F(n_param_sets);
  F(param_sets); F(stats_every);
  printf("RLFC_NUM_STATS %d\n", RLFC_NUM_STATS);
  printf("RLFC_STAT_UX %d\nRLFC_STAT_UY %d\nRLFC_STAT_P %d\nRLFC_STAT_UXUX %d\nRLFC_STAT_UYUY %d\nRLFC_STAT_PP %d\nRLFC_STAT_UV %d\n",
         RLFC_STAT_UX, RLFC_STAT_UY, RLFC_STAT_P, RLFC_STAT_UXUX, RLFC_STAT_UYUY, RLFC_STAT_PP, RLFC_STAT_UV);
  return 0;
}
