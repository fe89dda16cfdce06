/* tests/c/final_obs_abi_check.c -- the final-observation steps and the GAE scan
 * (include/marlnav_b200_final.h, included by marlnav_b200.h) from plain C: the declarations compile as
 * C99, every entry links, and a NULL / aliased final_obs, an unknown obs_dtype or a NULL GAE input comes
 * back as MARLNAV_ERR_BAD_ARG with a message (no GPU needed). */
#include <stdio.h>
#include <string.h>
#include "../../include/marlnav_b200.h"

int main(void) {
    void* entry[] = {(void*)marlnav_step_final_typed, (void*)marlnav_step_call_final_typed, (void*)marlnav_gae_f64};
    size_t i;
    for (i = 0; i < sizeof entry / sizeof entry[0]; ++i) if (!entry[i]) return 10;
    {
        marlnav_env_params p;
        marlnav_reset_spec rs;
        marlnav_step_call c;
        float dummy[4] = {0.f, 0.f, 0.f, 0.f};
        float obs[4], fin[4];
        unsigned char flags[4];
        double a[4], r[4];
        memset(&p, 0, sizeof p); memset(&rs, 0, sizeof rs); memset(&c, 0, sizeof c);
        p.struct_size = sizeof p; p.num_envs = 4; p.num_agents = 3; p.num_obstacles = 3;
        rs.struct_size = sizeof rs; rs.alias_first_step = 1;
        if (marlnav_step_final_typed(&p, &rs, dummy, dummy, dummy, dummy, flags, dummy, obs, MARLNAV_OBS_F32, NULL,
                                     dummy, flags, flags, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG) return 1;
        if (!strstr(marlnav_last_error(), "final_obs")) return 2;
        if (marlnav_step_final_typed(&p, &rs, dummy, dummy, dummy, dummy, flags, dummy, obs, MARLNAV_OBS_F16, obs,
                                     dummy, flags, flags, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG) return 3;
        if (!strstr(marlnav_last_error(), "different buffers")) return 4;
        if (marlnav_step_final_typed(&p, &rs, dummy, dummy, dummy, dummy, flags, dummy, obs, 7, fin,
                                     dummy, flags, flags, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG) return 5;
        if (!strstr(marlnav_last_error(), "obs_dtype")) return 6;
        c.struct_size = sizeof c; c.params = &p; c.reset = &rs; c.obs = obs;
        if (marlnav_step_call_final_typed(&c, MARLNAV_OBS_BF16, NULL) != MARLNAV_ERR_BAD_ARG) return 7;
        if (!strstr(marlnav_last_error(), "final_obs")) return 8;
        if (marlnav_step_call_final_typed(&c, -1, fin) != MARLNAV_ERR_BAD_ARG) return 9;
        if (!strstr(marlnav_last_error(), "obs_dtype")) return 11;
        if (marlnav_gae_f64(dummy, NULL, flags, flags, NULL, NULL, 0.99, 0.95, 1, 4, a, r, NULL) != MARLNAV_ERR_BAD_ARG)
            return 12;
        if (!strstr(marlnav_rollout_last_error(), "NULL")) return 13;
    }
    printf("final abi ok\n");
    return 0;
}
