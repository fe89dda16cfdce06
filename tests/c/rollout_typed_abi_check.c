/* tests/c/rollout_typed_abi_check.c -- the 16-bit rollout entry points (include/marlnav_b200_rollout_typed.h,
 * included by marlnav_b200.h) from plain C: the declarations compile as C99, every entry links, and an
 * unknown obs_dtype or a NULL pointer comes back as MARLNAV_ERR_BAD_ARG with a message (no GPU needed). */
#include <stdio.h>
#include <string.h>
#include "../../include/marlnav_b200.h"

int main(void) {
    void* entry[] = {(void*)marlnav_actor_sample_typed, (void*)marlnav_critic_value_typed,
                     (void*)marlnav_act_step_typed};
    size_t i;
    for (i = 0; i < sizeof entry / sizeof entry[0]; ++i) if (!entry[i]) return 10;
    {
        marlnav_env_params p;
        marlnav_reset_spec rs;
        float dummy[4] = {0.f, 0.f, 0.f, 0.f};
        memset(&p, 0, sizeof p); memset(&rs, 0, sizeof rs);
        p.struct_size = sizeof p; p.num_envs = 4; p.num_agents = 3; p.num_obstacles = 3;
        rs.struct_size = sizeof rs; rs.alias_first_step = 1;
        if (marlnav_actor_sample_typed(dummy, 3, 4, 12, 50, dummy, dummy, dummy, dummy, dummy, dummy, NULL, 0, 0,
                                       NULL, 0, dummy, dummy, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG) return 1;
        if (!strstr(marlnav_rollout_last_error(), "obs_dtype")) return 2;
        if (marlnav_critic_value_typed(dummy, -1, 4, 36, 50, dummy, dummy, dummy, dummy, dummy, NULL)
            != MARLNAV_ERR_BAD_ARG) return 3;
        if (!strstr(marlnav_rollout_last_error(), "obs_dtype")) return 4;
        if (marlnav_act_step_typed(&p, &rs, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, 255, NULL, NULL,
                                   NULL, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG) return 5;
        if (!strstr(marlnav_last_error(), "obs_dtype")) return 6;
        if (marlnav_actor_sample_typed(NULL, MARLNAV_OBS_F16, 4, 12, 50, dummy, dummy, dummy, dummy, dummy, dummy,
                                       NULL, 0, 0, NULL, 0, dummy, dummy, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG)
            return 7;
        if (!strstr(marlnav_rollout_last_error(), "NULL")) return 8;
        if (marlnav_critic_value_typed(NULL, MARLNAV_OBS_BF16, 4, 36, 50, dummy, dummy, dummy, dummy, dummy, NULL)
            != MARLNAV_ERR_BAD_ARG) return 9;
        if (!strstr(marlnav_rollout_last_error(), "NULL")) return 11;
        if (marlnav_act_step_typed(&p, &rs, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL,
                                   MARLNAV_OBS_F16, NULL, NULL, NULL, NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG)
            return 12;
        if (!strstr(marlnav_last_error(), "NULL")) return 13;
    }
    printf("rollout typed abi ok\n");
    return 0;
}
