/* tests/c/typed_abi_check.c -- the 16-bit observation entry points (include/marlnav_b200_typed.h, included
 * by marlnav_b200.h) from plain C: the declarations compile as C99, every entry links, and an unknown
 * obs_dtype or a NULL pointer comes back as MARLNAV_ERR_BAD_ARG with a message (no GPU needed). */
#include <stdio.h>
#include <string.h>
#include "../../include/marlnav_b200.h"

int main(void) {
    void* entry[] = {(void*)marlnav_observe_typed, (void*)marlnav_step_typed, (void*)marlnav_step_call_typed,
                     (void*)marlnav_step_host_typed};
    size_t i;
    for (i = 0; i < sizeof entry / sizeof entry[0]; ++i) if (!entry[i]) return 10;
    if (MARLNAV_OBS_F32 != 0 || MARLNAV_OBS_F16 != 1 || MARLNAV_OBS_BF16 != 2) return 1;
    {
        marlnav_env_params p;
        marlnav_reset_spec rs;
        marlnav_step_call call;
        float dummy[4] = {0.f, 0.f, 0.f, 0.f};
        memset(&p, 0, sizeof p); memset(&rs, 0, sizeof rs); memset(&call, 0, sizeof call);
        p.struct_size = sizeof p; p.num_envs = 4; p.num_agents = 3; p.num_obstacles = 3;
        rs.struct_size = sizeof rs; rs.alias_first_step = 1;
        call.struct_size = sizeof call; call.params = &p; call.reset = &rs;
        if (marlnav_observe_typed(&p, dummy, dummy, dummy, dummy, 3, NULL) != MARLNAV_ERR_BAD_ARG) return 2;
        if (!strstr(marlnav_last_error(), "obs_dtype")) return 3;
        if (marlnav_step_call_typed(&call, -1) != MARLNAV_ERR_BAD_ARG) return 4;
        if (!strstr(marlnav_last_error(), "obs_dtype")) return 5;
        if (marlnav_step_call_typed(&call, MARLNAV_OBS_F16) != MARLNAV_ERR_BAD_ARG) return 6;   /* NULL tensors */
        if (!strstr(marlnav_last_error(), "NULL")) return 7;
        if (marlnav_step_typed(&p, &rs, NULL, NULL, NULL, NULL, NULL, NULL, NULL, MARLNAV_OBS_BF16, NULL, NULL, NULL,
                               NULL, NULL, NULL) != MARLNAV_ERR_BAD_ARG) return 8;
        if (!strstr(marlnav_last_error(), "NULL")) return 9;
        if (marlnav_step_host_typed(NULL, &p, &rs, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL,
                                    NULL, NULL, NULL, NULL, NULL, NULL, NULL, 7) != MARLNAV_ERR_BAD_ARG) return 11;
        if (!strstr(marlnav_last_error(), "obs_dtype")) return 12;
    }
    printf("typed abi ok\n");
    return 0;
}
