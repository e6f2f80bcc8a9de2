/*
 * oracle_params.c -- TEST INFRASTRUCTURE ONLY.
 * The CPU oracle (oracle/bsk_oracle.c, included as it is) with the spacecraft parameters of a reference
 * `initial_conditions` dict settable per sim: the oracle builds every sim with the reference's values
 * (orc_leo_create: mass = 330, K = 7, ...), and the per-env parameter pools of the library
 * (bskenv_set_param_pool) need a reference for any other spacecraft.
 */
#include "../../oracle/bsk_oracle.c"

/* p[14] = mass, width, depth, height, baseDensity, scaleHeight, disturbance_magnitude, panelArea, panelEfficiency,
 * powerDraw, storageCapacity, K, P, hs_min (BSKENV_PARAM_DIM order).  Recomputes what orc_leo_create derives from those
 * keys (SIM:129-190): hub mass and inertia, the FSW inertia, atmosphere, disturbance torque, power, gains.  Call it right
 * after the sim is built, before the first run_sim. */
void orc_leo_set_params(orc_leo_sim *s, const double p[14])
{
    const double mass = p[0], width = p[1], depth = p[2], height = p[3];
    s->mHub = mass;
    memset(s->IHub, 0, sizeof(s->IHub));
    s->IHub[0][0] = 1. / 12. * mass * (pow(width, 2.) + pow(depth, 2.));
    s->IHub[1][1] = 1. / 12. * mass * (pow(depth, 2.) + pow(height, 2.));
    s->IHub[2][2] = 1. / 12. * mass * (pow(width, 2.) + pow(height, 2.));
    s->baseDensity = p[4]; s->scaleHeight = p[5];
    v3Scale(p[6], s->ic.disturbance_vector, s->extTorquePntB_B);         /* SIM:295 */
    s->panelArea = p[7]; s->panelEfficiency = p[8];
    s->nodePowerOut = p[9];
    s->storageCapacity = p[10];
    memcpy(s->ISC_fsw, s->IHub, sizeof(s->IHub));                          /* SIM:392-403 */
    s->K = p[11]; s->P = p[12]; s->hs_min = p[13];
}

/* orc_env_reset with the env's parameter set applied to the new sim (the reference builds every episode's sim from the
 * same dict) */
void orc_env_reset_params(orc_leo_env *e, const orc_leo_ic *ic, const double p[14], double ob[5])
{
    orc_env_reset(e, ic, ob);
    orc_leo_set_params(e->sim, p);
}
