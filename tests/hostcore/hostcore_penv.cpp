// hostcore_penv.cpp -- TEST INFRASTRUCTURE ONLY.
// The device core (basilisk_env_b200/csrc/leo_core.cuh) compiled for the HOST with g++, with the per-env parameter policy
// (leo::ParEnv) of the parameter-pool kernel: every env carries its own derived parameter block behind its state fields,
// exactly as in the library (leo_params.h: LeoPField), so that the CPU suite can compare the per-env arithmetic with the
// batch-global core and with the oracle.  Reference configuration (three wheels, DIAG) only, as the library builds it.
#include <stdint.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../basilisk_env_b200/csrc/leo_core.cuh"
#include "../../basilisk_env_b200/csrc/leo_host.h"

struct HCP {
    bskenv_config cfg;
    LeoParams P;
    int64_t n;
    std::vector<double> S;      // [LEO_ND + LEO_NPD][n]
    std::vector<int64_t> I;     // [LEO_NI][n]
    std::string err;
};

extern "C" {
HCP *hcp_create(const bskenv_config *cfg, int64_t n)
{
    HCP *h = new HCP();
    h->cfg = *cfg;
    if (!leo_host::build_params(*cfg, h->P).empty() || h->P.nrw != 3 || !h->P.diag) { delete h; return nullptr; }
    h->n = n;
    h->S.assign((size_t)(LEO_ND + LEO_NPD) * n, 0.0);
    h->I.assign((size_t)LEO_NI * n, 0);
    double raw[BSKENV_PARAM_DIM], row[LEO_NPD];           // every env starts on the batch configuration
    leo_host::param_row_get(*cfg, raw);
    leo_host::param_row_derive(h->P, raw, -1.0, row);
    for (int f = 0; f < LEO_NPD; f++)
        for (int64_t e = 0; e < n; e++) h->S[(size_t)(LEO_ND + f) * n + e] = row[f];
    return h;
}
void hcp_destroy(HCP *h) { delete h; }
const char *hcp_error(HCP *h) { return h->err.c_str(); }
// env e runs raw[e] (BSKENV_PARAM_DIM values); returns 0, or -1 with hcp_error set
int hcp_set_env_params(HCP *h, const double *raw)
{
    for (int64_t e = 0; e < h->n; e++) {
        double row[LEO_NPD];
        h->err = leo_host::param_row_build(h->cfg, raw + e * BSKENV_PARAM_DIM, (double)e, row);
        if (!h->err.empty()) return -1;
        for (int f = 0; f < LEO_NPD; f++) h->S[(size_t)(LEO_ND + f) * h->n + e] = row[f];
    }
    return 0;
}
void hcp_reset_ics(HCP *h, const double *ics, double *obs)
{
    for (int64_t e = 0; e < h->n; e++) {
        double ic[19];
        for (int k = 0; k < 19; k++) ic[k] = ics[e * 19 + k];
        leo::leo_reset_env<leo::ParEnv>(h->P, h->S.data(), h->I.data(), h->n, e, ic, obs ? obs + 5 * e : nullptr);
    }
}
// per_env = 1: leo_step_env with the per-env policy; 0: the batch-global core (its parameter block is ignored)
void hcp_step(HCP *h, int per_env, const int32_t *actions, double *obs, double *reward, uint8_t *done, uint8_t *reason)
{
    double bus[leo::LEO_NM_PENV];
    leo::MBus m; m.a = 0; m.p = bus;
    const int nch = leo_host::step_chunks(h->P);
    double *S = h->S.data();
    int64_t *I = h->I.data();
    for (int64_t e = 0; e < h->n; e++)
    for (int ch = 0; ch < nch; ch++) {
        leo::StepOut o;
        if (per_env) {
            if (h->P.use_j2) leo::leo_step_env<3, 1, true, false, leo::ParEnv>(h->P, S, I, h->n, e, m, actions[e], o, LeoParamsF(), ch, nch);
            else leo::leo_step_env<3, 0, true, false, leo::ParEnv>(h->P, S, I, h->n, e, m, actions[e], o, LeoParamsF(), ch, nch);
        } else {
            if (h->P.use_j2) leo::leo_step_env<3, 1, true>(h->P, S, I, h->n, e, m, actions[e], o, LeoParamsF(), ch, nch);
            else leo::leo_step_env<3, 0, true>(h->P, S, I, h->n, e, m, actions[e], o, LeoParamsF(), ch, nch);
        }
        if (ch + 1 < nch) continue;
        for (int k = 0; k < 5; k++) obs[5 * e + k] = o.ob[k];
        reward[e] = o.reward; done[e] = (uint8_t)o.done; reason[e] = (uint8_t)o.reason;
    }
}
// the LEO_ND state fields and the LEO_NI integer fields ([field][n])
void hcp_get_state(HCP *h, double *S, int64_t *I)
{
    memcpy(S, h->S.data(), sizeof(double) * LEO_ND * h->n);
    memcpy(I, h->I.data(), sizeof(int64_t) * LEO_NI * h->n);
}
int hcp_dims(int *nd, int *ni, int *npd) { *nd = LEO_ND; *ni = LEO_NI; *npd = LEO_NPD; return 0; }
// pool row selection of the library (leo::pool_row) for the assignment tests
int64_t hcp_pool_row(int64_t n_rows, int assign, uint64_t seed, int64_t global_env, int64_t episode)
{
    LeoPool pool; pool.rows = nullptr; pool.n_rows = (int32_t)n_rows; pool.assign = assign;
    return leo::pool_row(pool, seed, global_env, episode);
}
}
