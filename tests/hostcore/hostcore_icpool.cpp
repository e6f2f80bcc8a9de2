// hostcore_icpool.cpp -- TEST INFRASTRUCTURE ONLY.
// The initial-condition pool pieces of the device core (basilisk_env_b200/csrc/leo_core.cuh: ic_pool_row, pool_row,
// sample_ic; leo_host.h: ic_row_check) compiled for the HOST with g++, so that the CPU suite can check the row selection and
// the row validation the library uses.
#include <stdint.h>
#include <string.h>
#include <string>
#include "../../basilisk_env_b200/csrc/leo_core.cuh"
#include "../../basilisk_env_b200/csrc/leo_host.h"

extern "C" {
// leo::ic_pool_row: assign 0 = by index, 1 = per episode, 2 = the parameter row `param_row`
int64_t hci_ic_pool_row(int64_t n_rows, int assign, uint64_t seed, int64_t global_env, int64_t episode, int64_t param_row)
{
    IcPool pool; pool.rows = nullptr; pool.row_of = nullptr; pool.row_ep = nullptr; pool.n_rows = (int32_t)n_rows; pool.assign = assign;
    return leo::ic_pool_row(pool, seed, global_env, episode, param_row);
}
// leo::pool_row (the parameter pool), for the comparison of the two streams
int64_t hci_param_pool_row(int64_t n_rows, int assign, uint64_t seed, int64_t global_env, int64_t episode)
{
    LeoPool pool; pool.rows = nullptr; pool.n_rows = (int32_t)n_rows; pool.assign = assign;
    return leo::pool_row(pool, seed, global_env, episode);
}
// leo::sample_ic of the configuration `cfg` for (seed, global env, episode)
int hci_sample_ic(const bskenv_config *cfg, uint64_t seed, int64_t global_env, int64_t episode, double *ic)
{
    LeoParams P;
    if (!leo_host::build_params(*cfg, P).empty()) return -1;
    P.seed = seed;
    double out[19];
    leo::sample_ic(P, global_env, episode, out);
    memcpy(ic, out, sizeof(out));
    return 0;
}
// leo_host::ic_row_check: 0, or -1 with the message in msg
int hci_ic_row_check(const double *row, int dim, char *msg, int cap)
{
    const std::string err = leo_host::ic_row_check(row, dim);
    snprintf(msg, (size_t)cap, "%s", err.c_str());
    return err.empty() ? 0 : -1;
}
}
