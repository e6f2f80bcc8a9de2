/*
 * bskenv.h -- C ABI of the B200-native batched LEO power/attitude environment step.
 *
 * This is the drop-in boundary for ONE path of atharris/basilisk_env: everything below
 * `LEOPowerAttitudeSimulator.run_sim(action)` (reference: basilisk_env/simulators/
 * leoPowerAttitudeSimulator.py:535-644, i.e. the Basilisk `ExecuteSimulation()` call at :595 and the
 * message sampling at :598-642), plus the gym bookkeeping of `leoPowerAttEnv.step`
 * (basilisk_env/envs/leoPowerAttitudeEnvironment.py:65-145) and the simulator construction done in
 * `reset` (:172-191, simulators/...Simulator.py:67-117), vectorised over N independent environments.
 *
 * Plain pointers and sizes only; no torch / C++ types.  Device pointers are raw CUDA device
 * addresses in the handle's device (e.g. torch `tensor.data_ptr()`), streams are `cudaStream_t`
 * passed as `void*` (0 = legacy default stream).  Every function returns 0 on success or a negative
 * BSKENV_E* code; `bskenv_last_error` gives the message.  Nothing throws across this boundary and
 * there is NO CPU fallback: without a CUDA device `bskenv_create` fails.
 */
#ifndef BSKENV_H
#define BSKENV_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSKENV_ABI_VERSION 1

#define BSKENV_OK 0
#define BSKENV_EINVAL (-1)   /* bad argument / unsupported configuration */
#define BSKENV_ECUDA (-2)    /* CUDA runtime error (message in last_error) */
#define BSKENV_ENODEV (-3)   /* no usable CUDA device */

/* done_reason bitmask; replaces the reference's print() calls (envs/...Environment.py:110-127) */
#define BSKENV_DONE_MAXLEN 1 /* curr_step >= max_length          (:98-99)  */
#define BSKENV_DONE_WHEEL 2  /* ob[2] > 1, "wheel explosion"     (:110-115) */
#define BSKENV_DONE_POWER 4  /* ob[3] == 0, "ran out of power"   (:119-123) */
#define BSKENV_DONE_DECAY 8  /* sim_over, "orbit decayed"        (:125-127, simulators/...:641-642) */

#define BSKENV_OBS_DIM 5     /* [|sigma_BR|, |omega_BN_B|, |Omega_rw|/wheel_limit, Wh/power_max, shadowFactor] */
#define BSKENV_IC_DIM 19     /* rN(3) vN(3) sigma_init(3) omega_init(3) disturbance_vector(3) wheelSpeeds_rpm(3) storedCharge_Init */

/*
 * Batch-global configuration == the non-sampled entries of the reference's `initial_conditions`
 * dict (simulators/leoPowerAttitudeSimulator.py:127-191), the constructor arguments (:67) and the
 * env attributes (envs/leoPowerAttitudeEnvironment.py:25-42).  `bskenv_default_config` fills the
 * reference values; only the fields below are tunable, the module graph itself is fixed.
 */
typedef struct bskenv_config {
    int32_t abi_version;         /* BSKENV_ABI_VERSION */
    int32_t reserved0;
    /* LEOPowerAttitudeSimulator(dynRate, fswRate, step_duration) */
    double dynRate;              /* 0.1 s   */
    double fswRate;              /* 1.0 s   */
    double step_duration;        /* 180. s  */
    /* spacecraft ("mass", "width", "depth", "height") */
    double mass, width, depth, height;
    /* atmosphere ("planetRadius", "baseDensity", "scaleHeight") */
    double planetRadius, baseDensity, scaleHeight;
    double disturbance_magnitude;   /* 2e-4 */
    /* power ("nHat_B", "panelArea", "panelEfficiency", "powerDraw", "storageCapacity") */
    double nHat_B[3], panelArea, panelEfficiency, powerDraw, storageCapacity;
    /* FSW ("sigma_R0N", "K", "Ki", "P", "hs_min", "thrForceSign", "maxCounterValue", "thrMinFireTime") */
    double sigma_R0N[3], K, Ki, P, hs_min, thrMinFireTime;
    int32_t thrForceSign, maxCounterValue;
    /* env attributes */
    int32_t max_length;          /* 540 */
    int32_t auto_reset;          /* 0: gym single-env semantics; 1: re-sample ICs in-kernel when done */
    double wheel_limit_rpm;      /* 3000 */
    double power_max;            /* 20 */
    double failure_penalty;      /* 1 */
    /* documented deviations / switches (DESIGN.md): all 0 reproduces the reference wiring */
    int32_t use_j2;              /* SURVEY M1: reference has no J2; 1 only for the stress config */
    int32_t hill_cel_pun;        /* SURVEY Q3: 1 = hillPoint reads the SPICE message as an ephemeris message */
    int32_t rw_set;              /* 0: three HR16 along the body axes (reference LEO env, actuatorPrimatives.py:20-37);
                                    1: four HR16 in the opNav pyramid, elevation 40 deg, azimuth 45/135/225/315 deg
                                    (opNav_models/BSK_OpNavDynamics.py:269-293): BASELINE stress config.  The fourth
                                    wheel starts at the mean of the three sampled speeds. */
    int32_t precision;           /* 0: FP64 everywhere (the reference's arithmetic; every parity claim is about this setting).
                                    1: mixed precision for the accuracy / throughput trade-off of the stress config: the RK4 stage
                                    arithmetic, density, eclipse cone tests and panel projection in FP32; state accumulation,
                                    clocks, battery, flight software, wheel limits and thruster logic in FP64 */
    int32_t reserved[6];
} bskenv_config;

typedef struct bskenv_handle bskenv_handle;

int bskenv_abi_version(void);
void bskenv_default_config(bskenv_config *cfg);

/* One handle owns the persistent SoA state of `n_envs` environments on CUDA device `device`.
 * `first_env_index` is the global index of env 0 of this shard: per-env random streams are keyed by
 * (seed, global index, episode), so results do not depend on how envs are sharded across GPUs. */
int bskenv_create(const bskenv_config *cfg, int device, int64_t n_envs, int64_t first_env_index,
                  bskenv_handle **out);
int bskenv_destroy(bskenv_handle *h);
const char *bskenv_last_error(const bskenv_handle *h); /* h may be NULL: last create() error */
int64_t bskenv_num_envs(const bskenv_handle *h);

/* SURVEY 8(f)-4 -- optional force-model / ephemeris upgrades of a handle (all off = the reference wiring; call before
 * reset).  They close the gap to a SPICE-driven Basilisk run: the reference loads de430.bsp / pck00010.tpc through
 * Basilisk's spice_interface (simulators/leoPowerAttitudeSimulator.py:219-225); here the same data arrive as tables.
 *
 * bskenv_set_ephemeris: Chebyshev table in the layout of SPICE SPK type 2 / binary PCK type 2 records, host memory,
 * coef[n_seg][3][n_coef]; segment i covers sim time [t0 + i*seg_len, t0 + (i+1)*seg_len] seconds (sim time 0 = the
 * scenario epoch '2021 MAY 04 07:47:48.965 (UTC)', :219); value = sum_k a_k T_k(s), rate = its derivative.
 *   kind BSKENV_EPH_SUN    Sun position relative to Earth, J2000 axes [m]: replaces the analytic Sun (DESIGN D1)
 *   kind BSKENV_EPH_ORIENT Earth orientation angles RA, DEC, W [rad]: replaces the IAU rotation model
 * n_seg = 0 unloads the table.  The table must cover one episode, [0, (max_length + 1) * step_duration].
 *
 * bskenv_set_gravity_degree2: Earth's degree-2 field C20, C21, S21, C22, S22 (normalised, as gravity-model files
 * carry them; NULL = GGM03S-class defaults) evaluated in the planet-fixed frame, whose orientation comes with the
 * SPICE message every step_duration and is Euler-stepped in between (Basilisk GravBodyData::computeGravityInertial).
 * Overrides use_j2 (which keeps the zonal term on the inertial z axis). */
#define BSKENV_EPH_SUN 0
#define BSKENV_EPH_ORIENT 1
int bskenv_set_ephemeris(bskenv_handle *h, int kind, double t0, double seg_len, int n_seg, int n_coef, const double *coef);
int bskenv_set_gravity_degree2(bskenv_handle *h, int enable, const double *cbar /* [5] or NULL */);

/* Per-env spacecraft parameters (Monte Carlo dispersions, domain randomisation): in the reference every
 * LEOPowerAttitudeSimulator is built from its own `initial_conditions` dict (simulators/leoPowerAttitudeSimulator.py:127-191);
 * here a POOL of n_rows parameter sets is loaded into the handle and each env runs one row for a whole episode.  A row is
 * BSKENV_PARAM_DIM doubles, the reference's keys and units in this order:
 *   mass, width, depth, height, baseDensity, scaleHeight, disturbance_magnitude, panelArea, panelEfficiency, powerDraw,
 *   storageCapacity, K, P, hs_min
 * Everything else stays batch-global (bskenv_config).  The row is picked at reset -- bskenv_reset_seeded, bskenv_reset_ics
 * and the in-kernel auto-reset; bskenv_reset_init keeps the env's row, as the reference rebuilds from the same dict:
 *   BSKENV_PARAMS_BY_INDEX     row = (first_env_index + e) % n_rows  (n_rows = global env count: an explicit per-env table)
 *   BSKENV_PARAMS_PER_EPISODE  row drawn from a counter-based stream keyed by (seed, global env index, episode), separate
 *                              from the IC stream: the initial conditions are those of a run without a pool, and neither
 *                              depends on the sharding.  `episode` is the env's episode counter after the reset.
 * Loading a pool does not touch running envs until their next reset (envs that have not been reset under a pool run the
 * batch configuration, row -1).  n_rows = 0 unloads the pool: new resets use the batch configuration and bskenv_step*
 * returns to the batch-global kernels.  Each row is derived on the host exactly as bskenv_create derives the batch
 * configuration.  BSKENV_EINVAL for a non-positive mass, dimension, scaleHeight or storageCapacity, a non-finite value, an
 * unknown mode, and for configurations the per-env kernel is not built for: rw_set = 1, precision = 1, the degree-2 field
 * (bskenv_set_gravity_degree2) and BSKENV_ORG_SPLIT (which bskenv_set_organisation refuses while a pool is loaded).  With
 * a pool loaded, BSKENV_ORG_AUTO runs one thread per env at every batch size (kernel leo_step_penv_kernel). */
#define BSKENV_PARAM_DIM 14
#define BSKENV_PARAMS_BY_INDEX 0
#define BSKENV_PARAMS_PER_EPISODE 1
int bskenv_set_param_pool(bskenv_handle *h, int n_rows, const double *rows_host /* [n_rows][14] */, int assign);
/* The parameters every env runs with, double[n][BSKENV_PARAM_DIM] row-major, and its pool row (int32[n], may be NULL;
 * -1 = the batch configuration). */
int bskenv_get_env_params(bskenv_handle *h, double *params_dev /* [n][14] */, int32_t *row_dev /* [n] or NULL */, void *stream);

/* Per-episode initial conditions from a pool (Monte Carlo campaigns over dispersed start states, curricula, replayed failure
 * cases, fixed evaluation sets): the second half of the reference's `initial_conditions` dict, the state an episode starts
 * from.  n_rows rows of BSKENV_IC_DIM doubles, the layout of bskenv_reset_ics, are loaded into the handle (device memory);
 * resets that sample -- bskenv_reset_seeded and the auto-reset of bskenv_step* -- take a pool row instead of the built-in
 * sampler.  The row of each reset:
 *   BSKENV_ICS_BY_INDEX     row = (first_env_index + e) % n_rows
 *   BSKENV_ICS_PER_EPISODE  row drawn from a counter-based stream keyed by (seed, global env index, episode), separate from the
 *                           IC sampler, the parameter pool and the opNav noise streams: those are the draws of a run without
 *                           an IC pool, and nothing depends on the sharding.  `episode` is the counter after the reset.
 *   BSKENV_ICS_PARAM_ROW    row = the env's parameter-pool row of the same reset (LEO only): with a parameter pool of the same
 *                           n_rows the two pools are one scenario table of (initial conditions, parameters) pairs.
 * bskenv_reset_ics uses its explicit rows and records row -1; bskenv_reset_init replays the stored ICs and keeps the row;
 * bskenv_get_ics reports the pool values an env started from.  Loading a pool does not touch running envs until their next
 * reset; n_rows = 0 unloads it (new resets sample again and bskenv_step* returns to the in-kernel auto-reset).  With a pool and
 * auto_reset, bskenv_step* launches the step kernel without its in-kernel reset and then the reset kernel over the envs that
 * finished (mask = done): one more launch per step (bskenv_launch_count; bskenv_kernel_name still names the step kernel),
 * every organisation and configuration, the same results as bskenv_reset_seeded with mask = done after a step without
 * auto_reset.  BSKENV_EINVAL for a non-finite value or a zero position vector (the message names the row), an unknown mode,
 * BSKENV_ICS_PARAM_ROW without a loaded parameter pool of the same n_rows, and -- while such a paired pool is loaded --
 * bskenv_set_param_pool with another row count or an unload.  Refused while a host-buffer step is in flight.
 * bskenv_get_ic_rows: the pool row each env's current episode started from (int32[n], device memory); -1 = sampled or
 * explicit ICs, or a reset before the pool was loaded.  The row is not part of the state (bskenv_state_dims, get_state /
 * set_state): a checkpoint does not carry it. */
#define BSKENV_ICS_BY_INDEX 0
#define BSKENV_ICS_PER_EPISODE 1
#define BSKENV_ICS_PARAM_ROW 2
int bskenv_set_ic_pool(bskenv_handle *h, int n_rows, const double *ics_host /* [n_rows][19] */, int assign);
int bskenv_get_ic_rows(bskenv_handle *h, int32_t *rows_dev /* [n] */, void *stream);

/* reset(): sample fresh initial conditions on the device (distributions and clipping of
 * initial_conditions/leo_orbit.py:25-39, sc_attitudes.py:3-13, simulators/...Simulator.py:152-167).
 * `mask_dev` (uint8[n], may be NULL = all) selects the envs to reset.  `obs_dev` (double[n*5], may be
 * NULL) receives the normalised initial observation of the reset envs. */
int bskenv_reset_seeded(bskenv_handle *h, uint64_t seed, const uint8_t *mask_dev, double *obs_dev, void *stream);
/* reset with explicit initial conditions: `ics_dev` is double[n*19] row-major (BSKENV_IC_DIM). */
int bskenv_reset_ics(bskenv_handle *h, const double *ics_dev, const uint8_t *mask_dev, double *obs_dev, void *stream);
/* reset_init(): rebuild from the stored initial conditions (envs/...Environment.py:202-216). */
int bskenv_reset_init(bskenv_handle *h, const uint8_t *mask_dev, double *obs_dev, void *stream);
int bskenv_get_ics(bskenv_handle *h, double *ics_dev, void *stream);

/* step(): ONE kernel launch advances every env by one decision interval (step_duration of
 * simulated time: 1800 RK4 ticks + 1800 environment ticks + 180 flight-software ticks at the
 * reference rates) and evaluates reward/termination.  All buffers are caller-owned device memory:
 *   actions int32[n]; obs double[n*5]; reward double[n]; done uint8[n]; done_reason uint8[n].
 * With auto_reset, envs that finish are re-initialised inside the same launch; `obs` then holds the
 * first observation of the new episode and `term_obs_dev` (double[n*5], may be NULL) the terminal one. */
int bskenv_step(bskenv_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev,
                uint8_t *done_dev, uint8_t *done_reason_dev, double *term_obs_dev, void *stream);
/* Same call with HOST buffers (the reference-facing plugin path), synchronous: on return the results are in the
 * caller's buffers.  It is ordered after work queued earlier through the device-buffer entry points of this handle
 * (event on the stream of the last such call), so the two kinds of entry point can be mixed freely.  See
 * bskenv_step_host_async below for how the bytes move.  This is what bench.py times as `e2e`. */
int bskenv_step_host(bskenv_handle *h, const int32_t *actions, double *obs, double *reward,
                     uint8_t *done, uint8_t *done_reason);

/* SURVEY 8(f)-1 -- per-env episode bookkeeping of the reference's `info['episode'] = {'r': self.reward_total,
 * 'l': self.curr_step}` (envs/leoPowerAttitudeEnvironment.py:130-136).  bskenv_step with two more caller-owned device
 * outputs, written for EVERY env at every step (they are the episode record where done[e] != 0; with auto_reset they are
 * taken before the in-kernel reset):
 *   ep_return_dev double[n]  reward_total after this step (penalties included, :105,113,122)
 *   ep_length_dev int64[n]   curr_step before its increment (:144), i.e. the reference's 'l'
 * Both may be NULL (then this is bskenv_step). */
int bskenv_step_info(bskenv_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev,
                     uint8_t *done_dev, uint8_t *done_reason_dev, double *term_obs_dev, double *ep_return_dev,
                     int64_t *ep_length_dev, void *stream);

/* Host-buffer step, split in two (the shape of a VecEnv's step_async / step_wait): _async queues the launch on the handle's
 * own stream and returns; _wait blocks until the results are in the caller's buffers.  One step may be in flight per handle;
 * device-buffer calls on the same handle are refused until it has been waited for.  ep_return / ep_length as in
 * bskenv_step_info (host memory, may both be NULL).
 * ZERO-COPY: buffers that are page-locked and device-mapped (bskenv_alloc_host, cudaHostAlloc / cudaHostRegister, torch
 * pin_memory) are read and written by the kernel in place -- the 4 B in and 50 B out per env cross PCIe while the launch
 * runs, nothing is exposed after it.  Pageable buffers go through page-locked staging inside the handle and one memcpy
 * each.  bskenv_step_host == _async + _wait. */
int bskenv_step_host_async(bskenv_handle *h, const int32_t *actions, double *obs, double *reward, uint8_t *done,
                           uint8_t *done_reason, double *term_obs /* [n*5], may be NULL; rows of finished envs only */,
                           double *ep_return, int64_t *ep_length);
int bskenv_step_host_wait(bskenv_handle *h);
/* page-locked, device-mapped host memory for the host-buffer entry points (any handle, any device) */
int bskenv_alloc_host(size_t bytes, void **out);
int bskenv_free_host(void *p);

/* Checkpoint / parity injection: the whole persistent state as two SoA blocks,
 * double[n_double_fields][n] and int64[n_int_fields][n] (field-major). */
int bskenv_state_dims(const bskenv_handle *h, int32_t *n_double_fields, int32_t *n_int_fields);
int bskenv_get_state(bskenv_handle *h, double *dstate_dev, int64_t *istate_dev, void *stream);
int bskenv_set_state(bskenv_handle *h, const double *dstate_dev, const int64_t *istate_dev, void *stream);
/* index of a named state field (e.g. "r_BN_N", "sigma_BN", "Omega", "storedCharge"); -1 if unknown.
 * `is_int` receives 1 for int64 fields. */
int bskenv_state_field(const char *name, int32_t *is_int);

/* Episode statistics of this shard since the last call (sum of returns, sum of lengths, episodes
 * finished, finished by wheel / power / decay / max-length): int64/double[8] in `stats_host`.
 * (An optional NCCL all-reduce of these eight numbers is the only collective of the design.) */
int bskenv_episode_stats(bskenv_handle *h, double *stats_host);

/* Number of step-path kernel launches issued through this handle (bench.py's gpu_launches). */
int64_t bskenv_launch_count(const bskenv_handle *h);
/* Name of the step-kernel instantiation the last bskenv_step* call launched (as ncu lists it), "" before the first. */
const char *bskenv_kernel_name(const bskenv_handle *h);

/* Work organisation of the step kernel.  Both run the same arithmetic (the parity tests compare them with the oracle and
 * with each other); the choice only moves time.
 *   BSKENV_ORG_AUTO    pick by batch size (default)
 *   BSKENV_ORG_THREAD  one thread per env, one warp per 32 envs (throughput organisation; `north_star`: "thread ... owns
 *                      one spacecraft").  Batches beyond two blocks per SM are bucketed by action before the launch (a
 *                      warp takes 32 envs of one mode: the flight software of the three modes differs, leoPowerAttitude-
 *                      Simulator.py:543-588)
 *   BSKENV_ORG_THREAD_INDEX  the same without the bucketing: lanes in env-index order (measurement / test switch)
 *   BSKENV_ORG_SPLIT   two warps per group of 32 envs: a dynamics warp (RK4 and everything the next tick depends on) and a
 *                      companion warp (flight software, eclipse / panel / battery) on another SM sub-partition, handing
 *                      state over in shared memory once per tick -- the small-batch organisation (BASELINE configs[1]:
 *                      4096 envs), where one warp per group is bound by its own dependent-issue latency.  Takes batches
 *                      of at most 128 x SM-count envs (18944 on a B200), FP64, the reference or the stress configuration;
 *                      bskenv_step* returns BSKENV_EINVAL otherwise.
 * Replaces nothing in the reference (one Basilisk sim per Python process there, leoPowerAttitudeSimulator.py:75). */
#define BSKENV_ORG_AUTO 0
#define BSKENV_ORG_THREAD 1
#define BSKENV_ORG_SPLIT 2
#define BSKENV_ORG_THREAD_INDEX 3
int bskenv_set_organisation(bskenv_handle *h, int organisation);

/* FP64 FMA-pipe microbenchmark used as the roofline denominator (MEASURED_PEAKS.json has none):
 * returns achieved TFLOP/s of a register-resident DFMA chain kernel on `device`. */
int bskenv_fp64_peak(int device, double seconds, double *tflops);

/* ALGORITHMIC FP64 flop per env-decision-step for this configuration (DESIGN.md derivation). */
double bskenv_flops_per_step(const bskenv_handle *h);

/* =====================================================================================================
 * opNav environment (dynamics half + synthetic nav measurement + relative-OD filter, no rendering).
 *
 * Replaces everything below `scenario_OpNav.run_sim(action)` (reference: basilisk_env/simulators/
 * opNavSimulator.py:225-299: the Basilisk ExecuteSimulation() at :261 and the message sampling at :263-293) plus the
 * bookkeeping of `opNavEnv.step` / `reset` (basilisk_env/envs/opNavEnvironment.py:55-125, :153-168), vectorised over
 * N independent environments.  One launch = one decision interval of 50 min = 3000 ticks of 1 s: truth RK4 (hub +
 * four-wheel pyramid, Mars point mass), simple_nav error model, hillPoint / sunSafePoint guidance, MRP feedback,
 * wheel torque map, a pinhole circle measurement every 60 s, pixelLineConverter and the six-state SR-UKF.
 * ===================================================================================================== */
#define BSKENV_OPNAV_OBS_DIM 4    /* [cos(sun-Mars angle in body), sqrt(diag P_rr)/|r_nav| (3)]  (opNavSimulator.py:284-293) */
#define BSKENV_OPNAV_DEBUG_DIM 12 /* nav r(3), true r(3), true v(3), sigma_BN(3)                 (opNavSimulator.py:292) */
#define BSKENV_OPNAV_IC_DIM 12    /* rN(3) vN(3) rError(3) vError(3)                             (opNavSimulator.py:181-189) */
#define BSKENV_OPNAV_DONE_MAXLEN 1 /* curr_step >= max_length (opNavEnvironment.py:94-95) */
#define BSKENV_OPNAV_DONE_MODES 2  /* modeCounter >= numModes (opNavSimulator.py:296-297) */

typedef struct bskenv_opnav_config {
    int32_t abi_version;         /* BSKENV_ABI_VERSION */
    int32_t reserved0;
    double dynRate, fswRate;     /* 1.0, 1.0 s: scenario_OpNav(1., 1., step_duration) (opNavEnvironment.py:86) */
    double step_duration_min;    /* 50. minutes (opNavEnvironment.py:31, opNavSimulator.py:256-257) */
    int32_t max_length;          /* 40 (opNavEnvironment.py:23) */
    int32_t numModes;            /* 50 (opNavSimulator.py:149) */
    int32_t auto_reset;          /* 0: gym single-env semantics; 1: re-sample ICs in-kernel when done */
    int32_t nav_noise;           /* 1: simple_nav Gauss-Markov errors (BSK_OpNavDynamics.py:236-258); 0: truth */
    int32_t camera_reenable;     /* 0: reference behaviour (action 1 switches the camera off for the rest of the episode,
                                    opNavSimulator.py:239 is commented out); 1: action 0 switches it back on */
    int32_t sample_orbit;        /* 0: the fixed reference orbit (opNavSimulator.py:173-178); 1: the commented-out random
                                    element ranges (:166-171) for the device-side sampler */
    double pixel_noise_std;      /* synthetic circle finder: 1-sigma noise on centre / radius [px] */
    double circle_unc;           /* synthetic circle finder: CirclesOpNavMsg.uncertainty diagonal [px^2] */
    double reward_mult;          /* 1.0 (opNavEnvironment.py:32) */
    uint64_t noise_seed;         /* key of the per-env sensor-noise streams (counter-based; keyed by global env index
                                    and episode as well, so results do not depend on the sharding) */
    int32_t reserved[8];
} bskenv_opnav_config;

typedef struct bskenv_opnav_handle bskenv_opnav_handle;

void bskenv_opnav_default_config(bskenv_opnav_config *cfg);
int bskenv_opnav_create(const bskenv_opnav_config *cfg, int device, int64_t n_envs, int64_t first_env_index,
                        bskenv_opnav_handle **out);
int bskenv_opnav_destroy(bskenv_opnav_handle *h);
const char *bskenv_opnav_last_error(const bskenv_opnav_handle *h);
int64_t bskenv_opnav_num_envs(const bskenv_opnav_handle *h);
/* SURVEY 8(f)-4: Chebyshev table (layout as bskenv_set_ephemeris) of the Sun position relative to the Mars barycentre,
 * J2000 axes [m], sim time 0 = '2019 DECEMBER 12 18:00:00.0' (opNav_models/BSK_OpNavDynamics.py:396-401: de430.bsp through
 * spice_interface with zeroBase 'mars barycenter'); replaces the analytic Keplerian series.  n_seg = 0 unloads. */
int bskenv_opnav_set_ephemeris(bskenv_opnav_handle *h, double t0, double seg_len, int n_seg, int n_coef, const double *coef);
/* reset(): device-sampled ICs (filter initial error U(+-1e5 m), U(+-1e3 m/s), opNavSimulator.py:187-188; orbit fixed or
 * sampled); `obs_dev` (double[n*4], may be NULL) receives the initial observation (zeros, opNavSimulator.py:152). */
int bskenv_opnav_reset_seeded(bskenv_opnav_handle *h, uint64_t seed, const uint8_t *mask_dev, double *obs_dev, void *stream);
int bskenv_opnav_reset_ics(bskenv_opnav_handle *h, const double *ics_dev /* [n*12] */, const uint8_t *mask_dev,
                           double *obs_dev, void *stream);
int bskenv_opnav_reset_init(bskenv_opnav_handle *h, const uint8_t *mask_dev, double *obs_dev, void *stream);
int bskenv_opnav_get_ics(bskenv_opnav_handle *h, double *ics_dev, void *stream);
/* Initial-condition pool of the opNav batch: rows of BSKENV_OPNAV_IC_DIM doubles (rN vN rError vError), BSKENV_ICS_BY_INDEX or
 * BSKENV_ICS_PER_EPISODE; semantics, refusals and the extra launch of the step as bskenv_set_ic_pool / bskenv_get_ic_rows
 * (the auto-reset runs after the last kernel of the interval, in the two-kernel and the three-kernel form). */
int bskenv_opnav_set_ic_pool(bskenv_opnav_handle *h, int n_rows, const double *ics_host /* [n_rows][12] */, int assign);
int bskenv_opnav_get_ic_rows(bskenv_opnav_handle *h, int32_t *rows_dev /* [n] */, void *stream);
/* step(): ONE call = one decision interval for every env (two kernels: noise walk + dynamics / flight software, then the
 * filter; three -- the noise walk in a kernel of its own, feeding the dynamics through a device buffer of 120 B per env-tick,
 * allocated at the first step -- when the environment variable BSKENV_OPNAV_NOISE_SPLIT=1 is set at that time and the buffer
 * fits in 45 % of the free device memory; same results bit for bit).  Caller-owned device buffers:
 *   actions int32[n]; obs double[n*4]; reward double[n]; done uint8[n]; done_reason uint8[n];
 *   debug double[n*12] (may be NULL: info['full_states']); term_obs double[n*4] (may be NULL; auto_reset only). */
int bskenv_opnav_step(bskenv_opnav_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev,
                      uint8_t *done_dev, uint8_t *done_reason_dev, double *debug_dev, double *term_obs_dev, void *stream);
/* bskenv_opnav_step with the per-env episode record of `info['episode'] = {'r': self.reward_total, 'l': self.curr_step}`
 * (envs/opNavEnvironment.py:106-109) as two more device outputs, written for every env at every step (as bskenv_step_info) */
int bskenv_opnav_step_info(bskenv_opnav_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev,
                           uint8_t *done_dev, uint8_t *done_reason_dev, double *debug_dev, double *term_obs_dev,
                           double *ep_return_dev, int64_t *ep_length_dev, void *stream);
/* same with HOST buffers (zero-copy for page-locked caller buffers, staging for pageable ones, as bskenv_step_host;
 * synchronous): what bench.py times as e2e */
int bskenv_opnav_step_host(bskenv_opnav_handle *h, const int32_t *actions, double *obs, double *reward, uint8_t *done,
                           uint8_t *done_reason, double *debug);
int bskenv_opnav_state_dims(const bskenv_opnav_handle *h, int32_t *n_double_fields, int32_t *n_int_fields);
int bskenv_opnav_get_state(bskenv_opnav_handle *h, double *dstate_dev, int64_t *istate_dev, void *stream);
int bskenv_opnav_set_state(bskenv_opnav_handle *h, const double *dstate_dev, const int64_t *istate_dev, void *stream);
int bskenv_opnav_state_field(const char *name, int32_t *is_int);
/* [sum of returns, sum of lengths, episodes finished, by max_length, by numModes, env-steps, measurement updates,
 *  rejected filter updates] since the last call */
int bskenv_opnav_episode_stats(bskenv_opnav_handle *h, double *stats_host);
int64_t bskenv_opnav_launch_count(const bskenv_opnav_handle *h);
double bskenv_opnav_flops_per_step(const bskenv_opnav_handle *h);

#ifdef __cplusplus
}
#endif
#endif
