// bskenv.cu -- sm_100a kernels and the C ABI (include/bskenv.h) of the batched LEO environment step.
//
// Kernels:
//   leo_step_kernel   one thread = one spacecraft; ONE launch = one decision interval for all envs
//                     (replaces Basilisk ExecuteSimulation(), reference
//                     basilisk_env/simulators/leoPowerAttitudeSimulator.py:590-595, and the gym
//                     bookkeeping of basilisk_env/envs/leoPowerAttitudeEnvironment.py:65-145);
//                     warp-shuffle reduction of the episode statistics; optional in-kernel auto-reset.
//   leo_step_penv_kernel  the same body (leo_step_body) with per-env spacecraft parameters from a parameter pool.
//   leo_split_kernel  small batches: the same interval with the work of one env split over two warps (leo_split.cuh).
//   leo_reset_kernel  simulator construction + initial observation (reference ...Simulator.py:67-117,
//                     ...Environment.py:172-216) from explicit, stored or device-sampled ICs.
//   fp64_peak_kernel  DFMA microbenchmark = the roofline denominator.
// The lane bucketing before a step (bucket_count_kernel + bucket_fill_kernel) and the per-env state snapshot kernels
// (snapshot_gather_kernel, restore_scatter_kernel and their checks) are shared with the opNav batch (batch_common.cuh).
// There is no CPU path in this library.
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/bskenv.h"
#include "leo_core.cuh"
#include "leo_split.cuh"
#include "leo_host.h"
#include "batch_common.cuh"

#ifndef LEO_MIN_BLOCKS
#define LEO_MIN_BLOCKS 3        // resident blocks per SM: 3 x 128 threads x 168 registers
#endif
#define LEO_BUS_BYTES ((size_t)leo::LEO_NM * LEO_BLOCK * sizeof(double))   // shared-memory message bus of one block
#ifndef LEO_SPLIT_MAX_G
#define LEO_SPLIT_MAX_G 4       // groups per block of the two-warp organisation: 4 x 64 threads keep 255 registers per thread
#endif
#ifndef LEO_SPLIT_AUTO_G
#define LEO_SPLIT_AUTO_G 4      // ... and up to which it is selected automatically (groups <= SM count x this): measured on a
                                // B200 with one / two / four groups per block: 4096 envs 3.34 -> 2.39 ms, 8192 3.42 -> 2.49, 16384 3.76 -> 3.00
#endif
#define LEO_BUS_BYTES_PFIX ((size_t)leo::LEO_NM_PFIX * LEO_BLOCK * sizeof(double))   // ... of the planet-fixed gravity variant
#ifdef LEO_PENV_GLOBAL
#define LEO_BUS_BYTES_PENV LEO_BUS_BYTES                                               // ... of the per-env parameter kernel
#else
#define LEO_BUS_BYTES_PENV ((size_t)leo::LEO_NM_PENV * LEO_BLOCK * sizeof(double))
#endif

namespace {

enum { ST_RET = 0, ST_LEN, ST_COUNT, ST_WHEEL, ST_POWER, ST_DECAY, ST_MAXLEN, ST_STEPS, ST_N };

#ifdef LEO_MAXNREG
#define LEO_STEP_BOUNDS(MINB) __maxnreg__(LEO_MAXNREG)       // tuning builds: explicit register cap instead of an occupancy target
#else
#define LEO_STEP_BOUNDS(MINB) __launch_bounds__(LEO_BLOCK, MINB)
#endif

// Work distribution.  One warp steps one group of 32 consecutive envs through the whole decision interval and
// every group costs the same.  When there are more groups than resident warps (12 per SM: three 128-thread
// blocks of 168 registers), the grid is exactly one resident set of blocks and the warps pull groups from an
// atomic queue until it is empty: no block-granular waves, no warp waits for the slowest warp of its block, and
// the tail is spread over all SMs (131072 envs on 148 SMs: 16.15 ms with one block per 128 envs, 15.7 ms with
// the queue; an early-retiring third block per SM was measured as well and does not help).
//   sched[0] = queue head (zeroed before the launch)
// Work items of the queue are (chunk, group) pairs, chunk-major: the decision interval of a group is cut into n_chunks
// consecutive chunks (leo_core.cuh: leo_step_env; leo_host::step_chunks), so the tail of a launch is one chunk long instead
// of one interval long (131072 envs = 2.3 resident sets: the last 0.3 set used to run alone at one warp per sub-partition
// for 4.6 ms).  Chunk c of a group may start when chunk c - 1 has been published in progress[group] (release / acquire at
// GPU scope); its predecessor was handed out n_groups items earlier, so in practice nobody waits.  Without the queue
// (grid covers all groups) each warp runs the chunks of its own group back to back.
struct LeoSched { int *sched; int n_groups; int dynamic; int n_chunks; int *progress; const int32_t *perm; };

// Lane assignment of the throughput organisation.  The three modes run different flight software (hillPoint vs inertial3D;
// the desat chain, the thruster latch and the exact thruster steps only after action 2): a warp of mixed actions executes
// all of it, 180 times per interval.  Before the launch the envs are bucketed by action (batch_common.cuh:
// bucket_count_kernel + bucket_fill_kernel) and a warp takes 32 slots of the permutation: the state is gathered / scattered
// at the chunk boundaries (12 times per 1800 ticks), the tick loop diverges only in the at most three warps that straddle a
// bucket boundary.  Per-env arithmetic does not depend on the lane an env runs in: results are bit-identical with and
// without (tests/test_gpu_round2.py).  bucket[0..3] = sizes, bucket[4..7] = cursors, in bucket order: action 2 (the desat
// chain: the slowest warps), 0, 1, unknown -- the work queue hands out the long items first, so that the tail of a launch
// is made of the short ones.
struct LeoActionRank {
    const int32_t *actions;
    __device__ int operator()(int64_t e) const { const int a = actions[e]; return a == 2 ? 0 : (a == 0 ? 1 : (a == 1 ? 2 : 3)); }
};

__device__ __forceinline__ void chunk_publish(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" : : "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int chunk_peek(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// What follows the last chunk of a decision interval: results, per-env episode record, in-kernel auto-reset, episode statistics
// (warp-shuffle reduction, one atomic per warp and statistic).  Called by all 32 lanes of the warp that stepped the group.
// PA = ParEnv: the auto-reset also assigns the env's pool row for the new episode.
template <class PA = leo::ParBatch>
__device__ __forceinline__ void step_finish(const LeoParams &P, double *__restrict__ S, int64_t *__restrict__ I, double *__restrict__ ics,
                                            int64_t stride, int64_t e, bool valid, int lane, leo::StepOut &o, double *__restrict__ obs,
                                            double *__restrict__ reward, uint8_t *__restrict__ done, uint8_t *__restrict__ reason,
                                            double *__restrict__ term_obs, double *__restrict__ stats, double *__restrict__ ep_return,
                                            int64_t *__restrict__ ep_length, const LeoPool &pool = LeoPool{})
{
    double ep_ret = 0., ep_len = 0.;
    if (valid) {
        reward[e] = o.reward;
        done[e] = (uint8_t)o.done;
        reason[e] = (uint8_t)o.reason;
        if (o.done || ep_return) {
            ep_ret = S[(int64_t)F_EPRET * stride + e];
            ep_len = (double)I[(int64_t)I_STEP * stride + e];
        }
        if (ep_return) {       // ENV:130-136: info['episode'] = {'r': reward_total, 'l': curr_step (before its increment)}
            ep_return[e] = ep_ret;
            ep_length[e] = (int64_t)ep_len - 1;
        }
        if (o.done) {
            if (term_obs)
                for (int k = 0; k < 5; k++) term_obs[e * 5 + k] = o.ob[k];
            if (P.auto_reset) {
                // SB-VecEnv convention: the returned observation is the first one of the next episode
                int64_t ep = I[(int64_t)I_EPISODE * stride + e] + 1;
                I[(int64_t)I_EPISODE * stride + e] = ep;
                double ic[19];
                leo::sample_ic(P, P.first_env_index + e, ep, ic);
                for (int k = 0; k < 19; k++) ics[(int64_t)k * stride + e] = ic[k];
                if (!std::is_same<PA, leo::ParBatch>::value)
                    leo::pool_assign(pool, S, stride, e, leo::pool_row(pool, P.seed, P.first_env_index + e, ep));
                leo::leo_reset_env<PA>(P, S, I, stride, e, ic, o.ob);
            }
        }
        for (int k = 0; k < 5; k++) obs[e * 5 + k] = o.ob[k];
    }
    // episode statistics: warp-shuffle reduction, one atomic per warp and statistic
    if (stats) {
        const unsigned any_done = __ballot_sync(0xffffffffu, valid && o.done);
        if (any_done) {
            double v_ret = warp_sum(o.done ? ep_ret : 0.), v_len = warp_sum(o.done ? ep_len : 0.);
            int c_all = __popc(any_done);
            int c_w = __popc(__ballot_sync(0xffffffffu, valid && o.done && (o.reason & 2)));
            int c_p = __popc(__ballot_sync(0xffffffffu, valid && o.done && (o.reason & 4)));
            int c_d = __popc(__ballot_sync(0xffffffffu, valid && o.done && (o.reason & 8)));
            int c_m = __popc(__ballot_sync(0xffffffffu, valid && o.done && (o.reason & 1)));
            if (lane == 0) {
                atomicAdd(&stats[ST_RET], v_ret); atomicAdd(&stats[ST_LEN], v_len);
                atomicAdd(&stats[ST_COUNT], (double)c_all); atomicAdd(&stats[ST_WHEEL], (double)c_w);
                atomicAdd(&stats[ST_POWER], (double)c_p); atomicAdd(&stats[ST_DECAY], (double)c_d);
                atomicAdd(&stats[ST_MAXLEN], (double)c_m);
            }
        }
        const int c_valid = __popc(__ballot_sync(0xffffffffu, valid));
        if (lane == 0 && c_valid) atomicAdd(&stats[ST_STEPS], (double)c_valid);
    }
}

// One decision interval of the one-thread-per-env organisation, the body of both step kernels: work items from the queue
// or the warp's own group (LeoSched), slot -> env through the lane permutation, leo_step_env chunk by chunk with the
// chunk hand-over between work items, step_finish after the last chunk.  PA = the parameter accessor of leo_step_env
// (leo::ParBatch: the batch configuration; leo::ParEnv: per-env parameters, whose auto-reset assigns a row of `pool`).
// tid = threadIdx.x, read by the kernel: there the compiler knows its range from the launch bounds.
template <int NRW, int J2, bool DIAG, bool F32, class PA>
__device__ __forceinline__ void leo_step_body(unsigned tid, const LeoParams &P, const LeoParamsF &PF, const LeoPool &pool, double *__restrict__ S,
                                              int64_t *__restrict__ I, double *__restrict__ ics, int64_t stride, int64_t n,
                                              const int32_t *__restrict__ actions, double *__restrict__ obs, double *__restrict__ reward,
                                              uint8_t *__restrict__ done, uint8_t *__restrict__ reason, double *__restrict__ term_obs,
                                              double *__restrict__ stats, const LeoSched &sc, double *__restrict__ ep_return,
                                              int64_t *__restrict__ ep_length)
{
    extern __shared__ double bus_smem[];          // [LEO_NM (ParEnv: LEO_NM_PENV)][LEO_BLOCK]: per-thread message bus (leo_core.cuh: MBus)
    const int lane = tid & 31, warp = tid >> 5;
    leo::MBus bus;
    bus.p = nullptr;
    bus.a = (uint32_t)__cvta_generic_to_shared(bus_smem) + tid * (uint32_t)sizeof(double);
    for (bool more = true; more; more = sc.dynamic != 0) {
        int g, c_first = 0, c_end = sc.n_chunks;
        if (sc.dynamic) {
            g = 0;
            if (lane == 0) g = atomicAdd(&sc.sched[0], 1);
            g = __shfl_sync(0xffffffffu, g, 0);
            if (g >= sc.n_groups * sc.n_chunks) break;
            c_first = g / sc.n_groups; c_end = c_first + 1;
            g -= c_first * sc.n_groups;
            if (c_first > 0) {                                  // chunk c_first - 1 of this group must be in memory
                if (lane == 0)
                    while (chunk_peek(sc.progress + g) < c_first) __nanosleep(200);
                __syncwarp();
            }
        } else {
            g = blockIdx.x * (LEO_BLOCK / 32) + warp;
        }
        const int64_t slot = (int64_t)g * 32 + lane;
        const bool valid = slot < n;
        const int64_t e = (valid && sc.perm) ? (int64_t)sc.perm[slot] : slot;     // envs of one action per warp (see LeoSched)
        leo::StepOut o;
        o.done = 0; o.reason = 0; o.reward = 0.;
        for (int c = c_first; c < c_end; c++) {
            if (valid) leo::leo_step_env<NRW, J2, DIAG, F32, PA>(P, S, I, stride, e, bus, actions[e], o, PF, c, sc.n_chunks);
            if (c + 1 < sc.n_chunks) {                          // chunk boundary inside the interval: publish and go on
                if (sc.dynamic) {
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) chunk_publish(sc.progress + g, c + 1);
                }
                continue;
            }
            step_finish<PA>(P, S, I, ics, stride, e, valid, lane, o, obs, reward, done, reason, term_obs, stats, ep_return, ep_length, pool);
        }   // chunks of this item
        __syncwarp();
    }
}

// MINB = resident blocks per SM the register allocation is made for.  LEO_MIN_BLOCKS (3 blocks x 128 threads x 168 registers,
// a few spilled values) is the throughput organisation.  MINB = 1 is the SMALL-BATCH organisation (BASELINE configs[1], 4096
// envs): when the whole batch fits one block per SM anyway, every warp runs alone on its SM sub-partition at its dependent-
// issue latency, occupancy buys nothing and the full register file (255 registers, nothing spilled onto the dependency
// chain) is worth 20 % (DESIGN.md section 5b).
template <int NRW, int J2, bool DIAG, bool F32, int MINB>
__global__ void LEO_STEP_BOUNDS(MINB)
leo_step_kernel(const __grid_constant__ LeoParams P, const __grid_constant__ LeoParamsF PF, double *__restrict__ S, int64_t *__restrict__ I, double *__restrict__ ics,
                int64_t stride, int64_t n, const int32_t *__restrict__ actions, double *__restrict__ obs,
                double *__restrict__ reward, uint8_t *__restrict__ done, uint8_t *__restrict__ reason,
                double *__restrict__ term_obs, double *__restrict__ stats, const LeoSched sc,
                double *__restrict__ ep_return, int64_t *__restrict__ ep_length)
{
    leo_step_body<NRW, J2, DIAG, F32, leo::ParBatch>(threadIdx.x, P, PF, LeoPool{}, S, I, ics, stride, n, actions, obs, reward, done, reason, term_obs,
                                                     stats, sc, ep_return, ep_length);
}

// The same organisation with per-env spacecraft parameters (bskenv_set_param_pool): leo_step_env<..., ParEnv> reads each
// env's derived values from the parameter block behind its state (stage-rate values through its bus column, which is
// LEO_NM_PENV fields long), and the auto-reset assigns the pool row of the new episode.  Built for the reference
// configuration only (three wheels, DIAG, FP64).  A kernel of its own rather than a template argument of leo_step_kernel,
// so that the batch-global kernels stay exactly as they are.
template <int NRW, int J2, bool DIAG, int MINB>
__global__ void LEO_STEP_BOUNDS(MINB)
leo_step_penv_kernel(const __grid_constant__ LeoParams P, const LeoPool pool, double *__restrict__ S, int64_t *__restrict__ I,
                     double *__restrict__ ics, int64_t stride, int64_t n, const int32_t *__restrict__ actions,
                     double *__restrict__ obs, double *__restrict__ reward, uint8_t *__restrict__ done, uint8_t *__restrict__ reason,
                     double *__restrict__ term_obs, double *__restrict__ stats, const LeoSched sc, double *__restrict__ ep_return,
                     int64_t *__restrict__ ep_length)
{
    static_assert(NRW == 3 && DIAG && J2 != 2, "per-env parameters are built for the reference configuration");
    leo_step_body<NRW, J2, DIAG, false, leo::ParEnv>(threadIdx.x, P, LeoParamsF(), pool, S, I, ics, stride, n, actions, obs, reward, done, reason,
                                                     term_obs, stats, sc, ep_return, ep_length);
}

// Ragged batches in the split organisation: the lanes of the last group that have no env step a DUPLICATE of the last env
// (its state copied into the padding columns [n, stride) of the state blocks before every launch, the same action), so that
// every lane of a group takes the same barriers through the same code; nothing they compute leaves the padding columns.
__global__ void leo_pad_kernel(double *__restrict__ S, int64_t *__restrict__ I, int64_t stride, int64_t n)
{
    const int pads = (int)(stride - n);
    for (int t = threadIdx.x; t < (LEO_ND + LEO_NI) * pads; t += blockDim.x) {
        const int f = t / pads;
        const int64_t e = n + t % pads;
        if (f < LEO_ND) S[(int64_t)f * stride + e] = S[(int64_t)f * stride + n - 1];
        else I[(int64_t)(f - LEO_ND) * stride + e] = I[(int64_t)(f - LEO_ND) * stride + n - 1];
    }
}

// SMALL-BATCH organisation (leo_split.cuh): two warps per group of 32 envs -- a dynamics warp and a companion warp (flight
// software + EnvTask) -- on different SM sub-partitions of one block, G groups per block (block = 64 G threads; the G
// dynamics warps come first so that with G = 4 every sub-partition hosts one warp of each kind).  Every lane of a group
// steps an env (the spare lanes of a ragged last group a duplicate of the last one, see leo_pad_kernel): all 64 threads of a
// pair take every named barrier.  Chunks of the interval run back to back exactly as in the static path of leo_step_kernel.
template <int NRW, int J2, bool DIAG>
__global__ void __launch_bounds__(256, 1)
leo_split_kernel(const __grid_constant__ LeoParams P, double *__restrict__ S, int64_t *__restrict__ I, double *__restrict__ ics,
                 int64_t stride, int64_t n, const int32_t *__restrict__ actions, double *__restrict__ obs,
                 double *__restrict__ reward, uint8_t *__restrict__ done, uint8_t *__restrict__ reason,
                 double *__restrict__ term_obs, double *__restrict__ stats, int n_groups, int n_chunks,
                 double *__restrict__ ep_return, int64_t *__restrict__ ep_length)
{
    extern __shared__ double bus_smem[];          // [LEO_NM][LEO_BLOCK] message bus, then [SPLIT_NF][LEO_BLOCK] mailbox
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, G = blockDim.x >> 6;
    const int role = warp / G, q = warp - role * G;             // 0 = dynamics, 1 = companion; pair index within the block
    const int g = blockIdx.x * G + q;
    if (g >= n_groups) return;                                  // both warps of the pair leave: their barriers are never used
    const uint32_t col = (uint32_t)(q * 32 + lane) * (uint32_t)sizeof(double);
    leo::MBus bus, box;
    bus.p = box.p = nullptr;
    bus.a = (uint32_t)__cvta_generic_to_shared(bus_smem) + col;
    box.a = bus.a + (uint32_t)LEO_BUS_BYTES;
    const int bar = 1 + 2 * q;                                  // named barriers bar (TICK) and bar + 1 (FSW) of this pair
    const int64_t e = (int64_t)g * 32 + lane;
    const bool valid = e < n;
    const int action = actions[valid ? e : n - 1];
    if (role == 1) {
        for (int c = 0; c < n_chunks; c++) leo::split_env<NRW>(P, S, I, stride, e, bus, box, bar, action, c, n_chunks);
        return;
    }
    leo::StepOut o;
    o.done = 0; o.reason = 0; o.reward = 0.;
    for (int c = 0; c < n_chunks; c++) leo::split_dyn<NRW, J2, DIAG>(P, S, I, stride, e, bus, box, bar, action, o, c, n_chunks);
    step_finish(P, S, I, ics, stride, e, valid, lane, o, obs, reward, done, reason, term_obs, stats, ep_return, ep_length);
}

// mode 0: explicit ICs (row-major [n][19]); 1: stored ICs (reset_init); 2: device-sampled ICs, or a row of the IC pool.
// With a parameter pool (pool.n_rows > 0) modes 0 and 2 assign the env's pool row; mode 1 keeps it.  Mode 2 is also the
// auto-reset of a handle with an IC pool (launch_step: the step kernel runs without its in-kernel reset, then this kernel
// with mask = done): the same sequence as step_finish -- episode + 1, ICs, parameter row, leo_reset_env, observation.
// The parameter row is picked before the IC row, which BSKENV_ICS_PARAM_ROW takes from it.
__global__ void __launch_bounds__(256)
leo_reset_kernel(const __grid_constant__ LeoParams P, double *__restrict__ S, int64_t *__restrict__ I, double *__restrict__ ics,
                 int64_t stride, int64_t n, int mode, const double *__restrict__ ics_in, const uint8_t *__restrict__ mask,
                 double *__restrict__ obs, const LeoPool pool, const IcPool icp)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (mask && !mask[e]) return;
    const int64_t ge = P.first_env_index + e;
    int64_t ep = I[(int64_t)I_EPISODE * stride + e];
    if (mode == 2) I[(int64_t)I_EPISODE * stride + e] = ++ep;
    const int64_t prow = (pool.n_rows > 0 && mode != 1) ? leo::pool_row(pool, P.seed, ge, ep) : -1;
    double ic[19];
    reset_ics(mode, ics_in, ics, stride, e, ge, P.seed, ep, prow, icp, [&](double (&x)[19]) { leo::sample_ic(P, ge, ep, x); }, ic);
    double ob[5];
    if (pool.n_rows > 0) {
        if (mode != 1) leo::pool_assign(pool, S, stride, e, prow);
        leo::leo_reset_env<leo::ParEnv>(P, S, I, stride, e, ic, ob);
    } else {
        leo::leo_reset_env(P, S, I, stride, e, ic, ob);
    }
    if (obs)
        for (int k = 0; k < 5; k++) obs[e * 5 + k] = ob[k];
}

// bskenv_get_env_params: the reference values and the pool row of every env (the batch configuration, row -1, when the
// parameter block is not in use)
struct ParamRow { double v[BSKENV_PARAM_DIM]; };
__global__ void gather_params_kernel(const double *__restrict__ S, int64_t stride, int64_t n, int live, const ParamRow batch,
                                     double *__restrict__ out, int32_t *__restrict__ row)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int k = 0; k < BSKENV_PARAM_DIM; k++) out[e * BSKENV_PARAM_DIM + k] = live ? S[(int64_t)(LEO_ND + PE_RAW + k) * stride + e] : batch.v[k];
    if (row) row[e] = live ? (int32_t)S[(int64_t)(LEO_ND + PE_ROW) * stride + e] : -1;
}

// Snapshot records of the LEO batch (batch_common.cuh: SnapLayout; include/bskenv.h: BSKENV_SNAP_*).  The observation of a
// restored env is the one its source returned last: the reset's initial observation of the stored ICs while curr_step is 0
// (fresh from a reset or an auto-reset), else the last simulator observation F_OBS normalised as at the end of leo_step_env.
struct LeoSnap {
    using L = SnapLayout<BSKENV_SNAPSHOT_KIND_LEO, LEO_ND, LEO_NI, BSKENV_IC_DIM, LEO_NPD, PE_ROW, I_EPISODE>;
    using Params = LeoParams;
    enum : int { OD = BSKENV_OBS_DIM };
    __device__ static void obs(const LeoParams &P, const double *row, double *ob)
    {
        if (__double_as_longlong(row[L::OFF_I + I_STEP]) == 0) {
            double ic[19];
            for (int k = 0; k < 19; k++) ic[k] = row[L::OFF_IC + k];
            leo::reset_obs(P, ic, leo::ic_w4(ic), ob);
        } else {
            const double *f = row + L::OFF_S + F_OBS;
            ob[0] = f[0]; ob[1] = f[1]; ob[2] = f[2] / P.wheel_limit; ob[3] = f[3] / P.power_max; ob[4] = f[4];
        }
    }
};
static_assert(LeoSnap::L::OFF_S == BSKENV_SNAP_S && LeoSnap::L::OFF_I == BSKENV_SNAP_I && LeoSnap::L::OFF_IC == BSKENV_SNAP_ICS &&
              LeoSnap::L::OFF_P == BSKENV_SNAP_PARAMS && LeoSnap::L::OFF_ROW == BSKENV_SNAP_ICROW && LeoSnap::L::W == BSKENV_SNAPSHOT_W,
              "include/bskenv.h: the LEO record layout");

// The configuration fingerprint of snapshot records: the named fields of bskenv_config except the reserved words and
// auto_reset (handle policy)
static uint64_t leo_fingerprint(const bskenv_config &c)
{
    Fnv64 f;
    f.add(c.abi_version); f.add(c.dynRate); f.add(c.fswRate); f.add(c.step_duration);
    f.add(c.mass); f.add(c.width); f.add(c.depth); f.add(c.height);
    f.add(c.planetRadius); f.add(c.baseDensity); f.add(c.scaleHeight); f.add(c.disturbance_magnitude);
    f.add(c.nHat_B); f.add(c.panelArea); f.add(c.panelEfficiency); f.add(c.powerDraw); f.add(c.storageCapacity);
    f.add(c.sigma_R0N); f.add(c.K); f.add(c.Ki); f.add(c.P); f.add(c.hs_min); f.add(c.thrMinFireTime);
    f.add(c.thrForceSign); f.add(c.maxCounterValue); f.add(c.max_length);
    f.add(c.wheel_limit_rpm); f.add(c.power_max); f.add(c.failure_penalty);
    f.add(c.use_j2); f.add(c.hill_cel_pun); f.add(c.rw_set); f.add(c.precision);
    return f.h;
}

// 8 independent DFMA chains per thread, everything in registers
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *out, int iters, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    out[(int64_t)blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

thread_local std::string g_create_error;

}  // namespace

// The shared core (batch_common.cuh: BatchCore) and what only the LEO batch has.  The host-buffer step is complete when
// bskenv_step_host[_wait] returns; its staging slots are actions, obs, reward, done, reason, ep_return, ep_length, term_obs.
struct bskenv_handle : BatchCore {
    bskenv_config cfg;
    LeoParams P;
    LeoParamsF PF;
    int *sched;                 // work queue head of the step kernel
    int32_t *perm; int *bucket; // lane assignment of the throughput organisation (envs bucketed by action), bucket sizes / cursors
    void *pend_user[8]; size_t pend_bytes[8];   // the staged results of the host-buffer step in flight
    const char *kernel_name;    // the step-kernel instantiation of the last launch
    int organisation;           // BSKENV_ORG_*: 0 auto, 1 one thread per env, 2 two warps per env group (small batches)
    LeoPool pool;               // loaded parameter pool (n_rows = 0: none); rows in device memory
    int s_fields;               // double fields allocated per env in S: LEO_ND, or LEO_ND + LEO_NPD once a pool was loaded
};
#define NO_HOST_PENDING(h, what)                                                                                        \
    do {                                                                                                                \
        if ((h)->host_pending) { (h)->err = what ": a host-buffer step is in flight (call bskenv_step_host_wait first)"; return BSKENV_EINVAL; } \
    } while (0)

// Auto-reset of a handle with an IC pool: after the step kernel (which ran without its in-kernel reset), the reset kernel in
// its sampling mode over the envs the step finished -- mask = the step's `done`, obs = the step's `obs` (the terminal
// observation there is replaced by the first one of the new episode; term_obs, the episode record and the statistics were
// written by the step kernel before, exactly as before an in-kernel reset).  On the host-buffer paths both are the buffers
// the step kernel wrote: mapped caller memory or the staging blocks, which are copied back after this launch.
static int launch_follow_reset(bskenv_handle *h, const uint8_t *done, double *obs, cudaStream_t st)
{
    leo_reset_kernel<<<env_grid(h), 256, 0, st>>>(h->P, h->S, h->I, h->ics, h->stride, h->n, 2, nullptr, done, obs, h->pool, h->icp);
    CU_TRY(h, cudaGetLastError());
    h->launches++;
    return BSKENV_OK;
}

static int launch_step(bskenv_handle *h, const int32_t *act, double *obs, double *rew, uint8_t *done, uint8_t *reason,
                       double *term_obs, cudaStream_t st, double *ep_return = nullptr, int64_t *ep_length = nullptr)
{
    // With an IC pool the step kernels run on a copy of the parameter block without auto_reset (read only by step_finish) and
    // launch_follow_reset does the reset: every organisation and configuration, the step kernels as they are.
    const bool follow = h->icp.n_rows > 0 && h->P.auto_reset;
    LeoParams P_nr;
    if (follow) { P_nr = h->P; P_nr.auto_reset = 0; }
    const LeoParams &PK = follow ? P_nr : h->P;
    const int wpb = LEO_BLOCK / 32;
    const int64_t groups = (h->n + 31) / 32;
    const int resident = h->sm_count * LEO_MIN_BLOCKS;          // blocks of one full resident set
    int grid = (int)((groups + wpb - 1) / wpb);
#ifndef LEO_SMALL_BLOCKS
#define LEO_SMALL_BLOCKS 2      // two 128-thread blocks of the 255-register build fit one SM; measured against the 168-register
#endif                          // build: 18976 envs 4.35 -> 4.12 ms, 32768 envs 5.31 -> 5.02 ms (one block per SM before r02c)
    const bool small = grid <= h->sm_count * LEO_SMALL_BLOCKS;  // at most LEO_SMALL_BLOCKS blocks per SM: the 255-register build
    LeoSched sc;
    sc.sched = h->sched; sc.n_groups = (int)groups; sc.dynamic = 0;
    sc.n_chunks = leo_host::step_chunks(h->P); sc.progress = h->sched + 4; sc.perm = nullptr;
    if (grid > resident) {
        sc.dynamic = 1;
        grid = resident;
        CU_TRY(h, cudaMemsetAsync(h->sched, 0, sizeof(int) * (size_t)(4 + groups), st));    // queue head + chunk progress per group
    }
    // two warps per env group: whole groups only, the two configurations the small-batch kernels are built for
    const bool penv = h->pool.n_rows > 0;                      // per-env parameters: one thread per env at every batch size
    const bool split_cfg = !penv && !h->P.grav_pfix && !h->P.mixed && ((h->P.nrw == 3 && !h->cfg.use_j2 && h->P.diag) || (h->P.nrw == 4 && h->cfg.use_j2));
    const bool split_fit = split_cfg && groups <= (int64_t)h->sm_count * LEO_SPLIT_MAX_G;
    if (h->organisation == BSKENV_ORG_SPLIT && !split_fit) {
        h->err = "bskenv_step: the split organisation takes at most 128 * SM-count envs, FP64, and the reference or the stress configuration";
        return BSKENV_EINVAL;
    }
    if (split_fit && (h->organisation == BSKENV_ORG_SPLIT || (h->organisation == BSKENV_ORG_AUTO && groups <= (int64_t)h->sm_count * LEO_SPLIT_AUTO_G))) {
        int G = (int)((groups + h->sm_count - 1) / h->sm_count);
        G = G <= 1 ? 1 : (G == 2 ? 2 : 4);
        const int dgrid = (int)((groups + G - 1) / G);
        if (h->n % 32) leo_pad_kernel<<<1, 256, 0, st>>>(h->S, h->I, h->stride, h->n);
        const size_t smem = LEO_BUS_BYTES + LEO_SPLIT_BOX_BYTES;
        if (h->P.nrw == 3) {
            CU_TRY(h, allow_dynamic_smem<leo_split_kernel<3, 0, true>>(h->device, smem));
            h->kernel_name = "leo_split_kernel<3,0,true>";
            leo_split_kernel<3, 0, true><<<dgrid, 64 * G, smem, st>>>(PK, h->S, h->I, h->ics, h->stride, h->n, act, obs, rew, done, reason, term_obs,
                                                                 h->stats, (int)groups, sc.n_chunks, ep_return, ep_length);
        } else {
            CU_TRY(h, allow_dynamic_smem<leo_split_kernel<4, 1, false>>(h->device, smem));
            h->kernel_name = "leo_split_kernel<4,1,false>";
            leo_split_kernel<4, 1, false><<<dgrid, 64 * G, smem, st>>>(PK, h->S, h->I, h->ics, h->stride, h->n, act, obs, rew, done, reason, term_obs,
                                                                  h->stats, (int)groups, sc.n_chunks, ep_return, ep_length);
        }
        CU_TRY(h, cudaGetLastError());
        h->launches++;
        if (follow) { const int rc = launch_follow_reset(h, done, obs, st); if (rc) return rc; }
        if (st != h->own_stream || !st) CU_TRY(h, note_launch(h, st));
        return BSKENV_OK;
    }
    if (!small && h->organisation != BSKENV_ORG_THREAD_INDEX) {      // bucket the envs by action (LeoSched)
        const int bgrid = (int)((h->n + 255) / 256);
        const LeoActionRank rank{act};
        CU_TRY(h, cudaMemsetAsync(h->bucket, 0, sizeof(int) * 8, st));
        bucket_count_kernel<4><<<bgrid, 256, 0, st>>>(h->n, rank, h->bucket);
        bucket_fill_kernel<4><<<bgrid, 256, 0, st>>>(h->n, rank, h->bucket, h->perm);
        sc.perm = h->perm;
        h->launches += 2;
    }
#define LEO_STR_(x) #x
#define LEO_STR(x) LEO_STR_(x)
    // KERNEL<<<...>>>(PK, ARG2, ...): ARG2 = the reduced-precision parameter block of leo_step_kernel or the parameter pool of
    // leo_step_penv_kernel
#define LEO_LAUNCH_K(NAME, SMEM, ARG2, ...)                                                                                 \
    do {                                                                                                                   \
        CU_TRY(h, allow_dynamic_smem<__VA_ARGS__>(h->device, SMEM));                                                       \
        h->kernel_name = NAME;                                                                                             \
        __VA_ARGS__<<<grid, LEO_BLOCK, SMEM, st>>>(PK, ARG2, h->S, h->I, h->ics, h->stride, h->n, act, obs, rew, done, reason, \
                                                   term_obs, h->stats, sc, ep_return, ep_length);                         \
    } while (0)
#define LEO_LAUNCH_B(NRW, J2, DIAG, F32, MINB)                                                                         \
    LEO_LAUNCH_K("leo_step_kernel<" #NRW "," #J2 "," #DIAG "," #F32 "," LEO_STR(MINB) ">", (J2) == 2 ? LEO_BUS_BYTES_PFIX : LEO_BUS_BYTES, \
                 h->PF, leo_step_kernel<NRW, J2, DIAG, F32, MINB>)
#define LEO_LAUNCH(NRW, J2, DIAG, F32) LEO_LAUNCH_B(NRW, J2, DIAG, F32, LEO_MIN_BLOCKS)
#define LEO_LAUNCH_PENV(J2)                                                                                            \
    LEO_LAUNCH_K("leo_step_penv_kernel<3," #J2 ",true," LEO_STR(LEO_MIN_BLOCKS) ">", LEO_BUS_BYTES_PENV, h->pool,          \
                 leo_step_penv_kernel<3, J2, true, LEO_MIN_BLOCKS>)
    if (penv) { if (h->cfg.use_j2) LEO_LAUNCH_PENV(1); else LEO_LAUNCH_PENV(0); }    // (bskenv_set_param_pool checks the configuration)
    // small-batch organisation: built for the reference configuration and for the stress configuration
    else if (small &&!h->P.grav_pfix && !h->P.mixed && h->P.nrw == 3 && !h->cfg.use_j2 && h->P.diag) LEO_LAUNCH_B(3, 0, true, false, 1);
    else if (small && !h->P.grav_pfix && !h->P.mixed && h->P.nrw == 4 && h->cfg.use_j2) LEO_LAUNCH_B(4, 1, false, false, 1);
    else
    if (h->P.grav_pfix) {     // SURVEY 8(f)-4: degree-2 field in the planet-fixed frame (general EOM path)
        if (h->P.nrw == 4) LEO_LAUNCH(4, 2, false, false);
        else if (h->P.diag) LEO_LAUNCH(3, 2, true, false);
        else LEO_LAUNCH(3, 2, false, false);
    }
    else if (h->P.mixed) {         // mixed precision: built for the stress configuration and the reference configuration
        if (h->P.nrw == 4 && h->cfg.use_j2) LEO_LAUNCH(4, 1, false, true);
        else LEO_LAUNCH(3, 0, true, true);
    }
    else if (h->P.nrw == 4) { if (h->cfg.use_j2) LEO_LAUNCH(4, 1, false, false); else LEO_LAUNCH(4, 0, false, false); }
    else if (h->cfg.use_j2) { if (h->P.diag) LEO_LAUNCH(3, 1, true, false); else LEO_LAUNCH(3, 1, false, false); }
    else                    { if (h->P.diag) LEO_LAUNCH(3, 0, true, false); else LEO_LAUNCH(3, 0, false, false); }
#undef LEO_LAUNCH
#undef LEO_LAUNCH_B
#undef LEO_LAUNCH_PENV
#undef LEO_LAUNCH_K
    CU_TRY(h, cudaGetLastError());
    h->launches++;
    if (follow) { const int rc = launch_follow_reset(h, done, obs, st); if (rc) return rc; }
    if (st != h->own_stream || !st) CU_TRY(h, note_launch(h, st));
    return BSKENV_OK;
}

extern "C" {

int bskenv_abi_version(void) { return BSKENV_ABI_VERSION; }
void bskenv_default_config(bskenv_config *cfg) { leo_host::default_config(cfg); }
const char *bskenv_last_error(const bskenv_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }
int64_t bskenv_num_envs(const bskenv_handle *h) { return h ? h->n : 0; }
int64_t bskenv_launch_count(const bskenv_handle *h) { return h ? h->launches : 0; }
const char *bskenv_kernel_name(const bskenv_handle *h) { return (h && h->kernel_name) ? h->kernel_name : ""; }
double bskenv_flops_per_step(const bskenv_handle *h) { return h ? leo_host::flops_per_step(h->P) : 0.0; }

int bskenv_set_organisation(bskenv_handle *h, int organisation)
{
    if (!h) return BSKENV_EINVAL;
    if (organisation < BSKENV_ORG_AUTO || organisation > BSKENV_ORG_THREAD_INDEX) { h->err = "bskenv_set_organisation: unknown organisation"; return BSKENV_EINVAL; }
    if (organisation == BSKENV_ORG_SPLIT && h->pool.n_rows > 0) { h->err = "bskenv_set_organisation: the split organisation has no per-env parameters (a parameter pool is loaded)"; return BSKENV_EINVAL; }
    h->organisation = organisation;
    return BSKENV_OK;
}

int bskenv_create(const bskenv_config *cfg, int device, int64_t n_envs, int64_t first_env_index, bskenv_handle **out)
{
    const int rc = check_create("bskenv_create", cfg && out && n_envs > 0, device, g_create_error);
    if (rc) return rc;
    bskenv_handle *h = new bskenv_handle();
    h->cfg = *cfg;
    std::string perr = leo_host::build_params(*cfg, h->P);
    if (!perr.empty()) { g_create_error = "bskenv_create: " + perr; delete h; return BSKENV_EINVAL; }
    if (h->P.mixed && !((h->P.nrw == 4 && cfg->use_j2) || (h->P.nrw == 3 && !cfg->use_j2 && h->P.diag))) {
        g_create_error = "bskenv_create: precision = 1 is built for the reference configuration and for the stress configuration (rw_set = 1, use_j2 = 1)";
        delete h; return BSKENV_EINVAL;
    }
    leo_host::build_params_f(h->P, h->PF);
    h->P.first_env_index = first_env_index;
    h->fingerprint = leo_fingerprint(*cfg);
    h->s_fields = LEO_ND;       // (the handle is zero-initialised: no pools, BSKENV_ORG_AUTO)
    cudaError_t e = core_alloc(h, device, n_envs, LEO_ND, LEO_NI, 19, ST_N);
    if (e == cudaSuccess) e = cudaMalloc(&h->sched, sizeof(int) * (size_t)(4 + (n_envs + 31) / 32));
    if (e == cudaSuccess) e = cudaMalloc(&h->perm, sizeof(int32_t) * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->bucket, sizeof(int) * 8);
    if (e != cudaSuccess) {
        g_create_error = std::string("bskenv_create: ") + cudaGetErrorString(e);
        bskenv_destroy(h);
        return BSKENV_ECUDA;
    }
    *out = h;
    return BSKENV_OK;
}

int bskenv_destroy(bskenv_handle *h)
{
    if (!h) return BSKENV_OK;
    cudaSetDevice(h->device);
    cudaFree(h->sched); cudaFree(h->perm); cudaFree(h->bucket);
    cudaFree((void *)h->P.eph_sun.coef); cudaFree((void *)h->P.eph_orient.coef); cudaFree((void *)h->pool.rows);
    core_free(h);
    delete h;
    return BSKENV_OK;
}

int bskenv_set_gravity_degree2(bskenv_handle *h, int enable, const double *cbar)
{
    if (!h) return BSKENV_EINVAL;
    if (!enable) { h->P.grav_pfix = 0; return BSKENV_OK; }
    if (h->P.mixed) { h->err = "bskenv_set_gravity_degree2: not built for precision = 1"; return BSKENV_EINVAL; }
    if (h->pool.n_rows > 0) { h->err = "bskenv_set_gravity_degree2: not built with per-env parameters (a parameter pool is loaded)"; return BSKENV_EINVAL; }
    leo_host::set_degree2(h->P, cbar);
    return BSKENV_OK;
}

int bskenv_set_ephemeris(bskenv_handle *h, int kind, double t0, double seg_len, int n_seg, int n_coef, const double *coef)
{
    if (!h || kind < 0 || kind > 1) return BSKENV_EINVAL;
    // an episode runs from sim time 0 to (max_length + 1) decision intervals: the table has to cover it
    const double t_end = ((double)h->P.max_length + 1.0) * (double)h->P.step_ns * 1e-9;   // max_length may be INT_MAX
    return set_ephemeris(h, "bskenv_set_ephemeris", kind == 0 ? h->P.eph_sun : h->P.eph_orient, t_end, t0, seg_len, n_seg, n_coef, coef);
}

int bskenv_set_param_pool(bskenv_handle *h, int n_rows, const double *rows_host, int assign)
{
    if (!h) return BSKENV_EINVAL;
    NO_HOST_PENDING(h, "bskenv_set_param_pool");
    if (n_rows < 0 || (n_rows > 0 && !rows_host)) { h->err = "bskenv_set_param_pool: bad row count or null rows"; return BSKENV_EINVAL; }
    if (h->icp.n_rows > 0 && h->icp.assign == BSKENV_ICS_PARAM_ROW && n_rows != h->icp.n_rows) {
        h->err = "bskenv_set_param_pool: an IC pool of " + std::to_string(h->icp.n_rows) +
                 " rows is paired with the parameter pool (BSKENV_ICS_PARAM_ROW): unload it before changing the row count or unloading";
        return BSKENV_EINVAL;
    }
    if (n_rows > 0) {
        if (assign != BSKENV_PARAMS_BY_INDEX && assign != BSKENV_PARAMS_PER_EPISODE) { h->err = "bskenv_set_param_pool: unknown assignment mode"; return BSKENV_EINVAL; }
        if (h->P.nrw != 3 || !h->P.diag) { h->err = "bskenv_set_param_pool: per-env parameters are built for the three-wheel reference spacecraft (rw_set = 0)"; return BSKENV_EINVAL; }
        if (h->P.mixed) { h->err = "bskenv_set_param_pool: per-env parameters are not built for precision = 1"; return BSKENV_EINVAL; }
        if (h->P.grav_pfix) { h->err = "bskenv_set_param_pool: per-env parameters are not built for the degree-2 field"; return BSKENV_EINVAL; }
        if (h->organisation == BSKENV_ORG_SPLIT) { h->err = "bskenv_set_param_pool: the split organisation has no per-env parameters"; return BSKENV_EINVAL; }
    }
    std::vector<double> rows((size_t)LEO_NPD * n_rows), one(LEO_NPD);
    for (int r = 0; r < n_rows; r++) {
        const std::string err = leo_host::param_row_build(h->cfg, rows_host + (size_t)r * BSKENV_PARAM_DIM, (double)r, one.data());
        if (!err.empty()) { h->err = "bskenv_set_param_pool: row " + std::to_string(r) + ": " + err; return BSKENV_EINVAL; }
        for (int f = 0; f < LEO_NPD; f++) rows[(size_t)f * n_rows + r] = one[f];
    }
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());                         // a launch in flight may still read the old pool or the state block
    cudaFree((void *)h->pool.rows);
    h->pool.rows = nullptr;
    const bool was_loaded = h->pool.n_rows > 0;
    h->pool.n_rows = 0;
    if (n_rows == 0) return BSKENV_OK;                          // unloaded: the batch configuration, the batch-global kernels
    if (h->s_fields < LEO_ND + LEO_NPD) {                       // first pool of this handle: room for the parameter block
        double *S2 = nullptr;
        CU_TRY(h, cudaMalloc(&S2, sizeof(double) * (LEO_ND + LEO_NPD) * h->stride));
        CU_TRY(h, cudaMemcpy(S2, h->S, sizeof(double) * LEO_ND * h->stride, cudaMemcpyDeviceToDevice));
        cudaFree(h->S);
        h->S = S2; h->s_fields = LEO_ND + LEO_NPD;
    }
    if (!was_loaded) {                                          // running envs keep the batch values until their next reset
        double raw[BSKENV_PARAM_DIM];
        leo_host::param_row_get(h->cfg, raw);
        leo_host::param_row_derive(h->P, raw, -1.0, one.data());
        std::vector<double> blk((size_t)LEO_NPD * h->stride);
        for (int f = 0; f < LEO_NPD; f++)
            for (int64_t e = 0; e < h->stride; e++) blk[(size_t)f * h->stride + e] = one[f];
        CU_TRY(h, cudaMemcpy(h->S + (size_t)LEO_ND * h->stride, blk.data(), sizeof(double) * blk.size(), cudaMemcpyHostToDevice));
    }
    double *d_rows = nullptr;
    CU_TRY(h, cudaMalloc(&d_rows, sizeof(double) * rows.size()));
    CU_TRY(h, cudaMemcpy(d_rows, rows.data(), sizeof(double) * rows.size(), cudaMemcpyHostToDevice));
    h->pool.rows = d_rows; h->pool.n_rows = n_rows; h->pool.assign = assign;
    return BSKENV_OK;
}

int bskenv_get_env_params(bskenv_handle *h, double *params_dev, int32_t *row_dev, void *stream)
{
    if (!h || !params_dev) { if (h) h->err = "bskenv_get_env_params: null params"; return BSKENV_EINVAL; }
    CU_TRY(h, cudaSetDevice(h->device));
    ParamRow batch;
    leo_host::param_row_get(h->cfg, batch.v);
    gather_params_kernel<<<(int)((h->n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->S, h->stride, h->n, h->pool.n_rows > 0 ? 1 : 0,
                                                                                      batch, params_dev, row_dev);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

int bskenv_set_ic_pool(bskenv_handle *h, int n_rows, const double *ics_host, int assign)
{
    if (!h) return BSKENV_EINVAL;
    NO_HOST_PENDING(h, "bskenv_set_ic_pool");
    return set_ic_pool(h, "bskenv_set_ic_pool", n_rows, ics_host, BSKENV_IC_DIM, assign, [&]() -> std::string {
        if (assign != BSKENV_ICS_BY_INDEX && assign != BSKENV_ICS_PER_EPISODE && assign != BSKENV_ICS_PARAM_ROW)
            return "bskenv_set_ic_pool: unknown assignment mode";
        if (assign == BSKENV_ICS_PARAM_ROW && h->pool.n_rows != n_rows)
            return "bskenv_set_ic_pool: BSKENV_ICS_PARAM_ROW needs a loaded parameter pool of the same row count (" +
                   std::to_string(n_rows) + " IC rows, " + std::to_string(h->pool.n_rows) + " parameter rows)";
        return "";
    });
}

int bskenv_get_ic_rows(bskenv_handle *h, int32_t *rows_dev, void *stream)
{
    return h ? get_ic_rows(h, "bskenv_get_ic_rows", I_EPISODE, rows_dev, stream) : BSKENV_EINVAL;
}

static int do_reset(bskenv_handle *h, int mode, const double *ics_in, const uint8_t *mask, double *obs, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    NO_HOST_PENDING(h, "bskenv_reset");
    CU_TRY(h, cudaSetDevice(h->device));
    leo_reset_kernel<<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(h->P, h->S, h->I, h->ics, h->stride, h->n, mode, ics_in, mask, obs, h->pool, h->icp);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, note_launch(h, (cudaStream_t)stream));
    return BSKENV_OK;
}
int bskenv_reset_seeded(bskenv_handle *h, uint64_t seed, const uint8_t *mask_dev, double *obs_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    h->P.seed = seed;
    return do_reset(h, 2, nullptr, mask_dev, obs_dev, stream);
}
int bskenv_reset_ics(bskenv_handle *h, const double *ics_dev, const uint8_t *mask_dev, double *obs_dev, void *stream)
{
    if (!h || !ics_dev) { if (h) h->err = "bskenv_reset_ics: null ics"; return BSKENV_EINVAL; }
    return do_reset(h, 0, ics_dev, mask_dev, obs_dev, stream);
}
int bskenv_reset_init(bskenv_handle *h, const uint8_t *mask_dev, double *obs_dev, void *stream)
{
    return do_reset(h, 1, nullptr, mask_dev, obs_dev, stream);
}
int bskenv_get_ics(bskenv_handle *h, double *ics_dev, void *stream)
{
    return h ? get_ics<19>(h, ics_dev, stream) : BSKENV_EINVAL;
}

int bskenv_step(bskenv_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev, uint8_t *done_dev,
                uint8_t *done_reason_dev, double *term_obs_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions_dev || !obs_dev || !reward_dev || !done_dev || !done_reason_dev) { h->err = "bskenv_step: null buffer"; return BSKENV_EINVAL; }
    NO_HOST_PENDING(h, "bskenv_step");
    CU_TRY(h, cudaSetDevice(h->device));
    return launch_step(h, actions_dev, obs_dev, reward_dev, done_dev, done_reason_dev, term_obs_dev, (cudaStream_t)stream);
}

int bskenv_step_info(bskenv_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev, uint8_t *done_dev,
                     uint8_t *done_reason_dev, double *term_obs_dev, double *ep_return_dev, int64_t *ep_length_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions_dev || !obs_dev || !reward_dev || !done_dev || !done_reason_dev) { h->err = "bskenv_step_info: null buffer"; return BSKENV_EINVAL; }
    if ((ep_return_dev == nullptr) != (ep_length_dev == nullptr)) { h->err = "bskenv_step_info: ep_return and ep_length go together"; return BSKENV_EINVAL; }
    NO_HOST_PENDING(h, "bskenv_step_info");
    CU_TRY(h, cudaSetDevice(h->device));
    return launch_step(h, actions_dev, obs_dev, reward_dev, done_dev, done_reason_dev, term_obs_dev, (cudaStream_t)stream,
                       ep_return_dev, ep_length_dev);
}

// ---- host-buffer entry points (the reference-facing plugin path) ----------------------------------------------------
// Zero-copy (batch_common.cuh: host_map): 4 B in and 50 B out per env, spread over the whole launch, so no transfer is
// exposed after the kernel.

int bskenv_step_host_async(bskenv_handle *h, const int32_t *actions, double *obs, double *reward, uint8_t *done,
                           uint8_t *done_reason, double *term_obs, double *ep_return, int64_t *ep_length)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions || !obs || !reward || !done || !done_reason) { h->err = "bskenv_step_host: null buffer"; return BSKENV_EINVAL; }
    if ((ep_return == nullptr) != (ep_length == nullptr)) { h->err = "bskenv_step_host: ep_return and ep_length go together"; return BSKENV_EINVAL; }
    if (h->host_pending) { h->err = "bskenv_step_host_async: the previous host step has not been waited for"; return BSKENV_EINVAL; }
    CU_TRY(h, cudaSetDevice(h->device));
    const size_t n = (size_t)h->n;
    void *user[8] = {(void *)actions, obs, reward, done, done_reason, ep_return, ep_length, term_obs};
    const size_t bytes[8] = {n * sizeof(int32_t), n * 5 * sizeof(double), n * sizeof(double), n, n, n * sizeof(double), n * sizeof(int64_t), n * 5 * sizeof(double)};
    void *dev[8], *stage[8];
    int rc = host_step_begin(h, 8, user, bytes, dev, stage);
    if (rc) return rc;
    rc = launch_step(h, (const int32_t *)dev[0], (double *)dev[1], (double *)dev[2], (uint8_t *)dev[3], (uint8_t *)dev[4],
                     (double *)dev[7], h->own_stream, (double *)dev[5], (int64_t *)dev[6]);
    if (rc) return rc;
    for (int k = 0; k < 8; k++) { h->pend_user[k] = stage[k] ? user[k] : nullptr; h->pend_bytes[k] = bytes[k]; }
    h->host_pending = 1;
    return BSKENV_OK;
}

int bskenv_step_host_wait(bskenv_handle *h)
{
    if (!h) return BSKENV_EINVAL;
    if (!h->host_pending) return BSKENV_OK;
    h->host_pending = 0;
    CU_TRY(h, cudaStreamSynchronize(h->own_stream));
    host_step_copy_back(8, h->pend_user, h->h_stage, h->pend_bytes);
    return BSKENV_OK;
}

int bskenv_step_host(bskenv_handle *h, const int32_t *actions, double *obs, double *reward, uint8_t *done, uint8_t *done_reason)
{
    int rc = bskenv_step_host_async(h, actions, obs, reward, done, done_reason, nullptr, nullptr, nullptr);
    return rc ? rc : bskenv_step_host_wait(h);
}

int bskenv_alloc_host(size_t bytes, void **out)
{
    if (!out || bytes == 0) return BSKENV_EINVAL;
    if (cudaHostAlloc(out, bytes, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); *out = nullptr; return BSKENV_ECUDA; }
    return BSKENV_OK;
}
int bskenv_free_host(void *p)
{
    if (p && cudaFreeHost(p) != cudaSuccess) { cudaGetLastError(); return BSKENV_ECUDA; }
    return BSKENV_OK;
}

int bskenv_state_dims(const bskenv_handle *h, int32_t *nd, int32_t *ni)
{
    (void)h;
    if (nd) *nd = LEO_ND;
    if (ni) *ni = LEO_NI;
    return BSKENV_OK;
}
int bskenv_get_state(bskenv_handle *h, double *dstate_dev, int64_t *istate_dev, void *stream)
{
    return h ? get_state(h, LEO_ND, LEO_NI, dstate_dev, istate_dev, stream) : BSKENV_EINVAL;
}
int bskenv_set_state(bskenv_handle *h, const double *dstate_dev, const int64_t *istate_dev, void *stream)
{
    return h ? set_state(h, LEO_ND, LEO_NI, dstate_dev, istate_dev, stream) : BSKENV_EINVAL;
}
// ---- per-env state snapshots (batch_common.cuh: snapshot / restore) ----
static SnapCols leo_snap_cols(bskenv_handle *h)
{
    // the parameter block holds the envs' values only while a pool is loaded (as bskenv_get_env_params reads it); a pool
    // once loaded and unloaded leaves it allocated and stale
    return SnapCols{h->S, h->I, h->ics, h->icp.row_of, h->icp.row_ep, h->stride, h->n, h->P.first_env_index, h->fingerprint,
                    h->pool.n_rows > 0 ? 1 : 0};
}
int bskenv_snapshot_width(const bskenv_handle *h)
{
    (void)h;
    return BSKENV_SNAPSHOT_W;
}
int bskenv_snapshot(bskenv_handle *h, int64_t m, const int64_t *envs_dev, double *rec_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    SnapBlock<LEO_NPD> batch;   // the parameter block of the configuration itself, pool row -1 (as bskenv_set_param_pool derives it)
    double raw[BSKENV_PARAM_DIM];
    leo_host::param_row_get(h->cfg, raw);
    leo_host::param_row_derive(h->P, raw, -1.0, batch.v);
    return snapshot<LeoSnap::L>(h, "bskenv_snapshot", m, envs_dev, rec_dev, leo_snap_cols(h), batch, stream);
}
int bskenv_restore(bskenv_handle *h, int64_t m, const int64_t *envs_dev, const double *rec_dev, double *obs_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    NO_HOST_PENDING(h, "bskenv_restore");
    return restore<LeoSnap>(h, "bskenv_restore", m, envs_dev, rec_dev, obs_dev, leo_snap_cols(h), h->P, stream);
}

int bskenv_state_field(const char *name, int32_t *is_int)
{
    static const FieldEnt tab[] = {
        {"r_BN_N", F_R, 0}, {"v_BN_N", F_V, 0}, {"sigma_BN", F_SIG, 0}, {"omega_BN_B", F_OMG, 0}, {"Omega", F_WHL, 0},
        {"u_current", F_UCUR, 0}, {"density", F_RHO, 0}, {"storedCharge", F_E, 0}, {"shadowFactor", F_SHADOW, 0},
        {"extTorquePntB_B", F_LDIST, 0}, {"att_guidance", F_GUID, 0}, {"att_reference", F_REF, 0},
        {"commandedControlTorque", F_LR, 0}, {"rwTorqueCommand", F_RWCMD, 0}, {"wheelDeltaH", F_DELTAH, 0},
        {"ThrustOnCmd", F_THRON, 0}, {"ThrusterStartTime", F_THRSTART, 0}, {"thrOnTimeRemaining", F_THRREM, 0},
        {"OnTimeRequest", F_THRCMD, 0}, {"reward_total", F_EPRET, 0}, {"sim_obs", F_OBS, 0},
        {"tick", I_TICK, 1}, {"curr_step", I_STEP, 1}, {"task_mask", I_MASK, 1}, {"MRPSwitchCount", I_SWITCH, 1},
        {"thrFactorMask", I_THRFACTOR, 1}, {"initRequest", I_INITREQ, 1}, {"thrDumpingCounter", I_DUMPCNT, 1},
        {"dumpPriorTime", I_DUMPPRIOR, 1}, {"lastDeltaHInMsgTime", I_LASTDH, 1}, {"deltaHWriteTime", I_DHTIME, 1},
        {"episode", I_EPISODE, 1}, {"fireCounter", I_FIRE, 1}, {"thrActive", I_THRACTIVE, 1}, {"episode_over", I_OVER, 1},
        {"rwSat", I_RWSAT, 1}};
    return state_field(tab, name, is_int);
}

int bskenv_episode_stats(bskenv_handle *h, double *stats_host)
{
    return (h && stats_host) ? episode_stats(h, ST_N, stats_host) : BSKENV_EINVAL;
}

int bskenv_fp64_peak(int device, double seconds, double *tflops)
{
    if (!tflops) return BSKENV_EINVAL;
    if (cudaSetDevice(device) != cudaSuccess) return BSKENV_ENODEV;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return BSKENV_ECUDA;
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    double *out = nullptr;
    if (cudaMalloc(&out, sizeof(double) * blocks * threads) != cudaSuccess) return BSKENV_ECUDA;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    for (int w = 0; w < 3; w++) fp64_peak_kernel<<<blocks, threads>>>(out, iters, 0.999999, 1e-7);
    cudaDeviceSynchronize();
    double best = 0.0, spent = 0.0;
    const double flop = (double)blocks * threads * (double)iters * 64.0 * 2.0;
    int reps = 0;
    while ((spent < seconds || reps < 3) && reps < 10000) {
        cudaEventRecord(a);
        fp64_peak_kernel<<<blocks, threads>>>(out, iters, 0.999999, 1e-7);
        cudaEventRecord(b);
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        double tf = flop / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
        spent += ms * 1e-3; reps++;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(out);
    if (cudaGetLastError() != cudaSuccess) return BSKENV_ECUDA;
    *tflops = best;
    return BSKENV_OK;
}

}  // extern "C"
