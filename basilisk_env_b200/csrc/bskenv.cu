// bskenv.cu -- sm_100a kernels and the C ABI (include/bskenv.h) of the batched LEO environment step.
//
// Kernels:
//   leo_step_kernel   one thread = one spacecraft; ONE launch = one decision interval for all envs
//                     (replaces Basilisk ExecuteSimulation(), reference
//                     basilisk_env/simulators/leoPowerAttitudeSimulator.py:590-595, and the gym
//                     bookkeeping of basilisk_env/envs/leoPowerAttitudeEnvironment.py:65-145);
//                     warp-shuffle reduction of the episode statistics; optional in-kernel auto-reset.
//   leo_reset_kernel  simulator construction + initial observation (reference ...Simulator.py:67-117,
//                     ...Environment.py:172-216) from explicit, stored or device-sampled ICs.
//   fp64_peak_kernel  DFMA microbenchmark = the roofline denominator.
// There is no CPU path in this library.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/bskenv.h"
#include "leo_core.cuh"
#include "leo_split.cuh"
#include "leo_host.h"

#ifndef LEO_LANES
#define LEO_LANES 32            // envs per warp (tuning builds: 16 / 8 leave the upper lanes idle)
#endif
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

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

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
// all of it, 180 times per interval.  Before the launch the envs are bucketed by action (counting sort, warp-aggregated
// atomics: leo_bucket_count_kernel + leo_bucket_fill_kernel) and a warp takes 32 slots of the permutation: the state is
// gathered / scattered at the chunk boundaries (12 times per 1800 ticks), the tick loop diverges only in the at most three
// warps that straddle a bucket boundary.  Per-env arithmetic does not depend on the lane an env runs in: results are
// bit-identical with and without (tests/test_gpu_round2.py).  bucket[0..3] = sizes, bucket[4..7] = cursors.  Order of the
// buckets in the permutation: action 2 (the desat chain: the slowest warps), 0, 1, unknown -- the work queue hands out the
// long items first, so that the tail of a launch is made of the short ones.
__device__ __forceinline__ int leo_action_class(int action) { return (action >= 0 && action <= 2) ? action : 3; }
__global__ void __launch_bounds__(256)
leo_bucket_count_kernel(int64_t n, const int32_t *__restrict__ actions, int *__restrict__ bucket)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int cls = e < n ? leo_action_class(actions[e]) : -1;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const unsigned m = __ballot_sync(0xffffffffu, cls == c);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&bucket[c], __popc(m));
    }
}
__global__ void __launch_bounds__(256)
leo_bucket_fill_kernel(int64_t n, const int32_t *__restrict__ actions, int *__restrict__ bucket, int32_t *__restrict__ perm)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int cls = e < n ? leo_action_class(actions[e]) : -1;
    const int lane = threadIdx.x & 31;
    const int n0 = bucket[0], n1 = bucket[1], n2 = bucket[2];
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const unsigned m = __ballot_sync(0xffffffffu, cls == c);
        if (!m) continue;
        const int leader = __ffs(m) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(&bucket[4 + c], __popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        const int first = c == 2 ? 0 : (c == 0 ? n2 : (c == 1 ? n2 + n0 : n0 + n1 + n2));     // slowest bucket first in the queue
        if (cls == c) perm[first + base + __popc(m & ((1u << lane) - 1))] = (int32_t)e;
    }
}

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
    extern __shared__ double bus_smem[];          // [LEO_NM][LEO_BLOCK]: per-thread message bus (leo_core.cuh: MBus)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    leo::MBus bus;
    bus.p = nullptr;
    bus.a = (uint32_t)__cvta_generic_to_shared(bus_smem) + threadIdx.x * (uint32_t)sizeof(double);
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
        const int64_t slot = (int64_t)g * LEO_LANES + lane;
        const bool valid = lane < LEO_LANES && slot < n;
        const int64_t e = (valid && sc.perm) ? (int64_t)sc.perm[slot] : slot;     // envs of one action per warp (see LeoSched)
        leo::StepOut o;
        o.done = 0; o.reason = 0; o.reward = 0.;
        for (int c = c_first; c < c_end; c++) {
        if (valid) leo::leo_step_env<NRW, J2, DIAG, F32>(P, S, I, stride, e, bus, actions[e], o, PF, c, sc.n_chunks);
        if (c + 1 < sc.n_chunks) {                              // chunk boundary inside the interval: publish and go on
            if (sc.dynamic) {
                __threadfence();
                __syncwarp();
                if (lane == 0) chunk_publish(sc.progress + g, c + 1);
            }
            continue;
        }
        step_finish(P, S, I, ics, stride, e, valid, lane, o, obs, reward, done, reason, term_obs, stats, ep_return, ep_length);
        }   // chunks of this item
        __syncwarp();
    }
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
    extern __shared__ double bus_smem[];          // [LEO_NM_PENV][LEO_BLOCK]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    leo::MBus bus;
    bus.p = nullptr;
    bus.a = (uint32_t)__cvta_generic_to_shared(bus_smem) + threadIdx.x * (uint32_t)sizeof(double);
    for (bool more = true; more; more = sc.dynamic != 0) {
        int g, c_first = 0, c_end = sc.n_chunks;
        if (sc.dynamic) {
            g = 0;
            if (lane == 0) g = atomicAdd(&sc.sched[0], 1);
            g = __shfl_sync(0xffffffffu, g, 0);
            if (g >= sc.n_groups * sc.n_chunks) break;
            c_first = g / sc.n_groups; c_end = c_first + 1;
            g -= c_first * sc.n_groups;
            if (c_first > 0) {
                if (lane == 0)
                    while (chunk_peek(sc.progress + g) < c_first) __nanosleep(200);
                __syncwarp();
            }
        } else {
            g = blockIdx.x * (LEO_BLOCK / 32) + warp;
        }
        const int64_t slot = (int64_t)g * LEO_LANES + lane;
        const bool valid = lane < LEO_LANES && slot < n;
        const int64_t e = (valid && sc.perm) ? (int64_t)sc.perm[slot] : slot;
        leo::StepOut o;
        o.done = 0; o.reason = 0; o.reward = 0.;
        for (int c = c_first; c < c_end; c++) {
            if (valid) leo::leo_step_env<NRW, J2, DIAG, false, leo::ParEnv>(P, S, I, stride, e, bus, actions[e], o, LeoParamsF(), c, sc.n_chunks);
            if (c + 1 < sc.n_chunks) {
                if (sc.dynamic) {
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) chunk_publish(sc.progress + g, c + 1);
                }
                continue;
            }
            step_finish<leo::ParEnv>(P, S, I, ics, stride, e, valid, lane, o, obs, reward, done, reason, term_obs, stats, ep_return,
                                     ep_length, pool);
        }
        __syncwarp();
    }
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
#ifdef LEO_SPLIT_PROF
    long long tc[8]; tc[0] = clock64();
    for (int c = 0; c < n_chunks; c++) { leo::split_dyn<NRW, J2, DIAG>(P, S, I, stride, e, bus, box, bar, action, o, c, n_chunks); tc[c + 1] = clock64(); }
    step_finish(P, S, I, ics, stride, e, valid, lane, o, obs, reward, done, reason, term_obs, stats, ep_return, ep_length);
    if (lane == 0) printf("BLK %d total %lld chunks %lld %lld %lld %lld %lld %lld finish %lld\n", blockIdx.x, clock64() - tc[0], tc[1] - tc[0], tc[2] - tc[1], tc[3] - tc[2],
                          tc[4] - tc[3], tc[5] - tc[4], tc[6] - tc[5], clock64() - tc[6]);
#else
    for (int c = 0; c < n_chunks; c++) leo::split_dyn<NRW, J2, DIAG>(P, S, I, stride, e, bus, box, bar, action, o, c, n_chunks);
    step_finish(P, S, I, ics, stride, e, valid, lane, o, obs, reward, done, reason, term_obs, stats, ep_return, ep_length);
#endif
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
    if (mode == 0) {
        for (int k = 0; k < 19; k++) ic[k] = ics_in[e * 19 + k];
    } else if (mode == 1) {
        for (int k = 0; k < 19; k++) ic[k] = ics[(int64_t)k * stride + e];
    } else if (icp.n_rows > 0) {
        const int64_t r = leo::ic_pool_row(icp, P.seed, ge, ep, prow);
        for (int k = 0; k < 19; k++) ic[k] = icp.rows[r * 19 + k];
        icp.row_of[e] = (int32_t)r; icp.row_ep[e] = ep;
    } else {
        leo::sample_ic(P, ge, ep, ic);
    }
    if (icp.row_of && mode != 1 && !(mode == 2 && icp.n_rows > 0)) { icp.row_of[e] = -1; icp.row_ep[e] = ep; }
    for (int k = 0; k < 19; k++) ics[(int64_t)k * stride + e] = ic[k];
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

__global__ void gather_ics_kernel(const double *__restrict__ ics, int64_t stride, int64_t n, double *__restrict__ out)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int k = 0; k < 19; k++) out[e * 19 + k] = ics[(int64_t)k * stride + e];
}
// bskenv_get_ic_rows: the recorded row where it belongs to the env's current episode (an in-kernel reset after an unload
// advances the episode counter without touching the record)
__global__ void gather_ic_rows_kernel(const int32_t *__restrict__ row_of, const int64_t *__restrict__ row_ep, const int64_t *__restrict__ ep,
                                      int64_t n, int32_t *__restrict__ out)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    out[e] = row_ep[e] == ep[e] ? row_of[e] : -1;
}
// dense [fields][n] <-> padded [fields][stride]
template <typename T>
__global__ void copy_fields_kernel(const T *__restrict__ src, int64_t src_stride, T *__restrict__ dst, int64_t dst_stride,
                                   int64_t n, int fields)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int f = 0; f < fields; f++) dst[(int64_t)f * dst_stride + e] = src[(int64_t)f * src_stride + e];
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

struct bskenv_handle {
    bskenv_config cfg;
    LeoParams P;
    LeoParamsF PF;
    int device;
    int64_t n, stride;
    double *S, *ics, *stats;
    int64_t *I;
    int *sched;                 // work queue head of the step kernel
    int32_t *perm; int *bucket; // lane assignment of the throughput organisation (envs bucketed by action), bucket sizes / cursors
    double *d_eph[2];           // device copies of the ephemeris tables (Sun position, Earth orientation angles)
    int sm_count;
    // host-buffer entry points: page-locked staging (only for pageable caller buffers), own stream, ordering events
    void *h_stage[8];           // actions, obs, reward, done, reason, ep_return, ep_length, term_obs
    void *pend_user[8]; size_t pend_bytes[8]; int host_pending;
    cudaStream_t own_stream;
    cudaEvent_t ev_last;        // recorded after every launch queued through the device-buffer entry points
    int ev_valid;
    int64_t launches;
    const char *kernel_name;    // the step-kernel instantiation of the last launch
    int organisation;           // BSKENV_ORG_*: 0 auto, 1 one thread per env, 2 two warps per env group (small batches)
    LeoPool pool;               // loaded parameter pool (n_rows = 0: none); rows in device memory
    int s_fields;               // double fields allocated per env in S: LEO_ND, or LEO_ND + LEO_NPD once a pool was loaded
    IcPool icp;                 // loaded initial-condition pool (n_rows = 0: none); rows and per-env record in device memory
    std::string err;
};

#define CU_TRY(h, call)                                                                              \
    do {                                                                                             \
        cudaError_t _e = (call);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                            \
            return BSKENV_ECUDA;                                                                     \
        }                                                                                            \
    } while (0)

// Launches queued on the caller's streams are ordered before a later host-buffer step (which runs on the handle's own
// stream) through this event; the host-buffer step itself is complete when bskenv_step_host[_wait] returns.
static cudaError_t note_launch(bskenv_handle *h, cudaStream_t st)
{
    h->ev_valid = 1;
    return cudaEventRecord(h->ev_last, st);
}
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
    leo_reset_kernel<<<(int)((h->n + 255) / 256), 256, 0, st>>>(h->P, h->S, h->I, h->ics, h->stride, h->n, 2, nullptr, done, obs,
                                                                h->pool, h->icp);
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
    const int64_t groups = (h->n + LEO_LANES - 1) / LEO_LANES;
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
        static bool split_attr[64][2] = {{false}};
        const int which = h->P.nrw == 3 ? 0 : 1;
        if (!split_attr[h->device & 63][which]) {
            if (which == 0) CU_TRY(h, cudaFuncSetAttribute(leo_split_kernel<3, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            else CU_TRY(h, cudaFuncSetAttribute(leo_split_kernel<4, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            split_attr[h->device & 63][which] = true;
        }
        if (which == 0) {
            h->kernel_name = "leo_split_kernel<3,0,true>";
            leo_split_kernel<3, 0, true><<<dgrid, 64 * G, smem, st>>>(PK, h->S, h->I, h->ics, h->stride, h->n, act, obs, rew, done, reason, term_obs,
                                                                 h->stats, (int)groups, sc.n_chunks, ep_return, ep_length);
        } else {
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
        CU_TRY(h, cudaMemsetAsync(h->bucket, 0, sizeof(int) * 8, st));
        leo_bucket_count_kernel<<<bgrid, 256, 0, st>>>(h->n, act, h->bucket);
        leo_bucket_fill_kernel<<<bgrid, 256, 0, st>>>(h->n, act, h->bucket, h->perm);
        sc.perm = h->perm;
        h->launches += 2;
    }
#define LEO_STR_(x) #x
#define LEO_STR(x) LEO_STR_(x)
#define LEO_LAUNCH_B(NRW, J2, DIAG, F32, MINB)                                                                 \
    do {                                                                                                       \
        static bool attr_set[64] = {false};      /* opt in to > 48 KB of dynamic shared memory once per device */  \
        const size_t bus_bytes = (J2) == 2 ? LEO_BUS_BYTES_PFIX : LEO_BUS_BYTES;                                \
        if (!attr_set[h->device & 63]) {                                                                       \
            CU_TRY(h, cudaFuncSetAttribute(leo_step_kernel<NRW, J2, DIAG, F32, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bus_bytes)); \
            attr_set[h->device & 63] = true;                                                                   \
        }                                                                                                      \
        h->kernel_name = "leo_step_kernel<" #NRW "," #J2 "," #DIAG "," #F32 "," LEO_STR(MINB) ">";              \
        leo_step_kernel<NRW, J2, DIAG, F32, MINB><<<grid, LEO_BLOCK, bus_bytes, st>>>(PK, h->PF, h->S, h->I, h->ics, h->stride, h->n, act, obs, \
                                                                                 rew, done, reason, term_obs, h->stats, sc, ep_return, ep_length); \
    } while (0)
#define LEO_LAUNCH(NRW, J2, DIAG, F32) LEO_LAUNCH_B(NRW, J2, DIAG, F32, LEO_MIN_BLOCKS)
#define LEO_LAUNCH_PENV(J2)                                                                                    \
    do {                                                                                                       \
        static bool attr_set[64] = {false};                                                                    \
        if (!attr_set[h->device & 63]) {                                                                       \
            CU_TRY(h, cudaFuncSetAttribute(leo_step_penv_kernel<3, J2, true, LEO_MIN_BLOCKS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LEO_BUS_BYTES_PENV)); \
            attr_set[h->device & 63] = true;                                                                   \
        }                                                                                                      \
        h->kernel_name = "leo_step_penv_kernel<3," #J2 ",true," LEO_STR(LEO_MIN_BLOCKS) ">";                    \
        leo_step_penv_kernel<3, J2, true, LEO_MIN_BLOCKS><<<grid, LEO_BLOCK, LEO_BUS_BYTES_PENV, st>>>(PK, h->pool, h->S, h->I, h->ics, \
            h->stride, h->n, act, obs, rew, done, reason, term_obs, h->stats, sc, ep_return, ep_length);        \
    } while (0)
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
    if (!cfg || !out || n_envs <= 0) { g_create_error = "bskenv_create: bad arguments"; return BSKENV_EINVAL; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        g_create_error = "bskenv_create: no CUDA device (this library has no CPU path)";
        return BSKENV_ENODEV;
    }
    if (device < 0 || device >= ndev) { g_create_error = "bskenv_create: device index out of range"; return BSKENV_EINVAL; }
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
    h->device = device; h->n = n_envs; h->stride = (n_envs + 31) / 32 * 32; h->launches = 0; h->kernel_name = nullptr; h->organisation = BSKENV_ORG_AUTO;
    h->S = h->ics = h->stats = nullptr; h->I = nullptr; h->sched = nullptr; h->perm = nullptr; h->bucket = nullptr;
    h->d_eph[0] = h->d_eph[1] = nullptr;
    h->pool.rows = nullptr; h->pool.n_rows = 0; h->pool.assign = 0; h->s_fields = LEO_ND;
    h->icp.rows = nullptr; h->icp.row_of = nullptr; h->icp.row_ep = nullptr; h->icp.n_rows = 0; h->icp.assign = 0;
    for (int k = 0; k < 8; k++) { h->h_stage[k] = nullptr; h->pend_user[k] = nullptr; h->pend_bytes[k] = 0; }
    h->host_pending = 0; h->own_stream = nullptr; h->ev_last = nullptr; h->ev_valid = 0;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&h->sched, sizeof(int) * (size_t)(4 + (n_envs + LEO_LANES - 1) / LEO_LANES));
    if (e == cudaSuccess) e = cudaMalloc(&h->perm, sizeof(int32_t) * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->bucket, sizeof(int) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&h->S, sizeof(double) * LEO_ND * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->I, sizeof(int64_t) * LEO_NI * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->ics, sizeof(double) * 19 * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->stats, sizeof(double) * ST_N);
    if (e == cudaSuccess) e = cudaMemset(h->S, 0, sizeof(double) * LEO_ND * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->I, 0, sizeof(int64_t) * LEO_NI * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->ics, 0, sizeof(double) * 19 * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->stats, 0, sizeof(double) * ST_N);
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
    cudaFree(h->S); cudaFree(h->I); cudaFree(h->ics); cudaFree(h->stats); cudaFree(h->sched); cudaFree(h->perm); cudaFree(h->bucket);
    cudaFree(h->d_eph[0]); cudaFree(h->d_eph[1]); cudaFree((void *)h->pool.rows);
    cudaFree((void *)h->icp.rows); cudaFree(h->icp.row_of); cudaFree(h->icp.row_ep);
    if (h->own_stream) { cudaStreamSynchronize(h->own_stream); cudaStreamDestroy(h->own_stream); }
    for (int k = 0; k < 8; k++) cudaFreeHost(h->h_stage[k]);
    if (h->ev_last) cudaEventDestroy(h->ev_last);
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
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());                         // a launch in flight may still read the old table
    LeoEph &E = kind == 0 ? h->P.eph_sun : h->P.eph_orient;
    cudaFree(h->d_eph[kind]); h->d_eph[kind] = nullptr;
    E.coef = nullptr; E.nseg = 0; E.ncoef = 0; E.t0 = 0.; E.seg_len = 0.;
    if (n_seg <= 0) return BSKENV_OK;                           // back to the analytic model
    if (!coef || n_coef < 1 || n_coef > 64 || !(seg_len > 0.)) { h->err = "bskenv_set_ephemeris: bad table shape"; return BSKENV_EINVAL; }
    // an episode runs from sim time 0 to (max_length + 1) decision intervals: the table has to cover it
    const double t_end = ((double)h->P.max_length + 1.0) * (double)h->P.step_ns * 1e-9;   // max_length may be INT_MAX
    if (t0 > 0. || t0 + seg_len * n_seg < t_end) {
        h->err = "bskenv_set_ephemeris: the table does not cover one episode [0, (max_length + 1) * step_duration]";
        return BSKENV_EINVAL;
    }
    const size_t bytes = sizeof(double) * (size_t)n_seg * 3 * (size_t)n_coef;
    CU_TRY(h, cudaMalloc(&h->d_eph[kind], bytes));
    CU_TRY(h, cudaMemcpy(h->d_eph[kind], coef, bytes, cudaMemcpyHostToDevice));
    E.coef = h->d_eph[kind]; E.nseg = n_seg; E.ncoef = n_coef; E.t0 = t0; E.seg_len = seg_len;
    return BSKENV_OK;
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
    if (n_rows < 0 || (n_rows > 0 && !ics_host)) { h->err = "bskenv_set_ic_pool: bad row count or null rows"; return BSKENV_EINVAL; }
    if (n_rows > 0) {
        if (assign != BSKENV_ICS_BY_INDEX && assign != BSKENV_ICS_PER_EPISODE && assign != BSKENV_ICS_PARAM_ROW) {
            h->err = "bskenv_set_ic_pool: unknown assignment mode"; return BSKENV_EINVAL;
        }
        if (assign == BSKENV_ICS_PARAM_ROW && h->pool.n_rows != n_rows) {
            h->err = "bskenv_set_ic_pool: BSKENV_ICS_PARAM_ROW needs a loaded parameter pool of the same row count (" +
                     std::to_string(n_rows) + " IC rows, " + std::to_string(h->pool.n_rows) + " parameter rows)";
            return BSKENV_EINVAL;
        }
        for (int r = 0; r < n_rows; r++) {
            const std::string err = leo_host::ic_row_check(ics_host + (size_t)r * BSKENV_IC_DIM, BSKENV_IC_DIM);
            if (!err.empty()) { h->err = "bskenv_set_ic_pool: row " + std::to_string(r) + ": " + err; return BSKENV_EINVAL; }
        }
    }
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());                         // a launch in flight may still read the old pool
    cudaFree((void *)h->icp.rows);
    h->icp.rows = nullptr; h->icp.n_rows = 0;
    if (n_rows == 0) return BSKENV_OK;                          // unloaded: resets sample again, the in-kernel auto-reset
    if (!h->icp.row_of) {                                       // first pool of this handle: the per-env record, all -1
        CU_TRY(h, cudaMalloc(&h->icp.row_of, sizeof(int32_t) * h->stride));
        CU_TRY(h, cudaMalloc(&h->icp.row_ep, sizeof(int64_t) * h->stride));
        CU_TRY(h, cudaMemset(h->icp.row_of, 0xFF, sizeof(int32_t) * h->stride));
        CU_TRY(h, cudaMemset(h->icp.row_ep, 0, sizeof(int64_t) * h->stride));
    }
    double *d_rows = nullptr;
    const size_t bytes = sizeof(double) * (size_t)n_rows * BSKENV_IC_DIM;
    CU_TRY(h, cudaMalloc(&d_rows, bytes));
    CU_TRY(h, cudaMemcpy(d_rows, ics_host, bytes, cudaMemcpyHostToDevice));
    h->icp.rows = d_rows; h->icp.n_rows = n_rows; h->icp.assign = assign;
    return BSKENV_OK;
}

int bskenv_get_ic_rows(bskenv_handle *h, int32_t *rows_dev, void *stream)
{
    if (!h || !rows_dev) { if (h) h->err = "bskenv_get_ic_rows: null rows"; return BSKENV_EINVAL; }
    CU_TRY(h, cudaSetDevice(h->device));
    if (!h->icp.row_of) CU_TRY(h, cudaMemsetAsync(rows_dev, 0xFF, sizeof(int32_t) * h->n, (cudaStream_t)stream));
    else gather_ic_rows_kernel<<<(int)((h->n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->icp.row_of, h->icp.row_ep,
                                                                                             h->I + (size_t)I_EPISODE * h->stride, h->n, rows_dev);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

static int do_reset(bskenv_handle *h, int mode, const double *ics_in, const uint8_t *mask, double *obs, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    NO_HOST_PENDING(h, "bskenv_reset");
    CU_TRY(h, cudaSetDevice(h->device));
    const int grid = (int)((h->n + 255) / 256);
    leo_reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(h->P, h->S, h->I, h->ics, h->stride, h->n, mode, ics_in, mask, obs, h->pool, h->icp);
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
    if (!h || !ics_dev) return BSKENV_EINVAL;
    CU_TRY(h, cudaSetDevice(h->device));
    gather_ics_kernel<<<(int)((h->n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->ics, h->stride, h->n, ics_dev);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
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
// The step kernel reads the actions from and writes its results to PINNED HOST memory directly (zero-copy over PCIe:
// 4 B in and 50 B out per env, spread over the whole launch, so no transfer is exposed after the kernel).  Caller buffers
// that are already page-locked (bskenv_alloc_host, cudaHostRegister, torch pin_memory) are used in place; pageable ones go
// through page-locked staging owned by the handle plus one memcpy each.
namespace {
struct HostMap { void *dev; void *stage; };          // device-visible address, and the staging block behind it (or null)
bool host_pinned(const void *p, void **dev)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type != cudaMemoryTypeHost || !a.devicePointer) return false;
    *dev = a.devicePointer;
    return true;
}
}  // namespace

static int host_map(bskenv_handle *h, const void *user, size_t bytes, int slot, HostMap *m)
{
    m->stage = nullptr;
    if (host_pinned(user, &m->dev)) return BSKENV_OK;
    if (!h->h_stage[slot]) CU_TRY(h, cudaHostAlloc(&h->h_stage[slot], bytes, cudaHostAllocMapped));
    m->stage = h->h_stage[slot];
    CU_TRY(h, cudaHostGetDevicePointer(&m->dev, m->stage, 0));
    return BSKENV_OK;
}

int bskenv_step_host_async(bskenv_handle *h, const int32_t *actions, double *obs, double *reward, uint8_t *done,
                           uint8_t *done_reason, double *term_obs, double *ep_return, int64_t *ep_length)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions || !obs || !reward || !done || !done_reason) { h->err = "bskenv_step_host: null buffer"; return BSKENV_EINVAL; }
    if ((ep_return == nullptr) != (ep_length == nullptr)) { h->err = "bskenv_step_host: ep_return and ep_length go together"; return BSKENV_EINVAL; }
    if (h->host_pending) { h->err = "bskenv_step_host_async: the previous host step has not been waited for"; return BSKENV_EINVAL; }
    CU_TRY(h, cudaSetDevice(h->device));
    const size_t n = (size_t)h->n;
    if (!h->own_stream) CU_TRY(h, cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    cudaStream_t st = h->own_stream;
    HostMap m[8];
    int rc;
    if ((rc = host_map(h, actions, n * sizeof(int32_t), 0, &m[0]))) return rc;
    if ((rc = host_map(h, obs, n * 5 * sizeof(double), 1, &m[1]))) return rc;
    if ((rc = host_map(h, reward, n * sizeof(double), 2, &m[2]))) return rc;
    if ((rc = host_map(h, done, n, 3, &m[3]))) return rc;
    if ((rc = host_map(h, done_reason, n, 4, &m[4]))) return rc;
    m[5].dev = m[6].dev = m[7].dev = nullptr; m[5].stage = m[6].stage = m[7].stage = nullptr;
    if (term_obs && (rc = host_map(h, term_obs, n * 5 * sizeof(double), 7, &m[7]))) return rc;
    if (ep_return) {
        if ((rc = host_map(h, ep_return, n * sizeof(double), 5, &m[5]))) return rc;
        if ((rc = host_map(h, ep_length, n * sizeof(int64_t), 6, &m[6]))) return rc;
    }
    if (m[0].stage) memcpy(m[0].stage, actions, n * sizeof(int32_t));
    // order after whatever the caller queued through bskenv_step / reset / set_state on its own streams
    if (h->ev_valid) CU_TRY(h, cudaStreamWaitEvent(st, h->ev_last, 0));
    rc = launch_step(h, (const int32_t *)m[0].dev, (double *)m[1].dev, (double *)m[2].dev, (uint8_t *)m[3].dev, (uint8_t *)m[4].dev,
                     (double *)m[7].dev, st, (double *)m[5].dev, (int64_t *)m[6].dev);
    if (rc) return rc;
    void *user[8] = {nullptr, obs, reward, done, done_reason, ep_return, ep_length, term_obs};
    const size_t bytes[8] = {0, n * 5 * sizeof(double), n * sizeof(double), n, n, n * sizeof(double), n * sizeof(int64_t), n * 5 * sizeof(double)};
    for (int k = 0; k < 8; k++) { h->pend_user[k] = m[k].stage ? user[k] : nullptr; h->pend_bytes[k] = bytes[k]; }
    h->host_pending = 1;
    return BSKENV_OK;
}

int bskenv_step_host_wait(bskenv_handle *h)
{
    if (!h) return BSKENV_EINVAL;
    if (!h->host_pending) return BSKENV_OK;
    h->host_pending = 0;
    CU_TRY(h, cudaStreamSynchronize(h->own_stream));
    for (int k = 1; k < 8; k++)
        if (h->pend_user[k]) memcpy(h->pend_user[k], h->h_stage[k], h->pend_bytes[k]);
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
    if (!h) return BSKENV_EINVAL;
    CU_TRY(h, cudaSetDevice(h->device));
    const int grid = (int)((h->n + 255) / 256);
    if (dstate_dev) copy_fields_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(h->S, h->stride, dstate_dev, h->n, h->n, LEO_ND);
    if (istate_dev) copy_fields_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>(h->I, h->stride, istate_dev, h->n, h->n, LEO_NI);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}
int bskenv_set_state(bskenv_handle *h, const double *dstate_dev, const int64_t *istate_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    CU_TRY(h, cudaSetDevice(h->device));
    const int grid = (int)((h->n + 255) / 256);
    if (dstate_dev) copy_fields_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(dstate_dev, h->n, h->S, h->stride, h->n, LEO_ND);
    if (istate_dev) copy_fields_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>(istate_dev, h->n, h->I, h->stride, h->n, LEO_NI);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, note_launch(h, (cudaStream_t)stream));
    return BSKENV_OK;
}
int bskenv_state_field(const char *name, int32_t *is_int)
{
    struct Ent { const char *n; int idx; int is_int; };
    static const Ent tab[] = {
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
    if (!name) return -1;
    for (const Ent &t : tab)
        if (!strcmp(t.n, name)) { if (is_int) *is_int = t.is_int; return t.idx; }
    return -1;
}

int bskenv_episode_stats(bskenv_handle *h, double *stats_host)
{
    if (!h || !stats_host) return BSKENV_EINVAL;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());
    CU_TRY(h, cudaMemcpy(stats_host, h->stats, sizeof(double) * ST_N, cudaMemcpyDeviceToHost));
    CU_TRY(h, cudaMemset(h->stats, 0, sizeof(double) * ST_N));
    return BSKENV_OK;
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
