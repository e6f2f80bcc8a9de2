// opnav.cu -- sm_100a kernels and the C ABI (include/bskenv.h, bskenv_opnav_*) of the batched opNav environment step.
//
// Kernels:
//   opnav_pass1_kernel, opnav_pass2_kernel
//                       one thread = one spacecraft; the two launches are one 50-minute decision interval (3000 ticks) for
//                       all envs (replace Basilisk ExecuteSimulation(), reference simulators/opNavSimulator.py:256-261,
//                       and the gym bookkeeping of envs/opNavEnvironment.py:55-125): noise walk + dynamics / flight
//                       software, then the filter + observation / reward; warp-shuffle reduction of the episode
//                       statistics; optional in-kernel auto-reset.
//   opnav_reset_kernel  simulator construction + initial observation from explicit, stored or device-sampled ICs.
// There is no CPU path in this library.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>

#include "../../include/bskenv.h"
#include "opnav_core.cuh"
#include "opnav_host.h"

#ifndef ON_NZBUF_MAX_FRAC
#define ON_NZBUF_MAX_FRAC 0.45   // of the free device memory, for the noise buffer of the three-kernel interval
#endif
#ifndef ON_MIN_BLOCKS
#define ON_MIN_BLOCKS 3
#endif

namespace {

enum { OST_RET = 0, OST_LEN, OST_COUNT, OST_MAXLEN, OST_MODES, OST_STEPS, OST_MEAS, OST_BAD, OST_N };

__device__ __forceinline__ double warp_sum_d(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// One warp steps a group of 32 consecutive envs; when there are more groups than resident warps the grid is one
// resident set and the warps pull groups from an atomic queue (same scheme as the LEO step kernel).
struct OnSched { int *sched; int n_groups; int dynamic; };

#ifdef ON_MAXNREG
#define ON_STEP_BOUNDS(MINB) __maxnreg__(ON_MAXNREG)    // tuning builds: explicit register cap instead of an occupancy target
#else
#define ON_STEP_BOUNDS(MINB) __launch_bounds__(ON_BLOCK, MINB)
#endif

// Lane assignment.  The two flight-software task sets execute different code every tick (hillPoint + tracking error vs CSS +
// eclipse + cssWlsEst + sunSafePoint); with one env per lane in index order a warp of mixed actions runs both, 3000 times.
// Before the step, envs are therefore bucketed by the task set they WILL run (first-interval event, action, or the mode in
// force for an unknown action) and the warps of the step kernel take 32 envs of one bucket: the persistent state is read and
// written once per decision (gathered, 97 fields per env), the tick loop is divergence-free.  sched[1..2] = bucket sizes,
// sched[3..4] = bucket cursors.
__device__ __forceinline__ int opnav_task_set(const int64_t *__restrict__ I, int64_t stride, int64_t e, int action)
{
    if (I[(int64_t)OI_FIRST * stride + e]) return 0;
    // an unknown action keeps the mode in force; any non-zero mode field (also a foreign one injected through
    // bskenv_opnav_set_state) is the sun-safe set, so that every env lands in exactly one of the two buckets
    return action == 0 ? 0 : (action == 1 ? 1 : (I[(int64_t)OI_MODE * stride + e] != 0 ? 1 : 0));
}
__global__ void __launch_bounds__(256)
opnav_bucket_count_kernel(const int64_t *__restrict__ I, int64_t stride, int64_t n, const int32_t *__restrict__ actions, int *__restrict__ sched)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < n;
    const int cls = valid ? opnav_task_set(I, stride, e, actions[e]) : -1;
    const unsigned m0 = __ballot_sync(0xffffffffu, cls == 0);
    if ((threadIdx.x & 31) == 0 && m0) atomicAdd(&sched[1], __popc(m0));
}
__global__ void __launch_bounds__(256)
opnav_bucket_fill_kernel(const int64_t *__restrict__ I, int64_t stride, int64_t n, const int32_t *__restrict__ actions, int *__restrict__ sched,
                         int32_t *__restrict__ perm)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < n;
    const int cls = valid ? opnav_task_set(I, stride, e, actions[e]) : -1;
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int c = 0; c < 2; c++) {
        const unsigned m = __ballot_sync(0xffffffffu, cls == c);
        if (!m) continue;
        int base = 0;
        if (lane == __ffs(m) - 1) base = atomicAdd(&sched[3 + c], __popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (cls == c) perm[(c == 0 ? 0 : sched[1]) + base + __popc(m & ((1u << lane) - 1))] = (int32_t)e;
    }
}

__global__ void opnav_perm_identity_kernel(int32_t *__restrict__ perm, int64_t stride, int64_t n)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < stride) perm[e] = (int32_t)(e < n ? e : n - 1);
}

// Per-thread scratch in shared memory, one struct per pass, odd strides in doubles (conflict-free): first pass cold dynamics
// data (19) + walk states (15) + pad = 35, second pass the filter (33: the square-root factor is stored packed).
struct OnScratchA { opnav::Cold c; opnav::Walk w; double pad; };
struct OnScratchB { opnav::Ukf f; };

// One decision interval = two kernels (opnav_core.cuh: opnav_pass1 / opnav_pass2): noise walk + dynamics / flight software, then
// filter + observation / reward / termination, auto-reset and statistics.  One thread per env in both; the measurements of the
// interval cross in a global buffer.  Separate kernels give each pass its own register allocation: three blocks per SM (168
// registers) without the spills that the single interleaved loop had at that occupancy (and a warp-specialised form -- one
// warp per role, mailboxes in shared memory, git history -- could not have: one kernel, one allocation).
// MINB = resident blocks per SM the registers are allocated for: 2 (255 registers) or 3 (168 registers).  Three blocks deliver
// more per resident set but a set is larger and a partial set costs a whole one (the ticks are a latency-bound chain): the
// launcher picks the organisation with the shorter predicted launch.
__device__ __forceinline__ bool on_next_group(const OnSched &sc, int *head, int lane, int warp, int &g)
{
    if (sc.dynamic) {
        g = 0;
        if (lane == 0) g = atomicAdd(head, 1);
        g = __shfl_sync(0xffffffffu, g, 0);
        return g < sc.n_groups;
    }
    g = blockIdx.x * (ON_BLOCK / 32) + warp;
    return true;
}

template <int MINB>
__global__ void ON_STEP_BOUNDS(MINB)
opnav_pass1_kernel(const __grid_constant__ OpNavParams P, double *__restrict__ S, int64_t *__restrict__ I, int64_t stride, int64_t n,
                   const int32_t *__restrict__ actions, const OnSched sc, const int32_t *__restrict__ perm, double *__restrict__ mbuf)
{
    extern __shared__ double on_smem[];
    OnScratchA &scr = *reinterpret_cast<OnScratchA *>(on_smem + (size_t)threadIdx.x * (sizeof(OnScratchA) / sizeof(double)));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (bool more = true; more; more = sc.dynamic != 0) {
        int g;
        if (!on_next_group(sc, &sc.sched[0], lane, warp, g)) break;
        const int64_t slot = (int64_t)g * 32 + lane;
        if (slot < n) {
            const int64_t e = (int64_t)perm[slot];              // envs of one flight-software task set per warp
            opnav::MeasBuf mb;                                  // this env's column of the hand-over buffer
            mb.p = mbuf + e; mb.stride = stride;
            opnav::opnav_pass1(P, S, I, stride, e, actions[e], scr.c, scr.w, mb);
        }
        __syncwarp();
    }
}

// Three-kernel form (opnav_core.cuh: opnav_pass0 / opnav_pass1_fed): the noise walk of the whole interval first, one thread per
// slot of the lane permutation, a plain grid (every slot costs the same: no queue), registers allocated for ON_NOISE_BLOCKS
// blocks per SM; it writes the slot-major noise buffer that opnav_dyn_kernel -- the first pass without the walk -- consumes one
// tick ahead through its shared scratch.
#ifndef ON_NOISE_BLOCKS
#define ON_NOISE_BLOCKS 6      // 80 registers: 113664 slots are exactly one wave of 148 SMs x 6 blocks x 128 threads
#endif
struct OnScratchN { opnav::Walk w; };                                    // 15 doubles per thread (odd stride: conflict-free)
struct OnScratchD { opnav::Cold c; double feed[30]; };                   // 19 + 2 x 15 = 49 doubles per thread
__global__ void __launch_bounds__(ON_BLOCK, ON_NOISE_BLOCKS)
opnav_noise_kernel(const __grid_constant__ OpNavParams P, double *__restrict__ S, const int64_t *__restrict__ I, int64_t stride, int64_t n,
                   const int32_t *__restrict__ perm, double *__restrict__ nzbuf)
{
    extern __shared__ double on_smem[];
    OnScratchN &scr = *reinterpret_cast<OnScratchN *>(on_smem + (size_t)threadIdx.x * (sizeof(OnScratchN) / sizeof(double)));
    const int64_t slot = (int64_t)blockIdx.x * ON_BLOCK + threadIdx.x;
    if (slot >= n) return;
    opnav::opnav_pass0(P, S, I, stride, (int64_t)perm[slot], scr.w, nzbuf + slot, stride);
}

template <int MINB>
__global__ void ON_STEP_BOUNDS(MINB)
opnav_dyn_kernel(const __grid_constant__ OpNavParams P, double *__restrict__ S, int64_t *__restrict__ I, int64_t stride, int64_t n,
                 const int32_t *__restrict__ actions, const OnSched sc, const int32_t *__restrict__ perm, double *__restrict__ mbuf,
                 const double *__restrict__ nzbuf)
{
    extern __shared__ double on_smem[];
    OnScratchD &scr = *reinterpret_cast<OnScratchD *>(on_smem + (size_t)threadIdx.x * (sizeof(OnScratchD) / sizeof(double)));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (bool more = true; more; more = sc.dynamic != 0) {
        int g;
        if (!on_next_group(sc, &sc.sched[0], lane, warp, g)) break;
        const int64_t slot = (int64_t)g * 32 + lane;
        if (slot < n) {
            const int64_t e = (int64_t)perm[slot];
            opnav::MeasBuf mb;
            mb.p = mbuf + e; mb.stride = stride;
            opnav::NoiseFeed nf;
            nf.g = nzbuf + slot; nf.stride = stride; nf.buf = scr.feed;
            opnav::opnav_pass1_fed(P, S, I, stride, e, actions[e], scr.c, nf, mb);
        }
        __syncwarp();
    }
}

template <int MINB>
__global__ void ON_STEP_BOUNDS(MINB)
opnav_pass2_kernel(const __grid_constant__ OpNavParams P, double *__restrict__ S, int64_t *__restrict__ I, double *__restrict__ ics,
                   int64_t stride, int64_t n, const int32_t *__restrict__ actions, double *__restrict__ obs,
                   double *__restrict__ reward, uint8_t *__restrict__ done, uint8_t *__restrict__ reason,
                   double *__restrict__ debug, double *__restrict__ term_obs, double *__restrict__ stats, const OnSched sc,
                   const int32_t *__restrict__ perm, double *__restrict__ ep_return, int64_t *__restrict__ ep_length,
                   double *__restrict__ mbuf)
{
    extern __shared__ double on_smem[];
    OnScratchB &scr = *reinterpret_cast<OnScratchB *>(on_smem + (size_t)threadIdx.x * (sizeof(OnScratchB) / sizeof(double)));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (bool more = true; more; more = sc.dynamic != 0) {
        int g;
        if (!on_next_group(sc, &sc.sched[5], lane, warp, g)) break;
        const int64_t slot = (int64_t)g * 32 + lane;
        const bool valid = slot < n;
        const int64_t e = valid ? (int64_t)perm[slot] : 0;
        opnav::StepOut o;
        o.done = 0; o.reason = 0; o.reward = 0.;
        double ep_ret = 0., ep_len = 0., d_meas = 0., d_bad = 0.;
        if (valid) {
            const int64_t m0 = I[(int64_t)OI_NMEAS * stride + e], b0 = I[(int64_t)OI_NBAD * stride + e];
            opnav::MeasBuf mb;
            mb.p = mbuf + e; mb.stride = stride;
            opnav::opnav_pass2(P, S, I, stride, e, actions[e], o, scr.f, mb);
            d_meas = (double)(I[(int64_t)OI_NMEAS * stride + e] - m0); d_bad = (double)(I[(int64_t)OI_NBAD * stride + e] - b0);
            reward[e] = o.reward;
            done[e] = (uint8_t)o.done;
            reason[e] = (uint8_t)o.reason;
            if (debug)
                for (int k = 0; k < 12; k++) debug[e * 12 + k] = o.debug[k];
            if (o.done || ep_return) {
                ep_ret = S[(int64_t)OF_EPRET * stride + e];
                ep_len = (double)I[(int64_t)OI_STEP * stride + e];
            }
            if (ep_return) {       // opNavEnvironment.py:106-109: info['episode'] = {'r': reward_total, 'l': curr_step (before its increment)}
                ep_return[e] = ep_ret;
                ep_length[e] = (int64_t)ep_len - 1;
            }
            if (o.done) {
                if (term_obs)
                    for (int k = 0; k < 4; k++) term_obs[e * 4 + k] = o.ob[k];
                if (P.auto_reset) {
                    int64_t ep = I[(int64_t)OI_EPISODE * stride + e] + 1;
                    I[(int64_t)OI_EPISODE * stride + e] = ep;
                    double ic[OPNAV_IC_DIM];
                    opnav::sample_ic(P, P.first_env_index + e, ep, ic);
                    for (int k = 0; k < OPNAV_IC_DIM; k++) ics[(int64_t)k * stride + e] = ic[k];
                    opnav::opnav_reset_env(P, S, I, stride, e, ic, o.ob);
                }
            }
            for (int k = 0; k < 4; k++) obs[e * 4 + k] = o.ob[k];
        }
        if (stats) {
            const unsigned any_done = __ballot_sync(0xffffffffu, valid && o.done);
            if (any_done) {
                double v_ret = warp_sum_d(o.done ? ep_ret : 0.), v_len = warp_sum_d(o.done ? ep_len : 0.);
                int c_all = __popc(any_done);
                int c_m = __popc(__ballot_sync(0xffffffffu, valid && o.done && (o.reason & 1)));
                int c_s = __popc(__ballot_sync(0xffffffffu, valid && o.done && (o.reason & 2)));
                if (lane == 0) {
                    atomicAdd(&stats[OST_RET], v_ret); atomicAdd(&stats[OST_LEN], v_len);
                    atomicAdd(&stats[OST_COUNT], (double)c_all); atomicAdd(&stats[OST_MAXLEN], (double)c_m);
                    atomicAdd(&stats[OST_MODES], (double)c_s);
                }
            }
            const int c_valid = __popc(__ballot_sync(0xffffffffu, valid));
            double v_meas = warp_sum_d(d_meas), v_bad = warp_sum_d(d_bad);
            if (lane == 0 && c_valid) {
                atomicAdd(&stats[OST_STEPS], (double)c_valid);
                atomicAdd(&stats[OST_MEAS], v_meas);
                if (v_bad != 0.0) atomicAdd(&stats[OST_BAD], v_bad);
            }
        }
        __syncwarp();
    }
}

// mode 0: explicit ICs (row-major [n][12]); 1: stored ICs; 2: device-sampled ICs, or a row of the IC pool.  Mode 2 is also
// the auto-reset of a handle with an IC pool (opnav_launch_step: after the last kernel of the interval, mask = done), the
// same sequence as the in-kernel reset of opnav_pass2_kernel.
__global__ void __launch_bounds__(256)
opnav_reset_kernel(const __grid_constant__ OpNavParams P, double *__restrict__ S, int64_t *__restrict__ I, double *__restrict__ ics,
                   int64_t stride, int64_t n, int mode, const double *__restrict__ ics_in, const uint8_t *__restrict__ mask,
                   double *__restrict__ obs, const IcPool icp)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (mask && !mask[e]) return;
    int64_t ep = I[(int64_t)OI_EPISODE * stride + e];
    double ic[OPNAV_IC_DIM];
    if (mode == 0) {
        for (int k = 0; k < OPNAV_IC_DIM; k++) ic[k] = ics_in[e * OPNAV_IC_DIM + k];
    } else if (mode == 1) {
        for (int k = 0; k < OPNAV_IC_DIM; k++) ic[k] = ics[(int64_t)k * stride + e];
    } else {
        I[(int64_t)OI_EPISODE * stride + e] = ++ep;
        if (icp.n_rows > 0) {
            const int64_t r = leo::ic_pool_row(icp, P.seed, P.first_env_index + e, ep, -1);
            for (int k = 0; k < OPNAV_IC_DIM; k++) ic[k] = icp.rows[r * OPNAV_IC_DIM + k];
            icp.row_of[e] = (int32_t)r; icp.row_ep[e] = ep;
        } else {
            opnav::sample_ic(P, P.first_env_index + e, ep, ic);
        }
    }
    if (icp.row_of && mode != 1 && !(mode == 2 && icp.n_rows > 0)) { icp.row_of[e] = -1; icp.row_ep[e] = ep; }
    for (int k = 0; k < OPNAV_IC_DIM; k++) ics[(int64_t)k * stride + e] = ic[k];
    double ob[4];
    opnav::opnav_reset_env(P, S, I, stride, e, ic, ob);
    if (obs)
        for (int k = 0; k < 4; k++) obs[e * 4 + k] = ob[k];
}
__global__ void opnav_gather_ic_rows_kernel(const int32_t *__restrict__ row_of, const int64_t *__restrict__ row_ep,
                                            const int64_t *__restrict__ ep, int64_t n, int32_t *__restrict__ out)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    out[e] = row_ep[e] == ep[e] ? row_of[e] : -1;      // as bskenv.cu: gather_ic_rows_kernel
}
__global__ void opnav_gather_ics_kernel(const double *__restrict__ ics, int64_t stride, int64_t n, double *__restrict__ out)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int k = 0; k < OPNAV_IC_DIM; k++) out[e * OPNAV_IC_DIM + k] = ics[(int64_t)k * stride + e];
}
template <typename T>
__global__ void opnav_copy_fields_kernel(const T *__restrict__ src, int64_t src_stride, T *__restrict__ dst, int64_t dst_stride,
                                         int64_t n, int fields)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int f = 0; f < fields; f++) dst[(int64_t)f * dst_stride + e] = src[(int64_t)f * src_stride + e];
}

thread_local std::string g_opnav_create_error;

}  // namespace

struct bskenv_opnav_handle {
    bskenv_opnav_config cfg;
    OpNavParams P;
    int device;
    int64_t n, stride;
    double *S, *ics, *stats;
    int64_t *I;
    int *sched;
    int32_t *perm;              // lane assignment of the step kernel (envs bucketed by task set)
    double *mbuf;               // measurements of the interval, first pass -> second pass: [slot][ON_MEAS_W][stride]
    double *nzbuf;              // noise walk of the interval, noise kernel -> dynamics kernel: [ticks_per_step + 1][15][stride]
    int noise_split;            // -1 undecided, 0 fused first pass, 1 three-kernel form (nzbuf allocated)
    double *d_eph;              // device copy of the Sun ephemeris table
    int sm_count;
    void *h_stage[6];           // page-locked staging for pageable caller buffers: actions, obs, reward, done, reason, debug
    cudaStream_t own_stream;
    cudaEvent_t ev_last;        // recorded after every launch queued through the device-buffer entry points
    int ev_valid;
    int64_t launches;
    IcPool icp;                 // loaded initial-condition pool (n_rows = 0: none), as in the LEO handle
    std::string err;
};

#define ON_TRY(h, call)                                                                              \
    do {                                                                                             \
        cudaError_t _e = (call);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                            \
            return BSKENV_ECUDA;                                                                     \
        }                                                                                            \
    } while (0)

static int opnav_launch_step(bskenv_opnav_handle *h, const int32_t *act, double *obs, double *rew, uint8_t *done,
                             uint8_t *reason, double *debug, double *term_obs, cudaStream_t st, double *ep_return = nullptr,
                             int64_t *ep_length = nullptr)
{
    // With an IC pool the second pass runs without its in-kernel reset (auto_reset is read nowhere else) and the reset kernel
    // follows the interval, as in bskenv.cu: launch_follow_reset.
    const bool follow = h->icp.n_rows > 0 && h->P.auto_reset;
    OpNavParams P_nr;
    if (follow) { P_nr = h->P; P_nr.auto_reset = 0; }
    const OpNavParams &PK = follow ? P_nr : h->P;
    const int wpb = ON_BLOCK / 32;
    const int64_t groups = (h->n + 31) / 32;
    // First pass (noise + dynamics): 255 registers / two blocks per SM or 168 registers (with spills) / three; measured per full
    // resident set on a B200: 30.2 ms per 37888 envs against 37.9 ms per 56832, and a partial set costs a whole one (latency-
    // bound ticks) -> the shorter predicted launch wins.  Second pass (filter): 168 registers without spills, always three.
    const int64_t set2 = (int64_t)h->sm_count * 2 * ON_BLOCK, set3 = (int64_t)h->sm_count * 3 * ON_BLOCK;
    const int64_t n2 = (h->n + set2 - 1) / set2, n3 = (h->n + set3 - 1) / set3;
    const int minb1 = (ON_MIN_BLOCKS == 3 && n3 * 379 < n2 * 302) ? 3 : 2, minb2 = ON_MIN_BLOCKS == 3 ? 3 : 2;
#ifdef ON_DYN_FORCE_MINB
    const int minb1_dyn = ON_DYN_FORCE_MINB;
#else
    const int minb1_dyn = minb1;
#endif
    const int full = (int)((groups + wpb - 1) / wpb);
    OnSched sc;
    sc.sched = h->sched; sc.n_groups = (int)groups; sc.dynamic = 0;
    ON_TRY(h, cudaMemsetAsync(h->sched, 0, sizeof(int) * 8, st));
    {   // bucket the envs by flight-software task set (two small launches; see opnav_bucket_*_kernel)
        const int bgrid = (int)((h->n + 255) / 256);
        opnav_bucket_count_kernel<<<bgrid, 256, 0, st>>>(h->I, h->stride, h->n, act, h->sched);
        opnav_bucket_fill_kernel<<<bgrid, 256, 0, st>>>(h->I, h->stride, h->n, act, h->sched, h->perm);
    }
    OnSched s1 = sc, s2 = sc;
    const int r1 = h->sm_count * minb1, r2 = h->sm_count * minb2;
    s1.dynamic = full > r1; s2.dynamic = full > r2;
    const int grid1 = full > r1 ? r1 : full, grid2 = full > r2 ? r2 : full;
    const size_t smem_a = sizeof(OnScratchA) * ON_BLOCK, smem_b = sizeof(OnScratchB) * ON_BLOCK;
    static bool attr_set[64] = {false};             // opt in to the dynamic shared memory once per device
    if (!attr_set[h->device & 63]) {
        ON_TRY(h, cudaFuncSetAttribute(opnav_pass1_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a));
        ON_TRY(h, cudaFuncSetAttribute(opnav_pass1_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_a));
        ON_TRY(h, cudaFuncSetAttribute(opnav_pass2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        ON_TRY(h, cudaFuncSetAttribute(opnav_pass2_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        attr_set[h->device & 63] = true;
    }
    if (h->noise_split < 0) {
        // Three-kernel form: OPT-IN (BSKENV_OPNAV_NOISE_SPLIT=1), and only when the noise buffer fits -- 120 B per env-tick, at most
        // ON_NZBUF_MAX_FRAC of the free device memory (113664 envs x 3001 ticks = 40.9 GB).  Measured on a B200: 118.6 against
        // 122.4 ms per 113664 envs (+3 %), 83.1 against 89.1 ms per 75776 envs (+7 %), bit-identical -- for 40.9 GB of memory and
        // 84 GB of DRAM traffic per interval against 1.75 GB: not the default (DESIGN.md 6b).
        h->noise_split = 0;
        const char *split = getenv("BSKENV_OPNAV_NOISE_SPLIT");
        size_t free_b = 0, total_b = 0;
        const size_t need = sizeof(double) * 15 * (size_t)(h->P.ticks_per_step + 1) * (size_t)h->stride;
        if (h->P.nav_noise && split && split[0] == '1' && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess &&
            (double)need <= ON_NZBUF_MAX_FRAC * (double)free_b) {
            if (cudaMalloc(&h->nzbuf, need) == cudaSuccess) h->noise_split = 1;
            else { cudaGetLastError(); h->nzbuf = nullptr; }
        }
    }
    if (h->noise_split == 1) {
        const size_t smem_n = sizeof(OnScratchN) * ON_BLOCK, smem_d = sizeof(OnScratchD) * ON_BLOCK;
        static bool attr_d[64] = {false};
        if (!attr_d[h->device & 63]) {
            ON_TRY(h, cudaFuncSetAttribute(opnav_dyn_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_d));
            ON_TRY(h, cudaFuncSetAttribute(opnav_dyn_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_d));
            attr_d[h->device & 63] = true;
        }
        opnav_noise_kernel<<<(int)((h->n + ON_BLOCK - 1) / ON_BLOCK), ON_BLOCK, smem_n, st>>>(h->P, h->S, h->I, h->stride, h->n, h->perm, h->nzbuf);
        OnSched sd = sc;
        const int rd = h->sm_count * minb1_dyn, gridd = full > rd ? rd : full;
        sd.dynamic = full > rd;
        if (minb1_dyn == 3) opnav_dyn_kernel<3><<<gridd, ON_BLOCK, smem_d, st>>>(h->P, h->S, h->I, h->stride, h->n, act, sd, h->perm, h->mbuf, h->nzbuf);
        else opnav_dyn_kernel<2><<<gridd, ON_BLOCK, smem_d, st>>>(h->P, h->S, h->I, h->stride, h->n, act, sd, h->perm, h->mbuf, h->nzbuf);
        h->launches += 1;
    }
    else if (minb1 == 3) opnav_pass1_kernel<3><<<grid1, ON_BLOCK, smem_a, st>>>(h->P, h->S, h->I, h->stride, h->n, act, s1, h->perm, h->mbuf);
    else opnav_pass1_kernel<2><<<grid1, ON_BLOCK, smem_a, st>>>(h->P, h->S, h->I, h->stride, h->n, act, s1, h->perm, h->mbuf);
    if (minb2 == 3)
        opnav_pass2_kernel<3><<<grid2, ON_BLOCK, smem_b, st>>>(PK, h->S, h->I, h->ics, h->stride, h->n, act, obs, rew, done, reason, debug,
                                                          term_obs, h->stats, s2, h->perm, ep_return, ep_length, h->mbuf);
    else
        opnav_pass2_kernel<2><<<grid2, ON_BLOCK, smem_b, st>>>(PK, h->S, h->I, h->ics, h->stride, h->n, act, obs, rew, done, reason, debug,
                                                          term_obs, h->stats, s2, h->perm, ep_return, ep_length, h->mbuf);
    ON_TRY(h, cudaGetLastError());
    h->launches += 2;
    if (follow) {           // obs / done: the buffers the second pass wrote (device, mapped host or staging memory)
        opnav_reset_kernel<<<(int)((h->n + 255) / 256), 256, 0, st>>>(h->P, h->S, h->I, h->ics, h->stride, h->n, 2, nullptr, done, obs, h->icp);
        ON_TRY(h, cudaGetLastError());
        h->launches++;
    }
    if (st != h->own_stream || !st) { h->ev_valid = 1; ON_TRY(h, cudaEventRecord(h->ev_last, st)); }
    return BSKENV_OK;
}

extern "C" {

void bskenv_opnav_default_config(bskenv_opnav_config *cfg) { opnav_host::default_config(cfg); }
const char *bskenv_opnav_last_error(const bskenv_opnav_handle *h) { return h ? h->err.c_str() : g_opnav_create_error.c_str(); }
int64_t bskenv_opnav_num_envs(const bskenv_opnav_handle *h) { return h ? h->n : 0; }
int64_t bskenv_opnav_launch_count(const bskenv_opnav_handle *h) { return h ? h->launches : 0; }
double bskenv_opnav_flops_per_step(const bskenv_opnav_handle *h) { return h ? opnav_host::flops_per_step(h->P) : 0.0; }

int bskenv_opnav_create(const bskenv_opnav_config *cfg, int device, int64_t n_envs, int64_t first_env_index,
                        bskenv_opnav_handle **out)
{
    if (!cfg || !out || n_envs <= 0) { g_opnav_create_error = "bskenv_opnav_create: bad arguments"; return BSKENV_EINVAL; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        g_opnav_create_error = "bskenv_opnav_create: no CUDA device (this library has no CPU path)";
        return BSKENV_ENODEV;
    }
    if (device < 0 || device >= ndev) { g_opnav_create_error = "bskenv_opnav_create: device index out of range"; return BSKENV_EINVAL; }
    bskenv_opnav_handle *h = new bskenv_opnav_handle();
    h->cfg = *cfg;
    std::string perr = opnav_host::build_params(*cfg, h->P);
    if (!perr.empty()) { g_opnav_create_error = "bskenv_opnav_create: " + perr; delete h; return BSKENV_EINVAL; }
    h->P.first_env_index = first_env_index;
    h->device = device; h->n = n_envs; h->stride = (n_envs + 31) / 32 * 32; h->launches = 0;
    h->S = h->ics = h->stats = nullptr; h->I = nullptr; h->sched = nullptr; h->perm = nullptr; h->d_eph = nullptr; h->mbuf = nullptr; h->nzbuf = nullptr; h->noise_split = -1;
    for (int k = 0; k < 6; k++) h->h_stage[k] = nullptr;
    h->icp.rows = nullptr; h->icp.row_of = nullptr; h->icp.row_ep = nullptr; h->icp.n_rows = 0; h->icp.assign = 0;
    h->own_stream = nullptr; h->ev_last = nullptr; h->ev_valid = 0;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&h->sched, sizeof(int) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&h->perm, sizeof(int32_t) * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->mbuf, sizeof(double) * (size_t)opnav::opnav_meas_slots(h->P) * ON_MEAS_W * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->S, sizeof(double) * OPNAV_ND * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->I, sizeof(int64_t) * OPNAV_NI * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->ics, sizeof(double) * OPNAV_IC_DIM * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->stats, sizeof(double) * OST_N);
    if (e == cudaSuccess) e = cudaMemset(h->S, 0, sizeof(double) * OPNAV_ND * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->I, 0, sizeof(int64_t) * OPNAV_NI * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->ics, 0, sizeof(double) * OPNAV_IC_DIM * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->stats, 0, sizeof(double) * OST_N);
    if (e == cudaSuccess) {              // lane assignment starts as the identity (every slot names a valid env)
        opnav_perm_identity_kernel<<<(int)((h->stride + 255) / 256), 256>>>(h->perm, h->stride, h->n);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        g_opnav_create_error = std::string("bskenv_opnav_create: ") + cudaGetErrorString(e);
        bskenv_opnav_destroy(h);
        return BSKENV_ECUDA;
    }
    *out = h;
    return BSKENV_OK;
}

int bskenv_opnav_destroy(bskenv_opnav_handle *h)
{
    if (!h) return BSKENV_OK;
    cudaSetDevice(h->device);
    cudaFree(h->S); cudaFree(h->I); cudaFree(h->ics); cudaFree(h->stats); cudaFree(h->sched); cudaFree(h->perm); cudaFree(h->d_eph); cudaFree(h->mbuf); cudaFree(h->nzbuf);
    cudaFree((void *)h->icp.rows); cudaFree(h->icp.row_of); cudaFree(h->icp.row_ep);
    if (h->own_stream) { cudaStreamSynchronize(h->own_stream); cudaStreamDestroy(h->own_stream); }
    for (int k = 0; k < 6; k++) cudaFreeHost(h->h_stage[k]);
    if (h->ev_last) cudaEventDestroy(h->ev_last);
    delete h;
    return BSKENV_OK;
}

int bskenv_opnav_set_ephemeris(bskenv_opnav_handle *h, double t0, double seg_len, int n_seg, int n_coef, const double *coef)
{
    if (!h) return BSKENV_EINVAL;
    ON_TRY(h, cudaSetDevice(h->device));
    ON_TRY(h, cudaDeviceSynchronize());
    LeoEph &E = h->P.eph_sun;
    cudaFree(h->d_eph); h->d_eph = nullptr;
    E.coef = nullptr; E.nseg = 0; E.ncoef = 0; E.t0 = 0.; E.seg_len = 0.;
    if (n_seg <= 0) return BSKENV_OK;
    if (!coef || n_coef < 1 || n_coef > 64 || !(seg_len > 0.)) { h->err = "bskenv_opnav_set_ephemeris: bad table shape"; return BSKENV_EINVAL; }
    const double t_end = ((double)h->P.max_length + 1.0) * (double)h->P.ticks_per_step * h->P.dt;   // max_length may be INT_MAX
    if (t0 > 0. || t0 + seg_len * n_seg < t_end) {
        h->err = "bskenv_opnav_set_ephemeris: the table does not cover one episode [0, (max_length + 1) * step_duration]";
        return BSKENV_EINVAL;
    }
    const size_t bytes = sizeof(double) * (size_t)n_seg * 3 * (size_t)n_coef;
    ON_TRY(h, cudaMalloc(&h->d_eph, bytes));
    ON_TRY(h, cudaMemcpy(h->d_eph, coef, bytes, cudaMemcpyHostToDevice));
    E.coef = h->d_eph; E.nseg = n_seg; E.ncoef = n_coef; E.t0 = t0; E.seg_len = seg_len;
    return BSKENV_OK;
}

static int opnav_do_reset(bskenv_opnav_handle *h, int mode, const double *ics_in, const uint8_t *mask, double *obs, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    ON_TRY(h, cudaSetDevice(h->device));
    const int grid = (int)((h->n + 255) / 256);
    opnav_reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(h->P, h->S, h->I, h->ics, h->stride, h->n, mode, ics_in, mask, obs, h->icp);
    ON_TRY(h, cudaGetLastError());
    h->ev_valid = 1; ON_TRY(h, cudaEventRecord(h->ev_last, (cudaStream_t)stream));
    return BSKENV_OK;
}
int bskenv_opnav_reset_seeded(bskenv_opnav_handle *h, uint64_t seed, const uint8_t *mask_dev, double *obs_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    h->P.seed = seed;             // the IC stream and the sensor-noise streams share the key from here on
    return opnav_do_reset(h, 2, nullptr, mask_dev, obs_dev, stream);
}
int bskenv_opnav_reset_ics(bskenv_opnav_handle *h, const double *ics_dev, const uint8_t *mask_dev, double *obs_dev, void *stream)
{
    if (!h || !ics_dev) { if (h) h->err = "bskenv_opnav_reset_ics: null ics"; return BSKENV_EINVAL; }
    return opnav_do_reset(h, 0, ics_dev, mask_dev, obs_dev, stream);
}
int bskenv_opnav_reset_init(bskenv_opnav_handle *h, const uint8_t *mask_dev, double *obs_dev, void *stream)
{
    return opnav_do_reset(h, 1, nullptr, mask_dev, obs_dev, stream);
}
int bskenv_opnav_get_ics(bskenv_opnav_handle *h, double *ics_dev, void *stream)
{
    if (!h || !ics_dev) return BSKENV_EINVAL;
    ON_TRY(h, cudaSetDevice(h->device));
    opnav_gather_ics_kernel<<<(int)((h->n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->ics, h->stride, h->n, ics_dev);
    ON_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

int bskenv_opnav_set_ic_pool(bskenv_opnav_handle *h, int n_rows, const double *ics_host, int assign)
{
    if (!h) return BSKENV_EINVAL;
    if (n_rows < 0 || (n_rows > 0 && !ics_host)) { h->err = "bskenv_opnav_set_ic_pool: bad row count or null rows"; return BSKENV_EINVAL; }
    if (n_rows > 0) {
        if (assign != BSKENV_ICS_BY_INDEX && assign != BSKENV_ICS_PER_EPISODE) {
            h->err = "bskenv_opnav_set_ic_pool: unknown assignment mode (the opNav batch has no parameter pool to pair with)";
            return BSKENV_EINVAL;
        }
        for (int r = 0; r < n_rows; r++) {
            const std::string err = leo_host::ic_row_check(ics_host + (size_t)r * BSKENV_OPNAV_IC_DIM, BSKENV_OPNAV_IC_DIM);
            if (!err.empty()) { h->err = "bskenv_opnav_set_ic_pool: row " + std::to_string(r) + ": " + err; return BSKENV_EINVAL; }
        }
    }
    ON_TRY(h, cudaSetDevice(h->device));
    ON_TRY(h, cudaDeviceSynchronize());                         // a launch in flight may still read the old pool
    cudaFree((void *)h->icp.rows);
    h->icp.rows = nullptr; h->icp.n_rows = 0;
    if (n_rows == 0) return BSKENV_OK;
    if (!h->icp.row_of) {
        ON_TRY(h, cudaMalloc(&h->icp.row_of, sizeof(int32_t) * h->stride));
        ON_TRY(h, cudaMalloc(&h->icp.row_ep, sizeof(int64_t) * h->stride));
        ON_TRY(h, cudaMemset(h->icp.row_of, 0xFF, sizeof(int32_t) * h->stride));
        ON_TRY(h, cudaMemset(h->icp.row_ep, 0, sizeof(int64_t) * h->stride));
    }
    double *d_rows = nullptr;
    const size_t bytes = sizeof(double) * (size_t)n_rows * BSKENV_OPNAV_IC_DIM;
    ON_TRY(h, cudaMalloc(&d_rows, bytes));
    ON_TRY(h, cudaMemcpy(d_rows, ics_host, bytes, cudaMemcpyHostToDevice));
    h->icp.rows = d_rows; h->icp.n_rows = n_rows; h->icp.assign = assign;
    return BSKENV_OK;
}

int bskenv_opnav_get_ic_rows(bskenv_opnav_handle *h, int32_t *rows_dev, void *stream)
{
    if (!h || !rows_dev) { if (h) h->err = "bskenv_opnav_get_ic_rows: null rows"; return BSKENV_EINVAL; }
    ON_TRY(h, cudaSetDevice(h->device));
    if (!h->icp.row_of) ON_TRY(h, cudaMemsetAsync(rows_dev, 0xFF, sizeof(int32_t) * h->n, (cudaStream_t)stream));
    else opnav_gather_ic_rows_kernel<<<(int)((h->n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->icp.row_of, h->icp.row_ep,
                                                                                                  h->I + (size_t)OI_EPISODE * h->stride, h->n, rows_dev);
    ON_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

int bskenv_opnav_step(bskenv_opnav_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev, uint8_t *done_dev,
                      uint8_t *done_reason_dev, double *debug_dev, double *term_obs_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions_dev || !obs_dev || !reward_dev || !done_dev || !done_reason_dev) { h->err = "bskenv_opnav_step: null buffer"; return BSKENV_EINVAL; }
    ON_TRY(h, cudaSetDevice(h->device));
    return opnav_launch_step(h, actions_dev, obs_dev, reward_dev, done_dev, done_reason_dev, debug_dev, term_obs_dev, (cudaStream_t)stream);
}

int bskenv_opnav_step_info(bskenv_opnav_handle *h, const int32_t *actions_dev, double *obs_dev, double *reward_dev, uint8_t *done_dev,
                           uint8_t *done_reason_dev, double *debug_dev, double *term_obs_dev, double *ep_return_dev,
                           int64_t *ep_length_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions_dev || !obs_dev || !reward_dev || !done_dev || !done_reason_dev) { h->err = "bskenv_opnav_step_info: null buffer"; return BSKENV_EINVAL; }
    if ((ep_return_dev == nullptr) != (ep_length_dev == nullptr)) { h->err = "bskenv_opnav_step_info: ep_return and ep_length go together"; return BSKENV_EINVAL; }
    ON_TRY(h, cudaSetDevice(h->device));
    return opnav_launch_step(h, actions_dev, obs_dev, reward_dev, done_dev, done_reason_dev, debug_dev, term_obs_dev, (cudaStream_t)stream,
                             ep_return_dev, ep_length_dev);
}

// Host-buffer entry point: zero-copy, as bskenv_step_host (bskenv.cu) -- the kernel reads the actions from and writes its
// results to page-locked host memory directly; pageable caller buffers go through staging owned by the handle.
static int opnav_host_map(bskenv_opnav_handle *h, const void *user, size_t bytes, int slot, void **dev, void **stage)
{
    *stage = nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, user) == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer) { *dev = a.devicePointer; return BSKENV_OK; }
    cudaGetLastError();
    if (!h->h_stage[slot]) ON_TRY(h, cudaHostAlloc(&h->h_stage[slot], bytes, cudaHostAllocMapped));
    *stage = h->h_stage[slot];
    ON_TRY(h, cudaHostGetDevicePointer(dev, *stage, 0));
    return BSKENV_OK;
}

int bskenv_opnav_step_host(bskenv_opnav_handle *h, const int32_t *actions, double *obs, double *reward, uint8_t *done,
                           uint8_t *done_reason, double *debug)
{
    if (!h) return BSKENV_EINVAL;
    if (!actions || !obs || !reward || !done || !done_reason) { h->err = "bskenv_opnav_step_host: null buffer"; return BSKENV_EINVAL; }
    ON_TRY(h, cudaSetDevice(h->device));
    const size_t n = (size_t)h->n;
    if (!h->own_stream) ON_TRY(h, cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    cudaStream_t st = h->own_stream;
    void *user[6] = {(void *)actions, obs, reward, done, done_reason, debug};
    const size_t bytes[6] = {n * sizeof(int32_t), n * 4 * sizeof(double), n * sizeof(double), n, n, n * 12 * sizeof(double)};
    void *dev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}, *stage[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    for (int k = 0; k < 6; k++) {
        if (!user[k]) continue;
        int rc = opnav_host_map(h, user[k], bytes[k], k, &dev[k], &stage[k]);
        if (rc) return rc;
    }
    if (stage[0]) memcpy(stage[0], actions, bytes[0]);
    if (h->ev_valid) ON_TRY(h, cudaStreamWaitEvent(st, h->ev_last, 0));     // after the caller's device-buffer steps / resets
    int rc = opnav_launch_step(h, (const int32_t *)dev[0], (double *)dev[1], (double *)dev[2], (uint8_t *)dev[3], (uint8_t *)dev[4],
                               (double *)dev[5], nullptr, st);
    if (rc) return rc;
    ON_TRY(h, cudaStreamSynchronize(st));
    for (int k = 1; k < 6; k++)
        if (stage[k]) memcpy(user[k], stage[k], bytes[k]);
    return BSKENV_OK;
}

int bskenv_opnav_state_dims(const bskenv_opnav_handle *h, int32_t *nd, int32_t *ni)
{
    (void)h;
    if (nd) *nd = OPNAV_ND;
    if (ni) *ni = OPNAV_NI;
    return BSKENV_OK;
}
int bskenv_opnav_get_state(bskenv_opnav_handle *h, double *dstate_dev, int64_t *istate_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    ON_TRY(h, cudaSetDevice(h->device));
    const int grid = (int)((h->n + 255) / 256);
    if (dstate_dev) opnav_copy_fields_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(h->S, h->stride, dstate_dev, h->n, h->n, OPNAV_ND);
    if (istate_dev) opnav_copy_fields_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>(h->I, h->stride, istate_dev, h->n, h->n, OPNAV_NI);
    ON_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}
int bskenv_opnav_set_state(bskenv_opnav_handle *h, const double *dstate_dev, const int64_t *istate_dev, void *stream)
{
    if (!h) return BSKENV_EINVAL;
    ON_TRY(h, cudaSetDevice(h->device));
    const int grid = (int)((h->n + 255) / 256);
    if (dstate_dev) opnav_copy_fields_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(dstate_dev, h->n, h->S, h->stride, h->n, OPNAV_ND);
    if (istate_dev) opnav_copy_fields_kernel<int64_t><<<grid, 256, 0, (cudaStream_t)stream>>>(istate_dev, h->n, h->I, h->stride, h->n, OPNAV_NI);
    ON_TRY(h, cudaGetLastError());
    h->ev_valid = 1; ON_TRY(h, cudaEventRecord(h->ev_last, (cudaStream_t)stream));
    return BSKENV_OK;
}
int bskenv_opnav_state_field(const char *name, int32_t *is_int)
{
    struct Ent { const char *n; int idx; int is_int; };
    static const Ent tab[] = {
        {"r_BN_N", OF_R, 0}, {"v_BN_N", OF_V, 0}, {"sigma_BN", OF_SIG, 0}, {"omega_BN_B", OF_OMG, 0}, {"Omega", OF_WHL, 0},
        {"reactionwheel_cmds", OF_RWCMD, 0}, {"navErrors", OF_NAVERR, 0}, {"sun_point_data", OF_SUNPT, 0},
        {"shadowFactor", OF_SHADOW, 0}, {"filter_state", OF_FSTATE, 0}, {"filter_sBar", OF_FS, 0},
        {"reward_total", OF_EPRET, 0}, {"sim_obs", OF_OBS, 0}, {"sim_states", OF_DEBUG, 0},
        {"tick", OI_TICK, 1}, {"curr_step", OI_STEP, 1}, {"mode", OI_MODE, 1}, {"cameraIsOn", OI_CAMERA, 1},
        {"modeCounter", OI_MODECNT, 1}, {"first_run", OI_FIRST, 1}, {"MRPSwitchCount", OI_SWITCH, 1}, {"episode", OI_EPISODE, 1},
        {"episode_over", OI_OVER, 1}, {"n_meas", OI_NMEAS, 1}, {"n_bad", OI_NBAD, 1}, {"filter_tick", OI_FTICK, 1},
        {"sun_point_written", OI_SUNPT_W, 1}, {"n_images", OI_NIMG, 1}};
    if (!name) return -1;
    for (const Ent &t : tab)
        if (!strcmp(t.n, name)) { if (is_int) *is_int = t.is_int; return t.idx; }
    return -1;
}

int bskenv_opnav_episode_stats(bskenv_opnav_handle *h, double *stats_host)
{
    if (!h || !stats_host) return BSKENV_EINVAL;
    ON_TRY(h, cudaSetDevice(h->device));
    ON_TRY(h, cudaDeviceSynchronize());
    ON_TRY(h, cudaMemcpy(stats_host, h->stats, sizeof(double) * OST_N, cudaMemcpyDeviceToHost));
    ON_TRY(h, cudaMemset(h->stats, 0, sizeof(double) * OST_N));
    return BSKENV_OK;
}

}  // extern "C"
