// batch_common.cuh -- the handle layer the LEO batch (bskenv.cu) and the opNav batch (opnav.cu) share: the handle core,
// the IC choice of a reset, and the entry points around the step kernels that differ only in dimensions (create / destroy,
// ephemeris tables, IC pools, stored ICs, state blocks, statistics, host-buffer mapping, launch ordering), the lane
// bucketing before a step and the dynamic-shared-memory opt-in of the step kernels.
#pragma once
#include <cuda_runtime.h>
#include <string.h>
#include <string>

#include "../../include/bskenv.h"
#include "leo_core.cuh"
#include "leo_host.h"

#define CU_TRY(h, ...)         /* variadic: the call may name a template with several arguments */          \
    do {                                                                                             \
        cudaError_t _e = (__VA_ARGS__);                                                              \
        if (_e != cudaSuccess) {                                                                     \
            (h)->err = std::string(#__VA_ARGS__) + ": " + cudaGetErrorString(_e);                     \
            return BSKENV_ECUDA;                                                                     \
        }                                                                                            \
    } while (0)

// What every batch handle holds; bskenv_handle and bskenv_opnav_handle derive from it.
struct BatchCore {
    int device = 0;
    int64_t n = 0, stride = 0;  // envs, and the column pitch of the state blocks (n rounded up to whole warps)
    double *S = nullptr, *ics = nullptr, *stats = nullptr;
    int64_t *I = nullptr;
    int sm_count = 0;
    void *h_stage[8] = {};      // page-locked staging of the host-buffer entry points, one per buffer slot (pageable caller buffers)
    int host_pending = 0;       // a host-buffer step was queued and not waited for (LEO's bskenv_step_host_async; 0 for opNav)
    cudaStream_t own_stream = nullptr;  // the stream of the host-buffer entry points
    cudaEvent_t ev_last = nullptr;      // recorded after every launch queued through the device-buffer entry points
    int ev_valid = 0;
    int64_t launches = 0;
    IcPool icp{};               // loaded initial-condition pool (n_rows = 0: none); rows and per-env record in device memory
    uint64_t fingerprint = 0;   // of the configuration (snapshot records), set at create
    unsigned long long *snap_chk = nullptr;     // check words of snapshot / restore (allocated at first use)
    uint32_t *snap_owner = nullptr;             // [n]: lowest record position naming each env (restore with explicit indices)
    std::string err;
};

// FNV-1a, 64 bit: the configuration fingerprint of snapshot records, fed field by field (no padding or reserved words)
struct Fnv64 {
    uint64_t h = 14695981039346656037ull;
    template <typename T>
    void add(const T &v)
    {
        const unsigned char *p = reinterpret_cast<const unsigned char *>(&v);
        for (size_t i = 0; i < sizeof(T); i++) { h ^= p[i]; h *= 1099511628211ull; }
    }
    template <typename T, size_t N>
    void add(const T (&v)[N]) { for (size_t i = 0; i < N; i++) add(v[i]); }
};

namespace {

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// The initial conditions of a reset, stored into `ics`.  mode 0: explicit ICs (row-major [n][DIM]); 1: the stored ones
// (reset_init); 2: a row of the IC pool when one is loaded (row picked with the parameter row `prow` of this reset, -1 without
// one), else sample(ic).  The IC-pool record of the env becomes the drawn row, or -1 after explicit or sampled ICs; mode 1
// keeps it.  ep = the env's episode after the reset.
template <int DIM, class Sample>
__device__ __forceinline__ void reset_ics(int mode, const double *__restrict__ ics_in, double *__restrict__ ics, int64_t stride,
                                          int64_t e, int64_t global_env, uint64_t seed, int64_t ep, int64_t prow, const IcPool &icp,
                                          Sample sample, double (&ic)[DIM])
{
    if (mode == 0) {
        for (int k = 0; k < DIM; k++) ic[k] = ics_in[e * DIM + k];
    } else if (mode == 1) {
        for (int k = 0; k < DIM; k++) ic[k] = ics[(int64_t)k * stride + e];
    } else if (icp.n_rows > 0) {
        const int64_t r = leo::ic_pool_row(icp, seed, global_env, ep, prow);
        for (int k = 0; k < DIM; k++) ic[k] = icp.rows[r * DIM + k];
        icp.row_of[e] = (int32_t)r; icp.row_ep[e] = ep;
    } else {
        sample(ic);
    }
    if (icp.row_of && mode != 1 && !(mode == 2 && icp.n_rows > 0)) { icp.row_of[e] = -1; icp.row_ep[e] = ep; }
    for (int k = 0; k < DIM; k++) ics[(int64_t)k * stride + e] = ic[k];
}

template <int DIM>
__global__ void gather_ics_kernel(const double *__restrict__ ics, int64_t stride, int64_t n, double *__restrict__ out)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    for (int k = 0; k < DIM; k++) out[e * DIM + k] = ics[(int64_t)k * stride + e];
}
// get_ic_rows: the recorded row where it belongs to the env's current episode (an in-kernel reset after an unload advances
// the episode counter without touching the record)
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

// Lane bucketing before a step: a counting sort of the envs into the lane permutation `perm` of the step kernel, so that a
// warp takes 32 envs of one bucket (warp-aggregated atomics, one count and one fill launch).  rank(e) = the position of env
// e's bucket in the permutation, 0 .. NB - 1; bucket rank r starts after the sizes of all lower ranks.  bucket[0 .. NB-1] =
// sizes, bucket[NB .. 2 NB-1] = cursors, zeroed before the count launch.  Within a bucket the envs of a warp are in index
// order and the warps in the order they reach the cursor.
template <int NB, class Rank>
__global__ void __launch_bounds__(256) bucket_count_kernel(int64_t n, const Rank rank, int *__restrict__ bucket)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int r = e < n ? rank(e) : -1;
#pragma unroll
    for (int c = 0; c < NB; c++) {
        const unsigned m = __ballot_sync(0xffffffffu, r == c);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&bucket[c], __popc(m));
    }
}
template <int NB, class Rank>
__global__ void __launch_bounds__(256) bucket_fill_kernel(int64_t n, const Rank rank, int *__restrict__ bucket, int32_t *__restrict__ perm)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int r = e < n ? rank(e) : -1;
    const int lane = threadIdx.x & 31;
    int size[NB];                                               // final since the count launch: loaded before the first atomic
#pragma unroll
    for (int c = 0; c < NB; c++) size[c] = bucket[c];
    int first = 0;                                              // start of bucket c in the permutation
#pragma unroll
    for (int c = 0; c < NB; c++) {
        const unsigned m = __ballot_sync(0xffffffffu, r == c);
        if (m) {
            const int leader = __ffs(m) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(&bucket[NB + c], __popc(m));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (r == c) perm[first + base + __popc(m & ((1u << lane) - 1))] = (int32_t)e;
        }
        first += size[c];
    }
}

inline int env_grid(const BatchCore *h) { return (int)((h->n + 255) / 256); }

// Opts Kernel in to `bytes` of dynamic shared memory (beyond the 48 KB default) once per device; every launch of Kernel asks
// for the same amount.  One flag array per kernel.
template <auto Kernel>
cudaError_t allow_dynamic_smem(int device, size_t bytes)
{
    static bool done[64] = {};
    if (done[device & 63]) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) done[device & 63] = true;
    return e;
}

// Launches queued on the caller's streams are ordered before a later host-buffer step (which runs on the handle's own
// stream) through this event.
inline cudaError_t note_launch(BatchCore *h, cudaStream_t st)
{
    h->ev_valid = 1;
    return cudaEventRecord(h->ev_last, st);
}

// The checks of a create call before the handle exists; the message goes to `err`, the calling thread's create error.
inline int check_create(const char *what, bool args_ok, int device, std::string &err)
{
    if (!args_ok) { err = std::string(what) + ": bad arguments"; return BSKENV_EINVAL; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        err = std::string(what) + ": no CUDA device (this library has no CPU path)";
        return BSKENV_ENODEV;
    }
    if (device < 0 || device >= ndev) { err = std::string(what) + ": device index out of range"; return BSKENV_EINVAL; }
    return BSKENV_OK;
}

// The allocations every handle makes: the ordering event, the zeroed state blocks S [nd][stride] and I [ni][stride], the
// stored ICs [ic_dim][stride] and the n_stats episode statistics.
inline cudaError_t core_alloc(BatchCore *h, int device, int64_t n_envs, int nd, int ni, int ic_dim, int n_stats)
{
    h->device = device; h->n = n_envs; h->stride = (n_envs + 31) / 32 * 32;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaMalloc(&h->S, sizeof(double) * nd * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->I, sizeof(int64_t) * ni * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->ics, sizeof(double) * ic_dim * h->stride);
    if (e == cudaSuccess) e = cudaMalloc(&h->stats, sizeof(double) * n_stats);
    if (e == cudaSuccess) e = cudaMemset(h->S, 0, sizeof(double) * nd * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->I, 0, sizeof(int64_t) * ni * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->ics, 0, sizeof(double) * ic_dim * h->stride);
    if (e == cudaSuccess) e = cudaMemset(h->stats, 0, sizeof(double) * n_stats);
    return e;
}

// Frees what core_alloc and the shared entry points allocated (the current device is the handle's)
inline void core_free(BatchCore *h)
{
    cudaFree(h->S); cudaFree(h->I); cudaFree(h->ics); cudaFree(h->stats);
    cudaFree((void *)h->icp.rows); cudaFree(h->icp.row_of); cudaFree(h->icp.row_ep);
    cudaFree(h->snap_chk); cudaFree(h->snap_owner);
    if (h->own_stream) { cudaStreamSynchronize(h->own_stream); cudaStreamDestroy(h->own_stream); }
    for (void *p : h->h_stage) cudaFreeHost(p);
    if (h->ev_last) cudaEventDestroy(h->ev_last);
}

// Loads a Chebyshev ephemeris table into E (n_seg <= 0: none, back to the analytic model).  The table has to cover one
// episode, sim time 0 to t_end.  E.coef is the device copy.
inline int set_ephemeris(BatchCore *h, const char *what, LeoEph &E, double t_end, double t0, double seg_len, int n_seg, int n_coef,
                         const double *coef)
{
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());                         // a launch in flight may still read the old table
    cudaFree((void *)E.coef);
    E.coef = nullptr; E.nseg = 0; E.ncoef = 0; E.t0 = 0.; E.seg_len = 0.;
    if (n_seg <= 0) return BSKENV_OK;
    if (!coef || n_coef < 1 || n_coef > 64 || !(seg_len > 0.)) { h->err = std::string(what) + ": bad table shape"; return BSKENV_EINVAL; }
    if (t0 > 0. || t0 + seg_len * n_seg < t_end) {
        h->err = std::string(what) + ": the table does not cover one episode [0, (max_length + 1) * step_duration]";
        return BSKENV_EINVAL;
    }
    const size_t bytes = sizeof(double) * (size_t)n_seg * 3 * (size_t)n_coef;
    double *d = nullptr;
    CU_TRY(h, cudaMalloc(&d, bytes));
    E.coef = d;
    CU_TRY(h, cudaMemcpy(d, coef, bytes, cudaMemcpyHostToDevice));
    E.nseg = n_seg; E.ncoef = n_coef; E.t0 = t0; E.seg_len = seg_len;
    return BSKENV_OK;
}

// Loads n_rows IC rows of dim numbers each (n_rows = 0 unloads the pool: resets sample again, the in-kernel auto-reset).
// mode_error(): the batch's refusal of `assign` ("" = accepted), checked after the arguments and before the rows.
template <class ModeError>
int set_ic_pool(BatchCore *h, const char *what, int n_rows, const double *rows_host, int dim, int assign, ModeError mode_error)
{
    if (n_rows < 0 || (n_rows > 0 && !rows_host)) { h->err = std::string(what) + ": bad row count or null rows"; return BSKENV_EINVAL; }
    if (n_rows > 0) {
        const std::string merr = mode_error();
        if (!merr.empty()) { h->err = merr; return BSKENV_EINVAL; }
        for (int r = 0; r < n_rows; r++) {
            const std::string err = leo_host::ic_row_check(rows_host + (size_t)r * dim, dim);
            if (!err.empty()) { h->err = std::string(what) + ": row " + std::to_string(r) + ": " + err; return BSKENV_EINVAL; }
        }
    }
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());                         // a launch in flight may still read the old pool
    cudaFree((void *)h->icp.rows);
    h->icp.rows = nullptr; h->icp.n_rows = 0;
    if (n_rows == 0) return BSKENV_OK;
    if (!h->icp.row_of) {                                       // first pool of this handle: the per-env record, all -1
        CU_TRY(h, cudaMalloc(&h->icp.row_of, sizeof(int32_t) * h->stride));
        CU_TRY(h, cudaMalloc(&h->icp.row_ep, sizeof(int64_t) * h->stride));
        CU_TRY(h, cudaMemset(h->icp.row_of, 0xFF, sizeof(int32_t) * h->stride));
        CU_TRY(h, cudaMemset(h->icp.row_ep, 0, sizeof(int64_t) * h->stride));
    }
    double *d_rows = nullptr;
    const size_t bytes = sizeof(double) * (size_t)n_rows * dim;
    CU_TRY(h, cudaMalloc(&d_rows, bytes));
    CU_TRY(h, cudaMemcpy(d_rows, rows_host, bytes, cudaMemcpyHostToDevice));
    h->icp.rows = d_rows; h->icp.n_rows = n_rows; h->icp.assign = assign;
    return BSKENV_OK;
}

// ep_field: the episode counter's field in I
inline int get_ic_rows(BatchCore *h, const char *what, int ep_field, int32_t *rows_dev, void *stream)
{
    if (!rows_dev) { h->err = std::string(what) + ": null rows"; return BSKENV_EINVAL; }
    CU_TRY(h, cudaSetDevice(h->device));
    if (!h->icp.row_of) CU_TRY(h, cudaMemsetAsync(rows_dev, 0xFF, sizeof(int32_t) * h->n, (cudaStream_t)stream));
    else gather_ic_rows_kernel<<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(h->icp.row_of, h->icp.row_ep,
                                                                              h->I + (size_t)ep_field * h->stride, h->n, rows_dev);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

template <int DIM>
int get_ics(BatchCore *h, double *ics_dev, void *stream)
{
    if (!ics_dev) return BSKENV_EINVAL;
    CU_TRY(h, cudaSetDevice(h->device));
    gather_ics_kernel<DIM><<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(h->ics, h->stride, h->n, ics_dev);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

// The persistent state as dense [nd][n] doubles and [ni][n] integers (either may be null)
inline int get_state(BatchCore *h, int nd, int ni, double *dstate_dev, int64_t *istate_dev, void *stream)
{
    CU_TRY(h, cudaSetDevice(h->device));
    if (dstate_dev) copy_fields_kernel<double><<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(h->S, h->stride, dstate_dev, h->n, h->n, nd);
    if (istate_dev) copy_fields_kernel<int64_t><<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(h->I, h->stride, istate_dev, h->n, h->n, ni);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}
inline int set_state(BatchCore *h, int nd, int ni, const double *dstate_dev, const int64_t *istate_dev, void *stream)
{
    CU_TRY(h, cudaSetDevice(h->device));
    if (dstate_dev) copy_fields_kernel<double><<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(dstate_dev, h->n, h->S, h->stride, h->n, nd);
    if (istate_dev) copy_fields_kernel<int64_t><<<env_grid(h), 256, 0, (cudaStream_t)stream>>>(istate_dev, h->n, h->I, h->stride, h->n, ni);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, note_launch(h, (cudaStream_t)stream));
    return BSKENV_OK;
}

// Copies the n_stats episode statistics to the host and zeroes them (after everything queued on the device)
inline int episode_stats(BatchCore *h, int n_stats, double *stats_host)
{
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaDeviceSynchronize());
    CU_TRY(h, cudaMemcpy(stats_host, h->stats, sizeof(double) * n_stats, cudaMemcpyDeviceToHost));
    CU_TRY(h, cudaMemset(h->stats, 0, sizeof(double) * n_stats));
    return BSKENV_OK;
}

// Host-buffer entry points: the step kernels read the actions from and write their results to PINNED HOST memory directly
// (zero-copy over PCIe).  Caller buffers that are already page-locked (bskenv_alloc_host, cudaHostRegister, torch pin_memory)
// are used in place: *dev is their device-visible address, *stage null.  Pageable ones go through the handle's page-locked
// staging block of `slot` (*stage), and the caller copies in or out with one memcpy.
inline int host_map(BatchCore *h, const void *user, size_t bytes, int slot, void **dev, void **stage)
{
    *stage = nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, user) == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer) { *dev = a.devicePointer; return BSKENV_OK; }
    cudaGetLastError();
    if (!h->h_stage[slot]) CU_TRY(h, cudaHostAlloc(&h->h_stage[slot], bytes, cudaHostAllocMapped));
    *stage = h->h_stage[slot];
    CU_TRY(h, cudaHostGetDevicePointer(dev, *stage, 0));
    return BSKENV_OK;
}

// The start of a host-buffer step on the handle's own stream: maps the k caller buffers through host_map (slot s = user[s],
// null when not passed; dev[s] = the address the kernels use, stage[s] = its staging block or null), copies the actions
// (slot 0) into their stage, and orders the stream after whatever the caller queued on its own streams through the
// device-buffer entry points.
inline int host_step_begin(BatchCore *h, int k, void *const *user, const size_t *bytes, void **dev, void **stage)
{
    if (!h->own_stream) CU_TRY(h, cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    for (int s = 0; s < k; s++) {
        dev[s] = stage[s] = nullptr;
        if (!user[s]) continue;
        const int rc = host_map(h, user[s], bytes[s], s, &dev[s], &stage[s]);
        if (rc) return rc;
    }
    if (stage[0]) memcpy(stage[0], user[0], bytes[0]);
    if (h->ev_valid) CU_TRY(h, cudaStreamWaitEvent(h->own_stream, h->ev_last, 0));
    return BSKENV_OK;
}
// ... and its end, once the stream has completed: the staged results (slots 1 .. k-1 with both a caller buffer and a stage)
// copied to the caller
inline void host_step_copy_back(int k, void *const *user, void *const *stage, const size_t *bytes)
{
    for (int s = 1; s < k; s++)
        if (user[s] && stage[s]) memcpy(user[s], stage[s], bytes[s]);
}

// ---- per-env state snapshots (bskenv_snapshot / bskenv_restore and the opNav pair) ----------------------------------------
// A record is one row of L::W 8-byte words: header (kind << 16 | version, W, fingerprint, source global index), the ND double
// and NI integer state fields, the DIC stored ICs, the NPD-field parameter block (LEO; PROW = its pool-row field) and the
// IC-pool row.  EP = the episode counter's field in I.  The kernels move SNAP_ROWS records per block through a shared-memory
// tile of odd pitch (conflict-free 8-byte accesses both ways): state columns on one side -- one warp reads one field of 32
// records, coalesced when the envs are consecutive -- and one contiguous run of SNAP_ROWS * W record words on the other.
template <int KIND_, int ND_, int NI_, int DIC_, int NPD_, int PROW_, int EP_>
struct SnapLayout {
    enum : int {
        KIND = KIND_, ND = ND_, NI = NI_, DIC = DIC_, NPD = NPD_, PROW = PROW_, EP = EP_,
        OFF_S = 4, OFF_I = OFF_S + ND, OFF_IC = OFF_I + NI, OFF_P = OFF_IC + DIC, OFF_ROW = OFF_P + NPD, W = OFF_ROW + 1,
        PITCH = W | 1
    };
    static constexpr int64_t TAG = (int64_t)KIND << 16 | BSKENV_SNAPSHOT_VERSION;
};
#define SNAP_ROWS 32
#define SNAP_THREADS 256

// What the snapshot kernels address of a handle.  live: the parameter block behind the state fields holds each env's values
// (a parameter pool is loaded); otherwise a snapshot writes `batch` (SnapBlock) and a restore leaves the block alone.
struct SnapCols {
    double *S; int64_t *I; double *ics; int32_t *row_of; int64_t *row_ep;
    int64_t stride, n, first_env_index; uint64_t fingerprint; int live;
};
template <int NPD> struct SnapBlock { double v[NPD > 0 ? NPD : 1]; };

// Word w (>= 0) of env e's record
template <class L>
__device__ __forceinline__ double snap_word(const SnapCols &c, const SnapBlock<L::NPD> &batch, int64_t e, int w)
{
    const int64_t s = c.stride;
    if (w < L::OFF_S) {
        const int64_t v = w == 0 ? L::TAG : (w == 1 ? (int64_t)L::W : (w == 2 ? (int64_t)c.fingerprint : c.first_env_index + e));
        return __longlong_as_double(v);
    }
    if (w < L::OFF_I) return c.S[(int64_t)(w - L::OFF_S) * s + e];
    if (w < L::OFF_IC) return __longlong_as_double(c.I[(int64_t)(w - L::OFF_I) * s + e]);
    if (w < L::OFF_P) return c.ics[(int64_t)(w - L::OFF_IC) * s + e];
    if (w < L::OFF_ROW) return c.live ? c.S[(int64_t)(L::ND + w - L::OFF_P) * s + e] : batch.v[w - L::OFF_P];
    const int64_t row = (c.row_of && c.row_ep[e] == c.I[(int64_t)L::EP * s + e]) ? (int64_t)c.row_of[e] : -1;
    return __longlong_as_double(row);
}

// m records of the envs `envs` (null: envs 0 .. m-1) -> rec [m][W]
template <class L>
__global__ void __launch_bounds__(SNAP_THREADS)
snapshot_gather_kernel(const SnapCols c, const SnapBlock<L::NPD> batch, int64_t m, const int64_t *__restrict__ envs, double *__restrict__ rec)
{
    __shared__ double tile[SNAP_ROWS * L::PITCH];
    const int64_t r0 = (int64_t)blockIdx.x * SNAP_ROWS;
    const int rows = (int)(m - r0 < SNAP_ROWS ? m - r0 : SNAP_ROWS);
    for (int t = threadIdx.x; t < SNAP_ROWS * L::W; t += SNAP_THREADS) {     // a warp: one word of 32 records
        const int r = t % SNAP_ROWS, w = t / SNAP_ROWS;
        if (r < rows) tile[r * L::PITCH + w] = snap_word<L>(c, batch, envs ? envs[r0 + r] : r0 + r, w);
    }
    __syncthreads();
    double *out = rec + r0 * L::W;
    for (int t = threadIdx.x; t < rows * L::W; t += SNAP_THREADS) out[t] = tile[(t / L::W) * L::PITCH + t % L::W];
}

// rec [m][W] -> the envs `envs` (null: 0 .. m-1); obs (may be null) [n][B::OD] = B::obs of each restored env.  B = the batch's
// snapshot traits: layout L, parameter block type Params, observation dimension OD, obs(P, record row, out).
template <class B>
__global__ void __launch_bounds__(SNAP_THREADS)
restore_scatter_kernel(const __grid_constant__ typename B::Params P, const SnapCols c, int64_t m, const int64_t *__restrict__ envs,
                       const double *__restrict__ rec, double *__restrict__ obs)
{
    using L = typename B::L;
    __shared__ double tile[SNAP_ROWS * L::PITCH];
    const int64_t r0 = (int64_t)blockIdx.x * SNAP_ROWS;
    const int rows = (int)(m - r0 < SNAP_ROWS ? m - r0 : SNAP_ROWS);
    const double *in = rec + r0 * L::W;
    for (int t = threadIdx.x; t < rows * L::W; t += SNAP_THREADS) tile[(t / L::W) * L::PITCH + t % L::W] = in[t];
    __syncthreads();
    const int64_t s = c.stride;
    for (int t = threadIdx.x; t < SNAP_ROWS * (L::W - L::OFF_S); t += SNAP_THREADS) {
        const int r = t % SNAP_ROWS, w = L::OFF_S + t / SNAP_ROWS;
        if (r >= rows) continue;
        const int64_t e = envs ? envs[r0 + r] : r0 + r;
        const double v = tile[r * L::PITCH + w];
        if (w < L::OFF_I) c.S[(int64_t)(w - L::OFF_S) * s + e] = v;
        else if (w < L::OFF_IC) c.I[(int64_t)(w - L::OFF_I) * s + e] = __double_as_longlong(v);
        else if (w < L::OFF_P) c.ics[(int64_t)(w - L::OFF_IC) * s + e] = v;
        else if (w < L::OFF_ROW) { if (c.live) c.S[(int64_t)(L::ND + w - L::OFF_P) * s + e] = v; }
        else if (c.row_of) {
            c.row_of[e] = (int32_t)__double_as_longlong(v);
            c.row_ep[e] = __double_as_longlong(tile[r * L::PITCH + L::OFF_I + L::EP]);
        }
    }
    if (obs && (int)threadIdx.x < rows) {
        const int64_t e = envs ? envs[r0 + threadIdx.x] : r0 + threadIdx.x;
        B::obs(P, tile + threadIdx.x * L::PITCH, obs + e * B::OD);
    }
}

// Checks before a restore (rec != null) or a snapshot with explicit indices (rec == null).  chk[0] = the smallest
// (position << 8 | reason) over offending records, chk[1] = 1 when a record carries an IC-pool row; owner[e] = the lowest
// position naming env e (snapshot_dup_kernel then flags every later one).
enum { SNAP_BAD_KIND = 1, SNAP_BAD_WIDTH, SNAP_BAD_FINGERPRINT, SNAP_NO_PARAM_POOL, SNAP_BAD_INDEX, SNAP_DUP_INDEX };
template <class L>
__global__ void snapshot_check_kernel(int64_t m, const int64_t *__restrict__ envs, int64_t n, const double *__restrict__ rec,
                                      uint64_t fingerprint, int live, uint32_t *__restrict__ owner, unsigned long long *__restrict__ chk)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    int bad = 0;
    if (rec) {
        const double *row = rec + i * L::W;
        if (__double_as_longlong(row[0]) != L::TAG) bad = SNAP_BAD_KIND;
        else if (__double_as_longlong(row[1]) != (int64_t)L::W) bad = SNAP_BAD_WIDTH;
        else if ((uint64_t)__double_as_longlong(row[2]) != fingerprint) bad = SNAP_BAD_FINGERPRINT;
        else if (L::PROW >= 0 && !live && row[L::OFF_P + (L::PROW >= 0 ? L::PROW : 0)] >= 0.0) bad = SNAP_NO_PARAM_POOL;
        else if (__double_as_longlong(row[L::OFF_ROW]) >= 0) chk[1] = 1ull;
    }
    if (!bad && envs) {
        const int64_t e = envs[i];
        if (e < 0 || e >= n) bad = SNAP_BAD_INDEX;
        else if (owner) atomicMin(&owner[e], (uint32_t)i);
    }
    if (bad) atomicMin(&chk[0], (unsigned long long)i << 8 | (unsigned long long)bad);
}
__global__ void snapshot_dup_kernel(int64_t m, const int64_t *__restrict__ envs, int64_t n, const uint32_t *__restrict__ owner,
                                    unsigned long long *__restrict__ chk)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int64_t e = envs[i];
    if (e >= 0 && e < n && owner[e] < (uint32_t)i) atomicMin(&chk[0], (unsigned long long)i << 8 | SNAP_DUP_INDEX);
}

// Runs the checks on `st`, reads the check words back and waits for the stream.  *rows_needed: a record carries an IC-pool row.
template <class L>
int snapshot_checks(BatchCore *h, const char *what, int64_t m, const int64_t *envs, const double *rec, int live, cudaStream_t st,
                    bool *rows_needed)
{
    if (!h->snap_chk) CU_TRY(h, cudaMalloc(&h->snap_chk, 2 * sizeof(unsigned long long)));
    const bool dup = rec && envs;
    if (dup && !h->snap_owner) CU_TRY(h, cudaMalloc(&h->snap_owner, sizeof(uint32_t) * h->stride));
    CU_TRY(h, cudaMemsetAsync(h->snap_chk, 0xFF, sizeof(unsigned long long), st));
    CU_TRY(h, cudaMemsetAsync(h->snap_chk + 1, 0, sizeof(unsigned long long), st));
    if (dup) CU_TRY(h, cudaMemsetAsync(h->snap_owner, 0xFF, sizeof(uint32_t) * h->n, st));
    const int grid = (int)((m + 255) / 256);
    snapshot_check_kernel<L><<<grid, 256, 0, st>>>(m, envs, h->n, rec, h->fingerprint, live, dup ? h->snap_owner : nullptr, h->snap_chk);
    if (dup) snapshot_dup_kernel<<<grid, 256, 0, st>>>(m, envs, h->n, h->snap_owner, h->snap_chk);
    CU_TRY(h, cudaGetLastError());
    unsigned long long w[2];
    CU_TRY(h, cudaMemcpyAsync(w, h->snap_chk, sizeof(w), cudaMemcpyDeviceToHost, st));
    CU_TRY(h, cudaStreamSynchronize(st));
    if (w[0] != ~0ull) {
        static const char *why[] = {"", "not a record of this batch kind and format version", "record width differs",
                                    "configuration fingerprint differs from this handle's", "carries a parameter-pool row and no parameter pool is loaded",
                                    "env index outside [0, n)", "env index named twice"};
        h->err = std::string(what) + ": record " + std::to_string(w[0] >> 8) + ": " + why[w[0] & 0xFF];
        return BSKENV_EINVAL;
    }
    *rows_needed = w[1] != 0;
    return BSKENV_OK;
}

inline int snapshot_args(BatchCore *h, const char *what, int64_t m, const int64_t *envs, const void *rec)
{
    if (!rec || m < 1 || (!envs && m != h->n)) {
        h->err = std::string(what) + ": null records, m < 1, or no env indices and m != n";
        return BSKENV_EINVAL;
    }
    return BSKENV_OK;
}

// bskenv_snapshot / bskenv_opnav_snapshot: c = the handle's columns (row_of / row_ep included), batch = the parameter block of
// the configuration (LEO, written where c.live is 0)
template <class L>
int snapshot(BatchCore *h, const char *what, int64_t m, const int64_t *envs, double *rec, const SnapCols &c,
             const SnapBlock<L::NPD> &batch, void *stream)
{
    int rc = snapshot_args(h, what, m, envs, rec);
    if (rc) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const cudaStream_t st = (cudaStream_t)stream;
    bool unused;
    if (envs && (rc = snapshot_checks<L>(h, what, m, envs, nullptr, c.live, st, &unused))) return rc;
    snapshot_gather_kernel<L><<<(int)((m + SNAP_ROWS - 1) / SNAP_ROWS), SNAP_THREADS, 0, st>>>(c, batch, m, envs, rec);
    CU_TRY(h, cudaGetLastError());
    return BSKENV_OK;
}

// bskenv_restore / bskenv_opnav_restore: checks, then (the IC-pool record allocated at the first record that carries a row,
// as set_ic_pool does) the scatter
template <class B>
int restore(BatchCore *h, const char *what, int64_t m, const int64_t *envs, const double *rec, double *obs, SnapCols c,
            const typename B::Params &P, void *stream)
{
    int rc = snapshot_args(h, what, m, envs, rec);
    if (rc) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const cudaStream_t st = (cudaStream_t)stream;
    bool rows_needed = false;
    if ((rc = snapshot_checks<typename B::L>(h, what, m, envs, rec, c.live, st, &rows_needed))) return rc;
    if (rows_needed && !h->icp.row_of) {
        CU_TRY(h, cudaMalloc(&h->icp.row_of, sizeof(int32_t) * h->stride));
        CU_TRY(h, cudaMalloc(&h->icp.row_ep, sizeof(int64_t) * h->stride));
        CU_TRY(h, cudaMemsetAsync(h->icp.row_of, 0xFF, sizeof(int32_t) * h->stride, st));
        CU_TRY(h, cudaMemsetAsync(h->icp.row_ep, 0, sizeof(int64_t) * h->stride, st));
    }
    c.row_of = h->icp.row_of; c.row_ep = h->icp.row_ep;
    restore_scatter_kernel<B><<<(int)((m + SNAP_ROWS - 1) / SNAP_ROWS), SNAP_THREADS, 0, st>>>(P, c, m, envs, rec, obs);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, note_launch(h, st));
    return BSKENV_OK;
}

// bskenv_state_field / bskenv_opnav_state_field: the index of a named field in the batch's table (-1: none), is_int = which block
struct FieldEnt { const char *n; int idx; int is_int; };
template <size_t N>
int state_field(const FieldEnt (&tab)[N], const char *name, int32_t *is_int)
{
    if (!name) return -1;
    for (const FieldEnt &t : tab)
        if (!strcmp(t.n, name)) { if (is_int) *is_int = t.is_int; return t.idx; }
    return -1;
}

}  // namespace
