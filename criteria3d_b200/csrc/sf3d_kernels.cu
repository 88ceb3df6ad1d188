// sf3d_kernels.cu -- hand-written sm_100a kernels of the soilFluxes3D water time step and the
// device services behind sf3d_backend.h.
//
// All kernels are HBM-bandwidth bound sparse-stencil / streaming passes over structure-of-arrays
// state (no tensor cores: there is no dense contraction on this path).  Common shape:
//   * grid-stride loop, 256 threads per block, grid = min(ceil(n/256), 148 SMs x 8) so that the
//     grid is a whole number of waves on a B200 and the per-block partials stay small;
//   * consecutive threads own consecutive nodes -> every array access is a coalesced 256 B
//     request; neighbour gathers (x[j], H[j], K[j]) hit L1/L2 because links connect index
//     neighbours (+-1, +-cols, +-layer stride);
//   * reductions: warp shuffles -> shared memory -> one partial per block -> the LAST block
//     (atomic ticket) folds the partials in a fixed order and writes the scalar into the device
//     control block.  Deterministic for a given grid; no host round trip per reduction;
//   * the Jacobi sweep evaluates the reference's stopping rule on the device (last block), so a
//     batch of sweeps can be enqueued without synchronising; sweeps launched after convergence
//     return immediately.
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <algorithm>
#include "sf3d_backend.h"
#include "sf3d_rows_heat.h"
#include "sf3d_fields.h"

namespace sf3d {

#define SF3D_BLOCK 256
#ifndef SF3D_MAX_BLOCKS
#define SF3D_MAX_BLOCKS (148 * 8)           // grid cap of the sweep and of every other reducing / streaming kernel
#endif
#ifndef SF3D_WIDE_BLOCKS
#define SF3D_WIDE_BLOCKS (148 * 48)         // grid cap of the fp64-heavy node / assembly kernels (a multiple of every
                                            // residency below, short tail wave)
#endif

static cudaStream_t g_stream = nullptr;
static int g_device = -1;
static uint64_t g_launches = 0;
static Ctrl *g_ctrlPinned = nullptr;
static unsigned long long g_commNsSeen = 0, g_commCountSeen = 0;

#define CUDA_OK(call)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            fprintf(stderr, "[sf3d_b200] CUDA error %d (%s) at %s:%d: %s\n", (int)e_,          \
                    cudaGetErrorString(e_), __FILE__, __LINE__, #call);                        \
            throw DeviceError{(int)e_, cudaGetErrorString(e_), #call};                         \
        }                                                                                      \
    } while (0)

#define LAUNCH_CHECK()                                                                         \
    do { ++g_launches; CUDA_OK(cudaGetLastError()); } while (0)

static void ensure_device();
// ---- optional per-launch timing (CUDA events on the library's stream) ----------------------
struct ProfRec { int kind; cudaEvent_t a, b; };
static bool g_prof = false;
static std::vector<ProfRec> g_pending;
static std::vector<cudaEvent_t> g_eventPool;
static double g_profMs[SF3D_K_COUNT];
static uint64_t g_profN[SF3D_K_COUNT];

static cudaEvent_t prof_event()
{
    if (!g_eventPool.empty()) { cudaEvent_t e = g_eventPool.back(); g_eventPool.pop_back(); return e; }
    cudaEvent_t e; CUDA_OK(cudaEventCreate(&e)); return e;
}
static void prof_resolve()          // call only when the stream is idle
{
    for (const ProfRec &r : g_pending)
    {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { g_profMs[r.kind] += ms; g_profN[r.kind] += 1; }
        g_eventPool.push_back(r.a); g_eventPool.push_back(r.b);
    }
    g_pending.clear();
}
struct ProfScope {
    int kind; cudaEvent_t a{}, b{}; bool on;
    explicit ProfScope(int k) : kind(k), on(g_prof)
    { if (on) { a = prof_event(); b = prof_event(); cudaEventRecord(a, g_stream); } }
    ~ProfScope() { if (on) { cudaEventRecord(b, g_stream); g_pending.push_back(ProfRec{kind, a, b}); } }
};
void prof_enable(bool on)
{
    ensure_device();
    CUDA_OK(cudaStreamSynchronize(g_stream));
    prof_resolve();
    g_prof = on;
    for (int k = 0; k < SF3D_K_COUNT; ++k) { g_profMs[k] = 0.; g_profN[k] = 0; }
}
void prof_get(double ms[SF3D_K_COUNT], uint64_t n[SF3D_K_COUNT])
{
    ensure_device();
    CUDA_OK(cudaStreamSynchronize(g_stream));
    prof_resolve();
    for (int k = 0; k < SF3D_K_COUNT; ++k) { ms[k] = g_profMs[k]; n[k] = g_profN[k]; }
}

void dev_select(int device)
{
    if (g_stream && device == g_device) return;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
    {
        fprintf(stderr, "[sf3d_b200] no CUDA device available (%s). The B200 product has no CPU fallback.\n",
                cudaGetErrorString(e));
        throw DeviceError{(int)e, "no CUDA device", "dev_select"};
    }
    if (device < 0 || device >= count) throw DeviceError{-1, "bad device index", "dev_select"};
    CUDA_OK(cudaSetDevice(device));
    if (g_stream) { cudaStreamDestroy(g_stream); g_stream = nullptr; }
    CUDA_OK(cudaStreamCreateWithFlags(&g_stream, cudaStreamNonBlocking));
    if (!g_ctrlPinned) CUDA_OK(cudaMallocHost((void **)&g_ctrlPinned, sizeof(Ctrl)));
    g_device = device;
}
int dev_current() { return g_device; }
static void ensure_device() { if (!g_stream) dev_select(g_device < 0 ? 0 : g_device); }

void *dev_alloc(size_t bytes)
{
    ensure_device();
    void *p = nullptr;
    if (bytes == 0) bytes = 8;
    CUDA_OK(cudaMalloc(&p, bytes));
    CUDA_OK(cudaMemsetAsync(p, 0, bytes, g_stream));
    return p;
}
void dev_free(void *p) { if (p) cudaFree(p); }
void dev_zero(void *p, size_t bytes) { ensure_device(); CUDA_OK(cudaMemsetAsync(p, 0, bytes, g_stream)); }
void dev_copy(void *dst, const void *src, size_t bytes)
{ ensure_device(); CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, g_stream)); }
void h2d(void *dst, const void *src, size_t bytes)
{ ensure_device(); CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_stream)); CUDA_OK(cudaStreamSynchronize(g_stream)); }
void d2h(void *dst, const void *src, size_t bytes)
{ ensure_device(); CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_stream)); CUDA_OK(cudaStreamSynchronize(g_stream)); }
static cudaStream_t g_copyStream = nullptr;
static cudaEvent_t g_evReady = nullptr, g_evCopied[2] = {nullptr, nullptr};
static bool g_slotUsed[2] = {false, false};
static void ensure_copy_stream()
{
    ensure_device();
    if (g_copyStream) return;
    CUDA_OK(cudaStreamCreateWithFlags(&g_copyStream, cudaStreamNonBlocking));
    CUDA_OK(cudaEventCreateWithFlags(&g_evReady, cudaEventDisableTiming));
    for (int k = 0; k < 2; ++k) CUDA_OK(cudaEventCreateWithFlags(&g_evCopied[k], cudaEventDisableTiming));
}
void overlap_acquire(int slot)
{
    ensure_copy_stream();
    if (g_slotUsed[slot]) CUDA_OK(cudaStreamWaitEvent(g_stream, g_evCopied[slot], 0));
}
void d2h_overlapped(void *dst, const void *src, size_t bytes, int slot)
{
    ensure_copy_stream();
    CUDA_OK(cudaEventRecord(g_evReady, g_stream));
    CUDA_OK(cudaStreamWaitEvent(g_copyStream, g_evReady, 0));
    // in pieces, so that small copies of the library's stream (the control block after every batch of sweeps) can interleave
    const size_t piece = (size_t)4 << 20;
    for (size_t off = 0; off < bytes; off += piece)
        CUDA_OK(cudaMemcpyAsync((char *)dst + off, (const char *)src + off, (bytes - off < piece) ? bytes - off : piece,
                                cudaMemcpyDeviceToHost, g_copyStream));
    CUDA_OK(cudaEventRecord(g_evCopied[slot], g_copyStream));
    g_slotUsed[slot] = true;
}
void overlap_sync() { if (g_copyStream) CUDA_OK(cudaStreamSynchronize(g_copyStream)); }
void *pinned_alloc(size_t bytes) { ensure_device(); void *p = nullptr; CUDA_OK(cudaMallocHost(&p, bytes)); return p; }
void pinned_free(void *p) { if (p) cudaFreeHost(p); }
void dev_sync() { ensure_device(); CUDA_OK(cudaStreamSynchronize(g_stream)); }
uint64_t launches() { return g_launches; }
void *dev_stream() { ensure_device(); return (void *)g_stream; }

int wide_blocks(uint32_t n)
{
    long b = ((long)n + SF3D_BLOCK - 1) / SF3D_BLOCK;
    if (b < 1) b = 1;
    if (b > SF3D_WIDE_BLOCKS) b = SF3D_WIDE_BLOCKS;
    return (int)b;
}
int reduce_blocks(uint32_t n)
{
    long b = ((long)n + SF3D_BLOCK - 1) / SF3D_BLOCK;
    if (b < 1) b = 1;
    if (b > SF3D_MAX_BLOCKS) b = SF3D_MAX_BLOCKS;
    return (int)b;
}

// ------------------------------------------------------------------------------------------
// reduction helpers
// ------------------------------------------------------------------------------------------
template <bool IS_MAX>
__device__ __forceinline__ double warp_reduce(double v)
{
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        const double other = __shfl_down_sync(0xffffffffu, v, o);
        v = IS_MAX ? ((v < other) ? other : v) : (v + other);
    }
    return v;
}

// result valid in thread 0
template <bool IS_MAX>
__device__ __forceinline__ double block_reduce(double v, double *sh)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    v = warp_reduce<IS_MAX>(v);
    __syncthreads();
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    if (wid == 0)
    {
        v = (lane < (SF3D_BLOCK / 32)) ? sh[lane] : 0.0;   // identities: 0 for + and for max of non-negatives
        v = warp_reduce<IS_MAX>(v);
    }
    return v;
}

// elects the last block of the grid to finish; all its threads return true
__device__ __forceinline__ bool last_block(Ctrl *c)
{
    __shared__ int isLast;
    __threadfence();
    if (threadIdx.x == 0)
    {
        const unsigned t = atomicAdd(&c->ticket, 1u);
        isLast = (t == gridDim.x - 1);
    }
    __syncthreads();
    return isLast != 0;
}

// fold gridDim.x partials in a fixed order; result valid in thread 0
template <bool IS_MAX>
__device__ __forceinline__ double fold_partials(const double *part, double *sh)
{
    double acc = 0.0;
    for (unsigned k = threadIdx.x; k < gridDim.x; k += SF3D_BLOCK)
    {
        const double p = __ldcg(part + k);
        acc = IS_MAX ? ((acc < p) ? p : acc) : (acc + p);
    }
    return block_reduce<IS_MAX>(acc, sh);
}

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
// a halo copy of a row that another rank owns (multi-GPU slabs)
__device__ __forceinline__ bool sf3d_is_ghost(const SF3DView &v, uint32_t i) { return v.world > 1 && META_GHOST(v.meta[i]); }

__global__ void __launch_bounds__(SF3D_BLOCK) kern_link_geometry(SF3DView v, int *orderOk)
{
    const size_t N = v.N;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        const uint32_t m = v.meta[i];
        if ((META_SURFACE(m) != 0) != (i < v.Ns)) *orderOk = 0;
        #pragma unroll
        for (int c = 0; c < SF3D_NLINK; ++c)
        {
            const int slot = sf3d_slot_of_col(c);
            uint32_t j = i;
            double g = 0.;
            if (META_HAS_SLOT(m, slot))
            {
                j = v.lidx[(size_t)slot * N + i];
                g = sf3d_link_geom(v, i, j, slot, v.larea[(size_t)slot * N + i]);
            }
            v.mcol[(size_t)c * N + i] = j;
            v.lgeom[(size_t)c * N + i] = g;
        }
    }
}

// static heat geometry: atmospheric pressure at the node's altitude and the 3-D distance of every link
__global__ void __launch_bounds__(SF3D_BLOCK) kern_heat_geometry(SF3DView v)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_heat_geometry(v, i);
}

// ---- pattern compression of the column indices ------------------------------------------------
// For every node the ten column offsets (mcol[c][i] - i) form a "link pattern"; a DEM catchment has a
// few dozen distinct ones (interior, edges, corners x top/middle/bottom layer; more for ragged
// rasters).  Patterns are deduplicated in a small device hash table; each node keeps a 16-bit pattern
// id, so the sweep reads 2 bytes of index data per node instead of 40.  kern_verify_patterns then
// proves  i + pattern[pid[i]][c] == mcol[c][i]  for every entry (bit-exact integer map) or the
// explicit index array stays in use.
#define SF3D_PATTERN_SLOTS 1024
__device__ __forceinline__ unsigned long long pattern_hash(const int32_t *off)
{
    unsigned long long h = 0x9E3779B97F4A7C15ull;
    #pragma unroll
    for (int c = 0; c < SF3D_NLINK; ++c)
    {
        h ^= (unsigned long long)(uint32_t)off[c] + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
        h *= 0xBF58476D1CE4E5B9ull;
    }
    return h ? h : 1ull;            // 0 marks an empty slot
}
__global__ void __launch_bounds__(SF3D_BLOCK) kern_build_patterns(SF3DView v, unsigned long long *keys, int32_t *table,
                                                                  uint16_t *pid, int *overflow)
{
    const size_t N = v.N;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        if (sf3d_is_ghost(v, i)) { pid[i] = SF3D_GHOST_PID; continue; }
        int32_t off[SF3D_NLINK];
        bool fits = true;
        #pragma unroll
        for (int c = 0; c < SF3D_NLINK; ++c)
        {
            const long long d = (long long)v.mcol[(size_t)c * N + i] - (long long)i;
            if (d > 2147483647ll || d < -2147483647ll) fits = false;
            off[c] = (int32_t)d;
        }
        if (!fits) { *overflow = 1; pid[i] = 0; continue; }
        const unsigned long long h = pattern_hash(off);
        uint32_t slot = (uint32_t)(h % SF3D_PATTERN_SLOTS);
        bool placed = false;
        for (int probe = 0; probe < SF3D_PATTERN_SLOTS; ++probe)
        {
            const unsigned long long old = atomicCAS(&keys[slot], 0ull, h);
            if (old == 0ull)
            {
                #pragma unroll
                for (int c = 0; c < SF3D_NLINK; ++c) table[slot * SF3D_NLINK + c] = off[c];
                placed = true; break;
            }
            if (old == h) { placed = true; break; }
            slot = (slot + 1) % SF3D_PATTERN_SLOTS;
        }
        if (!placed) *overflow = 1;
        pid[i] = (uint16_t)slot;
    }
}
__global__ void __launch_bounds__(SF3D_BLOCK) kern_pattern_histogram(SF3DView v, const uint16_t *pid, unsigned int *count)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        // one atomic per warp and distinct pattern (interior warps share a single pattern)
        const unsigned p = pid[i];
        if (p == SF3D_GHOST_PID) continue;
        const unsigned peers = __match_any_sync(__activemask(), p);
        if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&count[p], (unsigned)__popc(peers));
    }
}
__global__ void __launch_bounds__(SF3D_BLOCK) kern_verify_patterns(SF3DView v, const int32_t *table, const uint16_t *pid, int *mismatch)
{
    const size_t N = v.N;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        if (pid[i] == SF3D_GHOST_PID) { if (!sf3d_is_ghost(v, i)) *mismatch = 1; continue; }
        const int32_t *off = table + (size_t)pid[i] * SF3D_NLINK;
        #pragma unroll
        for (int c = 0; c < SF3D_NLINK; ++c)
            if ((uint32_t)((int64_t)i + off[c]) != v.mcol[(size_t)c * N + i]) *mismatch = 1;
    }
}

#ifndef SF3D_POST_BLOCKS
#define SF3D_POST_BLOCKS 8
#endif
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_POST_BLOCKS) kern_begin_try(SF3DView v)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_begin_try(v, i);
}

__global__ void __launch_bounds__(SF3D_BLOCK) kern_restore_old(SF3DView v)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_restore_old(v, i);
}

#ifndef SF3D_NODE_BLOCKS
#define SF3D_NODE_BLOCKS 8
#endif
template <bool HEAT>
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_NODE_BLOCKS) kern_node_phase(SF3DView v, double dt, int withCapacity)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_node_phase<HEAT>(v, i, dt, withCapacity);
}

// ---- row-slab ranks: device side of the peer-memory all-reduce ---------------------------------------
// Every rank owns a mailbox that all ranks can write through CUDA IPC (NVLink peer stores).
#define SF3D_MAX_RANKS 16
// One 8-byte mailbox word carries 32 bits of payload and a 32-bit tag derived from the sequence number: an aligned
// 8-byte store is single-copy atomic, also over NVLink, so a reader that sees the expected tag has the payload of
// the same store and no fence is needed between "data" and "flag" (the scheme of NCCL's LL protocol).
struct Mbox {
    unsigned long long word[2][SF3D_MAX_RANKS][8];      // [parity][source rank][value k: low half 2k, high half 2k + 1]
    unsigned long long localSeq;        // all-reduces executed by THIS rank so far (only this rank touches it)
    int error; int pad;
};
// kernel parameter of the reducing kernels.  mine == nullptr: one GPU, or the NCCL transport (the host finishes the
// reduction over ranks, the kernel only leaves its local values in Ctrl::red)
struct CommDev { Mbox *mine; Mbox *const *peers; int rank, world; long long timeoutCycles; };

__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

// All-reduce of up to four doubles over peer memory, executed by ONE warp.  Every (destination rank, value, half)
// triple is one tagged 8-byte word; the lanes store this rank's words into all mailboxes over NVLink (one release
// fence at system scope first: it orders the halo rows every block of this kernel stored into peer memory -- the
// blocks' tickets were observed by this block -- before the words the peers wait for), then wait until every
// rank's words for the same sequence number have landed in the local mailbox; lanes k < count fold value k in rank
// order, so every rank obtains the bit-identical result and takes the same decisions.  The sequence number counts
// the all-reduces this rank has EXECUTED (device side: launches that return early on every rank, e.g. sweeps
// enqueued after convergence, do not consume one), so consecutive all-reduces use different parities and a rank can
// be at most one all-reduce ahead of its slowest peer.  The wait is bounded (SF3D_MAILBOX_TIMEOUT_S, default 20 s
// of SM clocks): on expiry Ctrl::commError is set and the status becomes SOLVE_COMM_ERROR, which the host turns
// into an error return (read_ctrl throws) -- never into a numerical "halve the time step" event.
__device__ __forceinline__ void p2p_allreduce_warp(const CommDev &cm, int count, int isMax, double *values, Ctrl *ctrl)
{
    const int lane = threadIdx.x & 31;
    unsigned long long seq = 0ull;
    int timedOut = 0;
    if (lane == 0) { seq = cm.mine->localSeq + 1ull; cm.mine->localSeq = seq; timedOut = cm.mine->error; }
    seq = __shfl_sync(0xffffffffu, seq, 0);
    timedOut = __shfl_sync(0xffffffffu, timedOut, 0);       // sticky: after one time-out no further waiting
    const int par = (int)(seq & 1ull);
    const unsigned long long tag = ((seq % 0xFFFFFFFFull) + 1ull) << 32;    // never 0 (a fresh mailbox is all zero)
    const int perRank = 2 * count, nWords = cm.world * perRank;
    if (!timedOut)
    {
        fence_acq_rel_sys();
        for (int w = lane; w < nWords; w += 32)
        {
            const int r = w / perRank, q = w - r * perRank;
            const unsigned long long bits = (unsigned long long)__double_as_longlong(values[q >> 1]);
            const unsigned long long half = (q & 1) ? (bits >> 32) : (bits & 0xFFFFFFFFull);
            *((volatile unsigned long long *)&cm.peers[r]->word[par][cm.rank][q]) = tag | half;
        }
        const long long t0 = clock64();
        for (int w = lane; w < nWords; w += 32)
        {
            const int r = w / perRank, q = w - r * perRank;
            while ((*((volatile unsigned long long *)&cm.mine->word[par][r][q]) & 0xFFFFFFFF00000000ull) != tag)
                if (clock64() - t0 > cm.timeoutCycles) { timedOut = 1; break; }
        }
    }
    timedOut = __any_sync(0xffffffffu, timedOut);
    fence_acq_rel_sys();
    if (timedOut)
    {
        if (lane == 0)
        {
            cm.mine->error = 1;
            if (ctrl) { ctrl->commError = 1; ctrl->status = SOLVE_COMM_ERROR; }
        }
    }
    else if (lane < count)
    {
        double acc = 0.;
        for (int r = 0; r < cm.world; ++r)
        {
            const unsigned long long lo = *((volatile unsigned long long *)&cm.mine->word[par][r][2 * lane]);
            const unsigned long long hi = *((volatile unsigned long long *)&cm.mine->word[par][r][2 * lane + 1]);
            const double x = __longlong_as_double((long long)((hi << 32) | (lo & 0xFFFFFFFFull)));
            acc = (r == 0) ? x : (isMax ? ((acc < x) ? x : acc) : (acc + x));
        }
        values[lane] = acc;
    }
    __syncwarp();
}
// called by EVERY thread of the block that finished last, after thread 0 wrote the local values into c->red[]:
// folds the all-reduce over ranks into the producing kernel (no extra launch per reduction)
__device__ __forceinline__ unsigned long long global_ns()
{ unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ void last_block_allreduce(const CommDev &cm, Ctrl *c, int count, int isMax)
{
    __syncthreads();
    if (threadIdx.x < 32)
    {
        const unsigned long long t0 = global_ns();
        p2p_allreduce_warp(cm, count, isMax, c->red, c);
        if (threadIdx.x == 0) { c->commNs += global_ns() - t0; c->commCount += 1ull; }
    }
    __syncthreads();
}

// ---- what each reducing kernel does with its reduced values ----------------------------------------------------
// count / isMax: the values and how they combine over the ranks; whileRunning: only while the solve runs (a sweep
// enqueued after the solve ended does nothing).  r[] holds the values reduced over all ranks.
struct CourantRule {            // kern_assemble
    static constexpr int count = 1; static constexpr bool isMax = true, whileRunning = false;
    double dt, dtMin;
    __device__ void operator()(Ctrl *c, const double *r) const
    {
        if (c->commError) { c->status = SOLVE_COMM_ERROR; return; }
        c->courantMax = r[0];
        const bool ok = (r[0] < 1.01) || (dt <= dtMin);      // CPUSolver::checkCourant, cpusolver.cpp:259
        c->status = ok ? SOLVE_RUNNING : SOLVE_COURANT_FAIL;
        c->sweeps = 0;
        c->bestNorm = 1.;       // solveLinearSystem: bestErrorNorm = 1 (cpusolver.cpp:674)
        c->lastNorm = 0.;
    }
};
struct WaterJacobiRule {        // the stopping rule of CPUSolver::solveLinearSystem (cpusolver.cpp:678-700)
    static constexpr int count = 1; static constexpr bool isMax = false, whileRunning = true;
    double nGlobal; int maxIter; double tol;
    __device__ void operator()(Ctrl *c, const double *r) const
    {
        if (c->commError) { c->status = SOLVE_COMM_ERROR; return; }
        const double curr = r[0] / nGlobal;                       // water.cpp:600
        c->lastNorm = curr;
        c->sweeps += 1;
        if (curr < tol) c->status = SOLVE_CONVERGED;              // cpusolver.cpp:692
        else if (curr > c->bestNorm * 10) c->status = SOLVE_DIVERGED;   // :695
        else
        {
            if (curr < c->bestNorm) c->bestNorm = curr;           // :698
            if (c->sweeps >= maxIter) c->status = SOLVE_MAXITER;
        }
    }
};
struct HeatJacobiRule {
    static constexpr int count = 1; static constexpr bool isMax = true, whileRunning = true;
    int maxIter; double tol;
    __device__ void operator()(Ctrl *c, const double *r) const
    {
        if (c->commError) { c->status = SOLVE_COMM_ERROR; return; }
        c->lastNorm = r[0];
        c->sweeps += 1;
        if (r[0] < tol) c->status = SOLVE_CONVERGED;              // cpusolver.cpp:692 (no divergence test for heat)
        else if (c->sweeps >= maxIter) c->status = SOLVE_MAXITER;
    }
};
template <bool HEAT>
__host__ __device__ inline auto jacobi_rule(const SF3DView &v, int maxIter, double tol)
{
    if constexpr (HEAT) return HeatJacobiRule{maxIter, tol};
    else return WaterJacobiRule{v.nGlobal, maxIter, tol};
}
struct WaterPostRule {
    static constexpr int count = 2; static constexpr bool isMax = false, whileRunning = false;
    __device__ void operator()(Ctrl *c, const double *r) const { c->storage = r[0]; c->sinkSum = r[1]; }
};
struct HeatPostRule {
    static constexpr int count = 2; static constexpr bool isMax = false, whileRunning = false;
    __device__ void operator()(Ctrl *c, const double *r) const { c->heatStorage = r[0]; c->heatSinkSum = r[1]; }
};
struct BoundaryTotalRule {
    static constexpr int count = 1; static constexpr bool isMax = false, whileRunning = false;
    __device__ void operator()(Ctrl *c, const double *r) const { c->boundarySum = r[0]; }
};
struct HeatCourantRule {
    static constexpr int count = 1; static constexpr bool isMax = true, whileRunning = false;
    __device__ void operator()(Ctrl *c, const double *r) const { c->heatCourantMax = r[0]; }
};

// The end of every reducing kernel, after thread 0 stored the block's partial(s) in v.partA (and v.partB): the block
// that finishes last folds the partials in a fixed order, then
//   * one GPU: applies the rule;
//   * peer transport (several ranks, cm.mine set): all-reduces the values over the ranks through the mailboxes, applies
//     the rule;
//   * NCCL transport: leaves the local values in Ctrl::red (the host all-reduces them and launches kern_rule);
// and resets the ticket.
template <class Rule>
__device__ __forceinline__ void finish_reduction(const SF3DView &v, double *sh, const CommDev &cm, const Rule &rule)
{
    Ctrl *c = v.ctrl;
    if (!last_block(c)) return;
    const bool peer = v.world > 1 && cm.mine != nullptr;
    double r[2];
    r[0] = fold_partials<Rule::isMax>(v.partA, sh);
    if (Rule::count == 2) r[1] = fold_partials<Rule::isMax>(v.partB, sh);
    if (peer)
    {
        if (threadIdx.x == 0) for (int k = 0; k < Rule::count; ++k) c->red[k] = r[k];
        last_block_allreduce(cm, c, Rule::count, Rule::isMax ? 1 : 0);
        if (threadIdx.x == 0) for (int k = 0; k < Rule::count; ++k) r[k] = c->red[k];
    }
    if (threadIdx.x == 0)
    {
        if (v.world == 1 || peer) rule(c, r);
        else for (int k = 0; k < Rule::count; ++k) c->red[k] = r[k];
        c->ticket = 0;
    }
}
// NCCL transport: the rule, applied after the host's all-reduce of Ctrl::red
template <class Rule>
__global__ void kern_rule(Ctrl *c, Rule rule)
{
    if (Rule::whileRunning && c->status != SOLVE_RUNNING) return;
    rule(c, c->red);
}

// link phase: conductances, diagonal, row normalisation, right-hand side, per-row Courant;
// the last block publishes max Courant and arms the on-device solver state
// (CPUSolver::checkCourant test, cpusolver.cpp:248-260).  Ghost rows are not assembled.
// Resident blocks per SM requested from ptxas.  These kernels are chains of dependent fp64 operations
// (pow / log / divisions) behind scattered gathers: measured on B200 they run 1.5-2x faster with 40 / 32
// registers and 1536 / 2048 resident threads per SM (a few spilled words) than unconstrained at 64 / 54
// registers (profiles/r01_occupancy_ab.json).
#ifndef SF3D_HEAT_ASSEMBLE_BLOCKS
#define SF3D_HEAT_ASSEMBLE_BLOCKS 6
#endif
#ifndef SF3D_HEAT_BLOCKS
#define SF3D_HEAT_BLOCKS 8          // same finding for the heat rows (profiles/r01_occupancy_ab.json)
#endif
#ifndef SF3D_ASSEMBLE_BLOCKS
#define SF3D_ASSEMBLE_BLOCKS 6
#endif
template <bool HEAT>
__global__ void __launch_bounds__(SF3D_BLOCK, HEAT ? SF3D_HEAT_ASSEMBLE_BLOCKS : SF3D_ASSEMBLE_BLOCKS) kern_assemble(SF3DView v, double dt, int approx, double dtMin, CommDev cm)
{
    __shared__ double sh[SF3D_BLOCK / 32];
    __shared__ double ksh[SF3D_NLINK * SF3D_BLOCK];          // ten conductances per thread, conflict-free layout
    double courant = 0.;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        if (sf3d_is_ghost(v, i)) continue;
        const double c = sf3d_row_assemble<HEAT>(v, i, dt, approx, ksh + threadIdx.x, SF3D_BLOCK);
        courant = (courant < c) ? c : courant;
    }
    courant = block_reduce<true>(courant, sh);
    if (threadIdx.x == 0) v.partA[blockIdx.x] = courant;
    finish_reduction(v, sh, cm, CourantRule{dt, dtMin});
}

// coupled heat: thermal liquid / vapour fluxes of every soil row (invariantFluxes of the water system), before the
// assembly of each approximation
#ifndef SF3D_THERMAL_BLOCKS
#define SF3D_THERMAL_BLOCKS 8
#endif
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_THERMAL_BLOCKS) kern_thermal_invariant(SF3DView v)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        if (!sf3d_is_ghost(v, i)) sf3d_row_thermal_invariant(v, i);
}

// one Jacobi sweep (Water::JacobiWaterCPU, sum of |dx|; heat: the infinity norm of heat.cpp:664-685) + the stopping
// rule of CPUSolver::solveLinearSystem (cpusolver.cpp:678-700) evaluated by the last block: one GPU, and the NCCL
// transport, which exchanges the halo and all-reduces the norm after this kernel.  Ghost rows are not swept.
#ifndef SF3D_JACOBI_BLOCKS
#define SF3D_JACOBI_BLOCKS 8
#endif
// this thread's rows of one sweep (grid-stride), except those skip(i) is true for; the rows' norm terms are added to
// norm (water) or raise it to their maximum (heat)
template <bool HEAT, bool COHERENT = false, class Skip>
__device__ __forceinline__ double sweep_rows(const SF3DView &v, const double *xin, double *xout, double norm, Skip skip)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        if (skip(i)) continue;
        const double d = HEAT ? sf3d_row_heat_jacobi(v, i, xin, xout) : sf3d_row_jacobi<COHERENT>(v, i, xin, xout);
        norm = HEAT ? ((norm < d) ? d : norm) : (norm + d);
    }
    return norm;
}
template <bool HEAT>
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_JACOBI_BLOCKS) kern_jacobi(SF3DView v, const double *__restrict__ xin,
                                                          double *__restrict__ xout, int maxIter, double tol)
{
    if (v.ctrl->status != SOLVE_RUNNING) return;
    __shared__ double sh[SF3D_BLOCK / 32];
    double norm = sweep_rows<HEAT>(v, xin, xout, 0., [&](uint32_t i) { return v.world > 1 && v.pid[i] == SF3D_GHOST_PID; });
    norm = block_reduce<HEAT>(norm, sh);
    if (threadIdx.x == 0) v.partA[blockIdx.x] = norm;
    finish_reduction(v, sh, CommDev{}, jacobi_rule<HEAT>(v, maxIter, tol));
}

// ---- small graphs: all sweeps of one solve in ONE launch -------------------------------------------------
// A catchment of a few ten thousand nodes (BASELINE config 1, CRITERIA-1D-sized callers) sweeps in ~1 us, so a solve of
// 30 sweeps is bound by 30 launches and by the batches' control-block reads.  This kernel is launched cooperatively
// (every block resident) and iterates on the device: sweep, block partial, grid-wide barrier, EVERY block folds the
// partials in the same fixed order and applies the stopping rule of kern_jacobi to its own copy of the solver state,
// so all blocks leave the loop in the same sweep without a second barrier; the partials alternate between two
// arrays, so a fast block's next partial never lands in the array a slow block is still folding.  Grid size, thread
// -> row mapping, partial sums and fold order are those of kern_jacobi: the residual norms, and with them the
// decisions, are bit-identical to the launch-per-sweep path.  xa holds the solution at entry.
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_JACOBI_BLOCKS) kern_jacobi_persistent(SF3DView v, double *xa, double *xb, int maxIter, double tol)
{
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    if (v.ctrl->status != SOLVE_RUNNING) return;        // Courant failure of the assembly: the same branch in every block
    __shared__ double sh[SF3D_BLOCK / 32];
    __shared__ int status;
    // thread 0's copy of the solver state (identical in every block), in registers: the rule is on the critical path of
    // every sweep
    Ctrl c = *v.ctrl;
    const auto rule = jacobi_rule<false>(v, maxIter, tol);
    for (int sweep = 0; ; ++sweep)
    {
        const double *xin = (sweep & 1) ? xb : xa;
        double *xout = (sweep & 1) ? xa : xb;
        double *part = (sweep & 1) ? v.partB : v.partA;
        double norm = sweep_rows<false, true>(v, xin, xout, 0., [](uint32_t) { return false; });
        norm = block_reduce<false>(norm, sh);
        if (threadIdx.x == 0) part[blockIdx.x] = norm;
        grid.sync();
        const double total = fold_partials<false>(part, sh);
        if (threadIdx.x == 0) { rule(&c, &total); status = c.status; }
        __syncthreads();
        if (status != SOLVE_RUNNING) break;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
    { v.ctrl->lastNorm = c.lastNorm; v.ctrl->sweeps = c.sweeps; v.ctrl->bestNorm = c.bestNorm; v.ctrl->status = c.status; }
}

// NCCL transport: gather owned boundary values into the send buffer / scatter received ones into the ghost rows
__global__ void __launch_bounds__(SF3D_BLOCK) kern_pack(const double *__restrict__ x, const uint32_t *__restrict__ idx,
                                                        uint32_t n, double *__restrict__ buf)
{
    for (uint32_t k = blockIdx.x * SF3D_BLOCK + threadIdx.x; k < n; k += gridDim.x * SF3D_BLOCK) buf[k] = x[idx[k]];
}
__global__ void __launch_bounds__(SF3D_BLOCK) kern_unpack(double *__restrict__ x, const uint32_t *__restrict__ idx,
                                                          uint32_t n, const double *__restrict__ buf)
{
    for (uint32_t k = blockIdx.x * SF3D_BLOCK + threadIdx.x; k < n; k += gridDim.x * SF3D_BLOCK) x[idx[k]] = buf[k];
}
// ---- peer transport: one launch per sweep on several GPUs ---------------------------------------------------
// The rows some neighbouring rank holds as ghosts ("boundary rows": the first / last owned DEM row of a slab, all
// layers) are swept FIRST and their new values stored straight into the neighbours' ghost rows (NVLink peer
// stores into the neighbour's output buffer of this sweep), so the halo travels while the interior rows are being
// swept.  Boundary and ghost rows carry SF3D_PID_SKIP in their pattern id, so the interior loop passes over them
// without an extra load.  The block that finishes last then all-reduces the residual through the mailboxes -- its
// system-scope fence orders every block's halo stores before the sequence number the peers wait for -- and
// applies the stopping rule (cpusolver.cpp:678-700).  A peer cannot be overtaken: rank r writes sweep s + 1 into
// a neighbour's buffer only after the all-reduce of sweep s, i.e. after that neighbour finished reading it.  This
// holds because every rank runs this kernel for every sweep: the transport is chosen once, the same on all ranks.
#define SF3D_MAX_HALO_PEERS 4
#define SF3D_NO_REMOTE 0xFFFFFFFFu
struct ExchangeDev {
    uint32_t nBoundary;                                 // owned rows that at least one peer holds as ghosts
    const uint32_t *bIdx;                               // their local ids (unique)
    int nPeers;
    const uint32_t *remote[SF3D_MAX_HALO_PEERS];        // [nBoundary] id of the row in peer p's numbering, or SF3D_NO_REMOTE
    double *peerX[SF3D_MAX_HALO_PEERS];                 // peer p's OUTPUT solution buffer of this sweep
};
template <bool HEAT>
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_JACOBI_BLOCKS) kern_jacobi_multi(SF3DView v, const double *__restrict__ xin,
                                                                                double *__restrict__ xout, int maxIter, double tol,
                                                                                ExchangeDev e, CommDev cm)
{
    if (v.ctrl->status != SOLVE_RUNNING) return;        // same decision on every rank: the status derives from all-reduced values
    __shared__ double sh[SF3D_BLOCK / 32];
    double norm = 0.;
    // (boundary row k goes to thread k / gridDim.x of block k % gridDim.x: every block takes the same share in its
    // lowest warps, so no block starts its interior rows a whole dependent-load chain later than the others;
    // measured against "one row per thread of the last blocks": 6.5 us per sweep)
    for (uint32_t k = threadIdx.x * gridDim.x + blockIdx.x; k < e.nBoundary; k += gridDim.x * SF3D_BLOCK)
    {
        const uint32_t i = e.bIdx[k];
        double xn;
        const double d = HEAT ? sf3d_row_heat_jacobi(v, i, xin, xout, &xn) : sf3d_row_jacobi(v, i, xin, xout, &xn);
        norm = HEAT ? ((norm < d) ? d : norm) : (norm + d);
        #pragma unroll
        for (int p = 0; p < SF3D_MAX_HALO_PEERS; ++p)
        {
            if (p >= e.nPeers) break;
            const uint32_t r = e.remote[p][k];
            if (r != SF3D_NO_REMOTE) e.peerX[p][r] = xn;
        }
        // system-scope fence by the threads that stored into peer memory, right here (early in the kernel, behind
        // other warps' work): these stores are then ordered before this block's ticket below and, through the last
        // block's own fence, before the sequence number the peers wait for
        __threadfence_system();
    }
    // ghost rows, and the boundary rows done above, are skipped
    norm = sweep_rows<HEAT>(v, xin, xout, norm, [&](uint32_t i) { return (v.pid[i] & SF3D_PID_SKIP) != 0; });
    norm = block_reduce<HEAT>(norm, sh);
    if (threadIdx.x == 0) v.partA[blockIdx.x] = norm;
    finish_reduction(v, sh, cm, jacobi_rule<HEAT>(v, maxIter, tol));
}
__global__ void __launch_bounds__(SF3D_BLOCK) kern_mark_boundary(uint16_t *pid, const uint32_t *__restrict__ idx, uint32_t n)
{
    for (uint32_t k = blockIdx.x * SF3D_BLOCK + threadIdx.x; k < n; k += gridDim.x * SF3D_BLOCK) pid[idx[k]] |= (uint16_t)SF3D_PID_SKIP;
}

// H = x, Se refresh, and the two mass-balance sums
// mode 3 ("follow the solve"): enqueued right behind a batch of sweeps, before the host has seen how the solve ended.  The
// kernel reads the outcome itself: it runs as mode 0 on the vector the last executed sweep wrote when the solve ended in a
// state the host goes on from (converged / sweep cap / diverged at the minimum time step: waterApproximationLoop,
// cpusolver.cpp:431-457), and returns at once otherwise (solve still running, Courant failure, divergence that halves the
// step).  One control-block read then tells the host both how the solve ended and the balance sums.  x = x0, xAlt = x1,
// start = index of the buffer that held the solution when the solve began; every block (and every rank: the status derives
// from all-reduced values) takes the same branch.
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_POST_BLOCKS) kern_post(SF3DView v, const double *__restrict__ x, double dt, int mode, CommDev cm,
                                                                        const double *__restrict__ xAlt = nullptr, int start = 0, double dtMin = 0.)
{
    if (mode == 3)
    {
        const int st = v.ctrl->status;
        const bool goesOn = st == SOLVE_CONVERGED || st == SOLVE_MAXITER || (st == SOLVE_DIVERGED && !(dt > dtMin));
        if (!goesOn) return;
        if ((start + v.ctrl->sweeps) & 1) x = xAlt;
        mode = 0;
    }
    __shared__ double sh[SF3D_BLOCK / 32];
    double storage = 0., sinkSum = 0.;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        double s, q;
        sf3d_row_post(v, i, x, dt, mode, &s, &q);
        if (sf3d_is_ghost(v, i)) continue;      // ghosts are counted by their owner
        storage += s;
        sinkSum += q;
    }
    storage = block_reduce<false>(storage, sh);
    sinkSum = block_reduce<false>(sinkSum, sh);
    if (threadIdx.x == 0) { v.partA[blockIdx.x] = storage; v.partB[blockIdx.x] = sinkSum; }
    finish_reduction(v, sh, cm, WaterPostRule{});
}

// PREP: the copies of the next try's first pass (kern_begin_try) ride on this pass (water-only runs: the heat step
// still reads the previous heads after the water step is accepted)
template <bool PREP>
__global__ void __launch_bounds__(SF3D_BLOCK) kern_accept(SF3DView v, double dt)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        if (!sf3d_is_ghost(v, i)) sf3d_row_accept(v, i, dt);
        if (PREP) sf3d_row_prepare_try(v, i);
    }
}

__global__ void __launch_bounds__(SF3D_BLOCK) kern_restore_best(SF3DView v)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_restore_best(v, i);
}

// getTotalBoundaryWaterFlow (soilFluxes3D.cpp:1240-1250)
__global__ void __launch_bounds__(SF3D_BLOCK) kern_total_boundary(SF3DView v, uint32_t bt, CommDev cm)
{
    __shared__ double sh[SF3D_BLOCK / 32];
    double sum = 0.;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        if (META_BT(v.meta[i]) == bt && !sf3d_is_ghost(v, i)) sum += v.bSum[i];
    sum = block_reduce<false>(sum, sh);
    if (threadIdx.x == 0) v.partA[blockIdx.x] = sum;
    finish_reduction(v, sh, cm, BoundaryTotalRule{});
}

// setNodeMatricPotential / setNodeTotalPotential over a range (soilFluxes3D.cpp:869-906)
__global__ void __launch_bounds__(SF3D_BLOCK) kern_set_potential(SF3DView v, uint32_t first, uint32_t count,
                                                                 const double *__restrict__ src, int isTotal)
{
    for (uint32_t k = blockIdx.x * SF3D_BLOCK + threadIdx.x; k < count; k += gridDim.x * SF3D_BLOCK)
    {
        const uint32_t i = first + k;
        const double z = v.z[i];
        const double H = isTotal ? src[k] : z + src[k];
        v.H[i] = H;
        v.oldH[i] = H;
        if (META_SURFACE(v.meta[i])) { v.Se[i] = 1.; v.K[i] = SF3D_NODATA; }
        else
        {
            const SoilRec &s = v.soil[v.tab[i]];
            const double se = sf3d_node_se(s, v.wrcModel, H, z);
            v.Se[i] = se;
            double K = sf3d_mualem(s, v.wrcModel, se);
            if (v.computeHeat && v.computeHeatVapor) K += sf3d_heat_vapor_K(v, i);
            v.K[i] = K;
        }
    }
}

// bulk getters: same value as the scalar getter of each node (soilFluxes3D.cpp:951-1234)
__global__ void __launch_bounds__(SF3D_BLOCK) kern_get_field(SF3DView v, int field, uint32_t first, uint32_t count,
                                                             double *__restrict__ dst)
{
    for (uint32_t k = blockIdx.x * SF3D_BLOCK + threadIdx.x; k < count; k += gridDim.x * SF3D_BLOCK)
        dst[k] = sf3d_field_value(v, field, first + k);
}

// raster-facing forcing / output maps, one thread per raster cell
__global__ void __launch_bounds__(SF3D_BLOCK) kern_forcing_rasters(SF3DView v, RasterDev g, ForcingDev f)
{
    const uint64_t cells = (uint64_t)g.rows * g.cols;
    for (uint64_t c = (uint64_t)blockIdx.x * SF3D_BLOCK + threadIdx.x; c < cells; c += (uint64_t)gridDim.x * SF3D_BLOCK)
        sf3d_cell_forcing(v, g, f, c);
}
__global__ void __launch_bounds__(SF3D_BLOCK) kern_layer_raster(SF3DView v, RasterDev g, int field, uint32_t layer, float nodata,
                                                                float *__restrict__ dst)
{
    const uint64_t cells = (uint64_t)g.rows * g.cols;
    for (uint64_t c = (uint64_t)blockIdx.x * SF3D_BLOCK + threadIdx.x; c < cells; c += (uint64_t)gridDim.x * SF3D_BLOCK)
        dst[c] = sf3d_cell_output(v, g, field, layer, nodata, c);
}

// DEM -> node/link graph (Project3D::setCrit3DTopography + setCrit3DNodeSoil,
// src/project3D/project3D.cpp:941-1103, 1164-1238), one thread per (layer, cell)
__global__ void __launch_bounds__(SF3D_BLOCK) kern_build_grid(SF3DView v, GridDev g)
{
    const size_t N = v.N;
    const uint64_t cells = (uint64_t)g.rows * g.cols;
    const uint64_t total = cells * g.layers;
    const double area = g.cell * g.cell;
    for (uint64_t t = (uint64_t)blockIdx.x * SF3D_BLOCK + threadIdx.x; t < total; t += (uint64_t)gridDim.x * SF3D_BLOCK)
    {
        const uint32_t layer = (uint32_t)(t / cells);
        const uint64_t cell = t % cells;
        const int32_t rank = g.rank[cell];
        if (rank < 0) continue;
        const uint32_t row = (uint32_t)(cell / g.cols), col = (uint32_t)(cell % g.cols);
        const uint32_t i = layer * g.nValid + (uint32_t)rank;

        const double thickness = g.layerThickness[layer];
        const double volume = area * thickness;
        const float lateralArea = (layer == 0) ? (float)g.cell : (float)(g.cell * thickness);
        const float bSlopeF = g.slope ? g.slope[cell] : 0.f;
        const float zf = g.dem[cell] - (float)g.layerDepth[layer];
        const bool outlet = g.outlet && g.outlet[cell];

        v.x[i] = g.xll + g.cell * ((double)col + 0.5);
        v.y[i] = g.yll + g.cell * ((double)(g.rows - row) - 0.5);
        v.z[i] = (double)zf;

        uint32_t bt = BT_NONE;
        double bSlope = 0., bSize = 0.;
        const bool surface = (layer == 0);
        if (surface)
        {
            v.size[i] = area;
            if (outlet && g.freeRunoff) { bt = BT_RUNOFF; bSlope = bSlopeF; bSize = (double)(float)g.cell; }
        }
        else
        {
            v.size[i] = volume;
            if (layer == g.layers - 1) { if (g.freeBottom) { bt = BT_FREE_DRAINAGE; bSlope = 0.; bSize = (double)(float)area; } }
            else if (outlet && g.freeLateral) { bt = BT_FREE_LATERAL; bSlope = bSlopeF; bSize = (double)lateralArea; }
            else if (layer == 1 && g.boundaryL1) bt = g.boundaryL1[cell];
            if (layer == 1 && g.heatSurfaceL1) { bt = BT_HEAT_SURFACE; bSlope = bSlopeF; bSize = area; }
        }
        if (bt != BT_NONE)          // setNodeBoundary (soilFluxes3D.cpp:689-725)
        {
            v.bSlope[i] = bSlope; v.bSize[i] = bSize;
            v.bRate[i] = 0.; v.bSum[i] = 0.; v.bPresc[i] = SF3D_NODATA;
            if (g.computeHeat)          // soilFluxes3D.cpp:705-722
            {
                v.hbHeightWind[i] = v.hbHeightT[i] = v.hbRough[i] = v.hbAero[i] = v.hbSoilCond[i] = SF3D_NODATA;
                v.hbT[i] = v.hbRH[i] = v.hbWind[i] = v.hbNetIrr[i] = v.hbFixT[i] = v.hbFixDepth[i] = SF3D_NODATA;
                v.hbRad[i] = v.hbLat[i] = v.hbSens[i] = v.hbAdv[i] = 0.;
            }
        }
        v.sink[i] = 0.;

        // links: slot 0 Up, slot 1 Down, slots 2.. Lateral in (dr,dc) order (-1,-1) .. (1,1)
        uint32_t mask = 0, nLat = 0;
        if (layer > 0)
        {
            v.lidx[i] = (layer - 1) * g.nValid + (uint32_t)rank;
            v.larea[i] = area; mask |= 1u;
        }
        if (layer < g.layers - 1)
        {
            v.lidx[N + i] = (layer + 1) * g.nValid + (uint32_t)rank;
            v.larea[N + i] = area; mask |= 2u;
        }
        for (int di = -1; di <= 1; ++di)
        for (int dj = -1; dj <= 1; ++dj)
        {
            if (di == 0 && dj == 0) continue;
            const long rr = (long)row + di, cc = (long)col + dj;
            if (rr < 0 || cc < 0 || rr >= (long)g.rows || cc >= (long)g.cols) continue;
            const int32_t lrank = g.rank[(uint64_t)rr * g.cols + (uint64_t)cc];
            if (lrank < 0) continue;
            const uint32_t slot = 2 + nLat;
            v.lidx[(size_t)slot * N + i] = layer * g.nValid + (uint32_t)lrank;
            v.larea[(size_t)slot * N + i] = lateralArea * 0.5;
            mask |= (1u << slot);
            ++nLat;
        }
        v.meta[i] = bt | ((surface ? 1u : 0u) << 4) | (nLat << 5) | (mask << 9);
        if (g.computeHeat)              // setNodeLink, soilFluxes3D.cpp:669-678
            for (uint32_t sl = 0; sl < SF3D_NLINK; ++sl)
                if ((mask >> sl) & 1u)
                {
                    v.lfluxes[(size_t)sl * N + i] = SF3D_NODATA;
                    if (v.hfSaveMode == 2) for (int t = 1; t < 9; ++t) v.lfluxes[((size_t)t * SF3D_NLINK + sl) * N + i] = SF3D_NODATA;
                }

        if (surface)
        {
            v.tab[i] = g.surfaceId ? g.surfaceId[cell] : 0;
            v.pond[i] = g.pond ? g.pond[cell] : (double)0.0001f;
        }
        else
        {
            const uint32_t sid = g.soilId ? g.soilId[cell] : 0;
            v.tab[i] = g.layerTab[(size_t)layer * g.nSoilIds + sid];
            if (g.computeHeat) { v.T[i] = 273.15 + 20; v.oldT[i] = 273.15 + 20; v.hFlux[i] = 0.; v.hSink[i] = 0.; }
        }
    }
}

// ------------------------------------------------------------------------------------------
// coupled heat (Heat::*, CPUSolver::heatLoop)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SF3D_BLOCK) kern_update_conductance(SF3DView v)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_update_conductance(v, i);
}
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_heat_coeffs(SF3DView v, double dtHeat, double dtWater)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        sf3d_row_heat_coeffs(v, i, dtHeat, dtWater);
}
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_save_water_fluxes(SF3DView v, double dtHeat, double dtWater)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        if (!sf3d_is_ghost(v, i)) sf3d_row_save_water_fluxes(v, i, dtHeat, dtWater);    // a ghost row has no link pattern
}
// updateBoundaryHeatData: heat flux per node + max heat-boundary Courant (heat.cpp:237-340)
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_boundary_heat(SF3DView v, double maxTimeStep, CommDev cm)
{
    __shared__ double sh[SF3D_BLOCK / 32];
    double courant = 0.;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        const double c = sf3d_row_boundary_heat(v, i, maxTimeStep);
        if (!sf3d_is_ghost(v, i)) courant = (courant < c) ? c : courant;
    }
    courant = block_reduce<true>(courant, sh);
    if (threadIdx.x == 0) v.partA[blockIdx.x] = courant;
    finish_reduction(v, sh, cm, HeatCourantRule{});
}
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_heat_begin(SF3DView v, double dtHeat, double dtWater)
{
    const size_t N = v.N;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        sf3d_row_heat_begin(v, i, dtHeat, dtWater);
        // resetFluxValues(true, false) (heat.cpp:55-78)
        // (save mode Total: the HeatTotal slots are reset by the heat assembly's own store, see sf3d_row_heat_assemble)
        if (v.hfSaveMode == 2)
            for (int t = 0; t < 5; ++t) for (int s = 0; s < SF3D_NLINK; ++s) v.lfluxes[((size_t)t * SF3D_NLINK + s) * N + i] = SF3D_NODATA;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
    { Ctrl *c = v.ctrl; c->status = SOLVE_RUNNING; c->sweeps = 0; c->lastNorm = 0.; }
}
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_heat_assemble(SF3DView v, double dtHeat, double dtWater)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        if (!sf3d_is_ghost(v, i)) sf3d_row_heat_assemble(v, i, dtHeat, dtWater);
}
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_heat_post(SF3DView v, const double *__restrict__ x, double dtHeat,
                                                             double dtWater, int mode, CommDev cm)
{
    __shared__ double sh[SF3D_BLOCK / 32];
    double storage = 0., sinkSum = 0.;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        double s, q;
        sf3d_row_heat_post(v, i, x, dtHeat, dtWater, mode, &s, &q);
        if (sf3d_is_ghost(v, i)) continue;
        storage += s; sinkSum += q;
    }
    storage = block_reduce<false>(storage, sh);
    sinkSum = block_reduce<false>(sinkSum, sh);
    if (threadIdx.x == 0) { v.partA[blockIdx.x] = storage; v.partB[blockIdx.x] = sinkSum; }
    finish_reduction(v, sh, cm, HeatPostRule{});
}
__global__ void __launch_bounds__(SF3D_BLOCK, SF3D_HEAT_BLOCKS) kern_heat_accept(SF3DView v, double dtHeat, double dtWater)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        if (!sf3d_is_ghost(v, i)) sf3d_row_heat_accept(v, i, dtHeat, dtWater);
}
// mode 0: oldT = T (accepted, cpusolver.cpp:598-602); mode 1: T = oldT (refused, :582-588)
__global__ void __launch_bounds__(SF3D_BLOCK) kern_heat_copy_T(SF3DView v, int mode)
{
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
    {
        if (i < v.Ns) continue;
        if (mode == 0) v.oldT[i] = v.T[i]; else v.T[i] = v.oldT[i];
    }
}
// resetFluxValues(false, true): water flux snapshots to NODATA in save mode All (heat.cpp:80-93)
__global__ void __launch_bounds__(SF3D_BLOCK) kern_reset_water_fluxes(SF3DView v)
{
    const size_t N = v.N;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        for (int t = 5; t < 9; ++t) for (int s = 0; s < SF3D_NLINK; ++s) v.lfluxes[((size_t)t * SF3D_NLINK + s) * N + i] = SF3D_NODATA;
}

__global__ void __launch_bounds__(SF3D_BLOCK) kern_count_links(SF3DView v, unsigned long long *out)
{
    unsigned long long n = 0;
    for (uint32_t i = blockIdx.x * SF3D_BLOCK + threadIdx.x; i < v.N; i += gridDim.x * SF3D_BLOCK)
        n += __popc(META_LINKMASK(v.meta[i]));
    for (int o = 16; o > 0; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(out, n);
}

__global__ void kern_fill(double *p, size_t n, double value)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = value;
}

// ------------------------------------------------------------------------------------------
// row-slab ranks: the two transports of the per-sweep halo of x and the scalar all-reduces (peer memory, or
// NCCL over NVLink; see transport()).  libnccl is resolved at run time (dlopen) so that single-GPU users need only libcudart; the
// few entry points used are declared here with the signatures of nccl.h (2.x ABI).
// ------------------------------------------------------------------------------------------
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { NCCL_SUM = 0, NCCL_MAX = 2, NCCL_FLOAT64 = 8 };
static struct {
    void *lib = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
} nccl;
static ncclComm_t g_comm = nullptr;
static int g_rank = 0, g_world = 1;
struct HaloPeer {
    int peer;
    std::vector<uint32_t> send, recv;   // my rows the peer holds as ghosts / my ghost rows the peer owns
    // peer transport: the peer's two solution buffers mapped through CUDA IPC, and where each send row lives in the
    // peer's numbering (its ghost row)
    double *peerX[2]; std::vector<uint32_t> remote;
};
static std::vector<HaloPeer> g_halo;
static double *g_localX[2] = {nullptr, nullptr};     // this rank's x0 / x1 (exported to the neighbours)
// peer transport: every rank owns a mailbox that all ranks can write through CUDA IPC
static Mbox *g_mbox = nullptr;                       // this rank's mailbox (device memory)
static Mbox *g_peerMbox[SF3D_MAX_RANKS] = {nullptr}; // host copy of the mapped pointers ([g_rank] = g_mbox)
static Mbox **g_peerMboxDev = nullptr;               // the same table in device memory, once every rank's mailbox is mapped
static long long g_timeoutCycles = 0;               // bound of the mailbox wait, SM clocks
// the unique boundary rows, marked in the pattern ids (comm_mark_boundary; null until marked for the current halo)
static uint32_t *g_bIdx = nullptr; static uint32_t g_nBoundary = 0;
// built by transport() for the transport it chose.  Peer: per peer, where each boundary row lives in the peer's
// numbering.  NCCL: the send / recv lists of all peers back to back and their staging buffers
static uint32_t *g_bRemote[SF3D_MAX_HALO_PEERS] = {nullptr};
static uint32_t *g_sendIdx = nullptr, *g_recvIdx = nullptr, g_nSend = 0, g_nRecv = 0;
static double *g_sendBuf = nullptr, *g_recvBuf = nullptr;
enum Transport { TRANSPORT_UNSET, TRANSPORT_SINGLE, TRANSPORT_PEER, TRANSPORT_NCCL };
static Transport g_transport = TRANSPORT_UNSET;
static uint32_t *upload(const std::vector<uint32_t> &a)
{
    uint32_t *d = (uint32_t *)dev_alloc(a.size() * 4);
    if (!a.empty()) h2d(d, a.data(), a.size() * 4);
    return d;
}
// forget the transport choice and the tables built for it (whenever the wiring changes)
static void reset_transport()
{
    for (int p = 0; p < SF3D_MAX_HALO_PEERS; ++p) { dev_free(g_bRemote[p]); g_bRemote[p] = nullptr; }
    dev_free(g_sendIdx); dev_free(g_recvIdx); dev_free(g_sendBuf); dev_free(g_recvBuf);
    g_sendIdx = g_recvIdx = nullptr; g_sendBuf = g_recvBuf = nullptr; g_nSend = g_nRecv = 0;
    g_transport = TRANSPORT_UNSET;
}

#define NCCL_OK(call)                                                                          \
    do {                                                                                       \
        int r_ = (call);                                                                       \
        if (r_ != 0) {                                                                         \
            fprintf(stderr, "[sf3d_b200] NCCL error %d (%s) at %s:%d: %s\n", r_,               \
                    nccl.GetErrorString ? nccl.GetErrorString(r_) : "?", __FILE__, __LINE__, #call); \
            throw DeviceError{r_, "NCCL", #call};                                              \
        }                                                                                      \
    } while (0)

static void nccl_load()
{
    if (nccl.lib) return;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) { nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (nccl.lib) break; }
    if (!nccl.lib) throw DeviceError{-1, "libnccl.so.2 not found", "dlopen"};
    auto sym = [&](const char *n) { void *p = dlsym(nccl.lib, n); if (!p) throw DeviceError{-1, "NCCL symbol missing", n}; return p; };
    nccl.GetUniqueId = (int (*)(ncclUniqueId *))sym("ncclGetUniqueId");
    nccl.CommInitRank = (int (*)(ncclComm_t *, int, ncclUniqueId, int))sym("ncclCommInitRank");
    nccl.CommDestroy = (int (*)(ncclComm_t))sym("ncclCommDestroy");
    nccl.AllReduce = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))sym("ncclAllReduce");
    nccl.Send = (int (*)(const void *, size_t, int, int, ncclComm_t, cudaStream_t))sym("ncclSend");
    nccl.Recv = (int (*)(void *, size_t, int, int, ncclComm_t, cudaStream_t))sym("ncclRecv");
    nccl.GroupStart = (int (*)())sym("ncclGroupStart");
    nccl.GroupEnd = (int (*)())sym("ncclGroupEnd");
    nccl.GetErrorString = (const char *(*)(int))sym("ncclGetErrorString");
}
void comm_unique_id(unsigned char out[128])
{
    nccl_load();
    ncclUniqueId id;
    NCCL_OK(nccl.GetUniqueId(&id));
    memcpy(out, id.internal, 128);
}
// idBytes == nullptr: no NCCL communicator (peer transport only: the solution buffers and the mailboxes must be
// wired before the first step; used where NCCL cannot run, e.g. several ranks sharing one device in the tests)
void comm_init(int rank, int world, const unsigned char idBytes[128])
{
    ensure_device();
    if (g_comm) { nccl.CommDestroy(g_comm); g_comm = nullptr; }
    if (idBytes)
    {
        nccl_load();
        ncclUniqueId id;
        memcpy(id.internal, idBytes, 128);
        NCCL_OK(nccl.CommInitRank(&g_comm, world, id, rank));
    }
    g_rank = rank; g_world = world;
    reset_transport();
    // bound of the mailbox wait in SM clocks
    double seconds = 20.;
    if (const char *e = getenv("SF3D_MAILBOX_TIMEOUT_S")) { const double t = atof(e); if (t > 0.) seconds = t; }
    int khz = 0;
    CUDA_OK(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g_device));
    g_timeoutCycles = (long long)(seconds * 1e3 * (double)khz);
}
int comm_world() { return g_world; }
int comm_rank() { return g_rank; }
void comm_clear_halo()
{
    for (HaloPeer &h : g_halo)
        for (int b = 0; b < 2; ++b) if (h.peerX[b]) cudaIpcCloseMemHandle(h.peerX[b]);
    g_halo.clear();
    for (int r = 0; r < SF3D_MAX_RANKS; ++r)
        if (g_peerMbox[r] && r != g_rank) { cudaIpcCloseMemHandle(g_peerMbox[r]); }
    for (int r = 0; r < SF3D_MAX_RANKS; ++r) g_peerMbox[r] = nullptr;
    dev_free(g_mbox); g_mbox = nullptr;             // a fresh mailbox starts with sequence 0 and no error
    dev_free(g_peerMboxDev); g_peerMboxDev = nullptr;
    dev_free(g_bIdx); g_bIdx = nullptr; g_nBoundary = 0;
    reset_transport();
}
// peer transport: export this rank's mailbox / import the others'
void comm_mailbox_export(unsigned char out[64])
{
    ensure_device();
    if (g_world > SF3D_MAX_RANKS) throw DeviceError{-1, "too many ranks for the mailbox all-reduce", "comm_mailbox_export"};
    if (!g_mbox) g_mbox = (Mbox *)dev_alloc(sizeof(Mbox));
    cudaIpcMemHandle_t h;
    CUDA_OK(cudaIpcGetMemHandle(&h, g_mbox));
    memcpy(out, &h, 64);
    g_peerMbox[g_rank] = g_mbox;
}
void comm_mailbox_import(int peer, const unsigned char handle[64])
{
    ensure_device();
    if (peer < 0 || peer >= g_world || peer >= SF3D_MAX_RANKS || peer == g_rank) throw DeviceError{-1, "bad mailbox peer", "comm_mailbox_import"};
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void *p = nullptr;
    CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    g_peerMbox[peer] = (Mbox *)p;
    reset_transport();
    bool all = g_mbox != nullptr;
    for (int r = 0; r < g_world; ++r) if (!g_peerMbox[r]) all = false;
    if (all)
    {
        if (!g_peerMboxDev) g_peerMboxDev = (Mbox **)dev_alloc(SF3D_MAX_RANKS * sizeof(Mbox *));
        h2d(g_peerMboxDev, g_peerMbox, SF3D_MAX_RANKS * sizeof(Mbox *));
    }
}
// peer transport: export this rank's solution buffers / import a neighbour's
void comm_ipc_export(double *x0, double *x1, unsigned char out[128])
{
    ensure_device();
    cudaIpcMemHandle_t h0, h1;
    CUDA_OK(cudaIpcGetMemHandle(&h0, x0));
    CUDA_OK(cudaIpcGetMemHandle(&h1, x1));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(out, &h0, 64); memcpy(out + 64, &h1, 64);
    g_localX[0] = x0; g_localX[1] = x1;
}
void comm_ipc_import(int peer, const unsigned char handles[128], uint32_t n, const uint32_t *remoteIdx)
{
    ensure_device();
    // the peer-transport sweep stores into at most SF3D_MAX_HALO_PEERS neighbours: with more, the wiring fails (and
    // mgpu.setup_slab puts every rank on NCCL)
    if (g_halo.size() > SF3D_MAX_HALO_PEERS) throw DeviceError{-1, "too many halo peers for the peer-memory halo", "comm_ipc_import"};
    for (HaloPeer &h : g_halo)
    {
        if (h.peer != peer) continue;
        if (n != h.send.size()) throw DeviceError{-1, "remote index list does not match the send list", "comm_ipc_import"};
        cudaIpcMemHandle_t hh[2];
        memcpy(&hh[0], handles, 64); memcpy(&hh[1], handles + 64, 64);
        for (int b = 0; b < 2; ++b)
        {
            void *p = nullptr;
            CUDA_OK(cudaIpcOpenMemHandle(&p, hh[b], cudaIpcMemLazyEnablePeerAccess));
            h.peerX[b] = (double *)p;
        }
        h.remote.assign(remoteIdx, remoteIdx + n);
        reset_transport();
        return;
    }
    throw DeviceError{-1, "unknown halo peer", "comm_ipc_import"};
}
void comm_finalize()
{
    comm_clear_halo();
    if (g_comm) { nccl.CommDestroy(g_comm); g_comm = nullptr; }
    g_world = 1; g_rank = 0;
}
void comm_add_halo_peer(int peer, uint32_t nSend, const uint32_t *sendIdx, uint32_t nRecv, const uint32_t *recvIdx)
{
    HaloPeer h{};
    h.peer = peer; h.peerX[0] = h.peerX[1] = nullptr;
    h.send.assign(sendIdx, sendIdx + nSend);
    h.recv.assign(recvIdx, recvIdx + nRecv);
    g_halo.push_back(h);
    dev_free(g_bIdx); g_bIdx = nullptr; g_nBoundary = 0;
    reset_transport();
}
// the unique boundary rows of this rank (union of the send lists, ascending)
static std::vector<uint32_t> boundary_rows()
{
    std::vector<uint32_t> all;
    for (const HaloPeer &h : g_halo) all.insert(all.end(), h.send.begin(), h.send.end());
    std::sort(all.begin(), all.end());
    all.erase(std::unique(all.begin(), all.end()), all.end());
    return all;
}
// pattern ids: boundary rows are skipped by the interior loop of the peer-transport sweep (harmless for every other
// kernel, which mask the bit).  Called after every (re)build of the pattern ids, whether or not the patterns are in
// use; the table is built even when it is empty.
void comm_mark_boundary(uint16_t *pid)
{
    if (g_world <= 1) return;
    const std::vector<uint32_t> rows = boundary_rows();
    dev_free(g_bIdx);
    g_bIdx = upload(rows);
    g_nBoundary = (uint32_t)rows.size();
    kern_mark_boundary<<<reduce_blocks(g_nBoundary), SF3D_BLOCK, 0, g_stream>>>(pid, g_bIdx, g_nBoundary); LAUNCH_CHECK();
}
// The transport of the row-slab steps, chosen once per wiring: peer memory iff the solution buffers of every halo
// peer and the mailboxes of every rank are mapped and there are at most SF3D_MAX_HALO_PEERS peers, NCCL otherwise.
// Nothing rank-specific enters (not the pattern compression, not the row counts), and mgpu.setup_slab makes the
// wiring all-or-none across the ranks, so every rank takes the same transport and launches the same kernels.
static Transport transport(const SF3DView &v)
{
    if (v.world <= 1) return TRANSPORT_SINGLE;
    if (g_transport != TRANSPORT_UNSET) return g_transport;
    bool peer = g_peerMboxDev != nullptr && g_halo.size() <= SF3D_MAX_HALO_PEERS;
    for (const HaloPeer &h : g_halo) if (!h.peerX[0] || !h.peerX[1]) peer = false;
    if (peer)
    {
        const std::vector<uint32_t> rows = boundary_rows();
        for (size_t p = 0; p < g_halo.size(); ++p)
        {
            const HaloPeer &h = g_halo[p];
            std::vector<uint32_t> rem(rows.size(), SF3D_NO_REMOTE);
            for (size_t k = 0; k < h.send.size(); ++k)
                rem[(size_t)(std::lower_bound(rows.begin(), rows.end(), h.send[k]) - rows.begin())] = h.remote[k];
            g_bRemote[p] = upload(rem);
        }
        g_transport = TRANSPORT_PEER;
        return g_transport;
    }
    if (!g_comm) throw DeviceError{-4, "no NCCL communicator and the peer-memory path is not wired", "row-slab step"};
    std::vector<uint32_t> send, recv;
    for (const HaloPeer &h : g_halo)
    {
        send.insert(send.end(), h.send.begin(), h.send.end());
        recv.insert(recv.end(), h.recv.begin(), h.recv.end());
    }
    g_sendIdx = upload(send); g_nSend = (uint32_t)send.size(); g_sendBuf = (double *)dev_alloc(send.size() * 8);
    g_recvIdx = upload(recv); g_nRecv = (uint32_t)recv.size(); g_recvBuf = (double *)dev_alloc(recv.size() * 8);
    g_transport = TRANSPORT_NCCL;
    return g_transport;
}
// what the reducing kernels receive: the mailboxes on the peer transport (the all-reduce over ranks runs inside the
// producing kernel), nothing otherwise
static CommDev comm_dev(const SF3DView &v)
{
    if (transport(v) != TRANSPORT_PEER) return CommDev{};
    return CommDev{g_mbox, g_peerMboxDev, g_rank, g_world, g_timeoutCycles};
}
static ExchangeDev exchange_dev(const double *xout)
{
    if (!g_bIdx) throw DeviceError{-1, "the boundary rows are not marked for the current halo", "k_jacobi"};
    const int b = (xout == g_localX[1]) ? 1 : 0;
    ExchangeDev e{};
    e.nBoundary = g_nBoundary; e.bIdx = g_bIdx; e.nPeers = (int)g_halo.size();
    for (size_t p = 0; p < g_halo.size(); ++p) { e.remote[p] = g_bRemote[p]; e.peerX[p] = g_halo[p].peerX[b]; }
    return e;
}
// NCCL transport: the boundary rows of x -> the neighbours' ghost rows (one pack and one unpack launch for all peers)
static void nccl_halo(double *x)
{
    kern_pack<<<reduce_blocks(g_nSend), SF3D_BLOCK, 0, g_stream>>>(x, g_sendIdx, g_nSend, g_sendBuf); LAUNCH_CHECK();
    NCCL_OK(nccl.GroupStart());
    size_t so = 0, ro = 0;
    for (const HaloPeer &h : g_halo)
    {
        if (!h.send.empty()) NCCL_OK(nccl.Send(g_sendBuf + so, h.send.size(), NCCL_FLOAT64, h.peer, g_comm, g_stream));
        if (!h.recv.empty()) NCCL_OK(nccl.Recv(g_recvBuf + ro, h.recv.size(), NCCL_FLOAT64, h.peer, g_comm, g_stream));
        so += h.send.size(); ro += h.recv.size();
    }
    NCCL_OK(nccl.GroupEnd());
    kern_unpack<<<reduce_blocks(g_nRecv), SF3D_BLOCK, 0, g_stream>>>(x, g_recvIdx, g_nRecv, g_recvBuf); LAUNCH_CHECK();
}
// NCCL transport: all-reduce the local values a reducing kernel left in Ctrl::red, then apply its rule
template <class Rule>
static void nccl_finish(const SF3DView &v, const Rule &rule)
{
    NCCL_OK(nccl.AllReduce(v.ctrl->red, v.ctrl->red, (size_t)Rule::count, NCCL_FLOAT64, Rule::isMax ? NCCL_MAX : NCCL_SUM, g_comm, g_stream));
    kern_rule<<<1, 1, 0, g_stream>>>(v.ctrl, rule); LAUNCH_CHECK();
}

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
#define GRID(n) reduce_blocks(n), SF3D_BLOCK, 0, g_stream
#define WIDE_GRID(n) wide_blocks(n), SF3D_BLOCK, 0, g_stream

void dev_fill_f64(double *p, size_t n, double value)
{ ensure_device(); kern_fill<<<reduce_blocks((uint32_t)(n > 0xFFFFFFFFull ? 0xFFFFFFFFull : n)), 256, 0, g_stream>>>(p, n, value); LAUNCH_CHECK(); }

void k_heat_geometry(const SF3DView &v)
{
    kern_heat_geometry<<<GRID(v.N)>>>(v); LAUNCH_CHECK();
}
void k_link_geometry(const SF3DView &v, int *surfaceOrderOk)
{
    int *flag = (int *)dev_alloc(sizeof(int));
    const int one = 1;
    h2d(flag, &one, sizeof one);
    kern_link_geometry<<<GRID(v.N)>>>(v, flag); LAUNCH_CHECK();
    d2h(surfaceOrderOk, flag, sizeof(int));
    dev_free(flag);
}
// returns true when the pattern-compressed index map reproduces mcol exactly
bool k_build_patterns(const SF3DView &v, uint16_t *pid, int32_t *table, uint32_t *hotPid, int32_t hotOff[SF3D_NLINK])
{
    unsigned long long *keys = (unsigned long long *)dev_alloc(SF3D_PATTERN_SLOTS * sizeof(unsigned long long));
    int *flags = (int *)dev_alloc(2 * sizeof(int));
    dev_zero(table, (size_t)SF3D_PATTERN_SLOTS * SF3D_NLINK * sizeof(int32_t));
    kern_build_patterns<<<GRID(v.N)>>>(v, keys, table, pid, flags); LAUNCH_CHECK();
    kern_verify_patterns<<<GRID(v.N)>>>(v, table, pid, flags + 1); LAUNCH_CHECK();
    int h[2] = {1, 1};
    d2h(h, flags, sizeof h);
    // most frequent pattern -> kernel parameters
    unsigned int *count = (unsigned int *)dev_alloc(SF3D_PATTERN_SLOTS * sizeof(unsigned int));
    kern_pattern_histogram<<<GRID(v.N)>>>(v, pid, count); LAUNCH_CHECK();
    std::vector<unsigned int> hc(SF3D_PATTERN_SLOTS);
    d2h(hc.data(), count, hc.size() * sizeof(unsigned int));
    uint32_t best = 0;
    for (uint32_t k = 1; k < SF3D_PATTERN_SLOTS; ++k) if (hc[k] > hc[best]) best = k;
    *hotPid = best;
    d2h(hotOff, table + (size_t)best * SF3D_NLINK, SF3D_NLINK * sizeof(int32_t));
    dev_free(keys); dev_free(flags); dev_free(count);
    return h[0] == 0 && h[1] == 0;
}
size_t pattern_table_bytes() { return (size_t)SF3D_PATTERN_SLOTS * SF3D_NLINK * sizeof(int32_t); }

void k_begin_try(const SF3DView &v) { ProfScope ps(SF3D_K_BEGIN_TRY); kern_begin_try<<<GRID(v.N)>>>(v); LAUNCH_CHECK(); }
void k_restore_old(const SF3DView &v) { ProfScope ps(SF3D_K_OTHER); kern_restore_old<<<GRID(v.N)>>>(v); LAUNCH_CHECK(); }
void k_node_phase(const SF3DView &v, double dt, int withCapacity)
{
    ProfScope ps(SF3D_K_NODE_PHASE);
    if (v.computeHeat) kern_node_phase<true><<<WIDE_GRID(v.N)>>>(v, dt, withCapacity);
    else kern_node_phase<false><<<WIDE_GRID(v.N)>>>(v, dt, withCapacity);
    LAUNCH_CHECK();
}
void k_assemble(const SF3DView &v, double dt, int approx, double dtMin)
{
    const CommDev cm = comm_dev(v);
    {
        ProfScope ps(SF3D_K_ASSEMBLE);
        if (v.computeHeat) { kern_thermal_invariant<<<GRID(v.N)>>>(v); LAUNCH_CHECK(); }
        if (v.computeHeat) kern_assemble<true><<<WIDE_GRID(v.N)>>>(v, dt, approx, dtMin, cm);
        else kern_assemble<false><<<WIDE_GRID(v.N)>>>(v, dt, approx, dtMin, cm);
        LAUNCH_CHECK();
    }
    if (transport(v) == TRANSPORT_NCCL) nccl_finish(v, CourantRule{dt, dtMin});
}
// the persistent solve is used for graphs one grid covers with one row per thread (beyond that a sweep takes much longer
// than a launch and the launch-per-sweep path overlaps its control reads with queued sweeps); SF3D_PERSISTENT_SOLVE=0
// disables it, =N sets the node limit
bool k_jacobi_persistent_ok(const SF3DView &v)
{
    static int maxCoopBlocks = -1;
    if (maxCoopBlocks < 0)
    {
        ensure_device();
        int coop = 0, perSm = 0, sms = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, g_device);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g_device);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, kern_jacobi_persistent, SF3D_BLOCK, 0) != cudaSuccess) { cudaGetLastError(); perSm = 0; }
        maxCoopBlocks = coop ? perSm * sms : 0;
    }
    const char *e = getenv("SF3D_PERSISTENT_SOLVE");        // read per solve: tests switch it inside one process
    const long limit = e ? atol(e) : (long)SF3D_MAX_BLOCKS * SF3D_BLOCK;
    return v.world == 1 && (long)v.N <= limit && reduce_blocks(v.N) <= maxCoopBlocks;
}
void k_jacobi_persistent(const SF3DView &v, double *xa, double *xb, int maxIter, double tol)
{
    ProfScope ps(SF3D_K_JACOBI);
    SF3DView vv = v;
    void *args[] = {(void *)&vv, (void *)&xa, (void *)&xb, (void *)&maxIter, (void *)&tol};
    CUDA_OK(cudaLaunchCooperativeKernel((const void *)kern_jacobi_persistent, dim3(reduce_blocks(v.N)), dim3(SF3D_BLOCK), args, 0, g_stream));
    LAUNCH_CHECK();
}
// one sweep.  Peer transport: one launch (boundary rows first with peer stores, interior rows, in-kernel all-reduce +
// stopping rule).  One GPU: one launch.  NCCL: the sweep, the halo exchange, the all-reduce of the norm and the rule.
template <bool HEAT>
static void jacobi_sweep(const SF3DView &v, const double *xin, double *xout, int maxIter, double tol, int kind)
{
    const Transport t = transport(v);
    {
        ProfScope ps(kind);
        if (t == TRANSPORT_PEER) kern_jacobi_multi<HEAT><<<GRID(v.N)>>>(v, xin, xout, maxIter, tol, exchange_dev(xout), comm_dev(v));
        else kern_jacobi<HEAT><<<GRID(v.N)>>>(v, xin, xout, maxIter, tol);
        LAUNCH_CHECK();
    }
    if (t == TRANSPORT_NCCL) { ProfScope ps(SF3D_K_COMM); nccl_halo(xout); nccl_finish(v, jacobi_rule<HEAT>(v, maxIter, tol)); }
}
void k_jacobi(const SF3DView &v, const double *xin, double *xout, int maxIter, double tol)
{ jacobi_sweep<false>(v, xin, xout, maxIter, tol, SF3D_K_JACOBI); }
void k_post(const SF3DView &v, const double *x, double dt, int mode)
{
    { ProfScope ps(SF3D_K_POST); kern_post<<<GRID(v.N)>>>(v, x, dt, mode, comm_dev(v)); LAUNCH_CHECK(); }
    if (transport(v) == TRANSPORT_NCCL) nccl_finish(v, WaterPostRule{});
}
// the post pass enqueued behind the sweeps (kern_post mode 3).  Not on the NCCL transport: its host-side all-reduce
// would run behind a skipped pass
bool k_post_can_follow_solve(const SF3DView &v) { return v.world == 1 || transport(v) == TRANSPORT_PEER; }
void k_post_follow_solve(const SF3DView &v, int start, double dt, double dtMin)
{
    ProfScope ps(SF3D_K_POST);
    kern_post<<<GRID(v.N)>>>(v, v.x0, dt, 3, comm_dev(v), v.x1, start, dtMin); LAUNCH_CHECK();
}
void k_accept(const SF3DView &v, double dt, bool prepareNextTry)
{
    ProfScope ps(SF3D_K_ACCEPT);
    if (prepareNextTry) kern_accept<true><<<GRID(v.N)>>>(v, dt); else kern_accept<false><<<GRID(v.N)>>>(v, dt);
    LAUNCH_CHECK();
}
void k_restore_best(const SF3DView &v) { ProfScope ps(SF3D_K_OTHER); kern_restore_best<<<GRID(v.N)>>>(v); LAUNCH_CHECK(); }
void k_total_boundary_flow(const SF3DView &v, uint32_t bt)
{
    kern_total_boundary<<<GRID(v.N)>>>(v, bt, comm_dev(v)); LAUNCH_CHECK();
    if (transport(v) == TRANSPORT_NCCL) nccl_finish(v, BoundaryTotalRule{});
}
void k_set_potential(const SF3DView &v, uint32_t first, uint32_t count, const double *src, int isTotal)
{ if (count) { kern_set_potential<<<GRID(count)>>>(v, first, count, src, isTotal); LAUNCH_CHECK(); } }
void k_get_field(const SF3DView &v, int field, uint32_t first, uint32_t count, double *dst)
{ if (count) { kern_get_field<<<GRID(count)>>>(v, field, first, count, dst); LAUNCH_CHECK(); } }
void k_forcing_rasters(const SF3DView &v, const RasterDev &g, const ForcingDev &f)
{
    const uint64_t cells = (uint64_t)g.rows * g.cols;
    kern_forcing_rasters<<<GRID((uint32_t)(cells > 0xFFFFFFFFull ? 0xFFFFFFFFull : cells))>>>(v, g, f); LAUNCH_CHECK();
}
void k_layer_raster(const SF3DView &v, const RasterDev &g, int field, uint32_t layer, float nodata, float *dst)
{
    const uint64_t cells = (uint64_t)g.rows * g.cols;
    kern_layer_raster<<<GRID((uint32_t)(cells > 0xFFFFFFFFull ? 0xFFFFFFFFull : cells))>>>(v, g, field, layer, nodata, dst); LAUNCH_CHECK();
}
void k_build_grid(const SF3DView &v, const GridDev &g)
{
    const uint64_t total = (uint64_t)g.rows * g.cols * g.layers;
    kern_build_grid<<<reduce_blocks((uint32_t)(total > 0xFFFFFFFFull ? 0xFFFFFFFFull : total)), SF3D_BLOCK, 0, g_stream>>>(v, g);
    LAUNCH_CHECK();
}

void k_update_conductance(const SF3DView &v) { ProfScope ps(SF3D_K_OTHER); kern_update_conductance<<<GRID(v.N)>>>(v); LAUNCH_CHECK(); }
void k_save_water_fluxes(const SF3DView &v, double dtHeat, double dtWater)
{
    { ProfScope ps(SF3D_K_HEAT_COEFFS); kern_heat_coeffs<<<GRID(v.N)>>>(v, dtHeat, dtWater); LAUNCH_CHECK(); }
    // Heat::saveNodeWaterFluxes (heat.cpp:109-138).  The snapshot is read by the advective terms only (computeAdvectiveFlux,
    // heat.cpp:606-621; boundary advection :273-287) and, in save mode All, by the per-type flux getters: without either the
    // pass has no observer and is not run (the reference computes it regardless)
    if (!(v.computeHeatAdvection || v.hfSaveMode == 2)) return;
    ProfScope ps(SF3D_K_HEAT_FLUX_SNAPSHOT);
    kern_save_water_fluxes<<<GRID(v.N)>>>(v, dtHeat, dtWater); LAUNCH_CHECK();
}
void k_reset_water_fluxes(const SF3DView &v) { if (v.hfSaveMode == 2) { kern_reset_water_fluxes<<<GRID(v.N)>>>(v); LAUNCH_CHECK(); } }
void k_boundary_heat(const SF3DView &v, double maxTimeStep)
{
    ProfScope ps(SF3D_K_HEAT_BOUNDARY);
    kern_boundary_heat<<<GRID(v.N)>>>(v, maxTimeStep, comm_dev(v)); LAUNCH_CHECK();
    if (transport(v) == TRANSPORT_NCCL) nccl_finish(v, HeatCourantRule{});
}
void k_heat_begin(const SF3DView &v, double dtHeat, double dtWater, bool coeffsAreCurrent)
{
    ProfScope ps(SF3D_K_HEAT_COEFFS);
    kern_heat_begin<<<GRID(v.N)>>>(v, dtHeat, dtWater); LAUNCH_CHECK();
    if (!coeffsAreCurrent) { kern_heat_coeffs<<<GRID(v.N)>>>(v, dtHeat, dtWater); LAUNCH_CHECK(); }
}
void k_heat_assemble(const SF3DView &v, double dtHeat, double dtWater)
{ ProfScope ps(SF3D_K_HEAT_ASSEMBLE); kern_heat_assemble<<<GRID(v.N)>>>(v, dtHeat, dtWater); LAUNCH_CHECK(); }
void k_heat_jacobi(const SF3DView &v, const double *xin, double *xout, int maxIter, double tol)
{ jacobi_sweep<true>(v, xin, xout, maxIter, tol, SF3D_K_HEAT_JACOBI); }
void k_heat_post(const SF3DView &v, const double *x, double dtHeat, double dtWater, int mode)
{
    ProfScope ps(SF3D_K_HEAT_POST);
    kern_heat_post<<<GRID(v.N)>>>(v, x, dtHeat, dtWater, mode, comm_dev(v)); LAUNCH_CHECK();
    if (transport(v) == TRANSPORT_NCCL) nccl_finish(v, HeatPostRule{});
}
void k_heat_accept(const SF3DView &v, double dtHeat, double dtWater)
{ ProfScope ps(SF3D_K_HEAT_ACCEPT); kern_heat_accept<<<GRID(v.N)>>>(v, dtHeat, dtWater); LAUNCH_CHECK(); }
void k_heat_copy_T(const SF3DView &v, int mode) { kern_heat_copy_T<<<GRID(v.N)>>>(v, mode); LAUNCH_CHECK(); }

uint64_t k_count_links(const SF3DView &v)
{
    unsigned long long *d = (unsigned long long *)dev_alloc(sizeof(unsigned long long));
    kern_count_links<<<GRID(v.N)>>>(v, d); LAUNCH_CHECK();
    unsigned long long h = 0;
    d2h(&h, d, sizeof h);
    dev_free(d);
    return (uint64_t)h;
}

void read_ctrl(const SF3DView &v, Ctrl *out)
{
    ensure_device();
    CUDA_OK(cudaMemcpyAsync(g_ctrlPinned, v.ctrl, sizeof(Ctrl), cudaMemcpyDeviceToHost, g_stream));
    CUDA_OK(cudaStreamSynchronize(g_stream));
    if (g_prof && g_pending.size() > 4096) prof_resolve();
    *out = *g_ctrlPinned;
    if (g_prof && out->commCount >= g_commCountSeen)
    {
        // device-side clocks of the in-kernel all-reduces since the last read (see Ctrl::commNs)
        g_profMs[SF3D_K_COMM] += (double)(out->commNs - g_commNsSeen) * 1e-6;
        g_profN[SF3D_K_COMM] += out->commCount - g_commCountSeen;
    }
    g_commNsSeen = out->commNs; g_commCountSeen = out->commCount;
    if (out->commError)
        throw DeviceError{-3, "a row-slab peer did not answer within the mailbox time-out (SF3D_MAILBOX_TIMEOUT_S): "
                              "the step was abandoned, the state is undefined", "all-reduce over ranks"};
}
void write_ctrl(const SF3DView &v, const Ctrl *in)
{
    ensure_device();
    CUDA_OK(cudaMemcpyAsync(v.ctrl, in, sizeof(Ctrl), cudaMemcpyHostToDevice, g_stream));
    CUDA_OK(cudaStreamSynchronize(g_stream));
}

}  // namespace sf3d
