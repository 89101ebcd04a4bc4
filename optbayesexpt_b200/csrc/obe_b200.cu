// obe_b200.cu -- libobe_b200.so: model-independent kernels, the C ABI (include/obe_b200.h),
// built-in model instantiations and the NVRTC path for user model source.  sm_100a only.
//
// Kernel inventory (reference call site -> kernel), all fp64 / HBM-streaming:
//   obe_base.py:381-394 + particlepdf.py:136-139,243-244,173-214  -> obe_update_body (obe_device.cuh)
//   particlepdf.py:330 cumsum (tile level)                        -> k_tile_scan
//   particlepdf.py:330-331 choice(p=w), K draws                   -> k_draw
//   particlepdf.py:330-331 choice(p=w), N draws (parity mode)     -> k_cdf + k_search + k_gather_jitter
//   particlepdf.py:286-310 resample, systematic comb (fast path)  -> k_sys_plan + k_sys_resample
//   obe_base.py:463-489,628-655,748                               -> obe_utility_body (obe_device.cuh)
//   obe_base.py:778-789 good_setting                              -> k_pick_weights + k_tile_scan + k_draw
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <nvrtc.h>
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include <cmath>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/obe_b200.h"
#include "obe_device.cuh"
#include "obe_models.cuh"

static_assert(OBE_TILE == OBE_TILE_SIZE, "tile size mismatch");
static_assert(OBE_STATS_LEN == OBE_STATS_DOUBLES, "stats length mismatch");
static_assert(OBE_TILE == OBE_THREADS * OBE_EPT, "tile geometry");

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
static int obe_fail(const char* fmt, const char* a = "", const char* b = "") {
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return -1;
}
#define OBE_CUDA(x)                                                                  \
    do {                                                                             \
        cudaError_t e_ = (x);                                                        \
        if (e_ != cudaSuccess) return obe_fail("%s: %s", #x, cudaGetErrorString(e_)); \
    } while (0)
#define OBE_LAUNCH_CHECK(what)                                                        \
    do {                                                                              \
        cudaError_t e_ = cudaGetLastError();                                          \
        if (e_ != cudaSuccess) return obe_fail("launch %s: %s", what, cudaGetErrorString(e_)); \
    } while (0)

static int g_sms[64] = {0};            // per device: a process may drive several (the current device decides)
static int obe_sms() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    if (g_sms[dev] == 0) {
        if (cudaDeviceGetAttribute(&g_sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) g_sms[dev] = 0;
    }
    return g_sms[dev];
}
#define OBE_BLOCKS_PER_SM 4
#define OBE_MAX_GRID 4096

// ---------------------------------------------------------------------------------------------
// scratch layout of a cloud
// ---------------------------------------------------------------------------------------------
struct Scratch {
    unsigned int* counter;   // 64 words
    double* partials;        // OBE_MAX_GRID * OBE_NACC_MAX
    long long* plan_h;       // n_tiles + 1
    int* unit_start;         // n_tiles + 2
    unsigned int* anc;       // n + 4 (ancestors of the offspring written INTO this cloud)
    int* unit_tile;          // n_tiles + n / OBE_WR_MIN_CHUNK + 4 (work unit -> input tile)
};
#define OBE_OUT_CHUNK_HOST 4096
#ifndef OBE_WR_CHUNK
#define OBE_WR_CHUNK 3200   /* most output slots per work unit of the one-kernel resample (k_sys_resample_warp) */
#endif
#define OBE_WR_GROUP_HOST 128
#define OBE_WR_MIN_CHUNK 128  /* small clouds get smaller units so that every SM has warps to run */
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static size_t scratch_bytes(int64_t n) {
    const int64_t nt = (n + OBE_TILE - 1) / OBE_TILE;
    size_t b = 256;
    b += align_up((size_t)OBE_MAX_GRID * OBE_NACC_MAX * sizeof(double), 256);
    b += align_up((size_t)(nt + 1) * sizeof(long long), 256);
    b += align_up((size_t)(nt + 2) * sizeof(int), 256);
    b += align_up((size_t)(n + 4) * sizeof(unsigned int), 256);
    b += align_up((size_t)(nt + n / OBE_WR_MIN_CHUNK + 4) * sizeof(int), 256);
    return b;
}
static Scratch scratch_of(const obe_cloud_t* c) {
    const int64_t nt = (c->n + OBE_TILE - 1) / OBE_TILE;
    char* p = (char*)c->scratch_dev;
    Scratch s;
    s.counter = (unsigned int*)p; p += 256;
    s.partials = (double*)p; p += align_up((size_t)OBE_MAX_GRID * OBE_NACC_MAX * sizeof(double), 256);
    s.plan_h = (long long*)p; p += align_up((size_t)(nt + 1) * sizeof(long long), 256);
    s.unit_start = (int*)p; p += align_up((size_t)(nt + 2) * sizeof(int), 256);
    s.anc = (unsigned int*)p; p += align_up((size_t)(c->n + 4) * sizeof(unsigned int), 256);
    s.unit_tile = (int*)p;
    return s;
}

// ---------------------------------------------------------------------------------------------
// generic (model-free) update kernels: y supplied / likelihood supplied / refresh
// ---------------------------------------------------------------------------------------------
template <int D, int SRC>
__global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) k_update_generic(const ObeUpdateArgs a) {
    obe_update_body<ObeNoModel, D, SRC>(a);
}
// dynamic shared memory of the update kernel for (d, source): mirrors ObeStage<NROWS>
static size_t update_smem_bytes(int d, int src) {
    const int nrows = 1 + d + (src == OBE_SRC_Y ? OBE_MAX_CH : 0) + (src == OBE_SRC_LIK ? 1 : 0);
    const int elems = nrows <= 4 ? 2048 : (nrows <= 8 ? 1024 : 512);
    const int bytes = nrows * elems * 8;
    int nst = OBE_SMEM_BUDGET / bytes;
    if (nst > 4) nst = 4;
    return (size_t)nst * bytes + 1024;
}
// cudaFuncAttributeMaxDynamicSharedMemorySize once per (kernel, device) and calling thread instead of before every
// launch: a small-cloud cycle is a chain of 5-10 us kernels and the host has to stay ahead of it.
// (Unloading a user model may hand its kernel addresses to the next one: g_smem_epoch drops every thread's cache.)
static std::atomic<int> g_smem_epoch{0};
static cudaError_t set_max_smem(const void* f, size_t smem) {
    struct Ent { const void* f; size_t smem; int dev; };
    static thread_local Ent cache[96];
    static thread_local int n_cached = 0;
    static thread_local int seen_epoch = 0;
    const int epoch = g_smem_epoch.load(std::memory_order_relaxed);
    if (seen_epoch != epoch) { seen_epoch = epoch; n_cached = 0; }
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = -1; }
    for (int i = 0; i < n_cached; ++i)
        if (cache[i].f == f && cache[i].dev == dev) {
            if (cache[i].smem == smem) return cudaSuccess;
            const cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) cache[i].smem = smem;
            return e;
        }
    const cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && dev >= 0 && n_cached < 96) cache[n_cached++] = Ent{f, smem, dev};
    return e;
}
// q: the per-record data of a non-Gaussian likelihood, the second argument of its update kernels
static int launch_update_kernel(const void* f, int d, int src, const ObeUpdateArgs& a, int grid, cudaStream_t st,
                                const ObeLikParams* q = nullptr) {
    const size_t smem = update_smem_bytes(d, src);
    cudaError_t e = set_max_smem(f, smem);
    if (e != cudaSuccess) return obe_fail("cudaFuncSetAttribute(max dynamic smem): %s%s", cudaGetErrorString(e));
    void* params[2] = {const_cast<ObeUpdateArgs*>(&a), const_cast<ObeLikParams*>(q)};
    e = cudaLaunchKernel(f, dim3(grid), dim3(OBE_UPDATE_THREADS), params, smem, st);
    if (e != cudaSuccess) return obe_fail("launch update kernel: %s%s", cudaGetErrorString(e));
    return 0;
}
template <int SRC>
static int launch_generic(int d, const ObeUpdateArgs& a, int grid, cudaStream_t st) {
    const void* f = nullptr;
    switch (d) {
        case 1: f = (const void*)k_update_generic<1, SRC>; break;
        case 2: f = (const void*)k_update_generic<2, SRC>; break;
        case 3: f = (const void*)k_update_generic<3, SRC>; break;
        case 4: f = (const void*)k_update_generic<4, SRC>; break;
        case 5: f = (const void*)k_update_generic<5, SRC>; break;
        case 6: f = (const void*)k_update_generic<6, SRC>; break;
        case 7: f = (const void*)k_update_generic<7, SRC>; break;
        case 8: f = (const void*)k_update_generic<8, SRC>; break;
        default: return obe_fail("n_params must be 1..8%s%s");
    }
    return launch_update_kernel(f, d, SRC, a, grid, st);
}

// ---------------------------------------------------------------------------------------------
// single-block scans over per-tile arrays
// ---------------------------------------------------------------------------------------------
#define OBE_SCAN_THREADS 1024

// Block-wide exclusive scans (1024 threads) of one value per thread; the per-array kernels below
// walk their array in coalesced chunks of 1024 with a running carry, so the association order
// (carry + (warp base + lane prefix)) depends only on the element index.
__device__ __forceinline__ double block_excl_sum_1024(double v, double* sm /*34*/, double* tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    __syncthreads();
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    if (warp == 0) {
        double xs = sm[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, xs, o);
            if (lane >= o) xs += y;
        }
        double ex = __shfl_up_sync(0xffffffffu, xs, 1);  // exclusive base of each warp
        if (lane == 0) ex = 0.0;
        sm[lane] = ex;
        if (lane == 31) sm[32] = xs;
    }
    __syncthreads();
    const double base = sm[warp];
    double ex = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) ex = 0.0;
    *tot = sm[32];
    return base + ex;
}

__device__ __forceinline__ int block_excl_isum_1024(int v, int* sm /*34*/, int* tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    __syncthreads();
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    if (warp == 0) {
        const int w = sm[lane];
        int xs = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, xs, o);
            if (lane >= o) xs += y;
        }
        sm[lane] = xs - w;
        if (lane == 31) sm[32] = xs;
    }
    __syncthreads();
    *tot = sm[32];
    return sm[warp] + (x - v);
}

// tile_prefix[k] = sum of tile_sums[0..k) in a fixed association; tile_prefix[n_tiles] is THE
// total every CDF consumer divides by.
__global__ void __launch_bounds__(OBE_SCAN_THREADS) k_tile_scan(const double* __restrict__ tile_sums,
                                                                long long n_tiles, double* __restrict__ prefix,
                                                                double* __restrict__ stats, int renormalise,
                                                                long long uniform, long long n,
                                                                const long long* __restrict__ n_dev = nullptr,
                                                                int implicit = 0) {
    __shared__ double sm[OBE_SCANW * (OBE_SCAN_THREADS / 32 + 1)];
    if (n_dev) { n = *n_dev; n_tiles = (n + OBE_TILE - 1) / OBE_TILE; }
    obe_tile_scan_block<OBE_SCAN_THREADS / 32>(tile_sums, n_tiles, prefix, stats, renormalise, uniform, n, implicit, sm, 0);
}

__global__ void k_fill_uniform(double* __restrict__ w, double* __restrict__ tile_sums, long long n,
                               long long n_tiles, int write_weights, long long n_total,
                               const long long* __restrict__ n_dev = nullptr) {
    if (n_dev) { n = *n_dev; n_tiles = (n + OBE_TILE - 1) / OBE_TILE; }
    const double v = 1.0 / (double)n_total;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (write_weights)
        for (long long i = i0; i < n; i += stride) w[i] = v;
    for (long long k = i0; k < n_tiles; k += stride) {
        const long long cnt = min((long long)OBE_TILE, n - k * OBE_TILE);
        tile_sums[k] = (double)cnt * v;
    }
}

__global__ void k_normalized_weights(const double* __restrict__ w, const double* __restrict__ stats,
                                     double* __restrict__ out, long long n, const long long* __restrict__ n_dev) {
    if (n_dev) n = *n_dev;
    const double inv = stats[OBE_ST_INVS], wuni = stats[OBE_ST_UNIFORM];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        out[i] = obe_nan_to_num((wuni > 0.0 ? wuni : w[i]) * inv);
}

__global__ void __launch_bounds__(OBE_THREADS) k_cdf(const double* __restrict__ w, const double* __restrict__ prefix,
                                                     long long n, long long n_tiles, double* __restrict__ cdf,
                                                     const double* __restrict__ stats) {
    __shared__ double sm[8];
    const double inv_total = 1.0 / prefix[n_tiles];
    const double wuni = stats ? stats[OBE_ST_UNIFORM] : 0.0;
    for (long long k = blockIdx.x; k < n_tiles; k += gridDim.x) {
        double cn[OBE_EPT];
        tile_cdf_blocked(w, prefix, k, n, inv_total, cn, sm, 0.0, true, wuni);
        const long long i0 = k * OBE_TILE + (long long)threadIdx.x * OBE_EPT;
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e)
            if (i0 + e < n) cdf[i0 + e] = cn[e];
        __syncthreads();
    }
}

// tile containing u: #{k in [0, n_tiles) : cdf(end of tile k) <= u}, clamped
__device__ __forceinline__ long long find_tile(const double* __restrict__ prefix, long long n_tiles,
                                               double inv_total, double u) {
    long long lo = 0, hi = n_tiles;  // first k whose end-of-tile CDF value is > u
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        const double c = (mid == n_tiles - 1) ? 1.0 : obe_mul(prefix[mid + 1], inv_total);
        if (c <= u) lo = mid + 1; else hi = mid;
    }
    return min(lo, n_tiles - 1);
}

// The same search by a whole block: every round the blockDim.x threads probe evenly spaced tiles and a block-wide
// count narrows the range by a factor blockDim.x -- 2 rounds (two dependent loads) for 65 536 tiles where the
// sequential search walks 16.  All threads must call it (block barriers inside); same answer in every thread.
__device__ __forceinline__ long long find_tile_block(const double* __restrict__ prefix, long long n_tiles,
                                                     double inv_total, double u) {
    long long lo = 0, hi = n_tiles;  // first k in [lo, hi) whose end-of-tile CDF value is > u, else hi
    while (lo < hi) {
        const long long span = hi - lo;
        const long long step = (span + blockDim.x - 1) / blockDim.x;
        const long long k = lo + (long long)threadIdx.x * step;
        bool le = false;
        if (k < hi) {
            const double c = (k == n_tiles - 1) ? 1.0 : obe_mul(prefix[k + 1], inv_total);
            le = c <= u;
        }
        const long long cnt = __syncthreads_count(le);           // the probes with c <= u are a prefix (monotone CDF)
        if (cnt == 0) { hi = lo; break; }
        const long long next = lo + cnt * step;                  // first probe with c > u (if it exists)
        lo = lo + (cnt - 1) * step + 1;
        hi = next < hi ? next : hi;
    }
    return min(lo, n_tiles - 1);
}

__global__ void k_search(const double* __restrict__ cdf, const double* __restrict__ prefix, long long n,
                         long long n_tiles, const double* __restrict__ u, long long m,
                         long long* __restrict__ idx) {
    const double inv_total = 1.0 / prefix[n_tiles];
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < m;
         q += (long long)gridDim.x * blockDim.x) {
        const double uq = u[q];
        const long long k = find_tile(prefix, n_tiles, inv_total, uq);
        long long lo = k * OBE_TILE, hi = min(n, lo + OBE_TILE);
        const long long last = hi - 1;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (cdf[mid] <= uq) lo = mid + 1; else hi = mid;
        }
        idx[q] = min(lo, last);
    }
}

// ---------------------------------------------------------------------------------------------
// Peer exchange over NVLink (sharded engines, one process per GPU): every rank owns one small buffer
// (cudaMalloc + CUDA IPC, mapped by all peers).  The producing kernels write their few doubles straight
// into every peer's buffer, then a system-scope release store of an epoch number; consumers spin on
// their OWN buffer (acquire loads) -- no NCCL launch, no stream hop.  Slots are double-buffered by the
// parity of the epoch: a rank can run at most one exchange ahead of the slowest one, because passing
// exchange e needs every peer's flag e, which a peer raises only after it has consumed e-1.
// Layout in 8-byte words:
// ---------------------------------------------------------------------------------------------
#define OBE_PEER_MAX 16
#define OBE_PEER_STATS 0                                  /* [2][OBE_PEER_MAX][64] stats blocks        */
#define OBE_PEER_DRAWS (2 * OBE_PEER_MAX * OBE_STATS_LEN)  /* [2][1024]  draws (d, K), d*K <= 1024      */
#define OBE_PEER_FLAGS (OBE_PEER_DRAWS + 2 * 1024)         /* [2 kinds][2][OBE_PEER_MAX] uint64 epochs  */
#define OBE_PEER_ERR (OBE_PEER_FLAGS + 4 * OBE_PEER_MAX)   /* != 0: a wait timed out                    */
#define OBE_PEER_WORDS (OBE_PEER_ERR + 8)
struct ObePeers { double* p[OBE_PEER_MAX]; };

__device__ __forceinline__ void obe_flag_store(unsigned long long* addr, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long obe_flag_load(const unsigned long long* addr) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(addr) : "memory");
    return v;
}
// false after ~20 s: a peer died or the ranks fell out of step; the caller flags it, nothing hangs
__device__ __forceinline__ bool obe_flag_wait(const unsigned long long* flag, unsigned long long epoch) {
    const long long t0 = clock64();
    while (obe_flag_load(flag) < epoch) {
        __nanosleep(40);
        if (clock64() - t0 > 40000000000ll) return false;
    }
    return true;
}
__device__ __forceinline__ unsigned long long* obe_peer_flags(double* buf, int kind, int parity) {
    return reinterpret_cast<unsigned long long*>(buf + OBE_PEER_FLAGS) + (kind * 2 + parity) * OBE_PEER_MAX;
}

// Device-side resample decision (obe_cycle, resample == 2): the update writes stats[OBE_ST_FIRED]; the kernels of the
// resample half run only when it is set (gate), the plain K-draw kernel only when it is not (gate_off).  Armed per
// calling thread by obe_cycle around the entry points it chains, like the deferred emission below.
static thread_local const double* g_gate_on = nullptr;
static thread_local const double* g_gate_off = nullptr;
static thread_local double g_update_gate_thr = 0.0, g_update_gate_n = 0.0;
// Zero-copy results of a closed-loop cycle (obe_cycle with stats_host / best_host): the update kernel's finishing block
// and the utility kernel's last block store straight into the caller's pinned host block (device-visible under UVA).
static thread_local double* g_update_stats_out = nullptr;
static thread_local long long* g_utility_best_out = nullptr;
static thread_local unsigned long long* g_utility_seq_out = nullptr;
static thread_local unsigned long long g_utility_seq_val = 0;

struct ObeDrawArgs {
    const double* gate_off;     // optional: skip the whole launch when *gate_off != 0 (a resample fired instead)
    const double* w; const double* prefix; long long n; long long n_tiles;
    const double* particles; long long ld; int d;
    double* draws; long long* idx; int k;
    const long long* n_dev;     // optional live count
    const double* plan;         // optional shard plan: this rank draws only the uniforms it owns
    const double* stats;        // optional: stats block (implicit uniform weights)
    int post;                   // use the post-resample shard totals of the plan
    // peer mode (peer_world > 0): the owner of a draw writes it into EVERY rank's buffer, the last CTA raises
    // this rank's flag there (instead of zeros + all-reduce)
    int peer_world, peer_rank;
    unsigned long long peer_epoch;
    unsigned int* peer_counter;
    ObePeers peers;
    double u[OBE_MAX_DRAWS];
};
// one block per draw: tile by binary search on the prefix, element by a canonical scan + count
__global__ void __launch_bounds__(OBE_THREADS) k_draw(const ObeDrawArgs a) {
    __shared__ double sm[8];
    __shared__ int cnt[OBE_THREADS / 32];
    const int q = blockIdx.x;
    obe_grid_dep_launch();
    obe_grid_dep_wait();                           // (a no-op unless launched with programmatic serialization)
    if (a.gate_off && *a.gate_off != 0.0) return;
    double uq = a.u[q];
    const long long n = a.n_dev ? *a.n_dev : a.n;
    const long long n_tiles = a.n_dev ? (n + OBE_TILE - 1) / OBE_TILE : a.n_tiles;
    bool mine = true;
    if (a.plan) {
        // sharded cloud: owner of u is the shard whose [offset, offset+total) holds u*T; the others
        // contribute zeros to the all-reduce that follows (NCCL mode) or nothing at all (peer mode)
        const int world = (int)a.plan[OBE_PL_WORLD], rank = (int)a.plan[OBE_PL_RANK];
        const double* off = a.plan + (a.post ? OBE_PL_POST_OFF : OBE_PL_PRE_OFF);
        const double* tot = a.plan + (a.post ? OBE_PL_POST_TOT : OBE_PL_PRE_TOT);
        const double target = uq * (a.post ? a.plan[OBE_PL_POST_TOTAL] : a.plan[OBE_PL_TOTAL]);
        int owner = 0;
        for (int g = 0; g < world; ++g)
            if (off[g] + tot[g] <= target) owner = g + 1;
        owner = min(owner, world - 1);
        while (owner > 0 && !(tot[owner] > 0.0)) --owner;
        mine = (owner == rank);
        if (!mine) {
            if (threadIdx.x == 0 && a.peer_world == 0) {
                if (a.idx) a.idx[q] = -1;
                for (int j = 0; j < a.d; ++j) a.draws[(long long)j * a.k + q] = 0.0;
            }
        } else {
            uq = (target - off[rank]) / tot[rank];
            uq = uq < 0.0 ? 0.0 : (uq > 0.99999999999999989 ? 0.99999999999999989 : uq);
        }
    }
    if (mine) {                                    // (uniform over the block)
        const double inv_total = 1.0 / a.prefix[n_tiles];
        const long long k = find_tile_block(a.prefix, n_tiles, inv_total, uq);
        double cn[OBE_EPT];
        tile_cdf_blocked(a.w, a.prefix, k, n, inv_total, cn, sm, 0.0, true, a.stats ? a.stats[OBE_ST_UNIFORM] : 0.0);
        const long long base = k * OBE_TILE;
        int c = 0;
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e) {
            const long long i = base + (long long)threadIdx.x * OBE_EPT + e;
            if (i < n && cn[e] <= uq) ++c;
        }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) c += __shfl_xor_sync(0xffffffffu, c, m);
        if ((threadIdx.x & 31) == 0) cnt[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w2 = 0; w2 < OBE_THREADS / 32; ++w2) tot += cnt[w2];
            const long long last = min(n, base + OBE_TILE) - 1;
            const long long i = min(base + tot, last);
            if (a.idx) a.idx[q] = i;
            if (a.peer_world > 0) {
                const int parity = (int)(a.peer_epoch & 1ull);
                for (int j = 0; j < a.d; ++j) {
                    const double v = a.particles[j * a.ld + i];
                    for (int g = 0; g < a.peer_world; ++g)
                        a.peers.p[g][OBE_PEER_DRAWS + parity * 1024 + j * a.k + q] = v;
                }
            } else {
                for (int j = 0; j < a.d; ++j) a.draws[(long long)j * a.k + q] = a.particles[j * a.ld + i];
            }
        }
    }
    if (a.peer_world > 0 && threadIdx.x == 0) {
        // every CTA reports in; the last one raises this rank's flag in every peer's buffer
        __threadfence_system();
        if (atomicAdd(a.peer_counter, 1u) == gridDim.x - 1) {
            __threadfence_system();
            const int parity = (int)(a.peer_epoch & 1ull);
            for (int g = 0; g < a.peer_world; ++g)
                obe_flag_store(obe_peer_flags(a.peers.p[g], 1, parity) + a.peer_rank, a.peer_epoch);
            *a.peer_counter = 0u;
        }
    }
}

// consumer side of the draw exchange: wait for every rank's flag of this epoch, then copy the (d, K) draws
// out of the local buffer
__global__ void k_peer_collect_draws(double* mine, int world, unsigned long long epoch, double* __restrict__ draws,
                                     int n_values) {
    const int parity = (int)(epoch & 1ull);
    bool ok = true;
    if ((int)threadIdx.x < world) ok = obe_flag_wait(obe_peer_flags(mine, 1, parity) + threadIdx.x, epoch);
    if (!ok) mine[OBE_PEER_ERR] = 1.0;
    __syncthreads();
    __threadfence_system();
    for (int q = threadIdx.x; q < n_values; q += blockDim.x) draws[q] = mine[OBE_PEER_DRAWS + parity * 1024 + q];
}

// Packed normal stream of the streaming resample kernels (k_sys_resample_warp, k_sys_move): the jitter normals of
// the whole cloud form ONE sequence, normal m = D * slot + j, four per Philox call (two Box-Muller pairs): call
// q = m >> 2, word m & 3.  A thread that owns 4 consecutive output slots starting at a multiple of 4 needs exactly
// the calls (slot0 / 4) * D ... + D - 1: D calls per 4 slots whatever D, none of the 128 bits wasted (the per-slot
// stream of device_normals spends 4 * ceil(D / 4) calls).  ctr = (q_lo, q_hi, 0x80000000 | D, epoch), key = seed.
// Slots are GLOBAL comb slots, so the jitter does not depend on how the cloud is sharded.  Restated in
// oracle/obe_oracle.py:device_normals_packed.  Implementations: jitter_group4 (4 aligned slots), packed_normals_slot.
// Liu-West move of one particle (particlepdf.py:296-307): x + z @ F, optional contraction
template <int D>
__device__ __forceinline__ void liu_west(double (&x)[D], const double (&z)[D], const double* __restrict__ F,
                                         const double* __restrict__ mean, double a_param, int scale) {
#pragma unroll
    for (int j = 0; j < D; ++j) {
        double nud = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) nud += z[k] * F[k * D + j];
        double v = x[j] + nud;
        if (scale) v = obe_add(obe_mul(v, a_param), obe_mul(mean[j], obe_sub(1.0, a_param)));
        x[j] = v;
    }
}

// The D normals of ONE output slot out of the packed stream (kernels that walk slots one at a time: the batched
// engines' sys_unit): normals m = D*slot .. D*slot + D-1 live in calls (D*slot) >> 2 .. (D*slot + D-1) >> 2, at most
// (D + 6) / 4 of them.  Same values as jitter_group4 uses for that slot.
template <int D>
__device__ __forceinline__ void packed_normals_slot(long long slot, unsigned long long seed, unsigned int epoch,
                                                    double (&z)[D]) {
    constexpr int NC = (D + 6) / 4;
    const unsigned long long m0 = (unsigned long long)slot * (unsigned long long)D;
    const unsigned long long q0 = m0 >> 2;
    const int w0 = (int)(m0 & 3ull);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        if (4 * c >= w0 + D) break;                              // (warp-divergent only through slot & 3)
        const unsigned long long q = q0 + (unsigned long long)c;
        unsigned int r[4];
        philox4x32_10((unsigned int)(q & 0xffffffffull), (unsigned int)(q >> 32), 0x80000000u | (unsigned int)D, epoch,
                      (unsigned int)(seed & 0xffffffffull), (unsigned int)(seed >> 32), r);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float rad = obe_sqrt_approx(-2.0f * __logf(u24(r[2 * h])));
            float sn, cs;
            __sincosf(6.2831853071795865f * u24(r[2 * h + 1]), &sn, &cs);
            const double zz[2] = {(double)(rad * cs), (double)(rad * sn)};
#pragma unroll
            for (int w = 0; w < 2; ++w) {
                const int k = 4 * c + 2 * h + w - w0;            // coordinate this normal belongs to
#pragma unroll
                for (int j = 0; j < D; ++j)
                    if (j == k) z[j] = zz[w];
            }
        }
    }
}

// Liu-West move of 4 consecutive output slots (global slots slot0 .. slot0+3, slot0 a multiple of 4) with the packed
// normal stream, STREAMING: every normal is folded into the D coordinates it nudges as soon as Box-Muller produces it
// (x_j <- fma(z_k, F[k][j], x_j)), so the 4*D normals are never all live -- 2*4*D registers less than building z
// first, which is what lets the resample kernels keep their gathers and the Philox state in registers.  z_out
// (tests): the normals are also stored, (n, D) row-major at output position o0 + u.
// R = slot0 & 3 (compile time): the 4 slots need the 4*D consecutive normals m = D*slot0 .. D*slot0 + 4*D - 1 of the
// packed stream, which start at word W = (D*R) & 3 of call (D*slot0) >> 2 and span D calls when W == 0, D + 1 otherwise.
// A shard whose first global slot is not a multiple of 4 aligns its emission groups to its OUTPUT (whole 32-byte
// sectors, plain 16-byte stores) and pays the one extra Philox call per 4 slots instead of shuffling values between
// lanes; the normals of a slot do not depend on the grouping, so the offspring are the same bits either way.
template <int D, int R>
__device__ __forceinline__ void jitter_group4_w(double (&xv)[4][D], long long slot0, unsigned long long seed,
                                                unsigned int epoch, const double* __restrict__ F,
                                                const double* __restrict__ mean, double a_param, int scale,
                                                double* __restrict__ z_out, long long o0, const bool (&ok)[4]) {
    constexpr int W = (D * R) & 3;
    constexpr int NC = D + (W ? 1 : 0);
    const unsigned int key0 = (unsigned int)(seed & 0xffffffffull), key1 = (unsigned int)(seed >> 32);
    const unsigned long long q0 = ((unsigned long long)slot0 * (unsigned long long)D) >> 2;
    unsigned int c0[NC], c1[NC], c2[NC], c3[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        const unsigned long long q = q0 + (unsigned long long)c;
        c0[c] = (unsigned int)(q & 0xffffffffull);
        c1[c] = (unsigned int)(q >> 32);
        c2[c] = 0x80000000u | (unsigned int)D; c3[c] = epoch;
    }
    unsigned int k0 = key0, k1 = key1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const unsigned int hi0 = __umulhi(0xD2511F53u, c0[c]), lo0 = 0xD2511F53u * c0[c];
            const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2[c]), lo1 = 0xCD9E8D57u * c2[c];
            const unsigned int n0 = hi1 ^ c1[c] ^ k0, n2 = hi0 ^ c3[c] ^ k1;
            c0[c] = n0; c1[c] = lo1; c2[c] = n2; c3[c] = lo0;
        }
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        const unsigned int r4[4] = {c0[c], c1[c], c2[c], c3[c]};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int f0 = 4 * c + 2 * h - W;                    // compile-time after unrolling: first of the pair
            if (f0 + 1 < 0 || f0 >= 4 * D) continue;             // both normals of the pair lie outside the 4 slots
            const float rad = obe_sqrt_approx(-2.0f * __logf(u24(r4[2 * h])));
            float sn, cs;
            __sincosf(6.2831853071795865f * u24(r4[2 * h + 1]), &sn, &cs);
            const double zz[2] = {(double)(rad * cs), (double)(rad * sn)};
#pragma unroll
            for (int w = 0; w < 2; ++w) {
                const int f = f0 + w;
                if (f < 0 || f >= 4 * D) continue;
                const int u = f / D, k = f % D;
                if (z_out && ok[u]) z_out[(o0 + u) * D + k] = zz[w];
#pragma unroll
                for (int j = 0; j < D; ++j) xv[u][j] = fma(zz[w], F[k * D + j], xv[u][j]);
            }
        }
    }
    if (scale) {
        const double b = obe_sub(1.0, a_param);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int j = 0; j < D; ++j) xv[u][j] = obe_add(obe_mul(xv[u][j], a_param), obe_mul(mean[j], b));
        }
    }
}
template <int D>
__device__ __forceinline__ void jitter_group4(double (&xv)[4][D], long long slot0, unsigned long long seed,
                                              unsigned int epoch, const double* __restrict__ F,
                                              const double* __restrict__ mean, double a_param, int scale,
                                              double* __restrict__ z_out, long long o0, const bool (&ok)[4]) {
    jitter_group4_w<D, 0>(xv, slot0, seed, epoch, F, mean, a_param, scale, z_out, o0, ok);
}

struct ObeResampleArgs {
    const double* pin; long long ld_in; const double* w_in; const double* prefix;
    long long n; long long n_tiles;
    double* pout; long long ld_out; double* w_out;
    const long long* idx_in;       // gather mode
    const double* z_in;            // gather mode, optional (n, d)
    const long long* plan_h; const int* unit_start; const int* unit_tile;  // systematic mode
    const double* stats;
    long long* idx_out; double* z_out;
    double u0, a_param;
    int scale, factor_from_stats, jitter;
    unsigned int epoch;
    unsigned long long seed;
    // shard of a multi-GPU cloud (sharded == 0: the cloud is whole and these are derived on device)
    int sharded, last_shard;
    long long n_total;             // particles over all shards = teeth of the comb
    long long slot_begin, slot_end; // global output slots owned by this shard's particles
    double cdf_offset;             // summed weight of the lower-ranked shards
    double cdf_total;              // global total weight
    const long long* n_dev_in;     // optional live count of the input shard
    const double* plan;            // optional device-resident shard plan (overrides the by-value shard fields)
    long long cap_out;             // capacity of the output buffers (planned mode)
    int implicit_out;              // 1: do not write the offspring weights, leave them implicit
    int chunk;                     // output slots per work unit the plan was made with
    unsigned int* unit_counter;    // one-kernel path: next unit to hand out (zeroed by the plan kernel); null: static stride
    unsigned int* anc;             // two-kernel path: ancestor (input index) of every output slot of this shard
    double* out_tile_sums; double* out_prefix; double* out_stats;   // CDF bookkeeping of the offspring cloud
    const double* gate;            // optional: the one-kernel resample and the pick run only when *gate != 0
    double factor[OBE_MAX_DIMS * OBE_MAX_DIMS];
    double mean[OBE_MAX_DIMS];
};

// F (z @ F convention) and mean into shared memory; from the host, or Cholesky of
// (1-a^2) * cov(stats) on the device: the "covariance computed in the same pass" path.
template <int D>
__device__ __forceinline__ void setup_factor(const ObeResampleArgs& a, double* sF, double* sMean) {
    if (threadIdx.x == 0) {
        if (a.plan) {
            for (int q = 0; q < D * D; ++q) sF[q] = a.plan[OBE_PL_FACTOR + q];
            for (int j = 0; j < D; ++j) sMean[j] = a.plan[OBE_PL_MEAN + j];
        } else if (!a.factor_from_stats) {
            for (int q = 0; q < D * D; ++q) sF[q] = a.factor[q];
            for (int j = 0; j < D; ++j) sMean[j] = a.mean[j];
        } else {
            const double st = a.stats[OBE_ST_SUMT], ssq = a.stats[OBE_ST_SUMSQ];
            const double fact = st - ssq / st;
            const double shrink = 1.0 - a.a_param * a.a_param;
            double cov[D][D], L[D][D];
            int q = 0;
            for (int j = 0; j < D; ++j) {
                sMean[j] = a.stats[OBE_ST_PIVOT + j] + a.stats[OBE_ST_M1 + j] / st;
                for (int k = j; k < D; ++k) {
                    const double c = (a.stats[OBE_ST_M2 + q] - a.stats[OBE_ST_M1 + j] * a.stats[OBE_ST_M1 + k] / st) / fact;
                    cov[j][k] = cov[k][j] = shrink * c;
                    ++q;
                }
            }
            for (int j = 0; j < D; ++j)
                for (int k = 0; k < D; ++k) L[j][k] = 0.0;
            for (int j = 0; j < D; ++j) {
                double s = cov[j][j];
                for (int k = 0; k < j; ++k) s -= L[j][k] * L[j][k];
                const double dj = s > 0.0 ? sqrt(s) : 0.0;
                L[j][j] = dj;
                for (int i = j + 1; i < D; ++i) {
                    double t = cov[i][j];
                    for (int k = 0; k < j; ++k) t -= L[i][k] * L[j][k];
                    L[i][j] = dj > 0.0 ? t / dj : 0.0;
                }
            }
            // x = z @ L^T  ->  F[k][j] = L[j][k]
            for (int k = 0; k < D; ++k)
                for (int j = 0; j < D; ++j) sF[k * D + j] = L[j][k];
        }
    }
    __syncthreads();
}

template <int D>
__global__ void __launch_bounds__(OBE_THREADS) k_gather_jitter(const ObeResampleArgs a) {
    __shared__ double sF[D * D];
    __shared__ double sMean[D];
    setup_factor<D>(a, sF, sMean);
    const double wv = 1.0 / (double)a.n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n;
         i += (long long)gridDim.x * blockDim.x) {
        const long long anc = a.idx_in[i];
        double x[D], z[D];
#pragma unroll
        for (int j = 0; j < D; ++j) x[j] = a.pin[j * a.ld_in + anc];
        if (a.jitter) {
            if (a.z_in) {
#pragma unroll
                for (int j = 0; j < D; ++j) z[j] = a.z_in[i * D + j];
            } else {
                device_normals<D>(i, a.seed, a.epoch, z);
            }
            if (a.z_out) {
#pragma unroll
                for (int j = 0; j < D; ++j) a.z_out[i * D + j] = z[j];
            }
            liu_west<D>(x, z, sF, sMean, a.a_param, a.scale);
        }
#pragma unroll
        for (int j = 0; j < D; ++j) a.pout[j * a.ld_out + i] = x[j];
        a.w_out[i] = wv;
    }
}

// ---- systematic comb --------------------------------------------------------------------------
// #{i in [0,n) : (i + u0) * inv_n < c}; the comb value is two IEEE ops (add, mul), monotone in i.
// Works on integer-valued doubles (exact below 2^53) to stay off the int<->fp conversion path.
// The real-valued answer is ceil(c*n - u0).  The comb's three roundings move a tooth by at most
// ~4.4e-16*n slots, so when c*n - u0 is farther than `tol` = 2e-15*n from an integer the estimate is
// already exact; only the (probability ~4e-15*n) near-boundary cases run the exact comparison loop.
__device__ __forceinline__ double comb_count_d(double c, double u0, double inv_n, double nd, double tol) {
    const double x = fma(c, nd, -u0);
    double i = ceil(x);
    // c is a CDF value in [0, 1 + few ulp], so ceil(x) lies in [0, nd] unless x is within tol of nd,
    // which the boundary test catches: the fast path needs no range test.
    if (fabs((i - x) - 0.5) > 0.5 - tol) {
        i = (i < 0.0) ? 0.0 : i;
        i = (i > nd) ? nd : i;
        while (i > 0.0 && obe_mul(obe_add(i - 1.0, u0), inv_n) >= c) i -= 1.0;
        while (i < nd && obe_mul(obe_add(i, u0), inv_n) < c) i += 1.0;
    }
    return i;
}

// exclusive max over the preceding warps of a block of 8 warps (values >= 0), totals in smx[0..8)
__device__ __forceinline__ int obe_prev_warps_max8(const int* smx, int warp, int lane) {
    int v = smx[lane & 7];
    v = ((lane & 7) < warp) ? v : 0;
    v = max(v, __shfl_xor_sync(0xffffffffu, v, 1));
    v = max(v, __shfl_xor_sync(0xffffffffu, v, 2));
    v = max(v, __shfl_xor_sync(0xffffffffu, v, 4));
    return v;
}

#define OBE_OUT_CHUNK 4096
static_assert(OBE_OUT_CHUNK == OBE_OUT_CHUNK_HOST, "scratch sizing");
#define OBE_SPT (OBE_OUT_CHUNK / OBE_THREADS) /* output slots per thread in the mark scan */
// plan: H[k] = first output slot owned by tile k (monotone), unit_start[k] = first work unit of
// tile k, one unit = up to OBE_OUT_CHUNK output slots of one input tile.
__global__ void __launch_bounds__(OBE_SCAN_THREADS) k_sys_plan(const double* __restrict__ prefix, long long n_tiles,
                                                               long long n_total, double u0, double cdf_offset,
                                                               double cdf_total, long long slot_begin,
                                                               long long slot_end, long long* __restrict__ H,
                                                               int* __restrict__ unit_start,
                                                               int* __restrict__ unit_tile,
                                                               const long long* __restrict__ n_dev = nullptr,
                                                               const double* __restrict__ plan = nullptr,
                                                               int chunk = OBE_OUT_CHUNK,
                                                               unsigned int* __restrict__ unit_counter = nullptr,
                                                               const double* __restrict__ gate = nullptr) {
    __shared__ long long sml[OBE_SCANW * (OBE_SCAN_THREADS / 32 + 1)];
    __shared__ int smi[OBE_SCANW * (OBE_SCAN_THREADS / 32 + 1)];
    const int t = threadIdx.x;
    obe_grid_dep_launch();
    obe_grid_dep_wait();
    if (gate && *gate == 0.0) return;                      // device-side resample test: it did not fire
    if (t == 0 && unit_counter) *unit_counter = 0u;        // the streaming kernel hands its units out dynamically
    if (n_dev) n_tiles = (*n_dev + OBE_TILE - 1) / OBE_TILE;
    if (plan) {
        n_total = (long long)plan[OBE_PL_NTOTAL]; u0 = plan[OBE_PL_U0];
        cdf_offset = plan[OBE_PL_OFFSET]; cdf_total = plan[OBE_PL_TOTAL];
        slot_begin = (long long)plan[OBE_PL_SLOT0]; slot_end = (long long)plan[OBE_PL_SLOT1];
    }
    const double inv_total = 1.0 / (cdf_total > 0.0 ? cdf_total : prefix[n_tiles]);
    const double nd = (double)n_total, inv_n = 1.0 / nd, tol = 2e-15 * nd;
    // raw H[k]: elementwise, coalesced, OBE_SCANW loads in flight per thread
    for (long long base = 0; base <= n_tiles; base += OBE_SCANW * OBE_SCAN_THREADS) {
        double pk[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            pk[e] = (k < n_tiles) ? prefix[k] : 0.0;
        }
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k > n_tiles) continue;
            long long h = (k == 0) ? slot_begin
                                   : (k == n_tiles ? slot_end
                                                   : (long long)comb_count_d(obe_mul(obe_add(cdf_offset, pk[e]), inv_total),
                                                                             u0, inv_n, nd, tol));
            H[k] = min(max(h, slot_begin), slot_end);
        }
    }
    __syncthreads();
    // The prefix can dip by an ulp where two association orders meet, so H is made monotone by a
    // running max (in place); then unit_start = exclusive scan of the units per tile.  Both scans walk
    // OBE_SCANW chunks of 1024 tiles per round.
    constexpr int NWP = OBE_SCAN_THREADS / 32;
    long long hcarry = slot_begin;
    for (long long base = 0; base < n_tiles; base += OBE_SCANW * OBE_SCAN_THREADS) {
        long long h[OBE_SCANW], ex[OBE_SCANW], tot[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            h[e] = (k < n_tiles) ? H[k] : -1;
        }
        obe_block_excl_scanw<long long, NWP>(h, ex, tot, sml, ObeOpMax(), -1ll, 0);
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k < n_tiles) H[k] = max(max(hcarry, ex[e]), h[e]);
            hcarry = max(hcarry, tot[e]);
        }
        __syncthreads();
    }
    int icarry = 0;
    for (long long base = 0; base < n_tiles; base += OBE_SCANW * OBE_SCAN_THREADS) {
        int units[OBE_SCANW], ex[OBE_SCANW], tot[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            units[e] = (k < n_tiles) ? (int)((max(H[k + 1] - H[k], 0ll) + chunk - 1) / chunk) : 0;
        }
        obe_block_excl_scanw<int, NWP>(units, ex, tot, smi, ObeOpSum(), 0, 0);
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k < n_tiles) {
                const int first = icarry + ex[e];
                unit_start[k] = first;
                if (unit_tile)
                    for (int u = 0; u < units[e]; ++u) unit_tile[first + u] = (int)k;
            }
            icarry += tot[e];
        }
        __syncthreads();
    }
    const int total_units = icarry;
    if (t == 0) unit_start[n_tiles] = total_units;
}

// The same plan for large clouds on a thread-block cluster of 8 CTAs: every CTA takes a contiguous
// segment of the tiles (48 829 tiles at 1e8 particles -> one round of 8 x 1024 per CTA instead of six rounds
// of a single CTA per pass), scans it locally, and the eight segment totals (running max of H, units) are
// exchanged through distributed shared memory -- each CTA writes its total into every CTA's copy, one
// cluster barrier, then every CTA folds the totals of the segments before it into its own results.
#define OBE_PLAN_CLUSTER 8
// Launch with the programmatic-stream-serialization attribute (obe_grid_dep_wait in the kernel): the launch latency and
// the prologue of a dependent kernel overlap the tail of its predecessor in the stream.
static int64_t g_pdl = 1;                         /* obe_set_option("pdl") */
template <class... KArgs, class... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

static int64_t g_utility_lane_fill = 50;          /* obe_set_option("utility_lane_fill"), percent of resident threads */
static int64_t g_plan_cluster_min_tiles = 8192;   /* obe_set_option("plan_cluster_min_tiles") */
static int64_t g_utility_cache = 1;               /* obe_set_option("utility_cache"): park the K curves in shared memory */
static int64_t g_utility_info_blocks = 0;         /* obe_set_option("utility_info_blocks"): > 0 caps the information-gain grid */
static int64_t g_resample_fused = 1;              /* obe_set_option("resample_fused"): 1 = k_sys_resample_warp, 0 = ancestors + move */
static int64_t g_resample_units_per_sm = 16;      /* obe_set_option("resample_units_per_sm"): work units per SM the chunk size aims at */
static int64_t g_resample_reserve = 0;            /* obe_set_option("resample_reserve_ctas"): CTA slots an early-select resample leaves to the selection kernels */
static int64_t g_resample_dynamic = 1;            /* obe_set_option("resample_dynamic"): units handed out by an atomic counter */
static int64_t g_zero_copy_out = 1;               /* obe_set_option("zero_copy_out"): kernels store stats / argmax into the pinned host block themselves */
static int64_t g_copy_out_side = 1;               /* obe_set_option("copy_out_side"): early-select cycles copy stats + argmax out on the selection stream */
static int64_t g_resample_blocks = 0;             /* obe_set_option("resample_blocks"): CTAs per SM of the fused kernel (0: default) */
#ifndef OBE_PLAN_CLUSTER_MIN_TILES
#define OBE_PLAN_CLUSTER_MIN_TILES 8192     /* below: one CTA does every pass in a single round anyway */
#endif
__global__ void __cluster_dims__(OBE_PLAN_CLUSTER, 1, 1) __launch_bounds__(OBE_SCAN_THREADS)
k_sys_plan_cluster(const double* __restrict__ prefix, long long n_tiles, long long n_total, double u0,
                   double cdf_offset, double cdf_total, long long slot_begin, long long slot_end,
                   long long* __restrict__ H, int* __restrict__ unit_start, int* __restrict__ unit_tile,
                   const long long* __restrict__ n_dev, const double* __restrict__ plan, int chunk,
                   unsigned int* __restrict__ unit_counter, const double* __restrict__ gate) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int r = (int)cluster.block_rank();
    obe_grid_dep_launch();
    obe_grid_dep_wait();
    if (gate && *gate == 0.0) return;                      // (every CTA of the cluster reads the same flag)
    if (r == 0 && threadIdx.x == 0 && unit_counter) *unit_counter = 0u;
    __shared__ long long sml[OBE_SCANW * (OBE_SCAN_THREADS / 32 + 1)];
    __shared__ int smi[OBE_SCANW * (OBE_SCAN_THREADS / 32 + 1)];
    __shared__ long long xmax[OBE_PLAN_CLUSTER];     // segment maxima of H, every CTA holds all eight
    __shared__ int xsum[OBE_PLAN_CLUSTER];           // segment unit counts
    __shared__ long long s_next;                     // raw H of the first tile after this segment
    const int t = threadIdx.x;
    if (n_dev) n_tiles = (*n_dev + OBE_TILE - 1) / OBE_TILE;
    if (plan) {
        n_total = (long long)plan[OBE_PL_NTOTAL]; u0 = plan[OBE_PL_U0];
        cdf_offset = plan[OBE_PL_OFFSET]; cdf_total = plan[OBE_PL_TOTAL];
        slot_begin = (long long)plan[OBE_PL_SLOT0]; slot_end = (long long)plan[OBE_PL_SLOT1];
    }
    const double inv_total = 1.0 / (cdf_total > 0.0 ? cdf_total : prefix[n_tiles]);
    const double nd = (double)n_total, inv_n = 1.0 / nd, tol = 2e-15 * nd;
    const long long seg = (n_tiles + OBE_PLAN_CLUSTER - 1) / OBE_PLAN_CLUSTER;
    const long long k_lo = min((long long)r * seg, n_tiles), k_hi = min(k_lo + seg, n_tiles);   // tiles [k_lo, k_hi)
    auto raw_h = [&](long long k, double pk) -> long long {
        const long long h = (k == 0) ? slot_begin
                                     : (k >= n_tiles ? slot_end
                                                     : (long long)comb_count_d(obe_mul(obe_add(cdf_offset, pk), inv_total),
                                                                               u0, inv_n, nd, tol));
        return min(max(h, slot_begin), slot_end);
    };
    constexpr int NWP = OBE_SCAN_THREADS / 32;
    constexpr long long ROUND = (long long)OBE_SCANW * OBE_SCAN_THREADS;
    // ---- raw H of the segment + local running max (first sweep; the carry starts at the identity)
    if (t == 0) {
        s_next = raw_h(k_hi, k_hi < n_tiles ? prefix[k_hi] : 0.0);
        if (k_hi == n_tiles) H[n_tiles] = slot_end;
    }
    long long hcarry = -1;
    for (long long base = k_lo; base < k_hi; base += ROUND) {
        double pk[OBE_SCANW];
        long long h[OBE_SCANW], ex[OBE_SCANW], tot[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            pk[e] = (k < k_hi) ? prefix[k] : 0.0;
        }
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            h[e] = (k < k_hi) ? raw_h(k, pk[e]) : -1;
        }
        obe_block_excl_scanw<long long, NWP>(h, ex, tot, sml, ObeOpMax(), -1ll, 0);
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k < k_hi) H[k] = max(max(hcarry, ex[e]), h[e]);
            hcarry = max(hcarry, tot[e]);
        }
        __syncthreads();
    }
    if (t < OBE_PLAN_CLUSTER) *cluster.map_shared_rank(&xmax[r], t) = hcarry;
    cluster.sync();
    long long floor_h = slot_begin;                  // running max of everything before this segment
    for (int j = 0; j < r; ++j) floor_h = max(floor_h, xmax[j]);
    const long long next_h = max(max(floor_h, hcarry), s_next);         // final H[k_hi]
    // ---- fold the floor in, count the units of every tile, local exclusive scan (second sweep)
    int icarry = 0;
    for (long long base = k_lo; base < k_hi; base += ROUND) {
        long long hf[OBE_SCANW];
        int units[OBE_SCANW], ex[OBE_SCANW], tot[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            hf[e] = (k < k_hi) ? max(H[k], floor_h) : 0;
        }
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            units[e] = 0;
            if (k < k_hi) {
                // H[k+1] of this segment still lacks the floor; the last tile's neighbour is next_h
                const long long h1 = (k + 1 < k_hi) ? max(H[k + 1], floor_h) : next_h;
                units[e] = (int)((max(h1 - hf[e], 0ll) + chunk - 1) / chunk);
            }
        }
        __syncthreads();                             // all reads of the un-floored H precede the writes below
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k < k_hi) H[k] = hf[e];
        }
        obe_block_excl_scanw<int, NWP>(units, ex, tot, smi, ObeOpSum(), 0, 0);
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k < k_hi) unit_start[k] = icarry + ex[e];           // segment-local; the offset follows
            icarry += tot[e];
        }
        __syncthreads();
    }
    if (t < OBE_PLAN_CLUSTER) *cluster.map_shared_rank(&xsum[r], t) = icarry;
    cluster.sync();
    int off = 0, total = 0;
    for (int j = 0; j < OBE_PLAN_CLUSTER; ++j) { if (j < r) off += xsum[j]; total += xsum[j]; }
    // ---- third sweep: global unit numbers, unit -> tile map
    for (long long k = k_lo + t; k < k_hi; k += OBE_SCAN_THREADS) {
        const int first = unit_start[k] + off;
        const long long h1 = (k + 1 < k_hi) ? H[k + 1] : next_h;
        const int units = (int)((max(h1 - H[k], 0ll) + chunk - 1) / chunk);
        unit_start[k] = first;
        if (unit_tile)
            for (int u = 0; u < units; ++u) unit_tile[first + u] = (int)k;
    }
    if (r == 0 && t == 0) unit_start[n_tiles] = total;
}

// One work unit = (input tile k, chunk of <= 2048 consecutive output slots owned by that tile).
//  1. canonical CDF of the tile (blocked scan) -> end slot hi_j of every particle (comb count),
//     made monotone by a running max and clamped to the tile's slot range [H_k, H_k+1)
//  2. every particle that owns at least one slot of the chunk marks the first of them with its
//     index; a max-scan over the chunk's slots turns the marks into the ancestor of every slot
//  3. slots are walked in coalesced order: gather the ancestor (L1-resident tile), jitter, store
// Everything one work unit needs, in registers.  Shared by the single-cloud / sharded kernel and the
// batched kernel (where it is rebuilt per instance).
struct SysCtx {
    const double* w_in;        // weights of this cloud / shard / instance (tile k starts at k * OBE_TILE)
    const double* prefix;      // its tile prefix row
    long long n_in;            // its live particle count
    double inv_total, cdf_offset;
    bool last_shard;
    double u0, inv_n, nd, tol, wv;
    const double* pin; long long ld_in, in_base;      // ancestor j of the cloud is pin[row*ld_in + in_base + j]
    double* pout; long long ld_out, out_base;         // output slot o goes to pout[row*ld_out + out_base + o]
    double* w_out;
    long long slot_begin, cap_out;
    unsigned long long seed; unsigned int epoch;
    int jitter, scale;
    double a_param;
    long long* idx_out; double* z_out;
    unsigned int mask_le, mask_lt;                     // batched: constraint applied to the offspring
    double wuni_in;                                    // > 0: the input weights are implicit (uniform)
};

// One work unit = (input tile k, chunk of <= 2048 consecutive output slots owned by that tile).
//  1. canonical CDF of the tile (blocked scan) -> end slot hi_j of every particle (comb count),
//     made monotone by a running max and clamped to the tile's slot range [H_k, H_k+1)
//  2. every particle that owns at least one slot of the chunk marks the first of them with its
//     index; a max-scan over the chunk's slots turns the marks into the ancestor of every slot
//  3. slots are walked in coalesced order: gather the ancestor (L1-resident tile), jitter, store
// Staging (D <= OBE_STAGE_MAX_D): while phases 1-2 run, the TMA engine copies the tile's D particle
// rows into shared memory (`xs`, one mbarrier), so the ancestor gathers of phase 3 are LDS instead of
// dependent global loads -- the top stall of the unstaged kernel.
#define OBE_STAGE_MAX_D 4
#ifndef OBE_RES_UNROLL
#define OBE_RES_UNROLL 1
#endif
// Phases 1-2 of a work unit: on return anc_s[q] is the in-tile index of the ancestor of the chunk's
// slot q (before the clamp to the tile's last live particle), visible to the whole block.
__device__ __forceinline__ void sys_unit_ancestors(const SysCtx& c, long long k, long long Hk, long long Hk1,
                                                   int rel_begin, double* sm, int* smx, unsigned short* anc_s) {
    // Barrier budget per unit: 5.  Every small shared array (sm, smx) and anc_s is written only after a barrier
    // that follows its previous readers, INCLUDING the readers of the previous unit (the caller's loop has no
    // barrier of its own): sm after (e) of the previous unit, the anc_s clear after (a), smx after (a)/(c).
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int span = (int)(Hk1 - Hk);
    const int n_chunk = min(rel_begin + OBE_OUT_CHUNK, span) - rel_begin;
    // ---- 1. end slot of every particle of the tile, in chunk coordinates [0, n_chunk]
    double cn[OBE_EPT];
    tile_cdf_blocked<false>(c.w_in, c.prefix, k, c.n_in, c.inv_total, cn, sm, c.cdf_offset, c.last_shard,
                            c.wuni_in);                                                        // barrier (a)
    // clear the marks of the slots in use (OBE_SPT per thread, 16-byte stores); the previous unit's readers of
    // anc_s are behind barrier (a)
    const bool my_slots_live = tid * OBE_SPT < n_chunk;
    if (my_slots_live) {
#pragma unroll
        for (int v = 0; v < OBE_SPT / 8; ++v)
            *reinterpret_cast<uint4*>(&anc_s[tid * OBE_SPT + 8 * v]) = make_uint4(0u, 0u, 0u, 0u);
    }
    const long long base = k * OBE_TILE;
    const int lastrel = (int)(min(c.n_in, base + OBE_TILE) - 1 - base);
    const double chunk0 = (double)(Hk + rel_begin);          // exact: < 2^53
    int r[OBE_EPT];
    int run = 0;
#pragma unroll
    for (int e = 0; e < OBE_EPT; ++e) {
        int h = n_chunk;                                     // the tile's last live particle owns the tail
        if (tid * OBE_EPT + e < lastrel) {
            const double hd = comb_count_d(cn[e], c.u0, c.inv_n, c.nd, c.tol) - chunk0;   // |hd| < 2^32
            h = min(max(__double2int_rz(hd), 0), n_chunk);   // the conversion saturates
        }
        run = max(run, h);
        r[e] = run;
    }
    int x = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = max(x, y);
    }
    int ex = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) ex = 0;
    if (lane == 31) smx[warp] = x;
    __syncthreads();                                         // barrier (b): smx; the cleared marks
    ex = max(ex, obe_prev_warps_max8(smx, warp, lane));
    // ---- 2. a particle that owns slots of the chunk marks the first of them
    int prev = ex;                         // end slot of the previous particle
#pragma unroll
    for (int e = 0; e < OBE_EPT; ++e) {
        const int end = max(r[e], ex);
        if (end > prev) anc_s[prev] = (unsigned short)(tid * OBE_EPT + e);
        prev = end;
    }
    __syncthreads();                                         // barrier (c): the marks
    // max-scan of the marks over the chunk's slots (blocked: OBE_SPT consecutive slots per thread); threads
    // whose slots lie beyond the chunk only take part in the shuffles
    {
        int m[OBE_SPT];
        int runm = 0;
        if (my_slots_live) {
#pragma unroll
            for (int v = 0; v < OBE_SPT / 8; ++v) {
                const uint4 raw = *reinterpret_cast<const uint4*>(&anc_s[tid * OBE_SPT + 8 * v]);
                const unsigned int wds[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int val = (int)((wds[e >> 1] >> ((e & 1) * 16)) & 0xffffu);
                    runm = max(runm, val);
                    m[8 * v + e] = runm;
                }
            }
        }
        int xm = runm;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, xm, o);
            if (lane >= o) xm = max(xm, y);
        }
        int exm = __shfl_up_sync(0xffffffffu, xm, 1);
        if (lane == 0) exm = 0;
        if (lane == 31) smx[warp] = xm;                      // (the readers of smx are behind barrier (c))
        __syncthreads();                                     // barrier (d)
        exm = max(exm, obe_prev_warps_max8(smx, warp, lane));
        if (my_slots_live) {
#pragma unroll
            for (int v = 0; v < OBE_SPT / 8; ++v) {
                unsigned int packed[4];
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                    const unsigned int a0 = (unsigned int)max(m[8 * v + e], exm), a1v = (unsigned int)max(m[8 * v + e + 1], exm);
                    packed[e >> 1] = a0 | (a1v << 16);
                }
                *reinterpret_cast<uint4*>(&anc_s[tid * OBE_SPT + 8 * v]) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
            }
        }
    }
    __syncthreads();                                         // barrier (e): the ancestors
}

template <int D, class FT>
__device__ __forceinline__ void sys_unit(const SysCtx& c, long long k, long long Hk, long long Hk1, int rel_begin,
                                         const FT& F, const double* sMean, double* sm, int* smx,
                                         unsigned short* anc_s, double* xs, unsigned long long* bar,
                                         unsigned int& phase, long long& staged_k) {
    const int tid = threadIdx.x;
    const int span = (int)(Hk1 - Hk);
    constexpr bool STAGE = (D <= OBE_STAGE_MAX_D);
    const bool reload = STAGE && (staged_k != k);
    if (reload && tid == 0) {
        const long long base0 = k * OBE_TILE;
        long long cnt = min(c.n_in, base0 + OBE_TILE) - base0;
        cnt += (cnt & 1);                                  // 16-byte granules; the pad element exists (ld is even)
        const unsigned row_bytes = (unsigned)cnt * 8u;
        obe_mbar_expect_tx(bar, row_bytes * (unsigned)D);
#pragma unroll
        for (int j = 0; j < D; ++j)
            obe_bulk_g2s(xs + j * OBE_TILE, c.pin + j * c.ld_in + c.in_base + base0, row_bytes, bar);
    }
    const int rel_end = min(rel_begin + OBE_OUT_CHUNK, span);
    sys_unit_ancestors(c, k, Hk, Hk1, rel_begin, sm, smx, anc_s);
    const long long base = k * OBE_TILE;
    const long long last = min(c.n_in, base + OBE_TILE) - 1;
    // ---- 3. outputs in coalesced order.  Staged: gathers are shared-memory reads.  Unstaged: the
    //         ancestor of the NEXT slot is gathered before the RNG / jitter arithmetic of this one.
    const int n_out = rel_end - rel_begin;
    const int lastrel = (int)(last - base);
    if (reload) {
        obe_mbar_wait(bar, phase);
        phase ^= 1u;
    }
    staged_k = k;
    constexpr int U = OBE_RES_UNROLL;                       // output slots per thread per iteration
    for (int q0 = tid; q0 < n_out; q0 += U * OBE_THREADS) {
        bool act[U];
        long long og[U], o[U];
        int rel[U];
        double xv[U][D], z[U][D];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int q = q0 + u * OBE_THREADS;
            act[u] = q < n_out;
            rel[u] = act[u] ? min((int)anc_s[q], lastrel) : 0;
            og[u] = Hk + rel_begin + q;                        // global slot: comb tooth, RNG counter
            o[u] = og[u] - c.slot_begin;                       // position in this shard's output
            act[u] = act[u] && (o[u] < c.cap_out);             // capacity overflow is flagged in the plan
#pragma unroll
            for (int j = 0; j < D; ++j)
                xv[u][j] = STAGE ? xs[j * OBE_TILE + rel[u]] : __ldg(c.pin + j * c.ld_in + c.in_base + base + rel[u]);
        }
        if (c.jitter) {
#pragma unroll
            for (int u = 0; u < U; ++u) packed_normals_slot<D>(og[u], c.seed, c.epoch, z[u]);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (c.z_out && act[u]) {
#pragma unroll
                    for (int j = 0; j < D; ++j) c.z_out[o[u] * D + j] = z[u][j];
                }
                liu_west<D>(xv[u], z[u], F, sMean, c.a_param, c.scale);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!act[u]) continue;
            double wo = c.wv;
            if (c.mask_le | c.mask_lt) {
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    if (((c.mask_le >> j) & 1u) && xv[u][j] <= 0.0) wo = 0.0;
                    if (((c.mask_lt >> j) & 1u) && xv[u][j] < 0.0) wo = 0.0;
                }
            }
#pragma unroll
            for (int j = 0; j < D; ++j) c.pout[j * c.ld_out + c.out_base + o[u]] = xv[u][j];
            if (c.w_out) c.w_out[c.out_base + o[u]] = wo;
            if (c.idx_out) c.idx_out[o[u]] = base + rel[u];
        }
    }
    __syncthreads();
}

// The per-launch context of the single-cloud / sharded kernels, from by-value arguments or the device plan.
__device__ __forceinline__ SysCtx sys_ctx_of(const ObeResampleArgs& a, long long& n_tiles_in) {
    const long long n_in = a.n_dev_in ? *a.n_dev_in : a.n;
    n_tiles_in = a.n_dev_in ? (n_in + OBE_TILE - 1) / OBE_TILE : a.n_tiles;
    const bool sharded = a.plan ? true : (a.sharded != 0);
    const double cdf_total = a.plan ? a.plan[OBE_PL_TOTAL] : a.cdf_total;
    const long long n_total = a.plan ? (long long)a.plan[OBE_PL_NTOTAL] : a.n_total;
    SysCtx c;
    c.w_in = a.w_in; c.prefix = a.prefix; c.n_in = n_in;
    c.inv_total = 1.0 / (sharded ? cdf_total : a.prefix[n_tiles_in]);
    c.cdf_offset = a.plan ? a.plan[OBE_PL_OFFSET] : (sharded ? a.cdf_offset : 0.0);
    c.last_shard = a.plan ? (a.plan[OBE_PL_LAST] != 0.0) : (sharded ? (a.last_shard != 0) : true);
    c.u0 = a.plan ? a.plan[OBE_PL_U0] : a.u0;
    c.nd = (double)n_total; c.inv_n = 1.0 / c.nd; c.wv = 1.0 / c.nd; c.tol = 2e-15 * c.nd;
    c.pin = a.pin; c.ld_in = a.ld_in; c.in_base = 0;
    c.pout = a.pout; c.ld_out = a.ld_out; c.out_base = 0; c.w_out = a.w_out;
    c.slot_begin = a.plan ? (long long)a.plan[OBE_PL_SLOT0] : a.slot_begin;
    c.cap_out = a.plan ? a.cap_out : (1ll << 62);
    c.seed = a.seed; c.epoch = a.epoch; c.jitter = a.jitter; c.scale = a.scale; c.a_param = a.a_param;
    c.idx_out = a.idx_out; c.z_out = a.z_out; c.mask_le = 0u; c.mask_lt = 0u;
    c.wuni_in = a.stats[OBE_ST_UNIFORM];
    if (a.implicit_out) c.w_out = nullptr;               // offspring weights stay implicit (1/n_total)
    return c;
}

// ---- two-kernel systematic resample ----------------------------------------------------------
// A fused kernel (sys_unit, still used by the batched engine whose instances are a few tiles each)
// spends ~3/4 of its instructions in phase 3 (gather, Philox, Box-Muller, Liu-West, store) but runs
// it at the occupancy phases 1-2 dictate (barriers, shared-memory marks): 1.62 ms at 1e8 x 3.
// Splitting at the ancestor array costs 8 bytes per particle of extra traffic (4 written, 4 read) and
// buys a barrier-free elementwise second kernel at full occupancy with vector stores (0.45 + 0.87 ms):
//   k_sys_ancestors : work units as above, phases 1-2, ancestors (uint32 input index) to global memory
//   k_sys_move<D>   : V consecutive output slots per thread: ancestors -> gather -> jitter -> store
#ifndef OBE_ANC_BLOCKS_PER_SM
#define OBE_ANC_BLOCKS_PER_SM 5
#endif
__global__ void __launch_bounds__(OBE_THREADS, OBE_ANC_BLOCKS_PER_SM) k_sys_ancestors(const ObeResampleArgs a) {
    __shared__ double sm[8];
    __shared__ int smx[OBE_THREADS / 32];
    __shared__ __align__(16) unsigned short anc_s[OBE_OUT_CHUNK];
    __shared__ SysCtx cs;                  // in shared memory so that nothing of it is recomputed per unit
    __shared__ int s_units;
    if (threadIdx.x == 0) {
        long long n_tiles_in;
        cs = sys_ctx_of(a, n_tiles_in);
        s_units = a.unit_start[n_tiles_in];
    }
    __syncthreads();
    const SysCtx& c = cs;
    if (blockIdx.x == gridDim.x - 1) {
        // One extra block, off the critical path: the offspring cloud has uniform weights 1/n_total, so
        // its tile sums, CDF prefix and stats are known before a single particle is written (saves the
        // fill + scan launches after the resample).
        __shared__ double smd[OBE_SCANW * (OBE_THREADS / 32 + 1)];
        const long long slot_end = a.plan ? (long long)a.plan[OBE_PL_SLOT1] : a.slot_end;
        const long long n_out = slot_end - c.slot_begin;
        const long long tiles_out = (n_out + OBE_TILE - 1) / OBE_TILE;
        const long long n_total = (long long)c.nd;
        for (long long k = threadIdx.x; k < tiles_out; k += OBE_THREADS) {
            const long long cnt = min((long long)OBE_TILE, n_out - k * OBE_TILE);
            a.out_tile_sums[k] = (double)cnt * c.wv;
        }
        __threadfence_block();
        __syncthreads();
        obe_tile_scan_block<OBE_THREADS / 32>(a.out_tile_sums, tiles_out, a.out_prefix, a.out_stats, 0, n_total, n_out,
                                              a.implicit_out, smd, 0);
        return;
    }
    const int n_units = s_units;
    const int n_work_blocks = (int)gridDim.x - 1;
    const int per_block = (n_units + n_work_blocks - 1) / n_work_blocks;
    const int unit_lo = min((int)blockIdx.x * per_block, n_units);
    const int unit_hi = min(unit_lo + per_block, n_units);
    int k32 = 0;
    if (!a.unit_tile && unit_lo < unit_hi) {   // no unit -> tile map: binary search, then a forward walk
        int lo = 0, hi = (int)((c.n_in + OBE_TILE - 1) / OBE_TILE);
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (a.unit_start[mid] <= unit_lo) lo = mid + 1; else hi = mid;
        }
        k32 = lo - 1;
    }
    for (int unit = unit_lo; unit < unit_hi; ++unit) {
        if (a.unit_tile) k32 = a.unit_tile[unit];
        else while (a.unit_start[k32 + 1] <= unit) ++k32;
        const int k = k32;
        const long long Hk = a.plan_h[k], Hk1 = a.plan_h[k + 1];
        const int rel_begin = (unit - a.unit_start[k]) * OBE_OUT_CHUNK;
        sys_unit_ancestors(c, k, Hk, Hk1, rel_begin, sm, smx, anc_s);
        const unsigned int base = (unsigned int)k * OBE_TILE;
        const long long o0 = Hk + rel_begin - c.slot_begin;
        const long long room = c.cap_out - o0;                 // capacity overflow is flagged in the plan
        int n_out = min(rel_begin + OBE_OUT_CHUNK, (int)(Hk1 - Hk)) - rel_begin;
        if (room < (long long)n_out) n_out = room > 0 ? (int)room : 0;
        unsigned int* __restrict__ dst = a.anc + o0;
        // (marks are indices of live particles, so no clamp; the next unit touches anc_s only behind its first
        // barrier, so no barrier here either)
        for (int q = threadIdx.x; q < n_out; q += OBE_THREADS) dst[q] = base + (unsigned int)anc_s[q];
    }
}

#define OBE_MOVE_V 4
#define OBE_MOVE_BLOCKS(d) ((d) <= 3 ? 4 : ((d) == 4 ? 3 : 2))   /* resident CTAs per SM the registers allow */
template <int D>
__global__ void __launch_bounds__(OBE_THREADS, OBE_MOVE_BLOCKS(D)) k_sys_move(const ObeResampleArgs a) {
    constexpr int V = OBE_MOVE_V;
    __shared__ double sF[D * D];
    __shared__ double sMean[D];
    setup_factor<D>(a, sF, sMean);
    const long long slot_begin = a.plan ? (long long)a.plan[OBE_PL_SLOT0] : a.slot_begin;
    long long n_out = a.plan ? (long long)a.plan[OBE_PL_SLOT1] - slot_begin : a.slot_end - a.slot_begin;
    if (a.plan && n_out > a.cap_out) n_out = a.cap_out;
    // groups of 4 consecutive GLOBAL slots starting at a multiple of 4 (the packed normal stream); the first group
    // of a shard whose slot_begin is not a multiple of 4 is partial
    const int sh = (int)(slot_begin & 3);
    const long long n_groups = (n_out + sh + V - 1) / V;
    for (long long g = (long long)blockIdx.x * OBE_THREADS + threadIdx.x; g < n_groups;
         g += (long long)gridDim.x * OBE_THREADS) {
        const long long o0 = g * V - sh;                         // position of the group in this shard's output
        const bool full = o0 >= 0 && o0 + V <= n_out;
        unsigned int anc[V];
        if (full && sh == 0) {
            const uint4 t = *reinterpret_cast<const uint4*>(a.anc + o0);
            anc[0] = t.x; anc[1] = t.y; anc[2] = t.z; anc[3] = t.w;
        } else {
            bool any = false;
            long long ofirst = 0;
#pragma unroll
            for (int u = V - 1; u >= 0; --u)
                if (o0 + u >= 0 && o0 + u < n_out) { any = true; ofirst = o0 + u; }
            if (!any) continue;
#pragma unroll
            for (int u = 0; u < V; ++u) anc[u] = (o0 + u >= 0 && o0 + u < n_out) ? a.anc[o0 + u] : a.anc[ofirst];
        }
        double xv[V][D];
        bool ok[V];
#pragma unroll
        for (int u = 0; u < V; ++u) {
            ok[u] = o0 + u >= 0 && o0 + u < n_out;
#pragma unroll
            for (int j = 0; j < D; ++j) xv[u][j] = __ldg(a.pin + j * a.ld_in + anc[u]);
        }
        if (a.jitter)
            jitter_group4<D>(xv, slot_begin + o0, a.seed, a.epoch, sF, sMean, a.a_param, a.scale, a.z_out, o0, ok);
        if (full && (sh & 1) == 0) {
#pragma unroll
            for (int j = 0; j < D; ++j) {
#pragma unroll
                for (int u = 0; u < V; u += 2)
                    *reinterpret_cast<double2*>(a.pout + j * a.ld_out + o0 + u) = make_double2(xv[u][j], xv[u + 1][j]);
            }
        } else {
#pragma unroll
            for (int u = 0; u < V; ++u) {
                if (o0 + u >= 0 && o0 + u < n_out) {
#pragma unroll
                    for (int j = 0; j < D; ++j) a.pout[j * a.ld_out + o0 + u] = xv[u][j];
                }
            }
        }
        if (a.idx_out) {
#pragma unroll
            for (int u = 0; u < V; ++u)
                if (o0 + u >= 0 && o0 + u < n_out) a.idx_out[o0 + u] = (long long)anc[u];
        }
    }
}

// ---- one-kernel systematic resample, warp-autonomous -------------------------------------------
// The two-kernel path above pays for the ancestor array twice (4 B written + 4 B read per particle) and its
// ancestors kernel is barrier/latency-bound (5 block barriers per unit, 87 instructions per particle, 0.43 of
// HBM).  Here ONE WARP owns a work unit (input tile k, <= OBE_OUT_CHUNK output slots) from the weights to the
// stores, so nothing in the unit needs a block barrier and the ancestors never leave the SM:
//   phase A  the warp walks the tile's eight canonical 256-particle segments in order (lane t owns particles
//            [8t, 8t+8) of the segment: the same blocked layout, Kogge-Stone lane scan and SEQUENTIAL carry over
//            the segments that tile_scan_blocked uses, so every CDF value has the canonical bits; the next
//            segment's weights are in flight while this one is scanned), turns the CDF values into end slots
//            (comb count, running max carried across segments in a register), and every particle that owns
//            slots of the chunk marks the first of them in the warp's private array of ushort marks;
//   phase B  the chunk's slots are emitted in groups of 128: 4 consecutive slots per lane, the marks are
//            max-scanned in registers (carry across groups in a register), ancestors gathered through L1
//            (monotone ancestors: the gathers walk the tile almost sequentially), Philox / Box-Muller /
//            Liu-West, 16-byte stores of 32 contiguous bytes per lane and row.  Groups are aligned to 4 slots of
//            the shard's OUTPUT (the chunk is shifted by A = o_base & 3), so every full group stores whole 32-byte
//            sectors; on a shard whose first global slot is not a multiple of 4 the groups then straddle the 4-slot
//            blocks of the packed normal stream and take one more Philox call (jitter_group4_w).
// Same arithmetic as sys_unit_ancestors + k_sys_move, so the ancestors and the offspring are bit-identical to
// the two-kernel path's.  Algorithmic traffic 8N(2d+1) instead of 8N(2d+2).
#define OBE_WR_GROUP 128
#define OBE_WR_MARKS (OBE_WR_CHUNK + OBE_WR_GROUP)       /* shifted chunk coordinates: A + n_chunk <= 3203 */
#define OBE_WR_SMEM ((OBE_THREADS / 32) * OBE_WR_MARKS * 2)
#ifndef OBE_WR_MINB
#define OBE_WR_MINB 3     /* measured: 3 CTAs x 80 registers beat 4 x 64 (spills) -- 1.08 vs 1.38 ms at 1e8 x 3 */
#endif
#ifndef OBE_WR_BLOCKS
/* resident CTAs per SM: 52 KB of marks each (4 would fit in the 227 KB of an SM); the registers decide */
#define OBE_WR_BLOCKS(d) ((d) <= 3 ? OBE_WR_MINB : ((d) == 4 ? 3 : 2))
#endif
#ifndef OBE_WR_SPLIT
#define OBE_WR_SPLIT 1      /* 1: the mark scan is its own pass (B1), the emission loop (B2) has no shuffles */
#endif
#ifndef OBE_WR_PREFETCH
#define OBE_WR_PREFETCH 1   /* B2 prefetches the next group's ancestor lines into L2 while this group is computed */
#endif

struct WrUnit { long long og_al, o_al, base; int q_emit_end, A, lastrel, rr; };

// ---- the comb arithmetic of one work unit, shared by the streaming kernel and the early-select pick kernel (so the
// ancestor of a slot is the same bits wherever it is computed)
// fast comb count: x2 = c*n - u0 + 1/2 in ONE fma of the un-normalised CDF value with K = n/total, rounded to
// the nearest integer by the 1.5*2^52 trick (the low word of x2 + M IS the integer: no FRND / F2I), which is
// ceil(c*n - u0) unless c*n - u0 lies within `tolw` of an integer.  The estimate carries 4 more roundings
// than comb_count_d's (K, the fused normalisation, the pre-added prefix, the +1/2): <= 1e-15*n in all
// against tolw = 3e-15*n, so outside the window it equals the exact comb count; a thread that sees ANY of
// its 8 particles inside the window (probability ~5e-14*n) redoes all 8 the canonical way.
struct WrComb {
    double p0, K, c_half, tolh, chunk0d;
    int c0a, n_chunk, A, q_end, lastrel;
};
__device__ __forceinline__ WrComb wr_comb_of(const SysCtx& c, double prefix_k, long long chunk0, int A, int n_chunk,
                                             int lastrel) {
    WrComb w;
    w.p0 = obe_add(c.cdf_offset, prefix_k);
    w.K = c.nd * c.inv_total; w.c_half = 0.5 - c.u0; w.tolh = 0.5 - 3e-15 * c.nd;
    w.chunk0d = (double)chunk0;
    w.c0a = (int)(unsigned int)(unsigned long long)(chunk0 - A);   // wraps: differences stay < 2^31
    w.n_chunk = n_chunk; w.A = A; w.q_end = A + n_chunk; w.lastrel = lastrel;
    return w;
}
// Kogge-Stone scan of the lanes' sums of one 256-particle segment: exclusive base of this lane, segment total
__device__ __forceinline__ void wr_segment_scan(double run, int lane, double& ex, double& seg_total) {
    double x = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    ex = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) ex = 0.0;
    seg_total = __shfl_sync(0xffffffffu, x, 31);
}
// end slot (shifted chunk coordinates, NOT yet monotone) of this lane's 8 particles i0 .. i0+7 of the tile
__device__ __forceinline__ void wr_end_slots(const WrComb& w, const SysCtx& c, const double (&incl)[OBE_EPT], double bs,
                                             int i0, int (&h)[OBE_EPT]) {
    const double MAGIC = 6755399441055744.0;
    const double bsp = w.p0 + bs;
    bool near = false;
#pragma unroll
    for (int e = 0; e < OBE_EPT; ++e) {
        const double x2 = fma(bsp + incl[e], w.K, w.c_half);
        const double tt = x2 + MAGIC;
        const double dd = x2 - (tt - MAGIC);
        near |= !(fabs(dd) <= w.tolh);
        h[e] = __double2loint(tt) - w.c0a;
    }
    if (near) {                                  // rare: the canonical CDF value and the exact comb count
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e) {
            const double cn = obe_mul(obe_add(w.p0, bs + incl[e]), c.inv_total);
            const double hd = comb_count_d(cn, c.u0, c.inv_n, c.nd, c.tol) - w.chunk0d;   // |hd| < 2^32
            h[e] = min(max(__double2int_rz(hd), 0), w.n_chunk) + w.A;             // the conversion saturates
        }
    }
    if (i0 + OBE_EPT > w.lastrel) {                // the tile's last live particle owns the tail
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e)
            if (i0 + e >= w.lastrel) h[e] = w.q_end;
    }
}

__device__ __forceinline__ void wr_load_segment(const double* __restrict__ wt, int i0, int cnt_tile, double wuni,
                                                double (&v)[OBE_EPT]) {
    if (wuni > 0.0) {
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e) v[e] = (i0 + e < cnt_tile) ? wuni : 0.0;
    } else if (i0 + OBE_EPT <= cnt_tile) {
#pragma unroll
        for (int e = 0; e < OBE_EPT; e += 2) {
            const double2 x2 = *reinterpret_cast<const double2*>(wt + i0 + e);
            v[e] = x2.x; v[e + 1] = x2.y;
        }
    } else {
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e) v[e] = (i0 + e < cnt_tile) ? wt[i0 + e] : 0.0;
    }
}

template <int D>
__global__ void __launch_bounds__(OBE_THREADS, OBE_WR_BLOCKS(D)) k_sys_resample_warp(const ObeResampleArgs a) {
    constexpr int NWARP = OBE_THREADS / 32;
    extern __shared__ __align__(16) unsigned short wr_marks[];     // [NWARP][OBE_WR_MARKS]
    __shared__ double sF[D * D];
    __shared__ double sMean[D];
    __shared__ SysCtx cs;
    __shared__ WrUnit wu[NWARP];
    __shared__ int s_units;
    __shared__ long long s_tiles_in;
    for (int q = threadIdx.x; q < NWARP * OBE_WR_MARKS / 2; q += OBE_THREADS)
        reinterpret_cast<unsigned int*>(wr_marks)[q] = 0u;
    obe_grid_dep_wait();                                 // (programmatic dependent launch: the plan kernel is done)
    if (a.gate && *a.gate == 0.0) return;                // device-side resample test: it did not fire
    if (threadIdx.x == 0) {
        long long n_tiles_in;
        cs = sys_ctx_of(a, n_tiles_in);
        s_units = a.unit_start[n_tiles_in];
        s_tiles_in = n_tiles_in;
    }
    setup_factor<D>(a, sF, sMean);                       // ends with a block barrier
    const SysCtx& c = cs;
    if (blockIdx.x == 0) {
        // bookkeeping block: tile sums, CDF prefix and stats of the offspring cloud.  It is block 0 of a grid that
        // fits the machine in ONE wave, so it is resident from the start and its single-CTA scan (24 rounds at 1e8
        // particles) hides behind the workers; as the LAST block of a grid one larger than the wave it could only
        // start when a worker retired, i.e. it ran as a serial tail after the whole resample.
        __shared__ double smd[OBE_SCANW * (OBE_THREADS / 32 + 1)];
        const long long slot_end = a.plan ? (long long)a.plan[OBE_PL_SLOT1] : a.slot_end;
        long long n_out = slot_end - c.slot_begin;
        if (n_out > c.cap_out) n_out = c.cap_out;
        const long long tiles_out = (n_out + OBE_TILE - 1) / OBE_TILE;
        const long long n_total = (long long)c.nd;
        for (long long k = threadIdx.x; k < tiles_out; k += OBE_THREADS) {
            const long long cnt = min((long long)OBE_TILE, n_out - k * OBE_TILE);
            a.out_tile_sums[k] = (double)cnt * c.wv;
        }
        __threadfence_block();
        __syncthreads();
        obe_tile_scan_block<OBE_THREADS / 32>(a.out_tile_sums, tiles_out, a.out_prefix, a.out_stats, 0, n_total, n_out,
                                              a.implicit_out, smd, 0);
        return;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned short* marks = wr_marks + warp * OBE_WR_MARKS;
    const int n_units = s_units;
    const int n_warps = ((int)gridDim.x - 1) * NWARP;
    // Units are handed out DYNAMICALLY (one atomic per unit, lane 0): the selection kernels of an early select share
    // the SMs with this kernel for its first ~30 us, so some CTAs start late, and with a static stride (unit_counter
    // == nullptr: warp w walks units w, w + n_warps, ...) the whole launch waited for them.
    const bool dynamic = a.unit_counter != nullptr;
    auto next_unit = [&](int prev) -> int {
        if (!dynamic) return prev + n_warps;
        int v = 0;
        if (lane == 0) v = (int)atomicAdd(a.unit_counter, 1u);
        return __shfl_sync(0xffffffffu, v, 0);
    };
#pragma unroll 1
    for (int unit = dynamic ? next_unit(0) : ((int)blockIdx.x - 1) * NWARP + warp; unit < n_units; unit = next_unit(unit)) {
        int k;
        if (a.unit_tile) {
            k = a.unit_tile[unit];
        } else {                                          // no unit -> tile map: last k with unit_start[k] <= unit
            int lo = 0, hi = (int)s_tiles_in;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (a.unit_start[mid] <= unit) lo = mid + 1; else hi = mid;
            }
            k = lo - 1;
        }
        const long long Hk = a.plan_h[k], Hk1 = a.plan_h[k + 1];
        const int rel_begin = (unit - a.unit_start[k]) * a.chunk;
        const int n_chunk = min(rel_begin + a.chunk, (int)(Hk1 - Hk)) - rel_begin;
        const long long chunk0 = Hk + rel_begin;                      // global slot of the chunk's first output
        const long long o_base = chunk0 - c.slot_begin;               // its position in this shard's output
        const int A = (int)(o_base & 3);                              // shifted chunk coordinate q' = q + A: groups of
                                                                      // 4 slots start at multiples of 4 OUTPUT positions
        const int q_end = A + n_chunk;
        const long long base = (long long)k * OBE_TILE;
        const int cnt_tile = (int)(min(c.n_in, base + OBE_TILE) - base);
        const int lastrel = cnt_tile - 1;
        // ---------------------------------------------------------------- phase A: marks
        {
            const double wuni = c.wuni_in;
            const double* __restrict__ wt = c.w_in + base;
            // the whole tile's weights (16 KB) are requested into L2 at once: the segment walk below keeps only one
            // 2 KB segment in flight, so without this every segment paid its own HBM latency
            if (wuni <= 0.0) {
#pragma unroll 1
                for (int i = lane * 16; i < cnt_tile; i += 32 * 16)      // one 128-byte line per lane and step
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(wt + i));
            }
            const WrComb cw = wr_comb_of(c, c.prefix[k], chunk0, A, n_chunk, lastrel);
            double wb = 0.0;                  // canonical sum of the totals of the segments before this one
            int carry_end = A;                // end slot of the last particle walked so far
            double vn[OBE_EPT];
            wr_load_segment(wt, lane * OBE_EPT, cnt_tile, wuni, vn);
#pragma unroll 1
            for (int seg = 0; seg < OBE_TILE / 256; ++seg) {
                if (seg * 256 > lastrel || carry_end >= q_end) break;
                const int i0 = seg * 256 + lane * OBE_EPT;
                double incl[OBE_EPT];
                double run = 0.0;
#pragma unroll
                for (int e = 0; e < OBE_EPT; ++e) { run += vn[e]; incl[e] = run; }
                if ((seg + 1) * 256 <= lastrel) wr_load_segment(wt, i0 + 256, cnt_tile, wuni, vn);   // in flight below
                // canonical scan of the segment (tile_scan_blocked with the warp loop made sequential in time)
                double ex, seg_total;
                wr_segment_scan(run, lane, ex, seg_total);
                const double bs = wb + ex;
                // end slot of every particle in shifted chunk coordinates (the running max supplies the lower clamp)
                int h[OBE_EPT];
                wr_end_slots(cw, c, incl, bs, i0, h);
                int runm = A;
#pragma unroll
                for (int e = 0; e < OBE_EPT; ++e) {
                    runm = max(runm, min(h[e], q_end));
                    h[e] = runm;
                }
                int xm = runm;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, xm, o);
                    if (lane >= o) xm = max(xm, y);
                }
                int exm = __shfl_up_sync(0xffffffffu, xm, 1);
                if (lane == 0) exm = A;
                exm = max(exm, carry_end);
                // a particle that owns slots marks the first of them with its in-tile index + 1
                if (runm > exm) {
                    int prev = exm;
#pragma unroll
                    for (int e = 0; e < OBE_EPT; ++e) {
                        const int end = max(h[e], exm);
                        if (end > prev) marks[prev] = (unsigned short)(i0 + e + 1);
                        prev = end;
                    }
                }
                carry_end = max(carry_end, __shfl_sync(0xffffffffu, xm, 31));
                wb = wb + seg_total;
            }
        }
        __syncwarp();
        // ---------------------------------------------------------------- phase B: emission
        // The per-unit scalars live in the warp's slot of `wu` (shared memory) and are re-read where they are used:
        // held in registers across the emission loop they pushed it over the 80-register budget of 3 CTAs per SM and
        // the spilled ones (local memory, long scoreboard) were the top stall of the loop.
        {
            const long long room = c.cap_out - o_base;                // capacity overflow is flagged in the plan
            const int n_emit = room < (long long)n_chunk ? (room > 0 ? (int)room : 0) : n_chunk;
            if (lane == 0) {
                WrUnit& w = wu[warp];
                w.og_al = chunk0 - A;                                 // global slot of q' = 0 (= slot_begin mod 4)
                w.o_al = chunk0 - A - c.slot_begin;                   // its position in this shard's output (multiple of 4)
                w.base = base;
                w.q_emit_end = A + n_emit; w.A = A; w.lastrel = lastrel;
                w.rr = (int)(c.slot_begin & 3);                       // launch-uniform
            }
            __syncwarp();
            const volatile WrUnit& vu = wu[warp];
            const volatile SysCtx& vc = cs;
            // Groups are aligned to the shard's OUTPUT, so every full group stores whole 32-byte sectors whatever
            // the shard's first global slot is; a shard with slot_begin % 4 != 0 draws the normals of its groups from
            // one more Philox call (jitter_group4_w) -- the normals of a slot do not depend on the grouping.
#if OBE_WR_SPLIT
            // B1: marks -> ancestors (index + 1) in place: max-scan over the chunk, the carry in a register
            {
                int last_anc = 0;
#pragma unroll 1
                for (int g0 = 0; g0 < q_end; g0 += OBE_WR_GROUP) {
                    unsigned int* rp = reinterpret_cast<unsigned int*>(marks + g0 + lane * 4);
                    const uint2 raw = *reinterpret_cast<const uint2*>(rp);
                    int m0 = (int)(raw.x & 0xffffu);
                    int m1 = max(m0, (int)(raw.x >> 16));
                    int m2 = max(m1, (int)(raw.y & 0xffffu));
                    int m3 = max(m2, (int)(raw.y >> 16));
                    int xs = m3;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int y = __shfl_up_sync(0xffffffffu, xs, o);
                        if (lane >= o) xs = max(xs, y);
                    }
                    int exs = __shfl_up_sync(0xffffffffu, xs, 1);
                    if (lane == 0) exs = 0;
                    exs = max(exs, last_anc);
                    last_anc = max(last_anc, __shfl_sync(0xffffffffu, xs, 31));
                    m0 = max(m0, exs); m1 = max(m1, exs); m2 = max(m2, exs); m3 = max(m3, exs);
                    *reinterpret_cast<uint2*>(rp) = make_uint2((unsigned int)m0 | ((unsigned int)m1 << 16),
                                                               (unsigned int)m2 | ((unsigned int)m3 << 16));
                }
            }
            // (every lane reads back only the four entries it wrote: no warp barrier needed)
#else
            int last_anc = 0;                 // mark of the owner of the last slot of the previous group
#endif
            // FULL: every slot of the group is a live output of this unit (warp-uniform): no per-slot predicates
            auto emit = [&](auto full_tag, const int emit_pos) {
                constexpr bool FULL = decltype(full_tag)::value;
                const int q0 = emit_pos + lane * 4;
                const double* __restrict__ pin = vc.pin + vu.base;
                const long long ld_in = vc.ld_in;
                unsigned int* rp = reinterpret_cast<unsigned int*>(marks + q0);
                const uint2 raw = *reinterpret_cast<const uint2*>(rp);
                *reinterpret_cast<uint2*>(rp) = make_uint2(0u, 0u);
                int m[4];
#if OBE_WR_SPLIT
                m[0] = (int)(raw.x & 0xffffu); m[1] = (int)(raw.x >> 16);
                m[2] = (int)(raw.y & 0xffffu); m[3] = (int)(raw.y >> 16);
#if OBE_WR_PREFETCH
                if (emit_pos + OBE_WR_GROUP < q_end) {               // the next group's first ancestor of this lane:
                    const int nxt = (int)marks[q0 + OBE_WR_GROUP];   // its lines will be in L2 when the loads come
                    const double* pf = pin + max(nxt - 1, 0);
#pragma unroll
                    for (int j = 0; j < D; ++j) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf + j * ld_in));
                }
#endif
#else
                m[0] = (int)(raw.x & 0xffffu);
                m[1] = max(m[0], (int)(raw.x >> 16));
                m[2] = max(m[1], (int)(raw.y & 0xffffu));
                m[3] = max(m[2], (int)(raw.y >> 16));
                int xs = m[3];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, xs, o);
                    if (lane >= o) xs = max(xs, y);
                }
                int exs = __shfl_up_sync(0xffffffffu, xs, 1);
                if (lane == 0) exs = 0;
                exs = max(exs, last_anc);
                last_anc = max(last_anc, __shfl_sync(0xffffffffu, xs, 31));
#pragma unroll
                for (int u = 0; u < 4; ++u) m[u] = max(m[u], exs);
#endif
                bool ok[4];
                int rel[4];
                double xv[4][D];
                bool any = false, all = true;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int qq = q0 + u;
                    ok[u] = FULL || (qq >= vu.A && qq < vu.q_emit_end);
                    any |= ok[u];
                    all &= ok[u];
                    // (marks are indices of live particles + 1: no clamp to the tile's last live particle needed)
                    rel[u] = FULL ? m[u] - 1 : min(max(m[u] - 1, 0), vu.lastrel);
                }
                if (!FULL && !any) return;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
#pragma unroll
                    for (int j = 0; j < D; ++j) xv[u][j] = __ldg(pin + j * ld_in + rel[u]);
                }
                if (vc.jitter) {
                    switch (vu.rr) {
                        case 0: jitter_group4_w<D, 0>(xv, vu.og_al + q0, vc.seed, vc.epoch, sF, sMean, vc.a_param, vc.scale,
                                                      vc.z_out, vu.o_al + q0, ok); break;
                        case 1: jitter_group4_w<D, 1>(xv, vu.og_al + q0, vc.seed, vc.epoch, sF, sMean, vc.a_param, vc.scale,
                                                      vc.z_out, vu.o_al + q0, ok); break;
                        case 2: jitter_group4_w<D, 2>(xv, vu.og_al + q0, vc.seed, vc.epoch, sF, sMean, vc.a_param, vc.scale,
                                                      vc.z_out, vu.o_al + q0, ok); break;
                        default: jitter_group4_w<D, 3>(xv, vu.og_al + q0, vc.seed, vc.epoch, sF, sMean, vc.a_param, vc.scale,
                                                       vc.z_out, vu.o_al + q0, ok); break;
                    }
                }
                const long long o0 = vu.o_al + q0;
                double* __restrict__ pout = vc.pout;
                double* __restrict__ w_out = vc.w_out;
                const long long ld_out = vc.ld_out;
                if (FULL || all) {
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        double* dst = pout + j * ld_out + o0;
                        *reinterpret_cast<double2*>(dst) = make_double2(xv[0][j], xv[1][j]);
                        *reinterpret_cast<double2*>(dst + 2) = make_double2(xv[2][j], xv[3][j]);
                    }
                    if (w_out) {
                        const double wv = vc.wv;
                        *reinterpret_cast<double2*>(w_out + o0) = make_double2(wv, wv);
                        *reinterpret_cast<double2*>(w_out + o0 + 2) = make_double2(wv, wv);
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (!ok[u]) continue;
#pragma unroll
                        for (int j = 0; j < D; ++j) pout[j * ld_out + o0 + u] = xv[u][j];
                        if (w_out) w_out[o0 + u] = vc.wv;
                    }
                }
                long long* idx_out = vc.idx_out;
                if (idx_out) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (ok[u]) idx_out[o0 + u] = vu.base + rel[u];
                }
            };
#pragma unroll 1
            for (int emit_pos = 0; emit_pos < q_end; emit_pos += OBE_WR_GROUP) {
                if (emit_pos >= vu.A && emit_pos + OBE_WR_GROUP <= vu.q_emit_end) emit(std::true_type{}, emit_pos);
                else emit(std::false_type{}, emit_pos);
            }
        }
        __syncwarp();
    }
}

// ---- early select: the K draws of the design half, straight from the resample plan -----------------------------
// The parameter draws opt_setting / good_setting ask for right after a resample are particles of the OFFSPRING cloud
// (uniform weights): draw q is the offspring in global output slot s_q = min(floor(u_q * n_total), n_total - 1).
// That offspring is a function of the PLAN alone: its ancestor is the first particle of the owning tile whose comb
// end slot exceeds s_q (what the marks + max-scan of the streaming kernel compute for every slot at once), and its
// jitter comes from the slot-indexed Philox stream.  One warp per draw: 32-ary search of H for the tile, the same
// segment walk / comb arithmetic as the streaming kernel (wr_segment_scan, wr_end_slots), stop at the first segment
// that holds the ancestor, gather, jitter_group4 on the aligned group of four slots, store d doubles.  The values are
// bit-identical to what k_sys_resample_warp stores in slot s_q (tests/test_gpu_early_select.py), but they exist
// ~10 us after the plan instead of after the whole resample, so the utility pass can overlap the streaming kernel.
// Sharded: a rank produces the draws whose slots it owns; the others store nothing (peer exchange: the owner writes
// into every rank's buffer and the last CTA raises the flags) or zeros (collective mode: an all-reduce follows).
struct ObePickArgs {
    int k; int ldk; double* out;
    int peer_world, peer_rank;
    unsigned long long peer_epoch;
    unsigned int* peer_counter;
    ObePeers peers;
    double u[OBE_MAX_DRAWS];
};
#define OBE_PICK_WARPS 2
template <int D>
__global__ void __launch_bounds__(OBE_PICK_WARPS * 32) k_sys_pick(const ObeResampleArgs a, const ObePickArgs pk) {
    __shared__ double sF[D * D];
    __shared__ double sMean[D];
    __shared__ SysCtx cs;
    __shared__ long long s_tiles_in;
    obe_grid_dep_launch();                               // the utility kernel may be scheduled; it waits for this grid
    obe_grid_dep_wait();                                 // (programmatic dependent launch: the plan kernel is done)
    if (a.gate && *a.gate == 0.0) return;                // device-side resample test: it did not fire
    if (threadIdx.x == 0) {
        long long n_tiles_in;
        cs = sys_ctx_of(a, n_tiles_in);
        s_tiles_in = n_tiles_in;
    }
    setup_factor<D>(a, sF, sMean);                       // ends with a block barrier
    const SysCtx& c = cs;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = (int)blockIdx.x * OBE_PICK_WARPS + warp;
    if (q < pk.k) {
        const long long n_total = (long long)c.nd;
        const long long slot_end = a.plan ? (long long)a.plan[OBE_PL_SLOT1] : a.slot_end;
        long long s = (long long)(pk.u[q] * c.nd);
        s = s < 0 ? 0 : (s >= n_total ? n_total - 1 : s);
        const bool mine = s >= c.slot_begin && s < slot_end && s - c.slot_begin < c.cap_out;
        if (!mine) {
            if (pk.peer_world == 0 && lane < D) pk.out[(long long)lane * pk.ldk + q] = 0.0;
        } else {
            // last tile k with H[k] <= s (H is monotone): 32 probes per round
            int lo = 0, hi = (int)s_tiles_in;             // the answer lies in [lo, hi)
            while (hi - lo > 1) {
                const int step = (hi - lo + 31) / 32;
                const int probe = lo + (lane + 1) * step;
                const bool le = probe < hi && a.plan_h[probe] <= s;
                const int cnt = __popc(__ballot_sync(0xffffffffu, le));
                lo += cnt * step;
                hi = min(lo + step, hi);
            }
            const int k = lo;
            const long long Hk = a.plan_h[k], Hk1 = a.plan_h[k + 1];
            const int rel_begin = (int)((s - Hk) / a.chunk) * a.chunk;
            const int n_chunk = min(rel_begin + a.chunk, (int)(Hk1 - Hk)) - rel_begin;
            const long long chunk0 = Hk + rel_begin;
            const int A = (int)(chunk0 & 3);
            const int qs = A + (int)(s - chunk0);          // the slot in shifted chunk coordinates, A <= qs < A + n_chunk
            const long long base = (long long)k * OBE_TILE;
            const int cnt_tile = (int)(min(c.n_in, base + OBE_TILE) - base);
            const int lastrel = cnt_tile - 1;
            const WrComb cw = wr_comb_of(c, c.prefix[k], chunk0, A, n_chunk, lastrel);
            const double* __restrict__ wt = c.w_in + base;
            double wb = 0.0;
            int anc = lastrel;
            double vn[OBE_EPT];
            wr_load_segment(wt, lane * OBE_EPT, cnt_tile, c.wuni_in, vn);
#pragma unroll 1
            for (int seg = 0; seg < OBE_TILE / 256; ++seg) {
                if (seg * 256 > lastrel) break;
                const int i0 = seg * 256 + lane * OBE_EPT;
                double incl[OBE_EPT];
                double run = 0.0;
#pragma unroll
                for (int e = 0; e < OBE_EPT; ++e) { run += vn[e]; incl[e] = run; }
                if ((seg + 1) * 256 <= lastrel) wr_load_segment(wt, i0 + 256, cnt_tile, c.wuni_in, vn);
                double ex, seg_total;
                wr_segment_scan(run, lane, ex, seg_total);
                const double bs = wb + ex;
                int h[OBE_EPT];
                wr_end_slots(cw, c, incl, bs, i0, h);
                // the ancestor of slot qs is the first particle (in tile order) whose end slot exceeds it
                int first = 1 << 30;
#pragma unroll
                for (int e = OBE_EPT - 1; e >= 0; --e)
                    if (h[e] > qs) first = i0 + e;
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, m));
                if (first < (1 << 30)) { anc = first; break; }
                wb = wb + seg_total;
            }
            anc = min(anc, lastrel);
            if (lane == 0) {
                const int us = (int)(s & 3);
                double xv[4][D];
                bool ok[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    ok[u] = true;
#pragma unroll
                    for (int j = 0; j < D; ++j) xv[u][j] = __ldg(c.pin + j * c.ld_in + base + anc);
                }
                if (c.jitter)
                    jitter_group4<D>(xv, s - us, c.seed, c.epoch, sF, sMean, c.a_param, c.scale, nullptr, 0, ok);
                double val[D];
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    val[j] = xv[0][j];
#pragma unroll
                    for (int u = 1; u < 4; ++u) val[j] = (us == u) ? xv[u][j] : val[j];
                }
                if (pk.peer_world > 0) {
                    const int parity = (int)(pk.peer_epoch & 1ull);
#pragma unroll
                    for (int j = 0; j < D; ++j)
                        for (int g = 0; g < pk.peer_world; ++g)
                            pk.peers.p[g][OBE_PEER_DRAWS + parity * 1024 + j * pk.ldk + q] = val[j];
                } else {
#pragma unroll
                    for (int j = 0; j < D; ++j) pk.out[(long long)j * pk.ldk + q] = val[j];
                }
            }
        }
    }
    if (pk.peer_world > 0) {
        // every CTA reports in; the last one raises this rank's flag in every rank's buffer (as k_draw does)
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            if (atomicAdd(pk.peer_counter, 1u) == gridDim.x - 1) {
                __threadfence_system();
                const int parity = (int)(pk.peer_epoch & 1ull);
                for (int g = 0; g < pk.peer_world; ++g)
                    obe_flag_store(obe_peer_flags(pk.peers.p[g], 1, parity) + pk.peer_rank, pk.peer_epoch);
                *pk.peer_counter = 0u;
            }
        }
    }
}

// ---- batched systematic resample: one CTA walks the instances of the compacted list -------------
struct ObeBResampleArgs {
    const double* particles[2];
    double* particles_w[2];
    double* weights[2];
    int* cur;                      // (B) flipped for every resampled instance
    const double* prefix;          // (B * (T + 1))
    const double* stats;           // (B * OBE_STATS_LEN)
    unsigned int* epoch;           // (B) resamples so far, the Philox epoch of the next one
    const int* inst_list; const int* n_list;
    long long ld, np, n;
    int tiles;
    unsigned long long seed;       // instance b uses seed + b for its normals
    unsigned long long useed;      // key of the uniform streams
    unsigned int cycle; int u0_index;
    double a_param; int scale;
    unsigned int mask_le, mask_lt;
};

template <int D>
__global__ void __launch_bounds__(OBE_THREADS, (D <= 4 ? 3 : 2)) k_bsys_resample(const ObeBResampleArgs a) {
    __shared__ double sF[D * D];
    __shared__ double sMean[D];
    __shared__ double sm[8];
    __shared__ int smx[OBE_THREADS / 32];
    __shared__ long long Hs[66];
    __shared__ __align__(16) unsigned short anc_s[OBE_OUT_CHUNK];
    __shared__ unsigned long long stage_bar;
    extern __shared__ __align__(128) unsigned char obe_dyn_smem[];
    double* xs = reinterpret_cast<double*>(obe_dyn_smem);
    if (threadIdx.x == 0) { obe_mbar_init(&stage_bar, 1); obe_mbar_fence_init(); }
    unsigned int phase = 0u;
    __syncthreads();
    const int tid = threadIdx.x;
    const int T = a.tiles;
    const int n_list = *a.n_list;
    for (int li = blockIdx.x; li < n_list; li += gridDim.x) {
        const long long b = a.inst_list[li];
        const int cb = a.cur[b];
        const double* pre = a.prefix + b * (T + 1);
        const double* st = a.stats + b * OBE_STATS_LEN;
        SysCtx c;
        c.w_in = a.weights[cb] + b * a.np; c.prefix = pre; c.n_in = a.n;
        c.inv_total = 1.0 / pre[T]; c.cdf_offset = 0.0; c.last_shard = true;
        c.u0 = obe_batch_uniform(a.useed, (unsigned int)b, a.cycle, (unsigned int)a.u0_index);
        c.nd = (double)a.n; c.inv_n = 1.0 / c.nd; c.wv = 1.0 / c.nd; c.tol = 2e-15 * c.nd;
        c.pin = a.particles[cb]; c.ld_in = a.ld; c.in_base = b * a.np;
        c.pout = a.particles_w[1 - cb]; c.ld_out = a.ld; c.out_base = b * a.np; c.w_out = a.weights[1 - cb];
        c.slot_begin = 0; c.cap_out = a.np;
        c.seed = a.seed + (unsigned long long)b; c.epoch = a.epoch[b] + 1u; c.jitter = 1; c.scale = a.scale;
        c.a_param = a.a_param; c.idx_out = nullptr; c.z_out = nullptr; c.mask_le = a.mask_le; c.mask_lt = a.mask_lt;
        c.wuni_in = 0.0;
        if (tid == 0) {
            // slot bounds of the instance's tiles (monotone), Liu-West factor from its own moments
            long long run = 0;
            for (int t = 0; t <= T; ++t) {
                long long h = (t == 0) ? 0 : (t == T ? a.n : (long long)comb_count_d(obe_mul(pre[t], c.inv_total), c.u0,
                                                                                     c.inv_n, c.nd, c.tol));
                run = max(run, min(h, (long long)a.n));
                Hs[t] = run;
            }
            const double stt = st[OBE_ST_SUMT], fact = stt - st[OBE_ST_SUMSQ] / stt;
            const double shrink = 1.0 - a.a_param * a.a_param;
            double cov[D][D], L[D][D];
            int q = 0;
            for (int j = 0; j < D; ++j) {
                sMean[j] = st[OBE_ST_PIVOT + j] + st[OBE_ST_M1 + j] / stt;
                for (int k = j; k < D; ++k) {
                    const double cc = (st[OBE_ST_M2 + q] - st[OBE_ST_M1 + j] * st[OBE_ST_M1 + k] / stt) / fact;
                    cov[j][k] = cov[k][j] = shrink * cc;
                    ++q;
                }
            }
            for (int j = 0; j < D; ++j)
                for (int k = 0; k < D; ++k) L[j][k] = 0.0;
            for (int j = 0; j < D; ++j) {
                double sdiag = cov[j][j];
                for (int k = 0; k < j; ++k) sdiag -= L[j][k] * L[j][k];
                const double dj = sdiag > 0.0 ? sqrt(sdiag) : 0.0;
                L[j][j] = dj;
                for (int i = j + 1; i < D; ++i) {
                    double t2 = cov[i][j];
                    for (int k = 0; k < j; ++k) t2 -= L[i][k] * L[j][k];
                    L[i][j] = dj > 0.0 ? t2 / dj : 0.0;
                }
            }
            for (int k = 0; k < D; ++k)
                for (int j = 0; j < D; ++j) sF[k * D + j] = L[j][k];
        }
        __syncthreads();
        long long staged_k = -1;
        for (int t = 0; t < T; ++t) {
            const long long Hk = Hs[t], Hk1 = Hs[t + 1];
            for (int rel = 0; rel < (int)(Hk1 - Hk); rel += OBE_OUT_CHUNK)
                sys_unit<D>(c, t, Hk, Hk1, rel, sF, sMean, sm, smx, anc_s, xs, &stage_bar, phase, staged_k);
        }
        __syncthreads();
        if (tid == 0) { a.cur[b] = 1 - cb; a.epoch[b] = c.epoch; }
        __syncthreads();
    }
}

// compact the resample flags into a list of instance numbers (order preserved) + its length
__global__ void __launch_bounds__(OBE_SCAN_THREADS) k_bcompact(const int* __restrict__ flag, long long n_inst,
                                                               int* __restrict__ list, int* __restrict__ n_list) {
    __shared__ int smi[34];
    int carry = 0;
    for (long long base = 0; base < n_inst; base += OBE_SCAN_THREADS) {
        const long long b = base + threadIdx.x;
        const int f = (b < n_inst && flag[b]) ? 1 : 0;
        int tot;
        const int ex = block_excl_isum_1024(f, smi, &tot);
        if (f) list[carry + ex] = (int)b;
        carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_list = carry;
}

// ---------------------------------------------------------------------------------------------
// Shard plan: everything a rank must know about the other shards, computed ON THE DEVICE from the
// all-gathered stats blocks so that update -> collective -> resample -> draws needs no host
// round-trip.  One thread: G <= 64 shards, d <= 8 (a few hundred flops).  Restated on the host by
// optbayesexpt_b200/sharded.py (combine_stats, moments_from, shard_slot_bounds), which the tests
// compare it with.
// ---------------------------------------------------------------------------------------------
// A block of OBE_STATS_LEN (64) threads.  Thread t sums column t of the gathered blocks in rank order (the same
// association as the host's combine_stats), the comb counts of the shard boundaries run one per thread on the
// second warp while thread 0 does the Cholesky factor, and only the short sequential pieces (the exclusive scan of
// G totals, the monotone clamp of the G bounds) are left to one thread -- reading shared memory, not global: the
// first version walked everything with a single thread through global read-modify-writes, ~40 us at 8 ranks.
__device__ void shard_plan_block(const double* __restrict__ gathered, int rank, int world, int d, double u0,
                                 long long n_total, double a_param, int lazy, long long cap_out,
                                 double* __restrict__ plan, double* __restrict__ stats_local,
                                 long long* __restrict__ n_out_dev) {
    __shared__ double gs_s[OBE_STATS_LEN];
    __shared__ double tot_s[OBE_MAX_SHARDS], off_s[OBE_MAX_SHARDS + 1];
    __shared__ long long end_s[OBE_MAX_SHARDS];
    const int t = threadIdx.x;
    const int nm2 = d * (d + 1) / 2;
    {
        double acc = 0.0;
        for (int g = 0; g < world; ++g) acc = acc + gathered[(long long)g * OBE_STATS_LEN + t];
        const bool summed = t == OBE_ST_SUMSQ || t == OBE_ST_SUMT || t == OBE_ST_NZERO ||
                            (t >= OBE_ST_M1 && t < OBE_ST_M1 + d) || (t >= OBE_ST_M2 && t < OBE_ST_M2 + nm2) ||
                            (t >= OBE_ST_NOISE && t < OBE_ST_NOISE + OBE_MAX_CH);
        double v = summed ? acc : 0.0;
        if (t >= OBE_ST_PIVOT && t < OBE_ST_PIVOT + d) v = gathered[t];          // rank 0's pivot (common to all)
        gs_s[t] = v;
        for (int g = t; g < world; g += OBE_STATS_LEN) tot_s[g] = gathered[(long long)g * OBE_STATS_LEN + OBE_ST_TOTAL];
    }
    __syncthreads();
    if (t == 0) {
        double acc = 0.0;
        for (int g = 0; g < world; ++g) {                 // the canonical inter-GPU exclusive scan
            off_s[g] = acc;
            acc = acc + tot_s[g];
        }
        off_s[world] = acc;
        gs_s[OBE_ST_TOTAL] = acc;
        gs_s[OBE_ST_INVS] = lazy ? 1.0 / acc : 1.0;
        gs_s[OBE_ST_NEFF] = (acc * acc) / gs_s[OBE_ST_SUMSQ];
    }
    __syncthreads();
    const double total = off_s[world];
    plan[OBE_PL_GSTATS + t] = gs_s[t];
    for (int g = t; g < world; g += OBE_STATS_LEN) {
        plan[OBE_PL_PRE_OFF + g] = off_s[g];
        plan[OBE_PL_PRE_TOT + g] = tot_s[g];
    }
    const double nd = (double)n_total, inv_n = 1.0 / nd, tol = 2e-15 * nd, inv_total = 1.0 / total;
    if (t >= 32) {                                        // raw slot bound between shards g and g+1
        for (int g = t - 32; g + 1 < world; g += 32)
            end_s[g] = (long long)comb_count_d(obe_mul(off_s[g + 1], inv_total), u0, inv_n, nd, tol);
    }
    if (t == 0) {
        stats_local[OBE_ST_INVS] = gs_s[OBE_ST_INVS];     // the GLOBAL normaliser for the next update
        // global mean, Cholesky factor of (1 - a^2) * cov
        const double st = gs_s[OBE_ST_SUMT], fact = st - gs_s[OBE_ST_SUMSQ] / st, shrink = 1.0 - a_param * a_param;
        double cov[OBE_MAX_DIMS][OBE_MAX_DIMS], L[OBE_MAX_DIMS][OBE_MAX_DIMS];
        int q = 0;
        for (int j = 0; j < d; ++j) {
            plan[OBE_PL_MEAN + j] = gs_s[OBE_ST_PIVOT + j] + gs_s[OBE_ST_M1 + j] / st;
            for (int k = j; k < d; ++k) {
                const double c = (gs_s[OBE_ST_M2 + q] - gs_s[OBE_ST_M1 + j] * gs_s[OBE_ST_M1 + k] / st) / fact;
                cov[j][k] = cov[k][j] = shrink * c;
                ++q;
            }
        }
        for (int j = 0; j < d; ++j)
            for (int k = 0; k < d; ++k) L[j][k] = 0.0;
        for (int j = 0; j < d; ++j) {
            double sdiag = cov[j][j];
            for (int k = 0; k < j; ++k) sdiag -= L[j][k] * L[j][k];
            const double dj = sdiag > 0.0 ? sqrt(sdiag) : 0.0;
            L[j][j] = dj;
            for (int i = j + 1; i < d; ++i) {
                double tt = cov[i][j];
                for (int k = 0; k < j; ++k) tt -= L[i][k] * L[j][k];
                L[i][j] = dj > 0.0 ? tt / dj : 0.0;
            }
        }
        for (int k = 0; k < d; ++k)
            for (int j = 0; j < d; ++j) plan[OBE_PL_FACTOR + k * d + j] = L[j][k];
    }
    __syncthreads();
    if (t != 0) return;
    // slot bounds of every shard: H_0 = 0, H_G = n_total, monotone
    long long prev = 0, mine0 = 0, mine1 = n_total;
    double post_acc = 0.0;
    const double wv = 1.0 / nd;
    for (int g = 0; g < world; ++g) {
        long long end = n_total;
        if (g + 1 < world) end = min(max(end_s[g], prev), n_total);
        if (g == rank) { mine0 = prev; mine1 = end; }
        plan[OBE_PL_COUNTS + g] = (double)(end - prev);
        plan[OBE_PL_POST_OFF + g] = post_acc;
        plan[OBE_PL_POST_TOT + g] = (double)(end - prev) * wv;
        post_acc = post_acc + (double)(end - prev) * wv;
        prev = end;
    }
    plan[OBE_PL_POST_TOTAL] = post_acc;
    plan[OBE_PL_OFFSET] = off_s[rank];
    plan[OBE_PL_TOTAL] = total;
    plan[OBE_PL_U0] = u0;
    plan[OBE_PL_NTOTAL] = nd;
    plan[OBE_PL_SLOT0] = (double)mine0;
    plan[OBE_PL_SLOT1] = (double)mine1;
    plan[OBE_PL_LAST] = (rank == world - 1) ? 1.0 : 0.0;
    plan[OBE_PL_RANK] = (double)rank;
    plan[OBE_PL_WORLD] = (double)world;
    long long cnt = mine1 - mine0;
    plan[OBE_PL_OVERFLOW] = (cnt > cap_out) ? 1.0 : 0.0;
    if (cnt > cap_out) cnt = cap_out;
    if (n_out_dev) *n_out_dev = cnt;
}

__global__ void __launch_bounds__(OBE_STATS_LEN) k_shard_plan(const double* __restrict__ gathered, int rank, int world,
                                                              int d, double u0, long long n_total, double a_param,
                                                              int lazy, long long cap_out, double* __restrict__ plan,
                                                              double* __restrict__ stats_local,
                                                              long long* __restrict__ n_out_dev) {
    shard_plan_block(gathered, rank, world, d, u0, n_total, a_param, lazy, cap_out, plan, stats_local, n_out_dev);
}

// The stats exchange fused into the plan kernel: publish this rank's stats block into every peer's buffer,
// raise the flag, wait for everybody's flag in the local buffer, plan.  One launch, no collective.
__global__ void __launch_bounds__(OBE_STATS_LEN) k_shard_plan_peer(const ObePeers peers, int rank, int world,
                                                                   unsigned long long epoch, int d, double u0,
                                                                   long long n_total, double a_param, int lazy,
                                                                   long long cap_out, double* __restrict__ plan,
                                                                   double* __restrict__ stats_local,
                                                                   long long* __restrict__ n_out_dev) {
    __shared__ int ok;
    const int t = threadIdx.x, parity = (int)(epoch & 1ull);
    obe_grid_dep_launch();
    obe_grid_dep_wait();
    double* mine = peers.p[rank];
    const double v = stats_local[t];
    for (int g = 0; g < world; ++g) peers.p[g][OBE_PEER_STATS + (parity * OBE_PEER_MAX + rank) * OBE_STATS_LEN + t] = v;
    if (t == 0) ok = 1;
    __threadfence_system();
    __syncthreads();
    if (t < world) {
        obe_flag_store(obe_peer_flags(peers.p[t], 0, parity) + rank, epoch);
        if (!obe_flag_wait(obe_peer_flags(mine, 0, parity) + t, epoch)) ok = 0;
    }
    __syncthreads();
    __threadfence_system();
    shard_plan_block(mine + OBE_PEER_STATS + parity * OBE_PEER_MAX * OBE_STATS_LEN, rank, world, d, u0, n_total, a_param,
                     lazy, cap_out, plan, stats_local, n_out_dev);
    if (t == 0 && !ok) { plan[OBE_PL_OVERFLOW] = 2.0; mine[OBE_PEER_ERR] = 1.0; }
}

// the resample kernels stage the tile's particle rows in dynamic shared memory when d <= OBE_STAGE_MAX_D
#define OBE_DIM_CASE(dd, KERNEL, grid, st, args)                                                          \
    case dd: {                                                                                            \
        const size_t smem_ = (dd <= OBE_STAGE_MAX_D) ? (size_t)dd * OBE_TILE * sizeof(double) : 0;        \
        set_max_smem((const void*)KERNEL<dd>, smem_);                                                      \
        KERNEL<dd><<<grid, OBE_THREADS, smem_, st>>>(args);                                                \
    } break;
#define OBE_DIM_SWITCH(d, KERNEL, grid, st, args)                                     \
    switch (d) {                                                                      \
        OBE_DIM_CASE(1, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(2, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(3, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(4, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(5, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(6, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(7, KERNEL, grid, st, args)                                       \
        OBE_DIM_CASE(8, KERNEL, grid, st, args)                                       \
        default: return obe_fail("n_params must be 1..8%s%s");                        \
    }

#define OBE_DIM_CASE_PLAIN(dd, KERNEL, grid, st, args) case dd: KERNEL<dd><<<grid, OBE_THREADS, 0, st>>>(args); break;
#define OBE_DIM_SWITCH_PLAIN(d, KERNEL, grid, st, args)                               \
    switch (d) {                                                                      \
        OBE_DIM_CASE_PLAIN(1, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(2, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(3, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(4, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(5, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(6, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(7, KERNEL, grid, st, args)                                 \
        OBE_DIM_CASE_PLAIN(8, KERNEL, grid, st, args)                                 \
        default: return obe_fail("n_params must be 1..8%s%s");                        \
    }

#define OBE_DIM_CASE_WR(dd, grid, st, args)                                                               \
    case dd:                                                                                              \
        set_max_smem((const void*)k_sys_resample_warp<dd>, OBE_WR_SMEM);                                  \
        launch_pdl(k_sys_resample_warp<dd>, dim3(grid), dim3(OBE_THREADS), OBE_WR_SMEM, st, args);           \
        break;
#define OBE_DIM_SWITCH_WR(d, grid, st, args)                                          \
    switch (d) {                                                                      \
        OBE_DIM_CASE_WR(1, grid, st, args) OBE_DIM_CASE_WR(2, grid, st, args)         \
        OBE_DIM_CASE_WR(3, grid, st, args) OBE_DIM_CASE_WR(4, grid, st, args)         \
        OBE_DIM_CASE_WR(5, grid, st, args) OBE_DIM_CASE_WR(6, grid, st, args)         \
        OBE_DIM_CASE_WR(7, grid, st, args) OBE_DIM_CASE_WR(8, grid, st, args)         \
        default: return obe_fail("n_params must be 1..8%s%s");                        \
    }

// ---------------------------------------------------------------------------------------------
// Sweeper selection (demos/sweeper/obe_sweeper.py:118-162): a sweep from setting index `start` to
// `stop` is worth the point utility integrated along the sweep, divided by its cost:
//   cum = cumsum(U);  U_pair = (cum[stop] - cum[start]) / ((stop - start) + cost_of_new_sweep)
// k_cumsum: one CTA, inclusive scan in coalesced chunks (fixed association, 8 chunks per round).
// k_sweep_pairs: one thread per (start, stop) pair + fused argmax (np.argmax semantics).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(OBE_SCAN_THREADS) k_cumsum(const double* __restrict__ v_in, long long n,
                                                             double* __restrict__ cum) {
    __shared__ double sm[OBE_SCANW * (OBE_SCAN_THREADS / 32 + 1)];
    const int t = threadIdx.x;
    double carry = 0.0;
    for (long long base = 0; base < n; base += OBE_SCANW * OBE_SCAN_THREADS) {
        double v[OBE_SCANW], ex[OBE_SCANW], tot[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            v[e] = (k < n) ? v_in[k] : 0.0;
        }
        obe_block_excl_scanw<double, OBE_SCAN_THREADS / 32>(v, ex, tot, sm, ObeOpSum(), 0.0, 0);
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * OBE_SCAN_THREADS + t;
            if (k < n) cum[k] = (carry + ex[e]) + v[e];
            carry += tot[e];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(OBE_THREADS) k_sweep_pairs(const double* __restrict__ cum, long long n_settings,
                                                             const int* __restrict__ pairs, long long n_pairs,
                                                             double cost_new, double* __restrict__ pair_utility,
                                                             double* part_val, long long* part_idx,
                                                             unsigned int* counter, long long* best_idx,
                                                             double* best_val) {
    __shared__ double bval[OBE_THREADS / 32];
    __shared__ long long bidx[OBE_THREADS / 32];
    __shared__ unsigned int is_last;
    const int tid = threadIdx.x;
    double best = 0.0;
    long long besti = -1;
    for (long long p = (long long)blockIdx.x * OBE_THREADS + tid; p < n_pairs; p += (long long)gridDim.x * OBE_THREADS) {
        const int2 se = *reinterpret_cast<const int2*>(pairs + 2 * p);
        const double cost = obe_add((double)(se.y - se.x), cost_new);
        const double u = obe_div(obe_sub(cum[se.y], cum[se.x]), cost);
        if (pair_utility) pair_utility[p] = u;
        obe_argmax_take(best, besti, u, p);
    }
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        part_val[blockIdx.x] = best;
        part_idx[blockIdx.x] = besti;
        __threadfence();
        is_last = (atomicAdd(counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    best = 0.0; besti = -1;
    for (unsigned int b = tid; b < gridDim.x; b += blockDim.x)
        obe_argmax_take(best, besti, __ldcg(part_val + b), __ldcg(part_idx + b));
    __syncthreads();
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) { *best_idx = besti; *best_val = best; *counter = 0u; }
}

// ---------------------------------------------------------------------------------------------
// good_setting: p_j = nan_to_num(U_j ** pickiness) as a weight vector with tile sums
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(OBE_THREADS) k_pick_weights(const double* __restrict__ util, long long n,
                                                              double pickiness, double* __restrict__ p,
                                                              double* __restrict__ tile_sums) {
    __shared__ double red[OBE_THREADS / 32];
    const long long n_tiles = (n + OBE_TILE - 1) / OBE_TILE;
    for (long long k = blockIdx.x; k < n_tiles; k += gridDim.x) {
        double s = 0.0;
        for (int e = 0; e < OBE_EPT; ++e) {
            const long long i = k * OBE_TILE + e * OBE_THREADS + threadIdx.x;
            if (i < n) {
                const double v = obe_nan_to_num(pow(util[i], pickiness));
                p[i] = v;
                s += v;
            }
        }
        const double tot = obe_block_sum(s, red);
        if (threadIdx.x == 0) tile_sums[k] = tot;
    }
}

// ---------------------------------------------------------------------------------------------
// models: built-in instantiations + NVRTC-compiled user functors
// ---------------------------------------------------------------------------------------------
template <class M, int D>
__global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) k_update_model(const ObeUpdateArgs a) {
    obe_update_body<M, D, OBE_SRC_MODEL>(a);
}
template <class M, int D>
__global__ void __launch_bounds__(OBE_THREADS) k_evalp_model(const ObeEvalArgs a) {
    obe_eval_params_body<M, D>(a);
}
template <class M>
__global__ void __launch_bounds__(OBE_THREADS) k_utility_model(const ObeUtilityArgs a) {
    obe_utility_body<M>(a);
}
template <class M>
__global__ void __launch_bounds__(OBE_THREADS) k_evals_model(const ObeEvalArgs a) {
    obe_eval_settings_body<M>(a);
}
template <class M, int D>
__global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) k_bupdate_model(const ObeBatchArgs a) {
    obe_update_batched_body<M, D, OBE_SRC_MODEL>(a);
}
template <int D>
__global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) k_brefresh(const ObeBatchArgs a) {
    obe_update_batched_body<ObeNoModel, D, OBE_SRC_NONE>(a);
}
template <class M>
__global__ void __launch_bounds__(OBE_THREADS) k_bselect_model(const ObeBSelectArgs a) {
    obe_bselect_body<M>(a);
}

template <class M, int D>
__global__ void __launch_bounds__(OBE_THREADS) k_multi_model(const ObeMultiArgs a) {
    obe_update_multi_body<M, D>(a);
}
template <class M>
__global__ void __launch_bounds__(OBE_THREADS) k_bsim_model(const ObeBSimArgs a) {
    obe_bsimulate_body<M>(a);
}

struct obe_model {
    int ns, np_model, ncons, nch, d;
    bool user;
    const void* f_update;   // kernel entry (host stub address, or cudaKernel_t for user models)
    const void* f_evalp;
    const void* f_utility;
    const void* f_evals;
    const void* f_bupdate;  // batched instances
    const void* f_bselect;
    const void* f_bsim;
    const void* f_multi;    // multi-point (sweep) update
    cudaLibrary_t lib;
    int lik;                // OBE_LIK_*: the measurement likelihood of the update kernels
    const void* f_update_y; // non-Gaussian handles: the update from a supplied y_model (OBE_SRC_Y)
    int design;             // f_utility is the likelihood-aware utility: obe_utility reads var_noise[c] as the aux a_c
    const void* f_utility_info;  // Poisson / binomial design handles: the information-gain utility (method 4)
};
#define OBE_LIK_GAUSS 0
#define OBE_LIK_POISSON 1
#define OBE_LIK_BINOMIAL 2
#define OBE_LIK_USER 3

template <class M, int D>
static void fill_model(obe_model* m) {
    m->ns = M::NS; m->np_model = M::NP; m->ncons = M::NCONS; m->nch = M::NCH; m->d = D;
    m->user = false; m->lib = nullptr;
    m->f_update = (const void*)k_update_model<M, D>;
    m->f_evalp = (const void*)k_evalp_model<M, D>;
    m->f_utility = (const void*)k_utility_model<M>;
    m->f_evals = (const void*)k_evals_model<M>;
    m->f_bupdate = (const void*)k_bupdate_model<M, D>;
    m->f_bselect = (const void*)k_bselect_model<M>;
    m->f_bsim = (const void*)k_bsim_model<M>;
    m->f_multi = (const void*)k_multi_model<M, D>;
}
template <class M>
static int make_builtin(int d, obe_model* m) {
    // pre-instantiated: the model's own parameter count plus up to 2 extra rows (noise parameters)
    if (d == M::NP) { fill_model<M, M::NP>(m); return 0; }
    if (d == M::NP + 1) { fill_model<M, M::NP + 1>(m); return 0; }
    if (d == M::NP + 2) { fill_model<M, (M::NP + 2 <= OBE_MAX_DIMS ? M::NP + 2 : OBE_MAX_DIMS)>(m); return 0; }
    return obe_fail("built-in model supports n_params in [NP, NP+2]; compile it from source for other sizes%s%s");
}

static int launch_kernel(const void* f, int grid, size_t smem, cudaStream_t st, const void* args_struct, bool pdl = false) {
    void* params[1] = {const_cast<void*>(args_struct)};
    cudaError_t e;
    if (pdl) {                                   // the kernel calls obe_grid_dep_wait() before it reads anything
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(OBE_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
        cfg.attrs = at; cfg.numAttrs = 1;
        e = cudaLaunchKernelExC(&cfg, f, params);
    } else {
        e = cudaLaunchKernel(f, dim3(grid), dim3(OBE_THREADS), params, smem, st);
    }
    if (e != cudaSuccess) return obe_fail("cudaLaunchKernel: %s%s", cudaGetErrorString(e));
    return 0;
}

// ---- NVRTC (loaded lazily so the library loads on machines without it) ----------------------
struct NvrtcApi {
    void* h;
    decltype(&nvrtcCreateProgram) create;
    decltype(&nvrtcCompileProgram) compile;
    decltype(&nvrtcGetCUBINSize) cubin_size;
    decltype(&nvrtcGetCUBIN) cubin;
    decltype(&nvrtcGetProgramLogSize) log_size;
    decltype(&nvrtcGetProgramLog) log;
    decltype(&nvrtcDestroyProgram) destroy;
    decltype(&nvrtcGetErrorString) errstr;
};
static NvrtcApi g_nvrtc = {};
static int load_nvrtc() {
    if (g_nvrtc.h) return 0;
    const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12",
                           "/usr/local/cuda/lib64/libnvrtc.so"};
    void* h = nullptr;
    for (const char* nm : names) {
        h = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
        if (h) break;
    }
    if (!h) return obe_fail("cannot load libnvrtc: %s%s", dlerror());
#define OBE_SYM(field, name)                                                   \
    g_nvrtc.field = (decltype(g_nvrtc.field))dlsym(h, name);                   \
    if (!g_nvrtc.field) return obe_fail("libnvrtc lacks %s%s", name);
    OBE_SYM(create, "nvrtcCreateProgram")
    OBE_SYM(compile, "nvrtcCompileProgram")
    OBE_SYM(cubin_size, "nvrtcGetCUBINSize")
    OBE_SYM(cubin, "nvrtcGetCUBIN")
    OBE_SYM(log_size, "nvrtcGetProgramLogSize")
    OBE_SYM(log, "nvrtcGetProgramLog")
    OBE_SYM(destroy, "nvrtcDestroyProgram")
    OBE_SYM(errstr, "nvrtcGetErrorString")
#undef OBE_SYM
    g_nvrtc.h = h;
    return 0;
}

static const char* k_src_device =
#include "obe_device_src.inc"
    ;
static const char* k_src_models =
#include "obe_models_src.inc"
    ;

// NVRTC: source -> sm_100a cubin; the compiler log goes to `log` and, on failure, into the error message
static int nvrtc_cubin(const std::string& src, const char* name, std::vector<char>& cubin, char* log, size_t log_len) {
    nvrtcProgram prog;
    const char* headers[2] = {k_src_device, k_src_models};
    const char* names[2] = {"obe_device.cuh", "obe_models.cuh"};
    nvrtcResult r = g_nvrtc.create(&prog, src.c_str(), name, 2, headers, names);
    if (r != NVRTC_SUCCESS) return obe_fail("nvrtcCreateProgram: %s%s", g_nvrtc.errstr(r));
    const char* opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo"};
    r = g_nvrtc.compile(prog, 3, opts);
    size_t lsz = 0;
    g_nvrtc.log_size(prog, &lsz);
    std::vector<char> lbuf(lsz + 1, 0);
    if (lsz > 1) g_nvrtc.log(prog, lbuf.data());
    if (log && log_len) {
        strncpy(log, lbuf.data(), log_len - 1);
        log[log_len - 1] = 0;
    }
    if (r != NVRTC_SUCCESS) {
        g_nvrtc.destroy(&prog);
        return obe_fail("NVRTC compile failed: %s\n%s", g_nvrtc.errstr(r), lbuf.data());
    }
    size_t csz = 0;
    g_nvrtc.cubin_size(prog, &csz);
    cubin.resize(csz);
    g_nvrtc.cubin(prog, cubin.data());
    g_nvrtc.destroy(&prog);
    return 0;
}
// loads the cubin into m->lib and looks up `n` kernels; on failure frees m
static int load_kernels(obe_model* m, const std::vector<char>& cubin, const char* const* names, const void** k, int n) {
    cudaError_t e = cudaLibraryLoadData(&m->lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) { delete m; return obe_fail("cudaLibraryLoadData: %s%s", cudaGetErrorString(e)); }
    for (int i = 0; i < n; ++i) {
        cudaKernel_t kk;
        e = cudaLibraryGetKernel(&kk, m->lib, names[i]);
        if (e != cudaSuccess) {
            cudaLibraryUnload(m->lib);
            delete m;
            return obe_fail("cudaLibraryGetKernel(%s): %s", names[i], cudaGetErrorString(e));
        }
        k[i] = (const void*)kk;
    }
    return 0;
}

template <class M>
static const char* builtin_dims(const char* name, obe_model* m) {
    m->ns = M::NS; m->np_model = M::NP; m->ncons = M::NCONS; m->nch = M::NCH;
    return name;
}
// the functor struct of a built-in model (NULL for an unknown name), and its dimensions into m
static const char* builtin_struct(const std::string& s, obe_model* m) {
    if (s == "lorentzian_hwhm") return builtin_dims<ObeLorentzianHWHM>("ObeLorentzianHWHM", m);
    if (s == "lorentzian_fwhm") return builtin_dims<ObeLorentzianFWHM>("ObeLorentzianFWHM", m);
    if (s == "lorentzian_4p") return builtin_dims<ObeLorentzian4P>("ObeLorentzian4P", m);
    if (s == "lorentzian_dip") return builtin_dims<ObeLorentzianDip>("ObeLorentzianDip", m);
    if (s == "line") return builtin_dims<ObeLine>("ObeLine", m);
    if (s == "rabi") return builtin_dims<ObeRabi>("ObeRabi", m);
    if (s == "lockin_coil") return builtin_dims<ObeLockinCoil>("ObeLockinCoil", m);
    return nullptr;
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int obe_abi_version(void) { return OBE_ABI_VERSION; }
const char* obe_last_error(void) { return g_err; }
int obe_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int64_t obe_num_tiles(int64_t n) { return (n + OBE_TILE - 1) / OBE_TILE; }
size_t obe_scratch_bytes(int64_t n) { return scratch_bytes(n); }
size_t obe_select_scratch_bytes(int64_t n_settings) {
    const int64_t nt = (n_settings + OBE_TILE - 1) / OBE_TILE;
    size_t b = 256;                                            // counter
    b += align_up((size_t)OBE_MAX_GRID * sizeof(double), 256);    // part_val
    b += align_up((size_t)OBE_MAX_GRID * sizeof(long long), 256); // part_idx
    b += align_up((size_t)n_settings * sizeof(double), 256);      // p
    b += align_up((size_t)nt * sizeof(double), 256);              // tile sums
    b += align_up((size_t)(nt + 1) * sizeof(double), 256);        // prefix
    return b;
}

int obe_set_option(const char* name, int64_t value) {
    if (!name) return obe_fail("null argument%s%s");
    const std::string s(name);
    if (s == "plan_cluster_min_tiles") { g_plan_cluster_min_tiles = value < 0 ? 0 : value; return 0; }
    if (s == "utility_lane_fill") { g_utility_lane_fill = value < 0 ? 0 : value; return 0; }
    if (s == "utility_cache") { g_utility_cache = value ? 1 : 0; return 0; }
    if (s == "utility_info_blocks") { g_utility_info_blocks = value < 0 ? 0 : value; return 0; }
    if (s == "resample_fused") { g_resample_fused = value ? 1 : 0; return 0; }
    if (s == "resample_blocks") { g_resample_blocks = value < 0 ? 0 : value; return 0; }
    if (s == "resample_reserve_ctas") { g_resample_reserve = value < 0 ? 0 : value; return 0; }
    if (s == "pdl") { g_pdl = value ? 1 : 0; return 0; }
    if (s == "copy_out_side") { g_copy_out_side = value ? 1 : 0; return 0; }
    if (s == "zero_copy_out") { g_zero_copy_out = value ? 1 : 0; return 0; }
    if (s == "resample_dynamic") { g_resample_dynamic = value ? 1 : 0; return 0; }
    if (s == "resample_units_per_sm") { g_resample_units_per_sm = value < 1 ? 1 : value; return 0; }
    return obe_fail("unknown option '%s'%s", name);
}

int obe_model_builtin(const char* name, int n_params, obe_model_t* out) {
    if (!name || !out) return obe_fail("null argument%s%s");
    obe_model* m = new obe_model();
    int rc;
    const std::string s(name);
    if (s == "lorentzian_hwhm") rc = make_builtin<ObeLorentzianHWHM>(n_params, m);
    else if (s == "lorentzian_fwhm") rc = make_builtin<ObeLorentzianFWHM>(n_params, m);
    else if (s == "lorentzian_4p") rc = make_builtin<ObeLorentzian4P>(n_params, m);
    else if (s == "lorentzian_dip") rc = make_builtin<ObeLorentzianDip>(n_params, m);
    else if (s == "line") rc = make_builtin<ObeLine>(n_params, m);
    else if (s == "rabi") rc = make_builtin<ObeRabi>(n_params, m);
    else if (s == "lockin_coil") rc = make_builtin<ObeLockinCoil>(n_params, m);
    else rc = obe_fail("unknown built-in model '%s'%s", name);
    if (rc) { delete m; return rc; }
    *out = m;
    return 0;
}

int obe_model_compile(const char* cuda_source, const char* entry, int n_settings, int n_params,
                      int n_model_params, int n_constants, int n_channels, obe_model_t* out, char* log,
                      size_t log_len) {
    if (log && log_len) log[0] = 0;
    if (!cuda_source || !entry || !out) return obe_fail("null argument%s%s");
    if (n_params < 1 || n_params > OBE_MAX_DIMS || n_model_params < 0 || n_model_params > n_params ||
        n_channels < 1 || n_channels > OBE_MAX_CH || n_settings < 0 || n_settings > OBE_MAX_SET ||
        n_constants < 0 || n_constants > OBE_MAX_CONS)
        return obe_fail("model dimensions out of range%s%s");
    if (load_nvrtc()) return -1;
    char tail[2048];
    snprintf(tail, sizeof(tail),
             "\nstruct ObeUserModel {\n"
             "    enum { NS = %d, NP = %d, NCONS = %d, NCH = %d };\n"
             "    __device__ static __forceinline__ void eval(const double* s, const double* p, const double* c, double* y) {\n"
             "        %s(s, p, c, y);\n    }\n};\n"
             "OBE_DEFINE_MODEL_KERNELS(ObeUserModel, %d, user)\n"
             "OBE_DEFINE_GRID_KERNELS(ObeUserModel, user)\n"
             "OBE_DEFINE_BATCH_KERNELS(ObeUserModel, %d, user)\n",
             n_settings, n_model_params, n_constants, n_channels, entry, n_params, n_params);
    std::string src = "#include \"obe_device.cuh\"\n#include \"obe_models.cuh\"\n";
    src += cuda_source;
    src += tail;
    std::vector<char> cubin;
    if (nvrtc_cubin(src, "obe_user_model.cu", cubin, log, log_len)) return -1;
    obe_model* m = new obe_model();
    m->ns = n_settings; m->np_model = n_model_params; m->ncons = n_constants; m->nch = n_channels;
    m->d = n_params; m->user = true;
    const void* k[8];
    const char* kn[8] = {"obe_k_update_user", "obe_k_evalp_user", "obe_k_utility_user", "obe_k_evals_user",
                         "obe_k_bupdate_user", "obe_k_bselect_user", "obe_k_bsim_user", "obe_k_multi_user"};
    if (load_kernels(m, cubin, kn, k, 8)) return -1;
    m->f_update = k[0]; m->f_evalp = k[1];
    m->f_utility = k[2]; m->f_evals = k[3];
    m->f_bupdate = k[4]; m->f_bselect = k[5]; m->f_bsim = k[6];
    m->f_multi = k[7];
    *out = m;
    return 0;
}

// A non-Gaussian handle.  noise_var_entry == NULL: the plain likelihood handle, whose utility is today's
// (var_noise[c] the noise variance).  design != 0: the same update kernels, and the likelihood-aware utility
// (obe_k_utility_design: var_noise[c] is the design aux a_c; noise_var_entry names a user likelihood's variance).
static int compile_likelihood(const char* builtin_name, const char* model_source, const char* model_entry,
                              int n_settings, int n_params, int n_model_params, int n_constants, int n_channels,
                              const char* likelihood, const char* likelihood_source, const char* likelihood_entry,
                              int design, const char* noise_var_entry, obe_model_t* out, char* log, size_t log_len) {
    if (log && log_len) log[0] = 0;
    if (!out || !likelihood || (!builtin_name && (!model_source || !model_entry)))
        return obe_fail("null argument%s%s");
    const std::string lk(likelihood);
    int kind;
    if (lk == "poisson") kind = OBE_LIK_POISSON;
    else if (lk == "binomial") kind = OBE_LIK_BINOMIAL;
    else if (lk == "user") kind = OBE_LIK_USER;
    else return obe_fail("unknown likelihood '%s' (poisson, binomial or user)%s", likelihood);
    if (kind == OBE_LIK_USER && (!likelihood_source || !likelihood_entry))
        return obe_fail("a user likelihood needs its source and entry%s%s");
    if (design && kind == OBE_LIK_USER && !noise_var_entry)
        return obe_fail("a likelihood-aware design with a user likelihood needs its noise_var entry%s%s");
    obe_model tmp = {};
    std::string model_def;
    if (builtin_name) {
        const char* st = builtin_struct(builtin_name, &tmp);
        if (!st) return obe_fail("unknown built-in model '%s'%s", builtin_name);
        model_def = std::string("typedef ") + st + " ObeLikModel;\n";
    } else {
        if (n_model_params < 0 || n_channels < 1 || n_channels > OBE_MAX_CH || n_settings < 0 ||
            n_settings > OBE_MAX_SET || n_constants < 0 || n_constants > OBE_MAX_CONS)
            return obe_fail("model dimensions out of range%s%s");
        tmp.ns = n_settings; tmp.np_model = n_model_params; tmp.ncons = n_constants; tmp.nch = n_channels;
        char def[1024];
        snprintf(def, sizeof(def),
                 "\nstruct ObeLikModel {\n"
                 "    enum { NS = %d, NP = %d, NCONS = %d, NCH = %d };\n"
                 "    __device__ static __forceinline__ void eval(const double* s, const double* p, const double* c, double* y) {\n"
                 "        %s(s, p, c, y);\n    }\n};\n",
                 n_settings, n_model_params, n_constants, n_channels, model_entry);
        model_def = std::string(model_source) + def;
    }
    if (n_params < 1 || n_params > OBE_MAX_DIMS || tmp.np_model > n_params)
        return obe_fail("n_params out of range (the model's parameters .. 8)%s%s");
    if (load_nvrtc()) return -1;
    std::string src = "#include \"obe_device.cuh\"\n#include \"obe_models.cuh\"\n";
    src += model_def;
    const char* lik_type = kind == OBE_LIK_POISSON ? "ObePoissonLik" : (kind == OBE_LIK_BINOMIAL ? "ObeBinomialLik" : "ObeUserLik");
    if (kind == OBE_LIK_USER) {
        src += likelihood_source;
        src += "\nstruct ObeUserPmf {\n"
               "    static constexpr bool NONPOS = false;\n"
               "    template <int NY>\n"
               "    __device__ static __forceinline__ double loglik(const double (&y)[NY], const double* ym,\n"
               "                                                    const ObeLikParams& q, int n) {\n"
               "        return ";
        src += likelihood_entry;
        src += "(y, ym, q.aux, n);\n    }\n};\ntypedef ObeLogLik<ObeUserPmf> ObeUserLik;\n";
        if (design) {
            src += "struct ObeUserNoise {\n"
                   "    static constexpr bool LIK = true;\n"
                   "    static constexpr bool NU_IS_Y = false;\n"
                   "    __device__ static __forceinline__ double nu(double y, double a) { return ";
            src += noise_var_entry;
            src += "(y, a); }\n"
                   "    __device__ static __forceinline__ bool ok(double, double v) { return v >= 0.0; }\n"
                   "    __device__ static __forceinline__ double finish(double m, double) { return m; }\n"
                   "    typedef ObeNoInfo Info;\n};\n";
        }
    }
    const char* noise_type = kind == OBE_LIK_POISSON ? "ObePoissonNoise"
                             : (kind == OBE_LIK_BINOMIAL ? "ObeBinomialNoise" : "ObeUserNoise");
    char tail[512];
    if (design)
        snprintf(tail, sizeof(tail),
                 "OBE_DEFINE_LIK_KERNELS(ObeLikModel, %s, %d)\n"
                 "OBE_DEFINE_DESIGN_KERNELS(ObeLikModel, %s)\n", lik_type, n_params, noise_type);
    else
        snprintf(tail, sizeof(tail),
                 "OBE_DEFINE_LIK_KERNELS(ObeLikModel, %s, %d)\n"
                 "OBE_DEFINE_GRID_KERNELS(ObeLikModel, lik)\n", lik_type, n_params);
    src += tail;
    std::vector<char> cubin;
    if (nvrtc_cubin(src, "obe_likelihood_model.cu", cubin, log, log_len)) return -1;
    obe_model* m = new obe_model(tmp);
    m->d = n_params; m->user = true; m->lik = kind; m->design = design ? 1 : 0;
    const void* k[6];
    const char* kn[6] = {"obe_k_update_lik", "obe_k_updatey_lik", "obe_k_evalp_lik", "obe_k_utility_lik",
                         "obe_k_evals_lik", "obe_k_utility_info"};
    if (design) { kn[3] = "obe_k_utility_design"; kn[4] = "obe_k_evals_design"; }
    // (the information gain needs a known support: Poisson and binomial design handles only)
    const int nk = design && kind != OBE_LIK_USER ? 6 : 5;
    if (load_kernels(m, cubin, kn, k, nk)) return -1;
    m->f_update = k[0]; m->f_update_y = k[1]; m->f_evalp = k[2]; m->f_utility = k[3]; m->f_evals = k[4];
    if (nk == 6) m->f_utility_info = k[5];
    *out = m;
    return 0;
}

int obe_model_compile_likelihood(const char* builtin_name, const char* model_source, const char* model_entry,
                                 int n_settings, int n_params, int n_model_params, int n_constants, int n_channels,
                                 const char* likelihood, const char* likelihood_source, const char* likelihood_entry,
                                 obe_model_t* out, char* log, size_t log_len) {
    return compile_likelihood(builtin_name, model_source, model_entry, n_settings, n_params, n_model_params,
                              n_constants, n_channels, likelihood, likelihood_source, likelihood_entry, 0, nullptr, out,
                              log, log_len);
}

int obe_model_compile_likelihood_design(const char* builtin_name, const char* model_source, const char* model_entry,
                                        int n_settings, int n_params, int n_model_params, int n_constants,
                                        int n_channels, const char* likelihood, const char* likelihood_source,
                                        const char* likelihood_entry, const char* noise_var_entry, obe_model_t* out,
                                        char* log, size_t log_len) {
    return compile_likelihood(builtin_name, model_source, model_entry, n_settings, n_params, n_model_params,
                              n_constants, n_channels, likelihood, likelihood_source, likelihood_entry, 1,
                              noise_var_entry, out, log, log_len);
}

int obe_model_info(obe_model_t m, int* ns, int* npm, int* nc, int* nch, int* np) {
    if (!m) return obe_fail("null model%s%s");
    if (ns) *ns = m->ns;
    if (npm) *npm = m->np_model;
    if (nc) *nc = m->ncons;
    if (nch) *nch = m->nch;
    if (np) *np = m->d;
    return 0;
}
void obe_model_free(obe_model_t m) {
    if (!m) return;
    if (m->user && m->lib) {
        cudaLibraryUnload(m->lib);
        g_smem_epoch.fetch_add(1, std::memory_order_relaxed);
    }
    delete m;
}

static int check_cloud(const obe_cloud_t* c) {
    if (!c || !c->particles_dev || !c->weights_dev || !c->tile_sums_dev || !c->tile_prefix_dev ||
        !c->stats_dev || !c->scratch_dev)
        return obe_fail("cloud has null device pointers%s%s");
    if (c->n < 1 || c->d < 1 || c->d > OBE_MAX_DIMS || c->ld < c->n || (c->ld & 1))
        return obe_fail("cloud geometry invalid (need 1<=d<=8, ld>=n, ld even)%s%s");
    if (((uintptr_t)c->particles_dev | (uintptr_t)c->weights_dev) & 15)
        return obe_fail("particles/weights must be 16-byte aligned%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    return 0;
}
static int update_grid(const obe_cloud_t* c) {
    // persistent: one warp-specialised CTA per SM (its stage ring takes most of the shared memory)
    const int64_t nt = obe_num_tiles(c->n);
    int64_t g = (int64_t)obe_sms();
    if (g > nt) g = nt;
    if (g > OBE_MAX_GRID) g = OBE_MAX_GRID;
    return (int)g;
}
static void base_update_args(const obe_cloud_t* c, ObeUpdateArgs& a, const double* pivot) {
    memset(&a, 0, sizeof(a));
    const Scratch s = scratch_of(c);
    a.particles = c->particles_dev; a.ld = c->ld; a.n = c->n; a.n_dev = (const long long*)c->n_dev;
    a.weights = c->weights_dev; a.tile_sums = c->tile_sums_dev;
    a.partials = s.partials; a.counter = s.counter; a.stats = c->stats_dev;
    a.tile_prefix = c->tile_prefix_dev; a.renormalise = 1;
    for (int j = 0; j < OBE_MAX_CH; ++j) a.noise_idx[j] = -1;
    if (pivot) for (int j = 0; j < c->d; ++j) a.pivot[j] = pivot[j];
    a.gate_thr = g_update_gate_thr; a.gate_n = g_update_gate_n;
    a.stats_out2 = g_update_stats_out;
}
static int finish_update(const obe_cloud_t*, int, cudaStream_t) {
    return 0;   // the update kernel's last block scans the tile sums itself (ObeUpdateArgs::tile_prefix)
}
static int fill_likelihood_args(ObeUpdateArgs& a, int d, int nch_avail, const double* y_meas, const double* sigma,
                                const int32_t* noise_index, int n_lik, int use_choke, double choke) {
    if (n_lik < 0 || n_lik > nch_avail || n_lik > OBE_MAX_CH) return obe_fail("n_lik_channels out of range%s%s");
    if (!y_meas) return obe_fail("y_meas is null%s%s");
    if (!sigma && !noise_index) return obe_fail("need sigma or noise_index%s%s");
    a.n_lik_channels = n_lik;
    for (int cidx = 0; cidx < n_lik; ++cidx) {
        a.y_meas[cidx] = y_meas[cidx];
        a.inv_sigma[cidx] = sigma ? 1.0 / sigma[cidx] : 1.0;
        if (noise_index) {
            if (noise_index[cidx] < 0 || noise_index[cidx] >= d) return obe_fail("noise_index out of range%s%s");
            a.noise_idx[cidx] = noise_index[cidx];
            a.n_noise = cidx + 1;
        }
    }
    a.use_choke = use_choke; a.choke = choke;
    return 0;
}

// The record of a non-Gaussian likelihood: y_meas[c] = the counts (the measured values for a user likelihood),
// aux[c] = the record's third element (binomial trial counts; anything a user likelihood reads; NULL for Poisson).
// The log-factorial terms of the counting pmfs are per-record constants, computed here once.
static int fill_lik_record(ObeUpdateArgs& a, ObeLikParams& q, int kind, int nch_avail, const double* y_meas,
                           const double* aux, const int32_t* noise_index, int n_lik, int use_choke, double choke) {
    if (n_lik < 0 || n_lik > nch_avail || n_lik > OBE_MAX_CH) return obe_fail("n_lik_channels out of range%s%s");
    if (!y_meas) return obe_fail("y_meas is null%s%s");
    if (noise_index) return obe_fail("a noise parameter needs the Gaussian likelihood%s%s");
    if (!aux && kind != OBE_LIK_POISSON) return obe_fail("this likelihood needs the record's third element%s%s");
    memset(&q, 0, sizeof(q));
    a.n_lik_channels = n_lik;
    for (int cidx = 0; cidx < n_lik; ++cidx) {
        const double k = y_meas[cidx];
        a.y_meas[cidx] = k;
        q.aux[cidx] = aux ? aux[cidx] : 0.0;
        if (kind == OBE_LIK_POISSON) {
            if (!(std::isfinite(k) && k >= 0.0 && k == std::floor(k)))
                return obe_fail("Poisson counts must be finite non-negative integers%s%s");
            q.lconst[cidx] = std::lgamma(k + 1.0);
        } else if (kind == OBE_LIK_BINOMIAL) {
            const double nt = aux[cidx];
            if (!(std::isfinite(k) && std::isfinite(nt) && k >= 0.0 && k <= nt && k == std::floor(k) && nt == std::floor(nt)))
                return obe_fail("binomial records need integers 0 <= k <= n_trials%s%s");
            q.lconst[cidx] = (std::lgamma(nt + 1.0) - std::lgamma(k + 1.0)) - std::lgamma(nt - k + 1.0);
        }
    }
    a.use_choke = use_choke; a.choke = choke;
    return 0;
}

int obe_set_uniform(const obe_cloud_t* c, void* stream) {
    if (check_cloud(c)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    int grid = obe_sms() * 8;
    k_fill_uniform<<<grid, 256, 0, st>>>(c->weights_dev, c->tile_sums_dev, c->n, obe_num_tiles(c->n), 1, c->n,
                                         (const long long*)c->n_dev);
    OBE_LAUNCH_CHECK("k_fill_uniform");
    OBE_CUDA(cudaMemsetAsync(c->stats_dev, 0, OBE_STATS_LEN * sizeof(double), st));
    k_tile_scan<<<1, OBE_SCAN_THREADS, 0, st>>>(c->tile_sums_dev, obe_num_tiles(c->n), c->tile_prefix_dev,
                                               c->stats_dev, 0, c->n, c->n, (const long long*)c->n_dev);
    OBE_LAUNCH_CHECK("k_tile_scan");
    return 0;
}

int obe_set_uniform_total(const obe_cloud_t* c, int64_t n_total, void* stream) {
    if (check_cloud(c)) return -1;
    if (n_total < 1 || (!c->n_dev && n_total < c->n)) return obe_fail("n_total < n%s%s");
    cudaStream_t st = (cudaStream_t)stream;
    k_fill_uniform<<<obe_sms() * 8, 256, 0, st>>>(c->weights_dev, c->tile_sums_dev, c->n, obe_num_tiles(c->n), 1, n_total,
                                                  (const long long*)c->n_dev);
    OBE_LAUNCH_CHECK("k_fill_uniform");
    OBE_CUDA(cudaMemsetAsync(c->stats_dev, 0, OBE_STATS_LEN * sizeof(double), st));
    k_tile_scan<<<1, OBE_SCAN_THREADS, 0, st>>>(c->tile_sums_dev, obe_num_tiles(c->n), c->tile_prefix_dev,
                                               c->stats_dev, 0, n_total, c->n, (const long long*)c->n_dev);
    OBE_LAUNCH_CHECK("k_tile_scan");
    return 0;
}

int obe_update(obe_model_t m, const obe_cloud_t* c, const double* setting, const double* constants,
               const double* y_meas, const double* sigma, const int32_t* noise_index, int n_lik_channels,
               int use_choke, double choke, const double* pivot, void* stream) {
    if (!m) return obe_fail("null model%s%s");
    if (check_cloud(c)) return -1;
    if (m->d != c->d) return obe_fail("model was built for a different n_params%s%s");
    ObeUpdateArgs a;
    base_update_args(c, a, pivot);
    a.scale_in = 1; a.write_weights = 1;
    for (int j = 0; j < m->ns; ++j) a.setting[j] = setting[j];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    if (m->lik != OBE_LIK_GAUSS) {
        ObeLikParams q;
        if (fill_lik_record(a, q, m->lik, m->nch, y_meas, sigma, noise_index, n_lik_channels, use_choke, choke)) return -1;
        if (launch_update_kernel(m->f_update, c->d, OBE_SRC_MODEL, a, update_grid(c), (cudaStream_t)stream, &q)) return -1;
        return finish_update(c, 1, (cudaStream_t)stream);
    }
    if (fill_likelihood_args(a, c->d, m->nch, y_meas, sigma, noise_index, n_lik_channels, use_choke, choke)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    if (launch_update_kernel(m->f_update, c->d, OBE_SRC_MODEL, a, update_grid(c), st)) return -1;
    return finish_update(c, 1, st);
}

int obe_update_from_y(const obe_cloud_t* c, const double* y_model_dev, int64_t ld_y, int n_channels,
                      const double* y_meas, const double* sigma, const int32_t* noise_index, int n_lik_channels,
                      int use_choke, double choke, const double* pivot, void* stream) {
    if (check_cloud(c)) return -1;
    if (!y_model_dev || (ld_y & 1) || ((uintptr_t)y_model_dev & 15)) return obe_fail("y_model must be 16-byte aligned with even ld%s%s");
    ObeUpdateArgs a;
    base_update_args(c, a, pivot);
    a.scale_in = 1; a.write_weights = 1;
    a.y_model = y_model_dev; a.ld_y = ld_y;
    if (fill_likelihood_args(a, c->d, n_channels, y_meas, sigma, noise_index, n_lik_channels, use_choke, choke)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    if (launch_generic<OBE_SRC_Y>(c->d, a, update_grid(c), st)) return -1;
    return finish_update(c, 1, st);
}

int obe_update_from_y_model(obe_model_t m, const obe_cloud_t* c, const double* y_model_dev, int64_t ld_y,
                            int n_channels, const double* y_meas, const double* sigma, const int32_t* noise_index,
                            int n_lik_channels, int use_choke, double choke, const double* pivot, void* stream) {
    if (!m) return obe_fail("null model%s%s");
    if (m->lik == OBE_LIK_GAUSS)
        return obe_update_from_y(c, y_model_dev, ld_y, n_channels, y_meas, sigma, noise_index, n_lik_channels, use_choke,
                                 choke, pivot, stream);
    if (check_cloud(c)) return -1;
    if (m->d != c->d) return obe_fail("model was built for a different n_params%s%s");
    if (!y_model_dev || (ld_y & 1) || ((uintptr_t)y_model_dev & 15)) return obe_fail("y_model must be 16-byte aligned with even ld%s%s");
    ObeUpdateArgs a;
    base_update_args(c, a, pivot);
    a.scale_in = 1; a.write_weights = 1;
    a.y_model = y_model_dev; a.ld_y = ld_y;
    ObeLikParams q;
    if (fill_lik_record(a, q, m->lik, n_channels, y_meas, sigma, noise_index, n_lik_channels, use_choke, choke)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    if (launch_update_kernel(m->f_update_y, c->d, OBE_SRC_Y, a, update_grid(c), st, &q)) return -1;
    return finish_update(c, 1, st);
}

int obe_update_from_likelihood(const obe_cloud_t* c, const double* likelihood_dev, const double* pivot, void* stream) {
    if (check_cloud(c)) return -1;
    if (!likelihood_dev || ((uintptr_t)likelihood_dev & 15)) return obe_fail("likelihood must be 16-byte aligned%s%s");
    ObeUpdateArgs a;
    base_update_args(c, a, pivot);
    a.scale_in = 1; a.write_weights = 1;
    a.lik = likelihood_dev;
    cudaStream_t st = (cudaStream_t)stream;
    if (launch_generic<OBE_SRC_LIK>(c->d, a, update_grid(c), st)) return -1;
    return finish_update(c, 1, st);
}

int obe_refresh(const obe_cloud_t* c, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index, int n_noise,
                const double* pivot, int renormalise, void* stream) {
    if (check_cloud(c)) return -1;
    ObeUpdateArgs a;
    base_update_args(c, a, pivot);
    a.scale_in = 0;
    a.write_weights = (mask_le | mask_lt) ? 1 : 0;
    a.mask_le = mask_le; a.mask_lt = mask_lt;
    if (noise_index)
        for (int j = 0; j < n_noise && j < OBE_MAX_CH; ++j) { a.noise_idx[j] = noise_index[j]; a.n_noise = j + 1; }
    cudaStream_t st = (cudaStream_t)stream;
    a.renormalise = renormalise;
    if (launch_generic<OBE_SRC_NONE>(c->d, a, update_grid(c), st)) return -1;
    return finish_update(c, renormalise, st);
}

int obe_fetch_stats(const obe_cloud_t* c, double* stats_host, void* stream) {
    if (!c || !stats_host) return obe_fail("null argument%s%s");
    cudaStream_t st = (cudaStream_t)stream;
    OBE_CUDA(cudaMemcpyAsync(stats_host, c->stats_dev, OBE_STATS_LEN * sizeof(double), cudaMemcpyDeviceToHost, st));
    OBE_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int obe_normalized_weights(const obe_cloud_t* c, double* out_dev, void* stream) {
    if (check_cloud(c)) return -1;
    k_normalized_weights<<<obe_sms() * 8, 256, 0, (cudaStream_t)stream>>>(c->weights_dev, c->stats_dev, out_dev, c->n,
                                                                          (const long long*)c->n_dev);
    OBE_LAUNCH_CHECK("k_normalized_weights");
    return 0;
}

__global__ void k_materialize(double* __restrict__ w, double* __restrict__ stats, long long n,
                              const long long* __restrict__ n_dev) {
    if (n_dev) n = *n_dev;
    const double wuni = stats[OBE_ST_UNIFORM];
    if (!(wuni > 0.0)) return;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        w[i] = wuni;
}
__global__ void k_clear_uniform(double* __restrict__ stats) { stats[OBE_ST_UNIFORM] = 0.0; }

int obe_materialize_weights(const obe_cloud_t* c, void* stream) {
    if (check_cloud(c)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    k_materialize<<<obe_sms() * 8, 256, 0, st>>>(c->weights_dev, c->stats_dev, c->n, (const long long*)c->n_dev);
    OBE_LAUNCH_CHECK("k_materialize");
    k_clear_uniform<<<1, 1, 0, st>>>(c->stats_dev);
    OBE_LAUNCH_CHECK("k_clear_uniform");
    return 0;
}

int obe_cdf(const obe_cloud_t* c, double* cdf_dev, void* stream) {
    if (check_cloud(c)) return -1;
    const int64_t nt = obe_num_tiles(c->n);
    int grid = (int)(nt < (int64_t)obe_sms() * 8 ? nt : (int64_t)obe_sms() * 8);
    k_cdf<<<grid, OBE_THREADS, 0, (cudaStream_t)stream>>>(c->weights_dev, c->tile_prefix_dev, c->n, nt, cdf_dev,
                                                          c->stats_dev);
    OBE_LAUNCH_CHECK("k_cdf");
    return 0;
}

int obe_search(const obe_cloud_t* c, const double* cdf_dev, const double* u_dev, int64_t m, int64_t* idx_dev,
               void* stream) {
    if (check_cloud(c)) return -1;
    if (m <= 0) return 0;
    int64_t blocks = (m + 255) / 256;
    if (blocks > (int64_t)obe_sms() * 16) blocks = (int64_t)obe_sms() * 16;
    k_search<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(cdf_dev, c->tile_prefix_dev, c->n, obe_num_tiles(c->n),
                                                           u_dev, m, (long long*)idx_dev);
    OBE_LAUNCH_CHECK("k_search");
    return 0;
}

struct ObePeerDraw { const ObePeers* peers; int rank, world; unsigned long long epoch; unsigned int* counter; };
static int draw_impl(const double* w, const double* prefix, int64_t n, const double* particles, int64_t ld, int d,
                     const double* u_host, int k, double* draws_dev, int64_t* idx_dev, cudaStream_t st,
                     int ld_draws = 0, const long long* n_dev = nullptr, const double* plan = nullptr, int post = 0,
                     const double* stats = nullptr, const ObePeerDraw* peer = nullptr) {
    if (k <= 0) return 0;
    for (int off = 0; off < k; off += OBE_MAX_DRAWS) {
        const int kk = (k - off) < OBE_MAX_DRAWS ? (k - off) : OBE_MAX_DRAWS;
        ObeDrawArgs a;
        memset(&a, 0, sizeof(a));
        if (peer) {
            a.peers = *peer->peers; a.peer_rank = peer->rank; a.peer_world = peer->world; a.peer_epoch = peer->epoch;
            a.peer_counter = peer->counter;
        }
        a.w = w; a.prefix = prefix; a.n = n; a.n_tiles = obe_num_tiles(n);
        a.particles = particles; a.ld = ld; a.d = d;
        a.draws = draws_dev ? draws_dev + off : nullptr;
        a.idx = idx_dev ? (long long*)idx_dev + off : nullptr;
        a.k = ld_draws > 0 ? ld_draws : k;
        a.n_dev = n_dev; a.plan = plan; a.post = post; a.stats = stats;
        a.gate_off = g_gate_off;
        for (int i = 0; i < kk; ++i) a.u[i] = u_host[off + i];
        launch_pdl(k_draw, dim3(kk), dim3(OBE_THREADS), 0, st, a);
        OBE_LAUNCH_CHECK("k_draw");
    }
    return 0;
}

int obe_draw(const obe_cloud_t* c, const double* u_host, int k, double* draws_dev, int64_t* idx_dev, void* stream) {
    if (check_cloud(c)) return -1;
    if (!u_host || !draws_dev) return obe_fail("null argument%s%s");
    return draw_impl(c->weights_dev, c->tile_prefix_dev, c->n, c->particles_dev, c->ld, c->d, u_host, k, draws_dev,
                     idx_dev, (cudaStream_t)stream, 0, (const long long*)c->n_dev, nullptr, 0, c->stats_dev);
}

int obe_draw_planned(const obe_cloud_t* c, const double* u_host, int k, double* draws_dev, const double* plan_dev,
                     int post, void* stream) {
    if (check_cloud(c)) return -1;
    if (!u_host || !draws_dev || !plan_dev) return obe_fail("null argument%s%s");
    return draw_impl(c->weights_dev, c->tile_prefix_dev, c->n, c->particles_dev, c->ld, c->d, u_host, k, draws_dev,
                     nullptr, (cudaStream_t)stream, 0, (const long long*)c->n_dev, plan_dev, post, c->stats_dev);
}

static int finish_resample(const obe_cloud_t* out, int64_t n_total, cudaStream_t st, int implicit = 0) {
    k_fill_uniform<<<obe_sms() * 2, 256, 0, st>>>(out->weights_dev, out->tile_sums_dev, out->n, obe_num_tiles(out->n), 0,
                                                 n_total, (const long long*)out->n_dev);
    OBE_LAUNCH_CHECK("k_fill_uniform");
    k_tile_scan<<<1, OBE_SCAN_THREADS, 0, st>>>(out->tile_sums_dev, obe_num_tiles(out->n), out->tile_prefix_dev,
                                               out->stats_dev, 0, n_total, out->n, (const long long*)out->n_dev, implicit);
    OBE_LAUNCH_CHECK("k_tile_scan");
    return 0;
}

static int fill_resample_args(const obe_cloud_t* in, const obe_cloud_t* out, const double* factor, const double* mean,
                              double a_param, int scale, uint64_t seed, uint32_t epoch, ObeResampleArgs& a) {
    if (check_cloud(in) || check_cloud(out)) return -1;
    if (in->d != out->d) return obe_fail("resample: in/out geometry differs%s%s");
    if (in->particles_dev == out->particles_dev || in->weights_dev == out->weights_dev)
        return obe_fail("resample is out-of-place: pass a second cloud%s%s");
    memset(&a, 0, sizeof(a));
    a.pin = in->particles_dev; a.ld_in = in->ld; a.w_in = in->weights_dev; a.prefix = in->tile_prefix_dev;
    a.n = in->n; a.n_tiles = obe_num_tiles(in->n);
    a.pout = out->particles_dev; a.ld_out = out->ld; a.w_out = out->weights_dev;
    a.stats = in->stats_dev;
    a.a_param = a_param; a.scale = scale; a.seed = seed; a.epoch = epoch; a.jitter = 1;
    a.gate = g_gate_on;
    if (factor) {
        if (scale && !mean) return obe_fail("resample: mean required with a host factor when scale is on%s%s");
        for (int q = 0; q < in->d * in->d; ++q) a.factor[q] = factor[q];
        if (mean) for (int j = 0; j < in->d; ++j) a.mean[j] = mean[j];
        a.factor_from_stats = 0;
    } else {
        a.factor_from_stats = 1;
    }
    return 0;
}

int obe_draw_strided(const obe_cloud_t* c, const double* u_host, int m, double* draws_dev, int ld_draws,
                     int64_t* idx_dev, void* stream) {
    if (check_cloud(c)) return -1;
    if (m == 0) return 0;
    if (!u_host || !draws_dev || ld_draws < m) return obe_fail("bad argument%s%s");
    return draw_impl(c->weights_dev, c->tile_prefix_dev, c->n, c->particles_dev, c->ld, c->d, u_host, m, draws_dev,
                     idx_dev, (cudaStream_t)stream, ld_draws, (const long long*)c->n_dev, nullptr, 0, c->stats_dev);
}

int obe_gather_jitter(const obe_cloud_t* in, const obe_cloud_t* out, const int64_t* idx_dev, const double* factor,
                      const double* mean, const double* z_dev, uint64_t seed, uint32_t epoch, double a_param, int scale,
                      void* stream) {
    ObeResampleArgs a;
    if (fill_resample_args(in, out, factor, mean, a_param, scale, seed, epoch, a)) return -1;
    if (in->n != out->n) return obe_fail("gather_jitter: in/out sizes differ%s%s");
    if (!idx_dev) return obe_fail("null ancestors%s%s");
    a.idx_in = (const long long*)idx_dev; a.z_in = z_dev;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t blocks = (in->n + OBE_THREADS - 1) / OBE_THREADS;
    if (blocks > (int64_t)obe_sms() * 8) blocks = (int64_t)obe_sms() * 8;
    const int grid = (int)blocks;
    OBE_DIM_SWITCH_PLAIN(in->d, k_gather_jitter, grid, st, a)
    OBE_LAUNCH_CHECK("k_gather_jitter");
    return finish_resample(out, out->n, st);
}

// the unit -> tile map lives in the input cloud's scratch, which is sized for in->n particles
// Output slots per work unit.  Two-kernel path: 4096 (the CTA-wide mark scan is built for it).  One-kernel path: one
// WARP owns a unit, so a cloud of a few tiles would keep a handful of warps busy for thousands of slots each; the
// chunk shrinks (multiples of the 128-slot emission group) until there are ~16 units per SM, at the price of one
// more CDF walk of the tile per extra unit.
static int plan_chunk(int64_t out_cap) {
    if (!g_resample_fused) return OBE_OUT_CHUNK;
    int64_t c = out_cap / ((int64_t)obe_sms() * g_resample_units_per_sm);
    c = (c + OBE_WR_GROUP_HOST - 1) / OBE_WR_GROUP_HOST * OBE_WR_GROUP_HOST;
    if (c < OBE_WR_MIN_CHUNK) c = OBE_WR_MIN_CHUNK;
    if (c > OBE_WR_CHUNK) c = OBE_WR_CHUNK;
    return (int)c;
}
static bool unit_map_fits(const obe_cloud_t* in, int64_t out_cap) {
    const int64_t nt = (in->n + OBE_TILE - 1) / OBE_TILE;
    const int chunk = plan_chunk(out_cap);
    return nt + (out_cap + chunk - 1) / chunk <= nt + in->n / OBE_WR_MIN_CHUNK + 4;
}

// ---- early select: plan now, pick the K draws, stream the cloud later -------------------------------------
// obe_resample_defer(1) arms the calling thread: its next systematic resample call (whole cloud, sharded or planned)
// launches only the plan kernel and PARKS the streaming kernel's arguments; obe_resample_pick() then produces the K
// parameter draws of the design half straight from the plan (k_sys_resample_warp<D, true>), and obe_resample_emit()
// launches the parked streaming kernel.  The caller may put the pick + utility pass and the emission on different
// streams (obe_stream_fork / obe_stream_join), which hides the whole selection behind the resample.
struct ObeParked {
    bool armed, parked;
    ObeResampleArgs a;
    int d, grid;
    unsigned int* counter;
};
static thread_local ObeParked g_parked = {};

// k_sys_ancestors + k_sys_move, after k_sys_plan
static int launch_sys_resample(const obe_cloud_t* in, const obe_cloud_t* out, ObeResampleArgs& a, int64_t out_cap,
                               cudaStream_t st) {
    const int64_t max_units = a.n_tiles + (out_cap + a.chunk - 1) / a.chunk;
    if (in->n >= (1ll << 32)) return obe_fail("systematic resample supports shards of < 2^32 particles%s%s");
    a.anc = scratch_of(out).anc;
    a.out_tile_sums = out->tile_sums_dev; a.out_prefix = out->tile_prefix_dev; a.out_stats = out->stats_dev;
    a.unit_counter = g_resample_dynamic ? scratch_of(in).counter + 18 : nullptr;
    if (g_resample_fused) {
        // one kernel: every warp owns work units from the weights to the stores (+ the bookkeeping block)
        const int per_sm = (g_resample_blocks > 0 && g_resample_blocks < OBE_WR_BLOCKS(in->d)) ? (int)g_resample_blocks
                                                                                              : OBE_WR_BLOCKS(in->d);
        int64_t g = (int64_t)obe_sms() * per_sm - 1;          // workers; + the bookkeeping block = one full wave
        const int64_t need = (max_units + OBE_THREADS / 32 - 1) / (OBE_THREADS / 32);
        if (g > need) g = need;
        if (g < 1) g = 1;
        const int grid = (int)g + 1;
        if (g_parked.armed) {                                  // early select: the emission waits for obe_resample_emit
            g_parked.armed = false; g_parked.parked = true;
            g_parked.a = a; g_parked.d = in->d; g_parked.grid = grid;
            g_parked.counter = scratch_of(in).counter + 17;
            return 0;
        }
        OBE_DIM_SWITCH_WR(in->d, grid, st, a)
        OBE_LAUNCH_CHECK("k_sys_resample_warp");
        return 0;
    }
    if (g_parked.armed) { g_parked.armed = false; return obe_fail("deferred emission needs the one-kernel resample (resample_fused=1)%s%s"); }
    {
        int64_t g = (int64_t)obe_sms() * OBE_ANC_BLOCKS_PER_SM;
        if (g > max_units) g = max_units;
        k_sys_ancestors<<<(int)g + 1, OBE_THREADS, 0, st>>>(a);    // + the bookkeeping block
        OBE_LAUNCH_CHECK("k_sys_ancestors");
    }
    {
        int64_t g = (out_cap + 3 + (int64_t)OBE_THREADS * OBE_MOVE_V - 1) / ((int64_t)OBE_THREADS * OBE_MOVE_V);
        const int64_t gmax = (int64_t)obe_sms() * OBE_MOVE_BLOCKS(in->d) * 4;
        if (g > gmax) g = gmax;
        if (g < 1) g = 1;
        const int grid = (int)g;
        OBE_DIM_SWITCH_PLAIN(in->d, k_sys_move, grid, st, a)
        OBE_LAUNCH_CHECK("k_sys_move");
    }
    return 0;
}

static int resample_systematic_impl(const obe_cloud_t* in, const obe_cloud_t* out, double u0, const double* factor,
                                    const double* mean, uint64_t seed, uint32_t epoch, double a_param, int scale,
                                    int64_t* idx_out_dev, double* z_out_dev, int sharded, int64_t n_total,
                                    int64_t slot_begin, int64_t slot_end, double cdf_offset, double cdf_total,
                                    int last_shard, void* stream) {
    ObeResampleArgs a;
    if (fill_resample_args(in, out, factor, mean, a_param, scale, seed, epoch, a)) return -1;
    if (!(u0 >= 0.0 && u0 < 1.0)) return obe_fail("u0 must be in [0,1)%s%s");
    if (n_total >= (1ll << 31)) return obe_fail("systematic resample supports n < 2^31%s%s");
    if (out->n != slot_end - slot_begin) return obe_fail("resample: out->n must equal the number of output slots%s%s");
    if (sharded && !factor) return obe_fail("sharded resample needs the (global) factor from the host%s%s");
    const Scratch s = scratch_of(in);
    a.plan_h = s.plan_h; a.unit_start = s.unit_start; a.u0 = u0;
    a.unit_tile = unit_map_fits(in, out->n) ? s.unit_tile : nullptr;
    a.idx_out = (long long*)idx_out_dev; a.z_out = z_out_dev; a.implicit_out = 1;
    a.sharded = sharded; a.last_shard = last_shard; a.n_total = n_total;
    a.slot_begin = slot_begin; a.slot_end = slot_end; a.cdf_offset = cdf_offset; a.cdf_total = cdf_total;
    cudaStream_t st = (cudaStream_t)stream;
    a.chunk = plan_chunk(out->n);
    if (a.n_tiles > g_plan_cluster_min_tiles)
        launch_pdl(k_sys_plan_cluster, dim3(OBE_PLAN_CLUSTER), dim3(OBE_SCAN_THREADS), 0, st,
                   (const double*)in->tile_prefix_dev, (long long)a.n_tiles, (long long)n_total, u0,
                   sharded ? cdf_offset : 0.0, sharded ? cdf_total : 0.0, (long long)slot_begin, (long long)slot_end,
                   s.plan_h, s.unit_start, (int*)a.unit_tile, (const long long*)nullptr, (const double*)nullptr, a.chunk,
                   s.counter + 18, g_gate_on);
    else
        launch_pdl(k_sys_plan, dim3(1), dim3(OBE_SCAN_THREADS), 0, st, (const double*)in->tile_prefix_dev,
                   (long long)a.n_tiles, (long long)n_total, u0, sharded ? cdf_offset : 0.0, sharded ? cdf_total : 0.0,
                   (long long)slot_begin, (long long)slot_end, s.plan_h, s.unit_start, (int*)a.unit_tile,
                   (const long long*)nullptr, (const double*)nullptr, a.chunk, s.counter + 18, g_gate_on);
    OBE_LAUNCH_CHECK("k_sys_plan");
    return launch_sys_resample(in, out, a, out->n, st);
}

int obe_resample_systematic(const obe_cloud_t* in, const obe_cloud_t* out, double u0, const double* factor,
                            const double* mean, uint64_t seed, uint32_t epoch, double a_param, int scale,
                            int64_t* idx_out_dev, double* z_out_dev, void* stream) {
    if (!in) return obe_fail("null cloud%s%s");
    return resample_systematic_impl(in, out, u0, factor, mean, seed, epoch, a_param, scale, idx_out_dev, z_out_dev, 0,
                                    in->n, 0, in->n, 0.0, 0.0, 1, stream);
}

int obe_resample_systematic_sharded(const obe_cloud_t* in, const obe_cloud_t* out, double u0, int64_t n_total,
                                    int64_t slot_begin, int64_t slot_end, double cdf_offset, double cdf_total,
                                    int last_shard, const double* factor, const double* mean, uint64_t seed,
                                    uint32_t epoch, double a_param, int scale, int64_t* idx_out_dev, double* z_out_dev,
                                    void* stream) {
    if (!in) return obe_fail("null cloud%s%s");
    if (slot_begin < 0 || slot_end <= slot_begin || slot_end > n_total) return obe_fail("bad slot range%s%s");
    return resample_systematic_impl(in, out, u0, factor, mean, seed, epoch, a_param, scale, idx_out_dev, z_out_dev, 1,
                                    n_total, slot_begin, slot_end, cdf_offset, cdf_total, last_shard, stream);
}

// ---- peer exchange (CUDA IPC) -----------------------------------------------------------------
size_t obe_peer_bytes(void) { return (size_t)OBE_PEER_WORDS * 8; }

int obe_peer_alloc(void** dev_ptr, unsigned char* handle64) {
    if (!dev_ptr || !handle64) return obe_fail("null argument%s%s");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void* p = nullptr;
    OBE_CUDA(cudaMalloc(&p, obe_peer_bytes()));
    OBE_CUDA(cudaMemset(p, 0, obe_peer_bytes()));
    OBE_CUDA(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return obe_fail("cudaIpcGetMemHandle: %s%s", cudaGetErrorString(e)); }
    memcpy(handle64, &h, 64);
    *dev_ptr = p;
    return 0;
}
int obe_peer_open(const unsigned char* handle64, void** dev_ptr) {
    if (!dev_ptr || !handle64) return obe_fail("null argument%s%s");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    OBE_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
int obe_peer_close(void* dev_ptr) {
    if (dev_ptr) OBE_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return 0;
}
int obe_peer_free(void* dev_ptr) {
    if (dev_ptr) OBE_CUDA(cudaFree(dev_ptr));
    return 0;
}
static int fill_peers(void* const* peer_bufs, int rank, int world, ObePeers& pp) {
    if (!peer_bufs) return obe_fail("null peer buffers%s%s");
    if (world < 1 || world > OBE_PEER_MAX || rank < 0 || rank >= world) return obe_fail("peer exchange: 1..16 ranks%s%s");
    memset(&pp, 0, sizeof(pp));
    for (int g = 0; g < world; ++g) {
        if (!peer_bufs[g]) return obe_fail("null peer buffer%s%s");
        pp.p[g] = (double*)peer_bufs[g];
    }
    return 0;
}

int obe_shard_plan_peer(void* const* peer_bufs, int rank, int world, uint64_t epoch, int d, double u0, int64_t n_total,
                        double a_param, int lazy, const obe_cloud_t* local, const obe_cloud_t* out, double* plan_dev,
                        void* stream) {
    if (!plan_dev || !local) return obe_fail("null argument%s%s");
    if (d < 1 || d > OBE_MAX_DIMS) return obe_fail("n_params must be 1..8%s%s");
    if (epoch == 0) return obe_fail("peer exchange epochs start at 1%s%s");
    ObePeers pp;
    if (fill_peers(peer_bufs, rank, world, pp)) return -1;
    launch_pdl(k_shard_plan_peer, dim3(1), dim3(OBE_STATS_LEN), 0, (cudaStream_t)stream, pp, rank, world,
               (unsigned long long)epoch, d, u0, (long long)n_total, a_param, lazy, out ? (long long)out->ld : (1ll << 62),
               plan_dev, local->stats_dev, out ? (long long*)out->n_dev : (long long*)nullptr);
    OBE_LAUNCH_CHECK("k_shard_plan_peer");
    return 0;
}

int obe_draw_planned_peer(const obe_cloud_t* c, const double* u_host, int k, void* const* peer_bufs, int rank, int world,
                          uint64_t epoch, const double* plan_dev, int post, double* draws_dev, void* stream) {
    if (check_cloud(c)) return -1;
    if (!u_host || !draws_dev || !plan_dev) return obe_fail("null argument%s%s");
    if (k < 1 || k > OBE_MAX_DRAWS || (int64_t)k * c->d > 1024) return obe_fail("peer draws: n_draws * n_params <= 1024%s%s");
    if (epoch == 0) return obe_fail("peer exchange epochs start at 1%s%s");
    ObePeers pp;
    if (fill_peers(peer_bufs, rank, world, pp)) return -1;
    const Scratch s = scratch_of(c);
    ObePeerDraw pd = {&pp, rank, world, epoch, s.counter + 16};
    cudaStream_t st = (cudaStream_t)stream;
    if (draw_impl(c->weights_dev, c->tile_prefix_dev, c->n, c->particles_dev, c->ld, c->d, u_host, k, nullptr, nullptr, st, 0,
                  (const long long*)c->n_dev, plan_dev, post, c->stats_dev, &pd))
        return -1;
    k_peer_collect_draws<<<1, 128, 0, st>>>(pp.p[rank], world, epoch, draws_dev, k * c->d);
    OBE_LAUNCH_CHECK("k_peer_collect_draws");
    return 0;
}

int obe_shard_plan(const double* gathered_stats_dev, int rank, int world, int d, double u0, int64_t n_total,
                   double a_param, int lazy, const obe_cloud_t* local, const obe_cloud_t* out, double* plan_dev,
                   void* stream) {
    if (!gathered_stats_dev || !plan_dev || !local) return obe_fail("null argument%s%s");
    if (world < 1 || world > OBE_MAX_SHARDS || rank < 0 || rank >= world) return obe_fail("bad rank/world%s%s");
    if (d < 1 || d > OBE_MAX_DIMS) return obe_fail("n_params must be 1..8%s%s");
    k_shard_plan<<<1, OBE_STATS_LEN, 0, (cudaStream_t)stream>>>(gathered_stats_dev, rank, world, d, u0, n_total, a_param, lazy,
                                                    out ? out->ld : (1ll << 62), plan_dev, local->stats_dev,
                                                    out ? (long long*)out->n_dev : nullptr);
    OBE_LAUNCH_CHECK("k_shard_plan");
    return 0;
}

int obe_resample_systematic_planned(const obe_cloud_t* in, const obe_cloud_t* out, const double* plan_dev,
                                    int64_t n_total, uint64_t seed, uint32_t epoch, double a_param, int scale,
                                    void* stream) {
    if (!plan_dev) return obe_fail("null plan%s%s");
    if (!out || !out->n_dev) return obe_fail("planned resample needs out->n_dev%s%s");
    ObeResampleArgs a;
    double dummy[OBE_MAX_DIMS * OBE_MAX_DIMS] = {0};
    if (fill_resample_args(in, out, dummy, dummy, a_param, scale, seed, epoch, a)) return -1;
    const Scratch s = scratch_of(in);
    a.plan_h = s.plan_h; a.unit_start = s.unit_start;
    a.unit_tile = unit_map_fits(in, out->ld) ? s.unit_tile : nullptr;
    a.plan = plan_dev; a.n_dev_in = (const long long*)in->n_dev; a.cap_out = out->ld;
    a.sharded = 1; a.n_total = n_total; a.implicit_out = 1;
    cudaStream_t st = (cudaStream_t)stream;
    a.chunk = plan_chunk(out->ld);
    if (a.n_tiles > g_plan_cluster_min_tiles)
        launch_pdl(k_sys_plan_cluster, dim3(OBE_PLAN_CLUSTER), dim3(OBE_SCAN_THREADS), 0, st,
                   (const double*)in->tile_prefix_dev, (long long)a.n_tiles, (long long)n_total, 0.0, 0.0, 1.0, 0ll, 0ll,
                   s.plan_h, s.unit_start, (int*)a.unit_tile, (const long long*)in->n_dev, plan_dev, a.chunk,
                   s.counter + 18, (const double*)nullptr);
    else
        launch_pdl(k_sys_plan, dim3(1), dim3(OBE_SCAN_THREADS), 0, st, (const double*)in->tile_prefix_dev,
                   (long long)a.n_tiles, (long long)n_total, 0.0, 0.0, 1.0, 0ll, 0ll, s.plan_h, s.unit_start,
                   (int*)a.unit_tile, (const long long*)in->n_dev, plan_dev, a.chunk, s.counter + 18,
                   (const double*)nullptr);
    OBE_LAUNCH_CHECK("k_sys_plan");
    return launch_sys_resample(in, out, a, out->ld, st);
}

int obe_resample_defer(int on) {
    g_parked.armed = on != 0;
    if (!on) g_parked.parked = false;
    return 0;
}

#define OBE_DIM_CASE_PICK(dd) \
    case dd: launch_pdl(k_sys_pick<dd>, dim3(grid), dim3(OBE_PICK_WARPS * 32), 0, st, g_parked.a, pk); break;

int obe_resample_pick(const double* u_host, int k, double* draws_dev, void* const* peer_bufs, int rank, int world,
                      uint64_t epoch, void* stream) {
    if (!g_parked.parked) return obe_fail("obe_resample_pick: no parked resample (obe_resample_defer + a systematic resample first)%s%s");
    if (!u_host || k < 1 || k > OBE_MAX_DRAWS) return obe_fail("obe_resample_pick: 1..128 draws%s%s");
    ObePickArgs pk;
    memset(&pk, 0, sizeof(pk));
    pk.k = k; pk.ldk = k; pk.out = draws_dev;
    if (peer_bufs) {
        if ((int64_t)k * g_parked.d > 1024) return obe_fail("peer draws: n_draws * n_params <= 1024%s%s");
        if (epoch == 0) return obe_fail("peer exchange epochs start at 1%s%s");
        if (fill_peers(peer_bufs, rank, world, pk.peers)) return -1;
        pk.peer_world = world; pk.peer_rank = rank; pk.peer_epoch = epoch; pk.peer_counter = g_parked.counter;
    } else if (!draws_dev) {
        return obe_fail("null argument%s%s");
    }
    for (int i = 0; i < k; ++i) pk.u[i] = u_host[i];
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (k + OBE_PICK_WARPS - 1) / OBE_PICK_WARPS;
    switch (g_parked.d) {
        OBE_DIM_CASE_PICK(1) OBE_DIM_CASE_PICK(2) OBE_DIM_CASE_PICK(3) OBE_DIM_CASE_PICK(4)
        OBE_DIM_CASE_PICK(5) OBE_DIM_CASE_PICK(6) OBE_DIM_CASE_PICK(7) OBE_DIM_CASE_PICK(8)
        default: return obe_fail("n_params must be 1..8%s%s");
    }
    OBE_LAUNCH_CHECK("k_sys_pick");
    if (peer_bufs && draws_dev) {
        k_peer_collect_draws<<<1, 128, 0, st>>>(pk.peers.p[rank], world, epoch, draws_dev, k * g_parked.d);
        OBE_LAUNCH_CHECK("k_peer_collect_draws");
    }
    return 0;
}

int obe_resample_emit(void* stream) {
    if (!g_parked.parked) return obe_fail("obe_resample_emit: no parked resample%s%s");
    g_parked.parked = false;
    cudaStream_t st = (cudaStream_t)stream;
    // The streaming kernel is persistent and fills every CTA slot of the machine; the selection kernels of the other
    // stream get in while it ramps up (pick) and as soon as its first CTAs run out of units (utility) -- the units are
    // handed out dynamically, so CTAs retire one by one over the last ~30 us instead of all at once.  Leaving slots
    // free from the start (resample_reserve_ctas > 0) was measured and costs more than it hides: 0 / 24 / 48 slots ->
    // 1.611 / 1.629 / 1.648 ms per cycle at 1e8 particles, 0.2783 / 0.2789 / 0.2800 ms at 1.25e7.
    int grid = g_parked.grid;
    if (grid == obe_sms() * OBE_WR_BLOCKS(g_parked.d)) grid -= (int)g_resample_reserve;
    if (grid < 2) grid = 2;
    OBE_DIM_SWITCH_WR(g_parked.d, grid, st, g_parked.a)
    OBE_LAUNCH_CHECK("k_sys_resample_warp");
    return 0;
}

// `to` waits for everything enqueued on `from` so far (one cached event per thread and direction)
static thread_local cudaEvent_t g_fork_ev[2] = {nullptr, nullptr};
static int stream_edge(int which, void* from, void* to) {
    if (!g_fork_ev[which]) OBE_CUDA(cudaEventCreateWithFlags(&g_fork_ev[which], cudaEventDisableTiming));
    OBE_CUDA(cudaEventRecord(g_fork_ev[which], (cudaStream_t)from));
    OBE_CUDA(cudaStreamWaitEvent((cudaStream_t)to, g_fork_ev[which], 0));
    return 0;
}
int obe_stream_fork(void* main_stream, void* side_stream) { return stream_edge(0, main_stream, side_stream); }
int obe_stream_join(void* main_stream, void* side_stream) { return stream_edge(1, side_stream, main_stream); }

int obe_stream_sync(void* stream) {
    OBE_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

// the results a closed loop waits for, copied into the caller's pinned host blocks behind the cycle's kernels
// device-side address of a pinned host block (identical under UVA; cached per block), NULL if it is not device-visible
static void* device_view(void* host) {
    static thread_local void* seen_host[4] = {nullptr, nullptr, nullptr, nullptr};
    static thread_local void* seen_dev[4] = {nullptr, nullptr, nullptr, nullptr};
    static thread_local int next = 0;
    if (!host || !g_zero_copy_out) return nullptr;
    for (int i = 0; i < 4; ++i)
        if (seen_host[i] == host) return seen_dev[i];
    void* dev = nullptr;
    if (cudaHostGetDevicePointer(&dev, host, 0) != cudaSuccess) { (void)cudaGetLastError(); dev = nullptr; }
    seen_host[next] = host; seen_dev[next] = dev;
    next = (next + 1) & 3;
    return dev;
}
struct CycleZeroCopy { double* stats; long long* best; unsigned long long* seq; };
static CycleZeroCopy cycle_zero_copy(const obe_cycle_t* c) {
    CycleZeroCopy z = {nullptr, nullptr, nullptr};
    // the update's own stats block only: a sharded cycle wants the COMBINED block of the plan (stats_src_dev)
    if (c->stats_host && !c->stats_src_dev) z.stats = (double*)device_view(c->stats_host);
    if (c->best_host && c->select) z.best = (long long*)device_view(c->best_host);
    if (z.best && c->seq_host) z.seq = (unsigned long long*)device_view(c->seq_host);
    return z;
}
static int cycle_copy_out(const obe_cycle_t* c, const obe_cloud_t* updated, void* stream, const CycleZeroCopy& z,
                          int what = 3) {
    cudaStream_t st = (cudaStream_t)stream;
    if ((what & 1) && c->best_host && c->select && !z.best)
        OBE_CUDA(cudaMemcpyAsync(c->best_host, c->best_dev, 16, cudaMemcpyDeviceToHost, st));
    if ((what & 2) && c->stats_host && !z.stats)
        OBE_CUDA(cudaMemcpyAsync(c->stats_host, c->stats_src_dev ? c->stats_src_dev : updated->stats_dev,
                                 OBE_STATS_LEN * sizeof(double), cudaMemcpyDeviceToHost, st));
    return 0;
}

// resample == 2: the resample test runs on the device.  The update's finishing block writes stats[FIRED]; plan, pick
// and the streaming resample are launched gated on it, the plain K-draw kernel gated on its complement, and the
// utility pass reads whichever draws were produced -- one stream, no host decision, the caller learns the outcome
// from stats_host[OBE_ST_FIRED] when it synchronises for the argmax (and swaps cloud / alt if it fired).
static int cycle_auto(const obe_cycle_t* c) {
    void* st = c->stream;
    const obe_cloud_t* live = c->cloud;
    if (c->plan_dev) return obe_fail("obe_cycle: the device-side resample test is for a whole (unsharded) cloud%s%s");
    if (c->phase != 1) {            // (phase 1 launches the update alone: the rest of the struct is filled in afterwards)
        if (!c->alt) return obe_fail("obe_cycle: resample needs the second buffer%s%s");
        if (!c->select || (c->mask_le | c->mask_lt) != 0u || c->noise_from_stats || c->method == 3 || c->k < 1 ||
            c->k > OBE_MAX_DRAWS || !g_resample_fused)
            return obe_fail("obe_cycle: resample == 2 needs select, no constraint masks, var_noise by value, a "
                            "variance/entropy utility, 1..128 draws and the one-kernel resample%s%s");
    }
    if (!(c->resample_threshold >= 0.0)) return obe_fail("obe_cycle: bad resample_threshold%s%s");
    const CycleZeroCopy z = cycle_zero_copy(c);
    if (c->phase != 2) {
        g_update_gate_thr = c->resample_threshold; g_update_gate_n = (double)live->n;
        g_update_stats_out = z.stats;
        const int rc_u = obe_update(c->model, live, c->setting, c->constants, c->y_meas, c->has_sigma ? c->sigma : nullptr,
                                    c->has_noise_index ? c->noise_index : nullptr, c->n_lik_channels, c->use_choke,
                                    c->choke, c->pivot, st);
        g_update_gate_thr = 0.0; g_update_gate_n = 0.0;
        g_update_stats_out = nullptr;
        if (rc_u) return -1;
        if (c->phase == 1) return 0;
    }
    const double* fired = live->stats_dev + OBE_ST_FIRED;
    g_gate_on = fired;
    obe_resample_defer(1);
    int rc = obe_resample_systematic(live, c->alt, c->u0, nullptr, nullptr, c->seed, c->epoch, c->a_param, c->scale, nullptr,
                                     nullptr, st);
    if (!rc) rc = obe_resample_pick(c->u, c->k, c->draws_dev, nullptr, 0, 1, 0, st);
    g_gate_on = nullptr;
    if (rc) { obe_resample_defer(0); return -1; }
    g_gate_off = fired;
    rc = obe_draw(live, c->u, c->k, c->draws_dev, nullptr, st);
    g_gate_off = nullptr;
    if (rc) { obe_resample_defer(0); return -1; }
    g_utility_best_out = z.best; g_utility_seq_out = z.seq; g_utility_seq_val = c->seq;
    const int rc_s = obe_utility(c->model, c->draws_dev, c->k, c->settings_dev, c->lds, c->n_settings, c->constants,
                                 c->var_noise, nullptr, c->cost_dev, c->method, c->log_form, c->kld_noise_dev, c->utility_dev,
                                 c->best_dev, c->select_scratch_dev, st);
    g_utility_best_out = nullptr; g_utility_seq_out = nullptr;
    if (rc_s) {
        obe_resample_defer(0);
        return -1;
    }
    if (obe_resample_emit(st)) return -1;
    return cycle_copy_out(c, live, st, z);
}

static int cycle_body(const obe_cycle_t* c, bool& copied, const CycleZeroCopy& z);
int obe_cycle(const obe_cycle_t* c) {
    if (!c || !c->cloud || !c->model) return obe_fail("obe_cycle: null argument%s%s");
    if (c->resample == 2) return cycle_auto(c);
    const CycleZeroCopy z = cycle_zero_copy(c);
    bool copied = false;
    g_utility_best_out = z.best;                 // (every path through cycle_body runs obe_utility at most once)
    g_utility_seq_out = z.seq; g_utility_seq_val = c->seq;
    const int rc = cycle_body(c, copied, z);
    g_utility_best_out = nullptr; g_utility_seq_out = nullptr;
    g_update_stats_out = nullptr;
    if (rc) return -1;
    return copied ? 0 : cycle_copy_out(c, c->cloud, c->stream, z);
}

static int cycle_body(const obe_cycle_t* c, bool& copied, const CycleZeroCopy& z) {
    void* st = c->stream;
    const obe_cloud_t* live = c->cloud;
    const int sharded = c->plan_dev != nullptr;
    if (sharded && !c->peer_bufs) return obe_fail("obe_cycle: a sharded cycle needs the peer exchange%s%s");
    if (c->phase != 2) {
        g_update_stats_out = z.stats;
        const int rc_u = obe_update(c->model, live, c->setting, c->constants, c->y_meas, c->has_sigma ? c->sigma : nullptr,
                                    c->has_noise_index ? c->noise_index : nullptr, c->n_lik_channels, c->use_choke,
                                    c->choke, c->pivot, st);
        g_update_stats_out = nullptr;          // (a constraint refresh further down must not overwrite the block)
        if (rc_u) return -1;
        if (c->phase == 1) { copied = true; return 0; }     // (nothing to copy out yet)
    }
    if (sharded &&
        obe_shard_plan_peer(c->peer_bufs, c->rank, c->world, c->epoch_stats, live->d, c->u0, c->n_total, c->a_param, 1,
                            live, c->alt, c->plan_dev, st))
        return -1;
    const bool masks = (c->mask_le | c->mask_lt) != 0u;
    const bool early = c->resample && c->select && !masks && !c->noise_from_stats && c->side_stream && c->method != 3 &&
                       c->k >= 1 && c->k <= OBE_MAX_DRAWS && g_resample_fused;
    const double* stats_for_utility = nullptr;
    if (c->resample) {
        if (!c->alt) return obe_fail("obe_cycle: resample needs the second buffer%s%s");
        if (early) obe_resample_defer(1);
        const int rc = sharded ? obe_resample_systematic_planned(live, c->alt, c->plan_dev, c->n_total, c->seed, c->epoch,
                                                                 c->a_param, c->scale, st)
                               : obe_resample_systematic(live, c->alt, c->u0, nullptr, nullptr, c->seed, c->epoch,
                                                         c->a_param, c->scale, nullptr, nullptr, st);
        if (rc) { obe_resample_defer(0); return -1; }
        if (early) {
            // side_stream == stream: the early order (plan, pick, utility, then the streaming kernel) on ONE stream --
            // for small clouds the fork / join events cost more than the overlap hides
            void* side = c->side_stream;
            const bool two_streams = side != st;
            if (two_streams && obe_stream_fork(st, side)) return -1;
            // a stats block that has to be COPIED (sharded: the combined block of the plan) goes first on the selection
            // stream, so that it has landed when the utility kernel raises the completion word
            if (g_copy_out_side && cycle_copy_out(c, c->cloud, side, z, 2)) return -1;
            if (obe_resample_pick(c->u, c->k, c->draws_dev, sharded ? c->peer_bufs : nullptr, c->rank, c->world,
                                  c->epoch_draws, side))
                return -1;
            if (obe_utility(c->model, c->draws_dev, c->k, c->settings_dev, c->lds, c->n_settings, c->constants,
                            c->var_noise, nullptr, c->cost_dev, c->method, c->log_form, c->kld_noise_dev, c->utility_dev,
                            c->best_dev, c->select_scratch_dev, side))
                return -1;
            // the copies a closed loop waits for ride the selection stream: they are done long before the streaming
            // kernel, so nothing trails it but the join (the stats block is final since the update / shard plan)
            if (g_copy_out_side) {
                if (cycle_copy_out(c, c->cloud, side, z, 1)) return -1;
                copied = true;
            }
            if (obe_resample_emit(st)) return -1;
            return two_streams ? obe_stream_join(st, side) : 0;
        }
        live = c->alt;
        if (masks) {
            if (sharded) return obe_fail("obe_cycle: constraint masks on a sharded cloud need a re-plan (not supported here)%s%s");
            if (obe_refresh(live, c->mask_le, c->mask_lt, c->n_noise > 0 ? c->noise_index : nullptr, c->n_noise, c->pivot, 1, st))
                return -1;
        }
    }
    if (!c->select) return 0;
    if (c->noise_from_stats) stats_for_utility = live->stats_dev;
    if (sharded) {
        if (obe_draw_planned_peer(live, c->u, c->k, c->peer_bufs, c->rank, c->world, c->epoch_draws, c->plan_dev,
                                  c->resample ? 1 : 0, c->draws_dev, st))
            return -1;
    } else if (obe_draw(live, c->u, c->k, c->draws_dev, nullptr, st)) {
        return -1;
    }
    return obe_utility(c->model, c->draws_dev, c->k, c->settings_dev, c->lds, c->n_settings, c->constants,
                       c->noise_from_stats ? nullptr : c->var_noise, stats_for_utility, c->cost_dev, c->method, c->log_form,
                       c->kld_noise_dev, c->utility_dev, c->best_dev, c->select_scratch_dev, st);
}

int64_t obe_comb_count(double c, double u0, int64_t n_total) {
    // host twin of the device comb count: #{i in [0,n) : (i + u0) * (1/n) < c}, same IEEE operations
    const double nd = (double)n_total, inv_n = 1.0 / nd;
    double i = ceil(c * nd - u0);
    i = (i < 0.0) ? 0.0 : i;
    i = (i > nd) ? nd : i;
    volatile double t;
    while (i > 0.0) { t = (i - 1.0) + u0; t = t * inv_n; if (t >= c) i -= 1.0; else break; }
    while (i < nd) { t = i + u0; t = t * inv_n; if (t < c) i += 1.0; else break; }
    return (int64_t)i;
}

struct SelectScratch {
    unsigned int* counter; double* part_val; long long* part_idx; double* p; double* tile_sums; double* prefix;
};
static SelectScratch select_scratch_of(void* base, int64_t n_settings) {
    const int64_t nt = (n_settings + OBE_TILE - 1) / OBE_TILE;
    char* p = (char*)base;
    SelectScratch s;
    s.counter = (unsigned int*)p; p += 256;
    s.part_val = (double*)p; p += align_up((size_t)OBE_MAX_GRID * sizeof(double), 256);
    s.part_idx = (long long*)p; p += align_up((size_t)OBE_MAX_GRID * sizeof(long long), 256);
    s.p = (double*)p; p += align_up((size_t)n_settings * sizeof(double), 256);
    s.tile_sums = (double*)p; p += align_up((size_t)nt * sizeof(double), 256);
    s.prefix = (double*)p;
    return s;
}

int obe_utility(obe_model_t m, const double* draws_dev, int k, const double* settings_dev, int64_t lds,
                int64_t n_settings, const double* constants, const double* var_noise, const double* stats_dev,
                const double* cost_dev, int method, int log_form, const double* kld_noise_dev, double* utility_dev,
                void* best_dev, void* select_scratch_dev, void* stream) {
    if (!m || !draws_dev || !settings_dev || !utility_dev || !best_dev || !select_scratch_dev)
        return obe_fail("null argument%s%s");
    if (method < 0 || method > 4) return obe_fail("unknown utility method%s%s");
    if (method == 4) {
        if (!m->design || !m->f_utility_info)
            return obe_fail("information gain utility: needs the likelihood-aware design handle of a Poisson or "
                            "binomial likelihood%s%s");
        if (m->nch != 1) return obe_fail("information gain utility: single-channel models only%s%s");
        if (k < 1 || k > OBE_MAX_DRAWS) return obe_fail("information gain utility: 1 <= n_draws <= 128%s%s");
        if (!var_noise) return obe_fail("information gain utility: needs the design aux in var_noise%s%s");
        if (m->lik == OBE_LIK_BINOMIAL && !(var_noise[0] >= 1.0 && var_noise[0] <= 9007199254740992.0 &&
                                            var_noise[0] == floor(var_noise[0]))) {
            char got[64];
            snprintf(got, sizeof(got), "%.17g", var_noise[0]);
            return obe_fail("information gain utility: the binomial trial count (design aux) must be an integer "
                            ">= 1, got %s%s", got);
        }
    }
    if ((method == 2 || method == 3) && (k < 3 || k > OBE_MAX_DRAWS))
        return obe_fail("entropy utilities need 3 <= n_draws <= 128%s%s");
    if (method == 3 && (!kld_noise_dev || m->nch != 1)) return obe_fail("full KLD utility: single-channel models, noise required%s%s");
    if (method == 3 && m->design)
        return obe_fail("full KLD utility: its noise samples are Gaussian; a likelihood-aware design handle has none%s%s");
    if (m->design && !var_noise) return obe_fail("a likelihood-aware design handle needs the design aux in var_noise%s%s");
    if (!var_noise && !stats_dev) return obe_fail("need var_noise or stats%s%s");
    if (k < 1) return obe_fail("n_draws must be >= 1%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    const SelectScratch s = select_scratch_of(select_scratch_dev, n_settings);
    ObeUtilityArgs a;
    memset(&a, 0, sizeof(a));
    a.draws = draws_dev; a.k = k; a.settings = settings_dev; a.lds = lds; a.n_settings = n_settings;
    a.cost = cost_dev; a.stats = stats_dev; a.utility = utility_dev;
    a.part_val = s.part_val; a.part_idx = s.part_idx; a.counter = s.counter;
    a.best_idx = (long long*)best_dev; a.best_val = (double*)((char*)best_dev + 8);
    a.noise_from_stats = var_noise ? 0 : 1;
    a.log_form = log_form; a.method = method; a.kld_noise = kld_noise_dev;
    a.best_out2 = g_utility_best_out;
    a.seq_out2 = g_utility_best_out ? g_utility_seq_out : nullptr; a.seq_val = g_utility_seq_val;
    if (var_noise) for (int c = 0; c < m->nch; ++c) a.var_noise[c] = var_noise[c];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    size_t smem = (size_t)k * (m->np_model > 0 ? m->np_model : 1) * sizeof(double);
    if (smem > 48 * 1024) return obe_fail("n_draws too large for shared memory%s%s");
    if (method == 4) {
        // one warp per setting, OBE_INFO_ARRAYS x K doubles of shared memory per warp beside the draws
        smem += (size_t)(OBE_THREADS / 32) * OBE_INFO_ARRAYS * k * sizeof(double);
        cudaError_t e = set_max_smem(m->f_utility_info, smem);
        if (e != cudaSuccess) return obe_fail("cudaFuncSetAttribute(max dynamic smem): %s%s", cudaGetErrorString(e));
        const int64_t per_block = OBE_THREADS / 32;
        int64_t blocks = (n_settings + per_block - 1) / per_block;
        if (blocks > (int64_t)obe_sms() * 8) blocks = (int64_t)obe_sms() * 8;
        if (g_utility_info_blocks > 0 && blocks > g_utility_info_blocks) blocks = g_utility_info_blocks;
        return launch_kernel(m->f_utility_info, (int)blocks, smem, (cudaStream_t)stream, &a, true);
    }
    // variance utility: several lanes per setting while the grid is too small to fill the GPU anyway (the
    // one-thread-per-setting walk is pure latency there; on a large grid the idle lanes of the sequential sums
    // would cost throughput: 1e5 settings take 42 us with one lane, 60 us with eight) and the K curves of a
    // CTA's settings fit in shared memory
    a.lanes = 1;
    const int64_t resident = (int64_t)obe_sms() * 8 * OBE_THREADS;
    for (int lanes = 8; lanes >= 2 && method == 0 && k >= 8; lanes >>= 1) {
        const size_t split = smem + (size_t)(OBE_THREADS / lanes) * m->nch * k * sizeof(double);
        if (n_settings * lanes <= resident * g_utility_lane_fill / 100 && split <= 48 * 1024) { a.lanes = lanes; smem = split; break; }
    }
    const int64_t per_block = OBE_THREADS / a.lanes;
    int64_t blocks = (n_settings + per_block - 1) / per_block;
    if (blocks > (int64_t)obe_sms() * 8) blocks = (int64_t)obe_sms() * 8;
    if (a.lanes == 1 && method == 0 && g_utility_cache) {
        // one thread per setting: park the K x NCH model values in shared memory between the two variance passes
        const size_t with_cache = smem + (size_t)k * m->nch * OBE_THREADS * sizeof(double);
        if (with_cache <= 100 * 1024) {
            if (with_cache > 48 * 1024) {
                cudaError_t e = set_max_smem(m->f_utility, with_cache);
                if (e != cudaSuccess) { (void)cudaGetLastError(); } else { a.cache = 1; smem = with_cache; }
            } else { a.cache = 1; smem = with_cache; }
        }
    }
    return launch_kernel(m->f_utility, (int)blocks, smem, (cudaStream_t)stream, &a, true);
}

int obe_pick(const double* utility_dev, int64_t n_settings, double pickiness, double u, int64_t* idx_dev,
             void* select_scratch_dev, void* stream) {
    if (!utility_dev || !idx_dev || !select_scratch_dev) return obe_fail("null argument%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    const SelectScratch s = select_scratch_of(select_scratch_dev, n_settings);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nt = obe_num_tiles(n_settings);
    int grid = (int)(nt < (int64_t)obe_sms() * 4 ? nt : (int64_t)obe_sms() * 4);
    k_pick_weights<<<grid, OBE_THREADS, 0, st>>>(utility_dev, n_settings, pickiness, s.p, s.tile_sums);
    OBE_LAUNCH_CHECK("k_pick_weights");
    k_tile_scan<<<1, OBE_SCAN_THREADS, 0, st>>>(s.tile_sums, nt, s.prefix, nullptr, 0, 0, n_settings);
    OBE_LAUNCH_CHECK("k_tile_scan");
    return draw_impl(s.p, s.prefix, n_settings, nullptr, 0, 0, &u, 1, nullptr, idx_dev, st);
}

int obe_update_multi(obe_model_t m, const obe_cloud_t* c, double* weights_out_dev, const double* records_dev,
                     int n_points, const double* constants, const int32_t* noise_index, int n_lik_channels,
                     const double* lik_scale, int use_choke, double choke, double threshold, int64_t n_total,
                     double* sums_dev, double* result_dev, void* stream) {
    if (!m || !weights_out_dev || !records_dev || !sums_dev || !result_dev) return obe_fail("null argument%s%s");
    if (m->lik != OBE_LIK_GAUSS)
        return obe_fail("obe_update_multi: the model handle has a non-Gaussian likelihood (only the single-cloud update takes one)%s%s");
    if (check_cloud(c)) return -1;
    if (m->d != c->d) return obe_fail("model was built for a different n_params%s%s");
    if (n_points < 1 || n_points > OBE_MULTI_MAX) return obe_fail("multi-point update takes 1..128 points per call%s%s");
    if (weights_out_dev == c->weights_dev) return obe_fail("multi-point update is out of place: pass another weight row%s%s");
    ObeMultiArgs a;
    memset(&a, 0, sizeof(a));
    a.particles = c->particles_dev; a.ld = c->ld; a.n = c->n; a.n_dev = (const long long*)c->n_dev;
    a.w_in = c->weights_dev; a.w_out = weights_out_dev; a.stats = c->stats_dev; a.records = records_dev;
    a.m_points = n_points; a.n_lik_channels = n_lik_channels; a.use_choke = use_choke; a.choke = choke;
    for (int ch = 0; ch < OBE_MAX_CH; ++ch) { a.noise_idx[ch] = -1; a.lik_scale[ch] = 1.0; }
    if (noise_index)
        for (int j = 0; j < n_lik_channels && j < OBE_MAX_CH; ++j) { a.noise_idx[j] = noise_index[j]; a.n_noise = j + 1; }
    if (lik_scale) for (int j = 0; j < m->nch; ++j) a.lik_scale[j] = lik_scale[j];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    const Scratch s = scratch_of(c);
    a.partials = s.partials; a.counter = s.counter + 8;
    a.sums = sums_dev; a.result = result_dev; a.threshold = threshold; a.n_total = n_total;
    int64_t blocks = (c->n + OBE_MULTI_NE * OBE_THREADS - 1) / (OBE_MULTI_NE * OBE_THREADS);
    int64_t cap = (int64_t)obe_sms() * 4;
    const int64_t fit = ((int64_t)OBE_MAX_GRID * OBE_NACC_MAX) / (2 * OBE_MULTI_MAX);
    if (cap > fit) cap = fit;
    if (blocks > cap) blocks = cap;
    return launch_kernel(m->f_multi, (int)blocks, 0, (cudaStream_t)stream, &a);
}

int obe_batch_simulate(obe_model_t m, const obe_batch_t* b, const double* settings_dev, int64_t lds,
                       const double* true_params_dev, int64_t ld_true, const double* constants,
                       const double* noise_level, const double* noise_level_dev, uint64_t seed, uint32_t cycle,
                       int write_sigma, void* stream) {
    if (!m || !b || !settings_dev || !true_params_dev) return obe_fail("null argument%s%s");
    if (m->lik != OBE_LIK_GAUSS)
        return obe_fail("obe_batch_simulate: the model handle has a non-Gaussian likelihood (only the single-cloud update takes one)%s%s");
    if (!noise_level && !noise_level_dev) return obe_fail("simulate: need a noise level%s%s");
    if (ld_true < b->n_inst) return obe_fail("simulate: ld_true < n_inst%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    ObeBSimArgs a;
    memset(&a, 0, sizeof(a));
    a.true_pars = true_params_dev; a.ld_true = ld_true; a.settings = settings_dev; a.lds = lds;
    a.last_idx = (const long long*)b->last_idx_dev; a.record = b->record_dev; a.n_inst = b->n_inst;
    a.noise_dev = noise_level_dev; a.seed = seed; a.cycle = cycle; a.write_sigma = write_sigma;
    if (noise_level) for (int c = 0; c < m->nch; ++c) a.noise[c] = noise_level[c];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    const int blocks = (int)((b->n_inst + OBE_THREADS - 1) / OBE_THREADS);
    return launch_kernel(m->f_bsim, blocks, 0, (cudaStream_t)stream, &a);
}

int obe_sweep_utility(const double* utility_dev, int64_t n_settings, const int32_t* pairs_dev, int64_t n_pairs,
                      double cost_of_new_sweep, double* cumsum_dev, double* pair_utility_dev, void* best_dev,
                      void* select_scratch_dev, void* stream) {
    if (!utility_dev || !pairs_dev || !cumsum_dev || !best_dev || !select_scratch_dev)
        return obe_fail("null argument%s%s");
    if (n_settings < 1 || n_pairs < 1) return obe_fail("sweep utility: empty settings or pairs%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    const SelectScratch s = select_scratch_of(select_scratch_dev, n_settings);
    cudaStream_t st = (cudaStream_t)stream;
    k_cumsum<<<1, OBE_SCAN_THREADS, 0, st>>>(utility_dev, n_settings, cumsum_dev);
    OBE_LAUNCH_CHECK("k_cumsum");
    int64_t blocks = (n_pairs + OBE_THREADS - 1) / OBE_THREADS;
    if (blocks > (int64_t)obe_sms() * 8) blocks = (int64_t)obe_sms() * 8;
    k_sweep_pairs<<<(int)blocks, OBE_THREADS, 0, st>>>(cumsum_dev, n_settings, pairs_dev, n_pairs, cost_of_new_sweep,
                                                      pair_utility_dev, s.part_val, s.part_idx, s.counter,
                                                      (long long*)best_dev, (double*)((char*)best_dev + 8));
    OBE_LAUNCH_CHECK("k_sweep_pairs");
    return 0;
}

int obe_eval_parameters(obe_model_t m, const obe_cloud_t* c, const double* setting, const double* constants,
                        double* y_dev, int64_t ldy, void* stream) {
    if (!m || !y_dev) return obe_fail("null argument%s%s");
    if (check_cloud(c)) return -1;
    if (m->d != c->d) return obe_fail("model was built for a different n_params%s%s");
    ObeEvalArgs a;
    memset(&a, 0, sizeof(a));
    a.a = c->particles_dev; a.ld = c->ld; a.n = c->n; a.y = y_dev; a.ldy = ldy;
    for (int j = 0; j < m->ns; ++j) a.fixed[j] = setting[j];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    int64_t blocks = (c->n + OBE_THREADS - 1) / OBE_THREADS;
    if (blocks > (int64_t)obe_sms() * 8) blocks = (int64_t)obe_sms() * 8;
    return launch_kernel(m->f_evalp, (int)blocks, 0, (cudaStream_t)stream, &a);
}

int obe_eval_settings(obe_model_t m, const double* settings_dev, int64_t lds, int64_t n_settings, const double* params,
                      const double* constants, double* y_dev, int64_t ldy, void* stream) {
    if (!m || !y_dev || !settings_dev) return obe_fail("null argument%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    ObeEvalArgs a;
    memset(&a, 0, sizeof(a));
    a.a = settings_dev; a.ld = lds; a.n = n_settings; a.y = y_dev; a.ldy = ldy;
    for (int j = 0; j < m->np_model; ++j) a.fixed[j] = params[j];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    int64_t blocks = (n_settings + OBE_THREADS - 1) / OBE_THREADS;
    if (blocks > (int64_t)obe_sms() * 8) blocks = (int64_t)obe_sms() * 8;
    return launch_kernel(m->f_evals, (int)blocks, 0, (cudaStream_t)stream, &a);
}

// ---------------------------------------------------------------------------------------------
// batched independent instances
// ---------------------------------------------------------------------------------------------
__global__ void k_batch_init(double* __restrict__ w0, int* __restrict__ cur, unsigned int* __restrict__ epoch,
                             long long* __restrict__ last_idx, int* __restrict__ flag, long long n_inst, long long n,
                             long long np) {
    const double v = 1.0 / (double)n;
    const long long total = n_inst * np;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        w0[i] = ((i % np) < n) ? v : 0.0;
        if (i < n_inst) { cur[i] = 0; epoch[i] = 0u; last_idx[i] = 0; flag[i] = 0; }
    }
}

static int check_batch(const obe_batch_t* b) {
    if (!b || !b->particles_dev[0] || !b->particles_dev[1] || !b->weights_dev[0] || !b->weights_dev[1] || !b->cur_dev ||
        !b->tile_sums_dev || !b->tile_prefix_dev || !b->stats_dev || !b->pivot_dev || !b->record_dev ||
        !b->last_idx_dev || !b->best_val_dev || !b->flag_dev || !b->list_dev || !b->n_list_dev || !b->epoch_dev)
        return obe_fail("batch has null device pointers%s%s");
    if (b->n_inst < 1 || b->n < 1 || b->d < 1 || b->d > OBE_MAX_DIMS) return obe_fail("batch geometry invalid%s%s");
    if (b->np % OBE_TILE || b->np < b->n || b->tiles != b->np / OBE_TILE || b->tiles > 64 || b->ld < b->n_inst * b->np)
        return obe_fail("batch: np must be n rounded up to whole tiles (<= 64 tiles), ld >= n_inst*np%s%s");
    if (obe_sms() <= 0) return obe_fail("no CUDA device: this library has no CPU fallback%s%s");
    return 0;
}
static void fill_batch_args(const obe_batch_t* b, ObeBatchArgs& a) {
    memset(&a, 0, sizeof(a));
    for (int j = 0; j < OBE_MAX_CH; ++j) a.u.noise_idx[j] = -1;
    a.u.n = b->n; a.u.ld = b->ld;
    a.particles[0] = b->particles_dev[0]; a.particles[1] = b->particles_dev[1];
    a.weights[0] = b->weights_dev[0]; a.weights[1] = b->weights_dev[1];
    a.cur = b->cur_dev; a.tile_sums = b->tile_sums_dev; a.prefix = b->tile_prefix_dev; a.stats = b->stats_dev;
    a.pivot = b->pivot_dev; a.rec_in = b->record_dev; a.last_idx = (const long long*)b->last_idx_dev;
    a.flag = b->flag_dev; a.n_inst = b->n_inst; a.np = b->np; a.tiles = b->tiles;
}
static int launch_batch_update(const void* f, int d, const ObeBatchArgs& a, int64_t n_inst, cudaStream_t st) {
    const size_t smem = update_smem_bytes(d, OBE_SRC_MODEL);
    cudaError_t e = set_max_smem(f, smem);
    if (e != cudaSuccess) return obe_fail("cudaFuncSetAttribute(max dynamic smem): %s%s", cudaGetErrorString(e));
    int64_t g = obe_sms();
    if (g > n_inst) g = n_inst;
    void* params[1] = {const_cast<ObeBatchArgs*>(&a)};
    e = cudaLaunchKernel(f, dim3((unsigned)g), dim3(OBE_UPDATE_THREADS), params, smem, st);
    if (e != cudaSuccess) return obe_fail("launch batched update kernel: %s%s", cudaGetErrorString(e));
    return 0;
}
static int batch_refresh_impl(const obe_batch_t* b, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index,
                              int n_noise, int only_listed, cudaStream_t st) {
    ObeBatchArgs a;
    fill_batch_args(b, a);
    a.u.scale_in = 0; a.u.write_weights = (mask_le | mask_lt) ? 1 : 0;
    a.u.mask_le = mask_le; a.u.mask_lt = mask_lt;
    a.flag = nullptr;
    if (noise_index)
        for (int j = 0; j < n_noise && j < OBE_MAX_CH; ++j) { a.u.noise_idx[j] = noise_index[j]; a.u.n_noise = j + 1; }
    if (only_listed) { a.inst_list = b->list_dev; a.n_list = b->n_list_dev; }
    const void* f = nullptr;
    switch (b->d) {
        case 1: f = (const void*)k_brefresh<1>; break;
        case 2: f = (const void*)k_brefresh<2>; break;
        case 3: f = (const void*)k_brefresh<3>; break;
        case 4: f = (const void*)k_brefresh<4>; break;
        case 5: f = (const void*)k_brefresh<5>; break;
        case 6: f = (const void*)k_brefresh<6>; break;
        case 7: f = (const void*)k_brefresh<7>; break;
        default: f = (const void*)k_brefresh<8>; break;
    }
    return launch_batch_update(f, b->d, a, b->n_inst, st);
}

int obe_batch_init(const obe_batch_t* b, const int32_t* noise_index, int n_noise, void* stream) {
    if (check_batch(b)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    k_batch_init<<<obe_sms() * 8, 256, 0, st>>>(b->weights_dev[0], b->cur_dev, b->epoch_dev, (long long*)b->last_idx_dev,
                                               b->flag_dev, b->n_inst, b->n, b->np);
    OBE_LAUNCH_CHECK("k_batch_init");
    OBE_CUDA(cudaMemsetAsync(b->stats_dev, 0, (size_t)b->n_inst * OBE_STATS_LEN * sizeof(double), st));
    OBE_CUDA(cudaMemsetAsync(b->pivot_dev, 0, (size_t)b->n_inst * OBE_MAX_DIMS * sizeof(double), st));
    // two refresh passes: the first finds the means, the second accumulates around them
    if (batch_refresh_impl(b, 0, 0, noise_index, n_noise, 0, st)) return -1;
    return batch_refresh_impl(b, 0, 0, noise_index, n_noise, 0, st);
}

int obe_batch_refresh(const obe_batch_t* b, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index, int n_noise,
                      void* stream) {
    if (check_batch(b)) return -1;
    return batch_refresh_impl(b, mask_le, mask_lt, noise_index, n_noise, 0, (cudaStream_t)stream);
}

int obe_batch_update(obe_model_t m, const obe_batch_t* b, const double* settings_dev, int64_t lds, int use_last,
                     const double* constants, const int32_t* noise_index, int n_lik_channels, int use_choke,
                     double choke, double resample_threshold, int force_resample, void* stream) {
    if (!m) return obe_fail("null model%s%s");
    if (m->lik != OBE_LIK_GAUSS)
        return obe_fail("obe_batch_update: the model handle has a non-Gaussian likelihood (only the single-cloud update takes one)%s%s");
    if (check_batch(b)) return -1;
    if (m->d != b->d) return obe_fail("model was built for a different n_params%s%s");
    if (use_last && !settings_dev) return obe_fail("use_last needs the setting grid%s%s");
    ObeBatchArgs a;
    fill_batch_args(b, a);
    a.u.scale_in = 1; a.u.write_weights = 1;
    for (int j = 0; j < m->ncons; ++j) a.u.cons[j] = constants[j];
    if (n_lik_channels < 0 || n_lik_channels > m->nch) return obe_fail("n_lik_channels out of range%s%s");
    a.u.n_lik_channels = n_lik_channels;
    if (noise_index)
        for (int c = 0; c < n_lik_channels; ++c) {
            if (noise_index[c] < 0 || noise_index[c] >= b->d) return obe_fail("noise_index out of range%s%s");
            a.u.noise_idx[c] = noise_index[c]; a.u.n_noise = c + 1;
        }
    a.u.use_choke = use_choke; a.u.choke = choke;
    a.settings = settings_dev; a.lds = lds; a.use_last = use_last; a.n_set = m->ns;
    a.resample_threshold = resample_threshold; a.force_resample = force_resample;
    return launch_batch_update(m->f_bupdate, b->d, a, b->n_inst, (cudaStream_t)stream);
}

int obe_batch_resample(const obe_batch_t* b, double a_param, int scale, uint64_t seed, uint64_t uniform_seed,
                       uint32_t cycle, int u0_index, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index,
                       int n_noise, void* stream) {
    if (check_batch(b)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    k_bcompact<<<1, OBE_SCAN_THREADS, 0, st>>>(b->flag_dev, b->n_inst, b->list_dev, b->n_list_dev);
    OBE_LAUNCH_CHECK("k_bcompact");
    ObeBResampleArgs a;
    memset(&a, 0, sizeof(a));
    a.particles[0] = b->particles_dev[0]; a.particles[1] = b->particles_dev[1];
    a.particles_w[0] = b->particles_dev[0]; a.particles_w[1] = b->particles_dev[1];
    a.weights[0] = b->weights_dev[0]; a.weights[1] = b->weights_dev[1];
    a.cur = b->cur_dev; a.prefix = b->tile_prefix_dev; a.stats = b->stats_dev; a.epoch = b->epoch_dev;
    a.inst_list = b->list_dev; a.n_list = b->n_list_dev;
    a.ld = b->ld; a.np = b->np; a.n = b->n; a.tiles = b->tiles;
    a.seed = seed; a.useed = uniform_seed; a.cycle = cycle; a.u0_index = u0_index;
    a.a_param = a_param; a.scale = scale; a.mask_le = mask_le; a.mask_lt = mask_lt;
    int64_t g = (int64_t)obe_sms() * OBE_BLOCKS_PER_SM;
    if (g > b->n_inst) g = b->n_inst;
    const int grid = (int)g;
    OBE_DIM_SWITCH(b->d, k_bsys_resample, grid, st, a)
    OBE_LAUNCH_CHECK("k_bsys_resample");
    // tile sums, CDF prefix, moments and noise sums of the new clouds (only the resampled instances)
    return batch_refresh_impl(b, 0, 0, noise_index, n_noise, 1, st);
}

int obe_batch_select(obe_model_t m, const obe_batch_t* b, const double* settings_dev, int64_t lds, int64_t n_settings,
                     const double* constants, int k, const double* var_noise, double cost_change, uint64_t uniform_seed,
                     uint32_t cycle, int method, int log_form, double* utility_dev, void* stream) {
    if (!m || !settings_dev) return obe_fail("null argument%s%s");
    if (m->lik != OBE_LIK_GAUSS)
        return obe_fail("obe_batch_select: the model handle has a non-Gaussian likelihood (only the single-cloud update takes one)%s%s");
    if (check_batch(b)) return -1;
    if (k < 1 || k > OBE_MAX_DRAWS) return obe_fail("n_draws must be 1..128 for batched engines%s%s");
    ObeBSelectArgs a;
    memset(&a, 0, sizeof(a));
    a.particles[0] = b->particles_dev[0]; a.particles[1] = b->particles_dev[1];
    a.weights[0] = b->weights_dev[0]; a.weights[1] = b->weights_dev[1];
    a.cur = b->cur_dev; a.prefix = b->tile_prefix_dev; a.stats = b->stats_dev;
    a.settings = settings_dev; a.lds = lds; a.n_settings = n_settings;
    a.ld = b->ld; a.np = b->np; a.n = b->n; a.n_inst = b->n_inst; a.tiles = b->tiles; a.k = k;
    a.last_idx = (long long*)b->last_idx_dev; a.best_val = b->best_val_dev; a.utility = utility_dev;
    a.seed = uniform_seed; a.cycle = cycle;
    a.noise_from_stats = var_noise ? 0 : 1; a.log_form = log_form; a.method = method; a.cost_change = cost_change;
    if (var_noise) for (int c = 0; c < m->nch; ++c) a.var_noise[c] = var_noise[c];
    for (int j = 0; j < m->ncons; ++j) a.cons[j] = constants[j];
    int64_t g = (int64_t)obe_sms() * 4;
    if (g > b->n_inst) g = b->n_inst;
    // (parking the K x NCH model values of a setting in shared memory, as obe_utility does, was measured here and
    // lost: 108 KB per CTA leaves 2 CTAs per SM and the kernel went from 0.44 to 0.57 ms -- occupancy matters more
    // than the second evaluation for this FP64-latency-bound body)
    const size_t smem = (size_t)(OBE_TILE + k * (m->np_model > 0 ? m->np_model : 1)) * sizeof(double);
    return launch_kernel(m->f_bselect, (int)g, smem, (cudaStream_t)stream, &a);
}

}  // extern "C"

#include "obe_summary.cuh"
