// gcs_b200_api.cu — C ABI (include/gcs_b200.h) over the sm_100a kernels.
//
// No torch types, no exceptions across the boundary, no CPU fallback: every compute entry point
// needs a CUDA device and reports GCS_E_NO_DEVICE otherwise.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/gcs_b200.h"
#include "newton_kernels.cuh"

using namespace gcsk;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(GCS_E_CUDA, "%s -> %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, \
                __LINE__);                                                                     \
    } while (0)

// GCS_VARIANT_DEFAULT: the sorted kernel from kSortedMinRuns Newton runs per launch (measured faster
// on every kind and seed count there, profiles/), the static kernel below (a sorted CTA lives
// twice as long as a static one, which shows while the launch does not fill the device).
// K4 (two linear equations: two updates per seed, then a selection that costs as much) runs one
// lane per sub-system with the seeds in sequence in both classes (K4, 2^19 sub-systems without
// parallel rows: 28.7 us against 43.0 sorted / 36.9 contracted static); so does the contracted
// 8-seed K1 (289 us against 371 per 2^20 x 8: a lane's eight runs add up to nearly the same
// total in every lane, so hardly a lane-slot idles).
constexpr long long kSortedMinRuns = 1ll << 18;
inline int resolve_variant(int variant, int kind, long long n, int n_seeds)
{
    if (variant == GCS_VARIANT_CONTRACTED) {
        // contracted arithmetic otherwise: the static kernel at every size (with a 55-cycle update the
        // sort's bookkeeping costs more than the idle lanes it removes: K1 51 vs 57 us, K3 68 vs 84 us per 2^19)
        // K4: a linear pair needs no iteration in this class (newton_linear_kernel)
        if (kind == GCS_KIND_PLL) return GCS_VARIANT_CONTRACTED_LINEAR;
        if (kind == GCS_KIND_PP && n_seeds == 8) return GCS_VARIANT_CONTRACTED_SEQ;
        return GCS_VARIANT_CONTRACTED_STATIC;
    }
    if (variant == GCS_VARIANT_CONTRACTED_LINEAR && kind != GCS_KIND_PLL) return resolve_variant(GCS_VARIANT_CONTRACTED, kind, n, n_seeds);
    if (variant != GCS_VARIANT_DEFAULT) return variant;
    if (kind == GCS_KIND_PLL && n * n_seeds >= (1ll << 17)) return GCS_VARIANT_SEQ;
    return n * n_seeds >= kSortedMinRuns ? GCS_VARIANT_SORTED : GCS_VARIANT_STATIC;
}
constexpr int kTicketSlots = 64;
constexpr int kRefillCH = 64;
constexpr int kRefillWarps = 4;

struct DeviceState {
    int device = -1;
    int sm_count = 0;
    unsigned* tickets = nullptr;  // kTicketSlots x 2 counters, zero between launches
    // a column of zeros the kernels read in place of the ABI's NULL anchor columns (grown on demand,
    // read-only afterwards: a few MB that stay in L2 and are shared by every NULL column of a batch)
    double* zeros = nullptr;
    size_t zeros_n = 0;
    // test hook (gcs_b200_debug_path_buffer): where device-resident contracted launches report how
    // each run was decided
    uint8_t* dbg_path = nullptr;
    long long dbg_path_cap = 0;
    std::atomic<unsigned> ticket_rr { 0 };
    // staging arena for the host-buffer entry points
    std::mutex arena_mu, zeros_mu;
    unsigned char* arena = nullptr;
    size_t arena_bytes = 0;
    size_t arena_used = 0;        // bump pointer; reset when the device is drained
    bool in_flight = false;       // host-buffer work enqueued and not yet waited for
    // gcs_b200_solve_many: launches beyond the first of a job go to these, forked from / joined
    // back into the caller's stream
    static constexpr int kSide = 3;
    std::mutex side_mu;
    cudaStream_t side[kSide] = {};
    cudaEvent_t side_fork = nullptr, side_join[kSide] = {};
    cudaStream_t stream = nullptr;  // kernels
    cudaStream_t h2d = nullptr;     // input copies  (own copy engine)
    cudaStream_t d2h = nullptr;     // output copies (the other copy engine)
    std::vector<cudaEvent_t> events;
    size_t ev_next = 0;
};

std::mutex g_mu;
std::vector<DeviceState*> g_devs;  // one per CUDA device, indexed by ordinal
std::vector<int> g_init_list;      // the devices of the last gcs_b200_init, in its order (what solve_sharded shards over)
std::atomic<long long> g_launches { 0 };

DeviceState* find_dev(int device)
{
    for (auto* d : g_devs)
        if (d->device == device) return d;
    return nullptr;
}

int ensure_init()
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_devs.empty()) return GCS_OK;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(GCS_E_NO_DEVICE, "no CUDA device (%s); this library has no CPU fallback",
            e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    for (int i = 0; i < n; ++i) {
        auto* d = new DeviceState();
        d->device = i;
        g_devs.push_back(d);
    }
    return GCS_OK;
}

int prepare_device(DeviceState* d)
{
    std::lock_guard<std::mutex> lk(g_mu);  // two first-time callers on one device must not both allocate
    if (d->tickets) return GCS_OK;
    CUDA_TRY(cudaSetDevice(d->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, d->device));
    d->sm_count = prop.multiProcessorCount;
    CUDA_TRY(cudaMalloc(&d->tickets, sizeof(unsigned) * 2 * kTicketSlots));
    CUDA_TRY(cudaMemset(d->tickets, 0, sizeof(unsigned) * 2 * kTicketSlots));
    CUDA_TRY(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&d->h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&d->d2h, cudaStreamNonBlocking));
    for (int k = 0; k < DeviceState::kSide; ++k) {
        CUDA_TRY(cudaStreamCreateWithFlags(&d->side[k], cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&d->side_join[k], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&d->side_fork, cudaEventDisableTiming));
    return GCS_OK;
}

}  // namespace

// for the other translation units of the library (sketch_program.cu)
namespace gcsk {
int api_fail(int code, const char* msg) { return fail(code, "%s", msg); }
void api_count_launch() { g_launches.fetch_add(1); }
}  // namespace gcsk

extern "C" int gcs_b200_column_may_be_null(int kind, int c)
{
    // columns that are identically zero in the anchored shapes of the zero-fixed solvers:
    // K1 ax, ay, by (point_point_solvers.cpp:48-50); K2 p1x, p1y, p2y (point_line_solvers.cpp:179-181);
    // K5 fdy, px, r2x, r2y (line_angle_solvers.cpp:249-274, :355-361)
    switch (kind) {
    case GCS_KIND_PP: return c == 0 || c == 1 || c == 4;
    case GCS_KIND_SDD: return c == 0 || c == 1 || c == 3;
    case GCS_KIND_ANG: return c == 1 || c == 7 || c == 10 || c == 11;
    }
    return 0;
}

namespace {

// device `d` current.  The zero column covers at least n sub-systems.
int ensure_zeros(DeviceState* d, size_t n)
{
    std::lock_guard<std::mutex> lk(d->zeros_mu);
    if (n <= d->zeros_n) return GCS_OK;
    size_t want = (size_t)1 << 16;
    while (want < n) want <<= 1;
    if (d->zeros) {
        CUDA_TRY(cudaDeviceSynchronize());  // launches in flight may still read the old one
        CUDA_TRY(cudaFree(d->zeros));
        d->zeros = nullptr, d->zeros_n = 0;
    }
    if (cudaMalloc(&d->zeros, want * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        return fail(GCS_E_NOMEM, "cudaMalloc(%zu) for the zero column failed", want * sizeof(double));
    }
    CUDA_TRY(cudaMemsetAsync(d->zeros, 0, want * sizeof(double), d->stream));
    CUDA_TRY(cudaStreamSynchronize(d->stream));
    d->zeros_n = want;
    return GCS_OK;
}

bool has_null_column(const gcs_b200_batch* b)
{
    const int nin = gcs_b200_kind_in_cols(b->kind);
    for (int c = 0; c < nin; ++c)
        if (!b->in[c]) return true;
    return false;
}

int validate(const gcs_b200_batch* b)
{
    if (!b) return fail(GCS_E_INVALID, "null batch");
    if (b->kind < 1 || b->kind > GCS_KIND_COUNT) return fail(GCS_E_INVALID, "unknown kind %d", b->kind);
    if (b->n < 0) return fail(GCS_E_INVALID, "negative n");
    if (b->variant < GCS_VARIANT_DEFAULT || b->variant > GCS_VARIANT_CONTRACTED_LINEAR)
        return fail(GCS_E_INVALID, "unknown variant %d", b->variant);
    const bool column_guess = (b->kind == GCS_KIND_SDD || b->kind == GCS_KIND_ANG);
    if (column_guess) {
        if (b->n_seeds != 2) return fail(GCS_E_INVALID, "kind %d takes exactly 2 seeds", b->kind);
    } else if (b->n_seeds != 2 && b->n_seeds != 8) {
        return fail(GCS_E_INVALID, "n_seeds must be 2 or 8 (got %d)", b->n_seeds);
    }
    if (b->n == 0) return GCS_OK;
    const int nin = gcs_b200_kind_in_cols(b->kind);
    for (int c = 0; c < nin; ++c)
        if (!b->in[c] && !gcs_b200_column_may_be_null(b->kind, c))
            return fail(GCS_E_INVALID, "input column %d of kind %d is null (only the anchor columns may be)", c, b->kind);
    if (!b->code) return fail(GCS_E_INVALID, "code column is null");
    const int nout = gcs_b200_kind_out_cols(b->kind);
    for (int c = 0; c < nout; ++c)
        if (!b->out[c]) return fail(GCS_E_INVALID, "output column %d is null", c);
    return GCS_OK;
}

BatchDev to_dev(const gcs_b200_batch* b)
{
    BatchDev p;
    memset(&p, 0, sizeof(p));
    for (int c = 0; c < GCS_MAX_IN_COLS; ++c) p.in[c] = b->in[c];
    p.code = b->code;
    p.guesses = b->guesses;
    for (int c = 0; c < GCS_MAX_OUT_COLS; ++c) p.out[c] = b->out[c];
    p.cand = b->cand;
    p.iters = b->iters;
    p.converged = b->converged;
    p.root = b->root_index;
    p.n = b->n;
    p.stride = b->n;
    return p;
}

// GCS_STATIC_BLOCK (tuning knob): lanes per CTA of the static kernel; anything but 32 / 64 / 96 / 128
// (whole warps within __launch_bounds__(128)) is ignored
inline int static_block_size()
{
    const char* e = getenv("GCS_STATIC_BLOCK");
    const int v = e ? atoi(e) : 128;
    return (v == 32 || v == 64 || v == 96 || v == 128) ? v : 128;
}

// GCS_B200_PREFETCH (tuning knob): waves of look-ahead of the L2 prefetch (0 = off, default 1)
inline int prefetch_waves()
{
    static const int v = [] {
        const char* e = getenv("GCS_B200_PREFETCH");
        const int w = e ? atoi(e) : 1;
        return (w >= 0 && w <= 8) ? w : 1;
    }();
    return v;
}

// sub-systems one wave of resident CTAs of `kern` covers on this device
template <typename Kern>
long long wave_subs(DeviceState* d, Kern kern, int block, int subs_per_block)
{
    int bps = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, block, 0) != cudaSuccess || bps < 1) {
        cudaGetLastError();
        return 0;
    }
    return (long long)d->sm_count * bps * subs_per_block;
}

template <int KIND, int NS, bool RLX = false>
int launch_static(DeviceState*, const BatchDev& p, cudaStream_t st)
{
    const long long threads = p.n * NS;
    static const int block = static_block_size();
    const long long grid = (threads + block - 1) / block;
    if (grid > 0x7fffffffLL) return fail(GCS_E_INVALID, "batch too large for one launch");
    newton_static_kernel<KIND, NS, RLX><<<(unsigned)grid, block, 0, st>>>(p);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

template <int KIND, int NS, bool RLX>
int launch_seq(DeviceState* d, BatchDev p, cudaStream_t st)
{
    const long long grid = (p.n + 127) / 128;
    if (grid > 0x7fffffffLL) return fail(GCS_E_INVALID, "batch too large for one launch");
    static thread_local long long wave[64] = {};
    if (prefetch_waves() > 0) {
        long long& w = wave[d->device & 63];
        if (w == 0) w = wave_subs(d, newton_seq_kernel<KIND, NS, RLX>, 128, 128);
        p.pf = w * prefetch_waves();
    }
    newton_seq_kernel<KIND, NS, RLX><<<(unsigned)grid, 128, 0, st>>>(p);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

template <int NS>
int launch_linear(DeviceState* d, BatchDev p, cudaStream_t st)
{
    const long long grid = (p.n + 127) / 128;
    if (grid > 0x7fffffffLL) return fail(GCS_E_INVALID, "batch too large for one launch");
    static thread_local long long wave[64] = {};
    if (prefetch_waves() > 0) {
        long long& w = wave[d->device & 63];
        if (w == 0) w = wave_subs(d, newton_linear_kernel<NS>, 128, 128);
        p.pf = w * prefetch_waves();
    }
    newton_linear_kernel<NS><<<(unsigned)grid, 128, 0, st>>>(p);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

template <int KIND>
int launch_pair(const BatchDev& p, cudaStream_t st)
{
    const long long grid = (p.n + 127) / 128;
    if (grid > 0x7fffffffLL) return fail(GCS_E_INVALID, "batch too large for one launch");
    newton_pair_kernel<KIND><<<(unsigned)grid, 128, 0, st>>>(p);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

template <int KIND, int NS, bool RLX = false>
int launch_sorted(const BatchDev& p, cudaStream_t st)
{
    constexpr int T = GCS_SORTED_THREADS, TILE = 2 * T / NS;  // two runs per lane
    const long long grid = (p.n + TILE - 1) / TILE;
    if (grid > 0x7fffffffLL) return fail(GCS_E_INVALID, "batch too large for one launch");
    newton_sorted_kernel<KIND, NS, TILE, T, RLX><<<(unsigned)grid, T, 0, st>>>(p);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

template <int KIND, int NS>
int launch_refill(DeviceState* d, const BatchDev& p, cudaStream_t st)
{
    constexpr int CH = kRefillCH, W = kRefillWarps;
    auto kern = newton_refill_kernel<KIND, NS, CH, W>;
    const size_t smem = refill_smem_bytes<KIND, NS, CH>(W);
    static thread_local int configured_dev[GCS_KIND_COUNT + 1][GCS_MAX_SEEDS + 1] = {};
    static thread_local int blocks_per_sm[GCS_KIND_COUNT + 1][GCS_MAX_SEEDS + 1] = {};
    if (configured_dev[KIND][NS] != d->device + 1) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int bps = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, W * 32, smem));
        if (bps < 1) return fail(GCS_E_CUDA, "refill kernel does not fit on an SM");
        blocks_per_sm[KIND][NS] = bps;
        configured_dev[KIND][NS] = d->device + 1;
    }
    const long long nchunks = (p.n + CH - 1) / CH;
    long long grid = (long long)d->sm_count * blocks_per_sm[KIND][NS];
    const long long need = (nchunks + W - 1) / W;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    bool aligned = p.code != nullptr && ((reinterpret_cast<uintptr_t>(p.code) & 15) == 0);
    for (int c = 0; c < Sys<KIND>::kCols; ++c)
        aligned = aligned && ((reinterpret_cast<uintptr_t>(p.in[c]) & 15) == 0);
    unsigned* tk = d->tickets + 2 * (d->ticket_rr.fetch_add(1) % kTicketSlots);
    kern<<<(unsigned)grid, W * 32, smem, st>>>(p, tk, aligned ? 1 : 0);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return GCS_OK;
}

template <int KIND>
int launch_kind(DeviceState* d, const gcs_b200_batch* b, const BatchDev& p, cudaStream_t st)
{
    const int variant = resolve_variant(b->variant, KIND, p.n, b->n_seeds);
    constexpr bool column_guess = (KIND == GCS_KIND_SDD || KIND == GCS_KIND_ANG);
    if constexpr (KIND == GCS_KIND_PLL) {
        if (variant == GCS_VARIANT_CONTRACTED_LINEAR) return b->n_seeds == 2 ? launch_linear<2>(d, p, st) : launch_linear<8>(d, p, st);
    }
    if (b->n_seeds == 2) {
        if (variant == GCS_VARIANT_CONTRACTED_SEQ) return launch_seq<KIND, 2, true>(d, p, st);
        if (variant == GCS_VARIANT_SEQ) return launch_seq<KIND, 2, false>(d, p, st);
        if (variant == GCS_VARIANT_CONTRACTED_SORTED) return launch_sorted<KIND, 2, true>(p, st);
        if (variant == GCS_VARIANT_CONTRACTED_STATIC) return launch_static<KIND, 2, true>(d, p, st);
        if (variant == GCS_VARIANT_SORTED) return launch_sorted<KIND, 2>(p, st);
        if (variant == GCS_VARIANT_PAIR) return launch_pair<KIND>(p, st);
        return variant == GCS_VARIANT_REFILL ? launch_refill<KIND, 2>(d, p, st) : launch_static<KIND, 2>(d, p, st);
    }
    if constexpr (!column_guess) {
        if (variant == GCS_VARIANT_CONTRACTED_SEQ) return launch_seq<KIND, 8, true>(d, p, st);
        if (variant == GCS_VARIANT_SEQ) return launch_seq<KIND, 8, false>(d, p, st);
        if (variant == GCS_VARIANT_CONTRACTED_SORTED) return launch_sorted<KIND, 8, true>(p, st);
        if (variant == GCS_VARIANT_CONTRACTED_STATIC) return launch_static<KIND, 8, true>(d, p, st);
        if (variant == GCS_VARIANT_SORTED) return launch_sorted<KIND, 8>(p, st);
        return variant == GCS_VARIANT_REFILL ? launch_refill<KIND, 8>(d, p, st) : launch_static<KIND, 8>(d, p, st);
    }
    return fail(GCS_E_INVALID, "unsupported seed count");
}

int solve_dev(DeviceState* d, const gcs_b200_batch* b, const BatchDev& p, cudaStream_t st)
{
    if (p.n == 0) return GCS_OK;
    switch (b->kind) {
    case GCS_KIND_PP: return launch_kind<GCS_KIND_PP>(d, b, p, st);
    case GCS_KIND_SDD: return launch_kind<GCS_KIND_SDD>(d, b, p, st);
    case GCS_KIND_PPL: return launch_kind<GCS_KIND_PPL>(d, b, p, st);
    case GCS_KIND_PLL: return launch_kind<GCS_KIND_PLL>(d, b, p, st);
    case GCS_KIND_ANG: return launch_kind<GCS_KIND_ANG>(d, b, p, st);
    }
    return fail(GCS_E_INVALID, "unknown kind");
}

int solve_on(DeviceState* d, const gcs_b200_batch* b, cudaStream_t st)
{
    if (b->n == 0) return GCS_OK;
    BatchDev p = to_dev(b);
    if (d->dbg_path && (long long)b->n * b->n_seeds <= d->dbg_path_cap) p.path = d->dbg_path;
    if (has_null_column(b)) {
        const int rc = ensure_zeros(d, (size_t)b->n);
        if (rc != GCS_OK) return rc;
        for (int c = 0; c < gcs_b200_kind_in_cols(b->kind); ++c)
            if (!p.in[c]) p.in[c] = d->zeros;
    }
    return solve_dev(d, b, p, st);
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- FP64 probes --------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) fp64_probe_kernel(double* out, int iters, double seed)
{
    // 8 independent chains per thread; MODE 0: DFMA, MODE 1: alternating DADD / DMUL
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3;
    double a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        if (MODE == 0) {
            a0 = __fma_rn(a0, m, c), a1 = __fma_rn(a1, m, c), a2 = __fma_rn(a2, m, c), a3 = __fma_rn(a3, m, c);
            a4 = __fma_rn(a4, m, c), a5 = __fma_rn(a5, m, c), a6 = __fma_rn(a6, m, c), a7 = __fma_rn(a7, m, c);
        } else {
            a0 = __dadd_rn(a0, c), a1 = __dmul_rn(a1, m), a2 = __dadd_rn(a2, c), a3 = __dmul_rn(a3, m);
            a4 = __dadd_rn(a4, c), a5 = __dmul_rn(a5, m), a6 = __dadd_rn(a6, c), a7 = __dmul_rn(a7, m);
        }
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

__global__ void fp64_latency_kernel(double* out, long long* cycles, int iters, double seed)
{
    double a = seed;
    const double m = 1.0000000001, c = 1e-9;
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
        a = __fma_rn(a, m, c), a = __fma_rn(a, m, c), a = __fma_rn(a, m, c), a = __fma_rn(a, m, c);
        a = __fma_rn(a, m, c), a = __fma_rn(a, m, c), a = __fma_rn(a, m, c), a = __fma_rn(a, m, c);
    }
    const long long t1 = clock64();
    out[threadIdx.x] = a;
    if (threadIdx.x == 0) *cycles = t1 - t0;
}

// DFMA lanes per SM per clock as a function of resident warps and per-thread ILP (one block per SM)
template <int ILP>
__global__ void fp64_curve_kernel(double* out, long long* cycles, int iters, double seed)
{
    double a[ILP];
#pragma unroll
    for (int k = 0; k < ILP; ++k) a[k] = seed + k + threadIdx.x;
    const double m = 1.0000000001, c = 1e-9;
    __syncthreads();
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int k = 0; k < ILP; ++k) a[k] = __fma_rn(a[k], m, c);
        }
    }
    __syncthreads();
    const long long t1 = clock64();
    double s = 0;
#pragma unroll
    for (int k = 0; k < ILP; ++k) s += a[k];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

}  // namespace

extern "C" {

int gcs_b200_kind_in_cols(int kind)
{
    static const int t[GCS_KIND_COUNT + 1] = { 0, 6, 9, 10, 12, 13 };
    return (kind >= 1 && kind <= GCS_KIND_COUNT) ? t[kind] : 0;
}

int gcs_b200_kind_out_cols(int kind)
{
    static const int t[GCS_KIND_COUNT + 1] = { 0, 2, 4, 2, 2, 4 };
    return (kind >= 1 && kind <= GCS_KIND_COUNT) ? t[kind] : 0;
}

void* gcs_b200_host_alloc(size_t bytes) { return gcs_b200_host_alloc_ex(bytes, 0); }

void* gcs_b200_host_alloc_ex(size_t bytes, int flags)
{
    if (bytes == 0 || ensure_init() != GCS_OK || g_devs.empty()) return nullptr;
    void* p = nullptr;
    const unsigned f = cudaHostAllocPortable | ((flags & GCS_HOST_WRITE_COMBINED) ? cudaHostAllocWriteCombined : 0u);
    if (cudaHostAlloc(&p, bytes, f) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void gcs_b200_host_free(void* p)
{
    if (p && cudaFreeHost(p) != cudaSuccess) cudaGetLastError();
}

int gcs_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int gcs_b200_init(int device_count, const int* devices)
{
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    const int avail = (int)g_devs.size();
    if (device_count <= 0) device_count = avail;
    std::vector<int> list;
    for (int i = 0; i < device_count; ++i) {
        const int dev = devices ? devices[i] : i;
        if (dev < 0 || dev >= avail) return fail(GCS_E_NO_DEVICE, "device %d out of range (%d present)", dev, avail);
        for (int seen : list)
            if (seen == dev) return fail(GCS_E_INVALID, "device %d listed twice", dev);
        rc = prepare_device(g_devs[dev]);
        if (rc != GCS_OK) return rc;
        list.push_back(dev);
    }
    std::lock_guard<std::mutex> lk(g_mu);
    g_init_list = list;
    return GCS_OK;
}

void gcs_b200_shutdown(void)
{
    std::lock_guard<std::mutex> lk(g_mu);
    for (auto* d : g_devs) {
        if (d->tickets || d->arena || d->stream) {
            cudaSetDevice(d->device);
            if (d->stream) cudaStreamSynchronize(d->stream), cudaStreamDestroy(d->stream);
            if (d->h2d) cudaStreamSynchronize(d->h2d), cudaStreamDestroy(d->h2d);
            if (d->d2h) cudaStreamSynchronize(d->d2h), cudaStreamDestroy(d->d2h);
            for (int k = 0; k < DeviceState::kSide; ++k) {
                if (d->side[k]) cudaStreamSynchronize(d->side[k]), cudaStreamDestroy(d->side[k]);
                if (d->side_join[k]) cudaEventDestroy(d->side_join[k]);
            }
            if (d->side_fork) cudaEventDestroy(d->side_fork);
            for (cudaEvent_t e : d->events) cudaEventDestroy(e);
            if (d->tickets) cudaFree(d->tickets);
            if (d->zeros) cudaFree(d->zeros);
            if (d->arena) cudaFree(d->arena);
        }
        delete d;
    }
    g_devs.clear();
    g_init_list.clear();
}

const char* gcs_b200_last_error(void) { return g_err; }

#ifndef GCS_SRC_HASH
#define GCS_SRC_HASH "unstamped"
#endif
// "src <hash>": sha256 prefix of csrc/*, the public header and the compiler flags this binary was
// built from (__graft_entry__.cuda_source_hash), so that a stale library is detectable
const char* gcs_b200_version(void) { return "gcs_b200 0.2.0 (sm_100a, fp64, fmad=false; src " GCS_SRC_HASH ")"; }

int64_t gcs_b200_launch_count(void) { return g_launches.load(); }

int gcs_b200_default_variant(int64_t n, int n_seeds) { return resolve_variant(GCS_VARIANT_DEFAULT, GCS_KIND_PP, n, n_seeds); }

int gcs_b200_resolve_variant(int variant, int kind, int64_t n, int n_seeds) { return resolve_variant(variant, kind, n, n_seeds); }

const char* gcs_b200_kernel_name(int kind, int n_seeds, int variant)
{
    static thread_local char name[96];
    variant = resolve_variant(variant, kind, kSortedMinRuns, n_seeds);  // default: named for a launch that fills the device
    const char* base = variant == GCS_VARIANT_REFILL ? "newton_refill_kernel"
        : variant == GCS_VARIANT_CONTRACTED_LINEAR   ? "newton_linear_kernel[contracted]"
        : variant == GCS_VARIANT_CONTRACTED_SEQ      ? "newton_seq_kernel[contracted]"
        : variant == GCS_VARIANT_SEQ                 ? "newton_seq_kernel"
        : variant == GCS_VARIANT_CONTRACTED_SORTED   ? "newton_sorted_kernel[contracted]"
        : variant == GCS_VARIANT_CONTRACTED_STATIC   ? "newton_static_kernel[contracted]"
        : variant == GCS_VARIANT_SORTED              ? "newton_sorted_kernel"
        : (variant == GCS_VARIANT_PAIR && n_seeds == 2) ? "newton_pair_kernel"
                                                     : "newton_static_kernel";
    snprintf(name, sizeof(name), "%s<K%d,%d seeds>", base, kind, n_seeds);
    return name;
}

int gcs_b200_solve(const gcs_b200_batch* b, int device, void* cuda_stream)
{
    int rc = validate(b);
    if (rc != GCS_OK) return rc;
    if (b->mem != GCS_MEM_DEVICE) return fail(GCS_E_INVALID, "gcs_b200_solve needs device pointers (mem=GCS_MEM_DEVICE)");
    rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    rc = prepare_device(d);
    if (rc != GCS_OK) return rc;
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    rc = solve_on(d, b, static_cast<cudaStream_t>(cuda_stream));
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    return rc;
}

int gcs_b200_solve_many(const gcs_b200_batch* const* batches, int count, int device, void* cuda_stream)
{
    if (count < 0 || (count > 0 && !batches)) return fail(GCS_E_INVALID, "bad batch list");
    for (int i = 0; i < count; ++i) {
        const int rc = validate(batches[i]);
        if (rc != GCS_OK) return rc;
        if (batches[i]->mem != GCS_MEM_DEVICE) return fail(GCS_E_INVALID, "gcs_b200_solve_many needs device pointers (batch %d)", i);
    }
    if (count == 0) return GCS_OK;
    if (count == 1) return gcs_b200_solve(batches[0], device, cuda_stream);
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    rc = prepare_device(d);
    if (rc != GCS_OK) return rc;
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    cudaStream_t user = static_cast<cudaStream_t>(cuda_stream);
    {
        // The batches are independent jobs: the first stays on the caller's stream, the others go
        // round-robin to side streams that start where the caller's stream stands now and are
        // joined back into it, so the call is stream-ordered as a whole while one kernel's ramp-up,
        // drain and literal re-runs are covered by its neighbours' throughput work.
        std::lock_guard<std::mutex> lk(d->side_mu);
        bool used[DeviceState::kSide] = {};
        rc = cudaEventRecord(d->side_fork, user) == cudaSuccess ? GCS_OK : fail(GCS_E_CUDA, "event record failed");
        for (int i = 0; i < count && rc == GCS_OK; ++i) {
            cudaStream_t st = user;
            if (i > 0) {
                const int k = (i - 1) % DeviceState::kSide;
                st = d->side[k];
                if (!used[k]) {
                    if (cudaStreamWaitEvent(st, d->side_fork, 0) != cudaSuccess) rc = fail(GCS_E_CUDA, "stream wait failed");
                    used[k] = true;
                }
            }
            if (rc == GCS_OK) rc = solve_on(d, batches[i], st);
        }
        for (int k = 0; k < DeviceState::kSide; ++k) {
            if (!used[k]) continue;  // joined even after a failure: nothing may be left running unordered
            if (cudaEventRecord(d->side_join[k], d->side[k]) != cudaSuccess || cudaStreamWaitEvent(user, d->side_join[k], 0) != cudaSuccess)
                if (rc == GCS_OK) rc = fail(GCS_E_CUDA, "joining the side streams failed");
        }
    }
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    return rc;
}

// ---- host-buffer path: chunked three-stage pipeline -------------------------------------
// A batch is cut into index ranges; range c+1 is on its way up (h2d stream, one copy engine)
// while range c is being solved (kernel stream) and range c-1 is on its way down (d2h stream,
// the other copy engine).  With pinned host buffers the three overlap and the call costs about
// max(H2D, D2H) instead of H2D + kernel + D2H; with pageable buffers the copies stage through
// the driver and the result is the same, only slower.
//
// (Recording the same calls as a CUDA graph and replaying it was measured too: 1.80 ms per bench
// step against 1.77 ms for plain stream calls - the enqueue cost, ~0.1 ms, already hides behind
// the transfers - so the plain form stayed.  Also measured and dropped: splitting the rows of a
// slab copy over two upload streams, 1.95 ms - the engines contend for the link; letting the
// kernel read and write the pinned buffers itself (zero copy, static kernel, no arena), 1.80 ms -
// SM loads pull ~45 GB/s over PCIe against ~47 GB/s for the copy engine on these row sizes; ranges
// that halve (n/2, n/4, n/8, n/8), 1.73 ms - the same as equal ranges; packed sub-batches of
// 131072 rows uploaded with one 1-D copy each, 1.70 ms - the same again.  Copies of pipeline-stage
// size (7-14 MB) reach ~48 GB/s on the box, the 55 GB/s of its PCIe link need 64 MB and more.)
namespace {

// GCS_B200_TRACE=1: timing events at the stage boundaries of the (non-graph) pipeline, printed at drain
struct TraceMark {
    cudaEvent_t ev;
    const char* what;
    int batch_kind;
    long long lo;
};
std::vector<TraceMark> g_trace;
cudaEvent_t g_trace_origin = nullptr;
bool trace_on()
{
    static const bool on = getenv("GCS_B200_TRACE") != nullptr;
    return on;
}
void trace_mark(cudaStream_t st, const char* what, int kind, long long lo)
{
    if (!trace_on()) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    g_trace.push_back({ e, what, kind, lo });
}
void trace_dump()
{
    if (!trace_on() || g_trace.empty()) return;
    for (auto& m : g_trace) {
        float ms = 0;
        cudaEventElapsedTime(&ms, g_trace[0].ev, m.ev);
        fprintf(stderr, "[trace] K%d lo=%-8lld %-10s %8.3f ms\n", m.batch_kind, m.lo, m.what, ms);
        }
    for (auto& m : g_trace) cudaEventDestroy(m.ev);
    g_trace.clear();
}

// Device bytes one index range of `count` sub-systems of batch `b` needs in the staging arena.
size_t arena_need(const gcs_b200_batch* b, int64_t count)
{
    const size_t n = (size_t)count;
    const int ns = b->n_seeds;
    const int nin = gcs_b200_kind_in_cols(b->kind), nout = gcs_b200_kind_out_cols(b->kind);
    int present = 0;
    for (int c = 0; c < nin; ++c) present += b->in[c] != nullptr;
    size_t need = align_up(n * 8, 256) * (size_t)(present + nout) + align_up(n, 256) * 2;  // columns, code, root
    if (b->guesses) need += align_up(n * 8 * 2 * ns, 256);
    if (b->cand) need += align_up(n * 8 * 2 * ns, 256);
    need += align_up(n * 2 * ns, 256) + align_up(n * ns, 256);  // iters + converged
    return need;
}

int drain(DeviceState* d)
{
    CUDA_TRY(cudaStreamSynchronize(d->h2d));
    CUDA_TRY(cudaStreamSynchronize(d->stream));
    CUDA_TRY(cudaStreamSynchronize(d->d2h));
    trace_dump();
    d->arena_used = 0;
    d->ev_next = 0;
    d->in_flight = false;
    return GCS_OK;
}

// makes room for `need` more arena bytes (may drain the device and grow the arena)
int reserve_arena(DeviceState* d, size_t need)
{
    if (d->arena_used + need <= d->arena_bytes) return GCS_OK;
    // Not enough room behind the batches already in flight: finish those, then size the arena
    // for what was asked for in total so that the same sequence of calls overlaps next time.
    const size_t want = d->arena_used + need;
    if (d->in_flight) {
        const int rc = drain(d);
        if (rc != GCS_OK) return rc;
    }
    if (d->arena) CUDA_TRY(cudaFree(d->arena));
    d->arena = nullptr, d->arena_bytes = 0;
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    size_t grow = want + want / 4;
    if (grow > free_b / 2) grow = want;
    if (grow > free_b / 2) grow = need;
    if (cudaMalloc(&d->arena, grow) != cudaSuccess) {
        cudaGetLastError();
        return fail(GCS_E_NOMEM, "cudaMalloc(%zu) for the staging arena failed", grow);
    }
    d->arena_bytes = grow;
    return GCS_OK;
}

int ensure_events(DeviceState* d, size_t count)
{
    while (d->events.size() < d->ev_next + count) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        d->events.push_back(e);
    }
    return GCS_OK;
}

int64_t chunk_len(int64_t n, bool slabs, size_t up_bytes_per_row)
{
    // Index ranges per batch.  Every copy costs a few microseconds of engine time whatever its
    // size, and copies below a few MB do not reach the link rate, so a range is sized by the BYTES
    // its upload moves (default 32 MB per stage, measured best of 4..32; GCS_B200_STAGE_MB), never below 32 Ki sub-systems
    // and never more than 16 ranges per batch (3 when every column needs its own copy call).  The
    // caller halves the last range, so what trails the final upload is 1/2 .. 1/32 of the batch.
    // Multiples of 128 keep every slice 16-byte aligned.
    static const int forced = getenv("GCS_B200_PARTS") ? atoi(getenv("GCS_B200_PARTS")) : 0;  // tuning knob, 1..64
    static const int stage_mb = getenv("GCS_B200_STAGE_MB") ? atoi(getenv("GCS_B200_STAGE_MB")) : 32;
    int64_t parts;
    if (forced > 0 && forced <= 64) {
        parts = forced;
    } else {
        const size_t stage = (size_t)(stage_mb > 0 && stage_mb <= 1024 ? stage_mb : 32) << 20;
        const size_t bytes = (size_t)n * (up_bytes_per_row ? up_bytes_per_row : 8);
        parts = (int64_t)((bytes + stage - 1) / stage);
        const int64_t max_parts = slabs ? 16 : 3;
        if (parts > max_parts) parts = max_parts;
        if (parts < 1) parts = 1;
    }
    int64_t c = (n + parts - 1) / parts;
    if (c < 32768) c = 32768;
    return (c + 127) / 128 * 128;
}

// Maximal runs of host columns at one constant positive spacing: such a run moves with ONE strided
// copy per index range.  runs[j] = length of the run starting at present-column j (0 inside a run).
void find_runs(const char* const* cols, int count, size_t row_bytes, int* runs, size_t* pitch)
{
    const bool off = getenv("GCS_B200_NOSLAB") != nullptr;
    for (int j = 0; j < count;) {
        int run = 1;
        size_t sp = 0;
        if (!off && j + 1 < count && cols[j + 1] > cols[j]) {
            sp = (size_t)(cols[j + 1] - cols[j]);
            if (sp >= row_bytes && sp <= 0x7fffffffull) {
                run = 2;
                while (j + run < count && cols[j + run] > cols[j + run - 1] && (size_t)(cols[j + run] - cols[j + run - 1]) == sp) ++run;
            }
        }
        runs[j] = run;
        pitch[j] = sp;
        for (int q = 1; q < run; ++q) runs[j + q] = 0;
        j += run;
    }
}

// Issues the whole pipeline of the index range [first, first + count) of host batch `b` on
// (h2d, stream, d2h), device buffers at arena + off.  The per-seed planes of the host batch keep
// the full batch's pitch (b->n), so several devices can fill disjoint ranges of the same arrays.
// Nothing joins the streams here: the next batch's upload may start at once (its buffers are a
// different arena region); gcs_b200_wait / drain synchronises all three.
int record_pipeline(DeviceState* d, const gcs_b200_batch* b, size_t off, int64_t first, int64_t count)
{
    const size_t n = (size_t)count, host_n = (size_t)b->n;
    const int ns = b->n_seeds;
    const int nin = gcs_b200_kind_in_cols(b->kind), nout = gcs_b200_kind_out_cols(b->kind);
    const size_t colb = align_up(n * 8, 256);
    unsigned char* cur_p = d->arena + off;
    auto take = [&](size_t bytes) {
        unsigned char* r = cur_p;
        cur_p += align_up(bytes, 256);
        return r;
    };
    // NULL input columns (all zeros, gcs_b200.h) have no device buffer and no copy
    double* din[GCS_MAX_IN_COLS] = {};
    double* dout[GCS_MAX_OUT_COLS] = {};
    int pres[GCS_MAX_IN_COLS], npres = 0;
    const char* hin[GCS_MAX_IN_COLS];
    for (int c = 0; c < nin; ++c) {
        if (!b->in[c]) continue;
        din[c] = reinterpret_cast<double*>(take(n * 8));
        hin[npres] = reinterpret_cast<const char*>(b->in[c] + first);
        pres[npres++] = c;
    }
    uint8_t* dcode = take(n);
    double* dguess = b->guesses ? reinterpret_cast<double*>(take(n * 8 * 2 * ns)) : nullptr;
    const char* hout[GCS_MAX_OUT_COLS];
    for (int c = 0; c < nout; ++c) {
        dout[c] = reinterpret_cast<double*>(take(n * 8));
        hout[c] = reinterpret_cast<const char*>(b->out[c] + first);
    }
    double* dcand = b->cand ? reinterpret_cast<double*>(take(n * 8 * 2 * ns)) : nullptr;
    int16_t* diters = reinterpret_cast<int16_t*>(take(n * 2 * ns));
    uint8_t* dconv = take(n * ns);
    uint8_t* droot = take(n);

    int in_runs[GCS_MAX_IN_COLS] = {}, out_runs[GCS_MAX_OUT_COLS] = {};
    size_t in_pitch[GCS_MAX_IN_COLS] = {}, out_pitch[GCS_MAX_OUT_COLS] = {};
    find_runs(hin, npres, n * 8, in_runs, in_pitch);
    find_runs(hout, nout, n * 8, out_runs, out_pitch);
    int in_calls = 0, out_calls = 0;
    for (int j = 0; j < npres; ++j) in_calls += in_runs[j] > 0;
    for (int j = 0; j < nout; ++j) out_calls += out_runs[j] > 0;
    const bool slabs = in_calls <= 2 && out_calls <= 2;

    // index ranges: equal steps, the last one halved so that less work trails the final upload
    const int64_t step = chunk_len(count, slabs, (size_t)npres * 8 + 1 + (b->guesses ? 16u * (size_t)ns : 0u));
    std::vector<std::pair<int64_t, int64_t>> ranges;
    for (int64_t lo = 0; lo < count; lo += step) ranges.push_back({ lo, (count - lo < step) ? (count - lo) : step });
    if (ranges.size() >= 2 && ranges.back().second >= 65536) {
        const auto last = ranges.back();
        const int64_t half = (last.second / 2 + 127) / 128 * 128;
        ranges.back() = { last.first, half };
        ranges.push_back({ last.first + half, last.second - half });
    }
    int rc = ensure_events(d, 2 * ranges.size());
    if (rc != GCS_OK) return rc;
    if (npres < nin) {
        rc = ensure_zeros(d, (size_t)step + 65536);
        if (rc != GCS_OK) return rc;
    }
    // the one-byte code column goes up whole, ahead of the first range: one copy instead of one
    // per range (every copy costs a few microseconds of engine time whatever its size)
    CUDA_TRY(cudaMemcpyAsync(dcode, b->code + first, n, cudaMemcpyHostToDevice, d->h2d));
    for (const auto& range : ranges) {
        const int64_t lo = range.first, len = range.second;
        const size_t m = (size_t)len;
        trace_mark(d->h2d, "up-begin", b->kind, lo);
        // up: columns that sit at a constant spacing in host memory (one [cols][n] slab) go up as
        // one strided copy (their device buffers are consecutive, pitch colb), anything else
        // column by column
        for (int j = 0; j < npres;) {
            const int run = in_runs[j];
            double* dst = din[pres[j]] + lo;
            const char* src = hin[j] + (size_t)lo * 8;
            if (run > 1) {
                CUDA_TRY(cudaMemcpy2DAsync(dst, colb, src, in_pitch[j], m * 8, (size_t)run, cudaMemcpyHostToDevice, d->h2d));
            } else {
                CUDA_TRY(cudaMemcpyAsync(dst, src, m * 8, cudaMemcpyHostToDevice, d->h2d));
            }
            j += run;
        }
        if (b->guesses)
            CUDA_TRY(cudaMemcpy2DAsync(dguess + lo, n * 8, b->guesses + first + lo, host_n * 8, m * 8, (size_t)(2 * ns),
                cudaMemcpyHostToDevice, d->h2d));
        cudaEvent_t up = d->events[d->ev_next++], done = d->events[d->ev_next++];
        CUDA_TRY(cudaEventRecord(up, d->h2d));
        trace_mark(d->h2d, "up-end", b->kind, lo);
        // solve
        CUDA_TRY(cudaStreamWaitEvent(d->stream, up, 0));
        BatchDev p;
        memset(&p, 0, sizeof(p));
        for (int c = 0; c < nin; ++c) p.in[c] = din[c] ? din[c] + lo : d->zeros;
        p.code = dcode + lo;
        p.guesses = dguess ? dguess + lo : nullptr;
        for (int c = 0; c < nout; ++c) p.out[c] = dout[c] + lo;
        p.cand = dcand ? dcand + lo : nullptr;
        p.iters = diters + lo;
        p.converged = dconv + lo;
        p.root = droot + lo;
        p.n = len;
        p.stride = count;
        rc = solve_dev(d, b, p, d->stream);
        if (rc != GCS_OK) return rc;
        CUDA_TRY(cudaEventRecord(done, d->stream));
        trace_mark(d->stream, "solved", b->kind, lo);
        // down
        CUDA_TRY(cudaStreamWaitEvent(d->d2h, done, 0));
        for (int j = 0; j < nout;) {
            const int run = out_runs[j];
            char* dst = const_cast<char*>(hout[j]) + (size_t)lo * 8;
            if (run > 1) {
                CUDA_TRY(cudaMemcpy2DAsync(dst, out_pitch[j], dout[j] + lo, colb, m * 8, (size_t)run, cudaMemcpyDeviceToHost, d->d2h));
            } else {
                CUDA_TRY(cudaMemcpyAsync(dst, dout[j] + lo, m * 8, cudaMemcpyDeviceToHost, d->d2h));
            }
            j += run;
        }
        if (b->cand)
            CUDA_TRY(cudaMemcpy2DAsync(b->cand + first + lo, host_n * 8, dcand + lo, n * 8, m * 8, (size_t)(2 * ns),
                cudaMemcpyDeviceToHost, d->d2h));
        if (b->iters)
            CUDA_TRY(cudaMemcpy2DAsync(b->iters + first + lo, host_n * 2, diters + lo, n * 2, m * 2, (size_t)ns, cudaMemcpyDeviceToHost, d->d2h));
        if (b->converged)
            CUDA_TRY(cudaMemcpy2DAsync(b->converged + first + lo, host_n, dconv + lo, n, m, (size_t)ns, cudaMemcpyDeviceToHost, d->d2h));
        if (b->root_index) CUDA_TRY(cudaMemcpyAsync(b->root_index + first + lo, droot + lo, m, cudaMemcpyDeviceToHost, d->d2h));
    }
    trace_mark(d->d2h, "flags-end", b->kind, -1);
    return GCS_OK;
}

// arena_mu held, device current
int enqueue_host(DeviceState* d, const gcs_b200_batch* b, int64_t first, int64_t count)
{
    const size_t need = arena_need(b, count);
    int rc = reserve_arena(d, need);
    if (rc != GCS_OK) return rc;
    const size_t off = d->arena_used;
    rc = record_pipeline(d, b, off, first, count);
    d->arena_used = off + need;
    d->in_flight = true;
    return rc;
}

// index range [first, first + count) of a validated host batch on `device`
int host_range_entry(const gcs_b200_batch* b, int device, int64_t first, int64_t count, bool wait)
{
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    rc = prepare_device(d);
    if (rc != GCS_OK) return rc;
    std::lock_guard<std::mutex> lk(d->arena_mu);
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    if (count > 0) rc = enqueue_host(d, b, first, count);
    if (rc != GCS_OK) {
        drain(d);  // leave nothing behind a failed call
    } else if (wait && d->in_flight) {
        rc = drain(d);
    }
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    return rc;
}

int host_entry(const gcs_b200_batch* b, int device, bool wait)
{
    int rc = validate(b);
    if (rc != GCS_OK) return rc;
    if (b->mem != GCS_MEM_HOST) return fail(GCS_E_INVALID, "this entry point needs host pointers (mem=GCS_MEM_HOST)");
    return host_range_entry(b, device, 0, b->n, wait);
}

}  // namespace

int gcs_b200_solve_host(const gcs_b200_batch* b, int device) { return host_entry(b, device, true); }

int gcs_b200_solve_host_async(const gcs_b200_batch* b, int device) { return host_entry(b, device, false); }

int gcs_b200_solve_host_range_async(const gcs_b200_batch* b, int device, int64_t first, int64_t count)
{
    int rc = validate(b);
    if (rc != GCS_OK) return rc;
    if (b->mem != GCS_MEM_HOST) return fail(GCS_E_INVALID, "this entry point needs host pointers (mem=GCS_MEM_HOST)");
    if (first < 0 || count < 0 || first > b->n || count > b->n - first)
        return fail(GCS_E_INVALID, "index range [%lld, %lld) outside the batch of %lld", (long long)first,
            (long long)(first + count), (long long)b->n);
    return host_range_entry(b, device, first, count, false);
}

int gcs_b200_wait(int device)
{
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    if (!d->tickets) return GCS_OK;  // never used
    std::lock_guard<std::mutex> lk(d->arena_mu);
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    rc = drain(d);
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    return rc;
}

int gcs_b200_solve_sharded(const gcs_b200_batch* b, int n_dev)
{
    int rc = validate(b);
    if (rc != GCS_OK) return rc;
    if (b->mem != GCS_MEM_HOST) return fail(GCS_E_INVALID, "gcs_b200_solve_sharded needs host pointers");
    rc = ensure_init();
    if (rc != GCS_OK) return rc;
    // the devices of the last gcs_b200_init, in its order; without one, ordinals 0..count-1
    std::vector<int> list;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        list = g_init_list;
    }
    if (list.empty())
        for (int i = 0; i < (int)g_devs.size(); ++i) list.push_back(i);
    const int avail = (int)list.size();
    if (n_dev <= 0) n_dev = avail;
    if (n_dev > avail) return fail(GCS_E_NO_DEVICE, "%d devices requested, %d initialised", n_dev, avail);
    // One pipeline per device, all enqueued from this thread before any is waited for; every
    // device fills its own index range of the caller's arrays (the per-seed planes keep the
    // full batch's pitch), so nothing is gathered afterwards and nothing crosses between devices.
    const int64_t n = b->n;
    int first_rc = GCS_OK;
    std::string first_msg;
    int enqueued = 0;
    for (int g = 0; g < n_dev && first_rc == GCS_OK; ++g) {
        const int64_t lo = n * g / n_dev, hi = n * (g + 1) / n_dev;
        rc = host_range_entry(b, list[g], lo, hi - lo, false);
        if (rc != GCS_OK) first_rc = rc, first_msg = "shard " + std::to_string(g) + " (device " + std::to_string(list[g]) + "): " + g_err;
        ++enqueued;
    }
    for (int g = 0; g < enqueued; ++g) {
        rc = gcs_b200_wait(list[g]);
        if (rc != GCS_OK && first_rc == GCS_OK) first_rc = rc, first_msg = "shard " + std::to_string(g) + ": " + g_err;
    }
    if (first_rc != GCS_OK) return fail(first_rc, "%s", first_msg.c_str());
    return GCS_OK;
}

int gcs_b200_contracted_stats_ex(int device, uint64_t out[8], int reset);

int gcs_b200_debug_path_buffer(int device, uint8_t* dev_buf, int64_t capacity)
{
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    if (capacity < 0) return fail(GCS_E_INVALID, "negative capacity");
    d->dbg_path = capacity > 0 ? dev_buf : nullptr;
    d->dbg_path_cap = d->dbg_path ? capacity : 0;
    return GCS_OK;
}

int gcs_b200_contracted_stats(int device, uint64_t out[2], int reset)
{
    uint64_t v[8] = {};
    const int rc = gcs_b200_contracted_stats_ex(device, v, reset);
    if (rc != GCS_OK) return rc;
    if (out) {
        out[1] = v[gcsk::kWhySelection];
        out[0] = 0;
        for (int k = 0; k < gcsk::kWhyCount; ++k)
            if (k != gcsk::kWhySelection) out[0] += v[k];
    }
    return GCS_OK;
}

int gcs_b200_contracted_stats_ex(int device, uint64_t out[8], int reset)
{
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaDeviceSynchronize());
    unsigned long long v[gcsk::kWhyCount] = {};
    CUDA_TRY(cudaMemcpyFromSymbol(v, gcsk::g_relax_reruns, sizeof(v)));
    if (reset) {
        const unsigned long long z[gcsk::kWhyCount] = {};
        CUDA_TRY(cudaMemcpyToSymbol(gcsk::g_relax_reruns, z, sizeof(z)));
    }
    if (out)
        for (int k = 0; k < gcsk::kWhyCount; ++k) out[k] = v[k];
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    return GCS_OK;
}

double gcs_b200_fp64_probe(int device, int what)
{
    int rc = ensure_init();
    if (rc != GCS_OK) return (double)rc;
    DeviceState* d = find_dev(device);
    if (!d) return (double)fail(GCS_E_NO_DEVICE, "device %d not present", device);
    rc = prepare_device(d);
    if (rc != GCS_OK) return (double)rc;
    if (cudaSetDevice(device) != cudaSuccess) return (double)GCS_E_CUDA;
    double* out = nullptr;
    const int blocks = d->sm_count * 8, threads = 256, iters = 20000;
    if (cudaMalloc(&out, sizeof(double) * blocks * threads + 64) != cudaSuccess) return (double)GCS_E_NOMEM;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0), cudaEventCreate(&e1);
    double result = 0.0;
    if (what == 0 || what == 1) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            cudaEventRecord(e0, d->stream);
            if (what == 0)
                fp64_probe_kernel<0><<<blocks, threads, 0, d->stream>>>(out, iters, 1.0);
            else
                fp64_probe_kernel<1><<<blocks, threads, 0, d->stream>>>(out, iters, 1.0);
            cudaEventRecord(e1, d->stream);
            cudaEventSynchronize(e1);
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep > 0 && ms < best) best = ms;
        }
        const double ops = (double)blocks * threads * (double)iters * 8.0;
        const double flops = ops * (what == 0 ? 2.0 : 1.0);
        result = flops / (best * 1e-3) / 1e12;
    } else if (what >= 1000) {
        // what = 1000 + 100*ILP + warps per SM  -> DFMA lanes per SM per clock
        const int ilp = (what / 100) % 10, warps = what % 100;
        if (warps < 1 || warps > 32) {
            cudaFree(out);
            return (double)fail(GCS_E_INVALID, "probe: warps per SM must be 1..32");
        }
        long long* cyc = nullptr;
        cudaMalloc(&cyc, sizeof(long long) * d->sm_count);
        const int it = 2000;
        for (int rep = 0; rep < 2; ++rep) {
            switch (ilp) {
            case 1: fp64_curve_kernel<1><<<d->sm_count, warps * 32, 0, d->stream>>>(out, cyc, it, 1.0); break;
            case 2: fp64_curve_kernel<2><<<d->sm_count, warps * 32, 0, d->stream>>>(out, cyc, it, 1.0); break;
            case 4: fp64_curve_kernel<4><<<d->sm_count, warps * 32, 0, d->stream>>>(out, cyc, it, 1.0); break;
            default: fp64_curve_kernel<8><<<d->sm_count, warps * 32, 0, d->stream>>>(out, cyc, it, 1.0); break;
            }
        }
        cudaStreamSynchronize(d->stream);
        long long h = 0;
        cudaMemcpy(&h, cyc, sizeof(h), cudaMemcpyDeviceToHost);
        cudaFree(cyc);
        const int eff_ilp = (ilp == 1 || ilp == 2 || ilp == 4) ? ilp : 8;
        result = (double)warps * 32.0 * it * 8.0 * eff_ilp / (double)h;
    } else {
        long long* cyc = reinterpret_cast<long long*>(out + (size_t)blocks * threads);
        fp64_latency_kernel<<<1, 32, 0, d->stream>>>(out, cyc, 4096, 1.0);
        fp64_latency_kernel<<<1, 32, 0, d->stream>>>(out, cyc, 4096, 1.0);
        cudaStreamSynchronize(d->stream);
        long long h = 0;
        cudaMemcpy(&h, cyc, sizeof(h), cudaMemcpyDeviceToHost);
        result = (double)h / (4096.0 * 8.0);
    }
    cudaError_t e = cudaGetLastError();
    cudaEventDestroy(e0), cudaEventDestroy(e1);
    cudaFree(out);
    if (e != cudaSuccess) return (double)fail(GCS_E_CUDA, "fp64 probe: %s", cudaGetErrorString(e));
    return result;
}

// Copy-only probe of the host link: what the host-buffer entry points could reach at best with the
// same byte counts.  Pinned (optionally write-combined) host buffers, `pieces` equal copies per
// direction (1 = one contiguous copy; the pipeline moves stage-sized pieces), the two directions on
// the library's two copy streams.  out[0] = H2D alone GB/s, out[1] = D2H alone GB/s, out[2] =
// milliseconds for both directions issued together (best of `reps`), out[3] = the same, median.
int gcs_b200_pcie_probe(int device, size_t bytes_up, size_t bytes_down, int pieces, int write_combined, int reps, double out[4])
{
    if (!out || pieces < 1 || reps < 1 || bytes_up == 0 || bytes_down == 0) return fail(GCS_E_INVALID, "bad probe arguments");
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    rc = prepare_device(d);
    if (rc != GCS_OK) return rc;
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    void *hu = nullptr, *hd = nullptr, *du = nullptr, *dd = nullptr;
    cudaEvent_t e[4] = {};
    auto cleanup = [&]() {
        if (hu) cudaFreeHost(hu);
        if (hd) cudaFreeHost(hd);
        if (du) cudaFree(du);
        if (dd) cudaFree(dd);
        for (auto ev : e)
            if (ev) cudaEventDestroy(ev);
        if (cur != device && cur >= 0) cudaSetDevice(cur);
    };
    cudaError_t ce = cudaHostAlloc(&hu, bytes_up, cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u));
    if (ce == cudaSuccess) ce = cudaHostAlloc(&hd, bytes_down, cudaHostAllocPortable);
    if (ce == cudaSuccess) ce = cudaMalloc(&du, bytes_up);
    if (ce == cudaSuccess) ce = cudaMalloc(&dd, bytes_down);
    for (int k = 0; k < 4 && ce == cudaSuccess; ++k) ce = cudaEventCreate(&e[k]);
    if (ce != cudaSuccess) {
        cleanup();
        return fail(GCS_E_NOMEM, "pcie probe: %s", cudaGetErrorString(ce));
    }
    memset(hu, 1, bytes_up);
    auto up = [&]() {
        const size_t piece = (bytes_up / pieces + 255) / 256 * 256;
        for (size_t o = 0; o < bytes_up; o += piece)
            cudaMemcpyAsync((char*)du + o, (char*)hu + o, bytes_up - o < piece ? bytes_up - o : piece, cudaMemcpyHostToDevice, d->h2d);
    };
    auto down = [&]() {
        const size_t piece = (bytes_down / pieces + 255) / 256 * 256;
        for (size_t o = 0; o < bytes_down; o += piece)
            cudaMemcpyAsync((char*)hd + o, (char*)dd + o, bytes_down - o < piece ? bytes_down - o : piece, cudaMemcpyDeviceToHost, d->d2h);
    };
    std::vector<double> both;
    double best_up = 1e30, best_down = 1e30;
    for (int r = 0; r < reps + 1; ++r) {
        float ms = 0;
        cudaEventRecord(e[0], d->h2d), up(), cudaEventRecord(e[1], d->h2d);
        cudaEventSynchronize(e[1]);
        cudaEventElapsedTime(&ms, e[0], e[1]);
        if (r > 0 && ms < best_up) best_up = ms;
        cudaEventRecord(e[2], d->d2h), down(), cudaEventRecord(e[3], d->d2h);
        cudaEventSynchronize(e[3]);
        cudaEventElapsedTime(&ms, e[2], e[3]);
        if (r > 0 && ms < best_down) best_down = ms;
        // both directions at once: from the common start to the later of the two ends
        cudaEventRecord(e[0], d->h2d);
        cudaStreamWaitEvent(d->d2h, e[0], 0);
        up(), down();
        cudaEventRecord(e[1], d->h2d), cudaEventRecord(e[3], d->d2h);
        cudaEventSynchronize(e[1]), cudaEventSynchronize(e[3]);
        float a = 0, b2 = 0;
        cudaEventElapsedTime(&a, e[0], e[1]), cudaEventElapsedTime(&b2, e[0], e[3]);
        if (r > 0) both.push_back(a > b2 ? a : b2);
    }
    ce = cudaGetLastError();
    std::sort(both.begin(), both.end());
    out[0] = (double)bytes_up / (best_up * 1e-3) / 1e9;
    out[1] = (double)bytes_down / (best_down * 1e-3) / 1e9;
    out[2] = both.front();
    out[3] = both[both.size() / 2];
    cleanup();
    if (ce != cudaSuccess) return fail(GCS_E_CUDA, "pcie probe: %s", cudaGetErrorString(ce));
    return GCS_OK;
}

int gcs_b200_selftest_launch(uint64_t seed, long long n, unsigned long long* dev_counts, int sm_count);  // selftest.cu

int gcs_b200_selftest(int device, uint64_t seed, int64_t n, uint64_t counts[8])
{
    if (!counts || n < 0) return fail(GCS_E_INVALID, "bad selftest arguments");
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    DeviceState* d = find_dev(device);
    if (!d) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    rc = prepare_device(d);
    if (rc != GCS_OK) return rc;
    CUDA_TRY(cudaSetDevice(device));
    unsigned long long* dc = nullptr;
    CUDA_TRY(cudaMalloc(&dc, 8 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(dc, 0, 8 * sizeof(unsigned long long)));
    rc = gcs_b200_selftest_launch(seed, (long long)n, dc, d->sm_count);
    g_launches.fetch_add(1);
    cudaError_t e = cudaDeviceSynchronize();
    unsigned long long h[8] = {};
    if (e == cudaSuccess) e = cudaMemcpy(h, dc, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(dc);
    if (rc != 0 || e != cudaSuccess) return fail(GCS_E_CUDA, "selftest: %s", cudaGetErrorString(e));
    for (int k = 0; k < 8; ++k) counts[k] = h[k];
    return GCS_OK;
}

int gcs_b200_synth_pp_launch(void* cuda_stream, uint64_t seed, int64_t first, int64_t n,
    int perturb_of, double* const cols[6], uint8_t* code);  // synth.cu

int gcs_b200_synth_pp(int device, void* cuda_stream, uint64_t seed, int64_t first, int64_t n,
    int perturb_of, double* const cols[6], uint8_t* code)
{
    if (n < 0 || !cols || !code) return fail(GCS_E_INVALID, "bad synth arguments");
    for (int c = 0; c < 6; ++c)
        if (!cols[c]) return fail(GCS_E_INVALID, "synth column %d is null", c);
    int rc = ensure_init();
    if (rc != GCS_OK) return rc;
    if (!find_dev(device)) return fail(GCS_E_NO_DEVICE, "device %d not present", device);
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != device) CUDA_TRY(cudaSetDevice(device));
    rc = gcs_b200_synth_pp_launch(cuda_stream, seed, first, n, perturb_of, cols, code);
    g_launches.fetch_add(1);
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    if (rc != 0) return fail(GCS_E_CUDA, "synth launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return GCS_OK;
}

}  // extern "C"
