// sketch_program.cu — sketch programs (include/gcs_b200.h, "sketch programs"): the wave plan of a
// decomposed sketch kept on the device and run for K instances of its constraint values.
//
// Device layout.  The caller's tables are instance-major (values [K][n_values], positions
// [K][n_slots][4]).  The kind batches of a wave put the K instances of one row next to each other
// (sub-system (row r, instance j) at index r*K + j of its kind's batch), so the threads of a warp
// share a row recipe and write consecutive column entries.  The gather (gather_row, run by the
// gather kernel) is the device copy of the numeric half of the host packer (Gcs::B200 packNumeric,
// host/src/b200/leaf_batch.cpp): same reads, same operations in the same order, built with
// --fmad=false like every kernel of the library, so the columns it writes are the host's bit for bit.
//
// Tangent runs (gcs_b200_program_run_tangents) add one launch per wave after the scatter: the
// tangent kernel, one thread per (row, instance, direction t) with t fastest, so that consecutive
// threads read and write consecutive doubles of the instance-major tangent tables (dvalues
// [K][n_values][T], dpositions [K][n_slots][4][T]).  It runs gather_row on the tangents to form the
// row's input-column tangents, linearises the row at its chosen root (csrc/newton_tangent.cuh) and
// writes the target's tangents.  The K2 / K5 batches then also keep their candidate planes, whose
// chosen normal is the row's unknown.
//
// Recorded runs (gcs_b200_program_run_recorded) place every (wave, kind) batch at its own offset of
// one tape allocation (tape_layout) instead of reusing one set of batches for every wave, so that
// the batches of all waves (columns, flags, K2 / K5 candidate planes) survive the run.  The adjoint
// sweep (gcs_b200_program_adjoints) reads them back, waves from last to first, with two launches per
// wave: the adjoint kernel, one thread per (row, instance, cotangent t) with t fastest, takes the
// adjoints of what the row wrote (its target, and the anchors of a zero-fixed row), zeroes them and
// writes the row's contributions to the slots and values it read (gather_row_transpose) into a
// contribution buffer; the
// reduce kernel adds those into the working slot-adjoint table and the value adjoints, each table
// entry's contributions in ascending (row, role) order from reader lists built at create time.  No
// atomics: the result does not depend on K, the stream or the schedule.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <type_traits>
#include <vector>

#include "../../include/gcs_b200.h"
#include "newton_adjoint.cuh"

namespace gcsk {
int api_fail(int code, const char* msg);  // gcs_b200_api.cu: sets gcs_b200_last_error()
void api_count_launch();
}  // namespace gcsk

namespace {

int failf(int code, const char* fmt, ...)
{
    char buf[400];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    return gcsk::api_fail(code, buf);
}

#define PROG_TRY(expr)                                                                                    \
    do {                                                                                                  \
        cudaError_t e_ = (expr);                                                                          \
        if (e_ != cudaSuccess) return failf(GCS_E_CUDA, "%s -> %s (%s:%d)", #expr, cudaGetErrorString(e_), \
            __FILE__, __LINE__);                                                                          \
    } while (0)

#define PROG_RC(expr)                  \
    do {                               \
        const int rc_ = (expr);        \
        if (rc_ != GCS_OK) return rc_; \
    } while (0)

constexpr int kKinds = GCS_KIND_COUNT;
constexpr int kThreads = 256;

// Gcs::B200::kindOf / the roles' element types / the values each solver reads, by solver id
constexpr int kKindOfSolver[9] = { 0, GCS_KIND_PP, GCS_KIND_SDD, GCS_KIND_ANG, GCS_KIND_PP, GCS_KIND_SDD, GCS_KIND_PPL,
    GCS_KIND_PLL, GCS_KIND_ANG };
constexpr bool kRoleIsLine[9][3] = { {}, { 0, 0, 0 }, { 0, 0, 1 }, { 1, 0, 1 }, { 0, 0, 0 }, { 0, 0, 1 }, { 0, 1, 0 },
    { 1, 1, 0 }, { 1, 0, 1 } };
constexpr bool kReads[9][3] = { {}, { 1, 1, 1 }, { 1, 1, 1 }, { 1, 1, 1 }, { 0, 1, 1 }, { 0, 1, 1 }, { 0, 1, 1 },
    { 0, 1, 1 }, { 1, 0, 1 } };

// f(std::integral_constant<int, kind>()): f sees a kind known at run time as a compile-time
// constant.  The host (in_cols, out_cols) and the kernels' device lambdas share it; the pragma lets
// the one template call either.
#pragma nv_exec_check_disable
template <class F>
__host__ __device__ __forceinline__ auto with_kind(int kind, F&& f)
{
    switch (kind) {
    case GCS_KIND_PP: return f(std::integral_constant<int, GCS_KIND_PP>());
    case GCS_KIND_SDD: return f(std::integral_constant<int, GCS_KIND_SDD>());
    case GCS_KIND_PPL: return f(std::integral_constant<int, GCS_KIND_PPL>());
    case GCS_KIND_PLL: return f(std::integral_constant<int, GCS_KIND_PLL>());
    default: return f(std::integral_constant<int, GCS_KIND_ANG>());
    }
}

// a kind's input and output columns
__host__ __device__ __forceinline__ int in_cols(int kind)
{
    return with_kind(kind, [](auto K) { return gcsk::Sys<decltype(K)::value>::kCols; });
}

__host__ __device__ __forceinline__ int out_cols(int kind)
{
    return with_kind(kind, [](auto K) { return gcsk::Sys<decltype(K)::value>::kOut; });
}

// one wave: rows [seg[0], seg[5]) of the program relative to `rows`, kind k + 1 at [seg[k], seg[k+1])
struct WaveArgs {
    const gcs_b200_program_row* rows;
    long long seg[kKinds + 1];
    long long K;
    double* cols[kKinds];      // kind batch: input columns, then output columns, `cap` apart
    long long cap[kKinds];
    uint8_t* code[kKinds];
    uint8_t* root[kKinds];
    uint8_t* conv[kKinds];     // [2][n] of the launch
    double* cand[kKinds];      // [2][2][n] of the launch, K2 and K5 of tangent runs only
    double* pos;               // [K][n_slots][4]
    const double* val;         // [K][n_values]
    long long n_slots, n_values;
    uint32_t* nonconverged;    // [K] or null
    long long T;               // directions of a tangent run, cotangents of a sweep (0: plain run)
    double* dpos;              // [K][n_slots][4][T]
    const double* dval;        // [K][n_values][T]
    // adjoint sweep
    double* apos;              // working slot adjoints [K][n_slots][4][T]
    double* scon;              // slot contributions [rows][role a, b][4][K][T]
    double* vcon;              // value contributions [rows][v0, v1, v2][K][T]
    uint8_t* flag;             // [K][T]: a row without a root has a non-zero output adjoint
};

struct Where {
    long long r, j, i;  // row (relative to the wave), instance, index in the kind batch
    int k;              // kind - 1
};

// sub-system s = r * K + j of the wave
__device__ __forceinline__ void place(const WaveArgs& w, long long s, Where& at)
{
    at.r = s / w.K;
    at.j = s - at.r * w.K;
    int k = 0;
    while (at.r >= w.seg[k + 1]) ++k;
    at.k = k;
    at.i = (at.r - w.seg[k]) * w.K + at.j;
}

__device__ __forceinline__ bool locate(const WaveArgs& w, Where& at)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= w.seg[kKinds] * w.K) return false;
    place(w, t, at);
    return true;
}

// The gather of one row, solver by solver: its input columns and, for the zero-fixed solvers 1-3,
// the anchors it writes into the positions.  S provides
//   slot(role, q)  coordinate q of role a (0) or b (1), as a double&;
//   value(q)       v0 .. v2;
//   cst(i)         canvas constant i;
//   in(col, v)     writes input column col.
// program_gather_kernel runs it on the positions and values (GatherColumns), program_tangent_kernel
// on their tangents (GatherTangents, where every canvas constant is 0), so that each statement of the
// latter is the exact derivative of the former's.
template <class S>
__device__ __forceinline__ void gather_row(const gcs_b200_program_row& row, S& s)
{
    auto pa = [&](int q) -> double& { return s.slot(0, q); };
    auto pb = [&](int q) -> double& { return s.slot(1, q); };
    auto cst = [&](int i) { return s.cst(i); };
    auto in = [&](int col, double v) { s.in(col, v); };
    const double v0 = s.value(0), v1 = s.value(1), v2 = s.value(2);
    switch (row.solver) {
    case 1:  // ZeroFixedPointsTriangle: P1 -> (0, 0), P2 -> (d12, 0)
        pa(0) = 0.0, pa(1) = 0.0, pb(0) = v0, pb(1) = 0.0;
        in(0, 0.0), in(1, 0.0), in(2, v1), in(3, v0), in(4, 0.0), in(5, v2);
        break;
    case 4:  // TwoFixedPointsDistance
        in(0, pa(0)), in(1, pa(1)), in(2, v1), in(3, pb(0)), in(4, pb(1)), in(5, v2);
        break;
    case 2:  // ZeroFixedPPLTriangle
        pa(0) = 0.0, pa(1) = 0.0, pb(0) = v0, pb(1) = 0.0;
        in(0, 0.0), in(1, 0.0), in(2, v0), in(3, 0.0);
        in(4, row.sign[1] * v1), in(5, row.sign[2] * v2), in(6, cst(0)), in(7, cst(1)), in(8, cst(2));
        break;
    case 5:  // TwoFixedPointsLine
        in(0, pa(0)), in(1, pa(1)), in(2, pb(0)), in(3, pb(1));
        in(4, row.sign[1] * v1), in(5, row.sign[2] * v2), in(6, cst(0)), in(7, cst(1)), in(8, cst(2));
        break;
    case 6:  // FixedPointAndLineFreePoint: a point, b line
        in(0, pa(0)), in(1, pa(1)), in(2, v1), in(3, pb(0)), in(4, pb(1)), in(5, pb(2)), in(6, pb(3));
        in(7, row.sign[2] * v2), in(8, cst(0)), in(9, cst(1));
        break;
    case 7:  // TwoFixedLinesFreePoint
        in(0, pa(0)), in(1, pa(1)), in(2, pa(2)), in(3, pa(3)), in(4, row.sign[1] * v1);
        in(5, pb(0)), in(6, pb(1)), in(7, pb(2)), in(8, pb(3)), in(9, row.sign[2] * v2);
        in(10, cst(0)), in(11, cst(1));
        break;
    case 3: {  // ZeroFixedLLPAngleTriangle: line1 -> (x1, 0)-(x2, 0), point -> (0, sign * d(P, line1)); v0 holds cos(angle)
        const double sd1 = row.sign[1] * v1;
        pa(0) = cst(7), pa(1) = 0.0, pa(2) = cst(8), pa(3) = 0.0;
        pb(0) = 0.0, pb(1) = sd1;
        in(0, cst(5)), in(1, cst(6)), in(2, v0), in(3, cst(0)), in(4, cst(1)), in(5, cst(2)), in(6, cst(3));
        in(7, 0.0), in(8, sd1), in(9, row.sign[2] * v2), in(10, 0.0), in(11, 0.0), in(12, cst(4));
        break;
    }
    case 8: {  // FixedLineAndPointFreeLine: a fixed line, b point; v0 holds cos(angle)
        const double p1x = pa(0), p1y = pa(1), p2x = pa(2), p2y = pa(3);
        in(0, p2x - p1x), in(1, p2y - p1y), in(2, v0), in(3, cst(0)), in(4, cst(1)), in(5, cst(2)), in(6, cst(3));
        in(7, pb(0)), in(8, pb(1)), in(9, row.sign[2] * v2), in(10, (p1x + p2x) / 2.0), in(11, (p1y + p2y) / 2.0);
        in(12, cst(4));
        break;
    }
    }
}

// The transpose of gather_row, for program_adjoint_kernel: from the input-column adjoints kb and the
// adjoint `anchor` of the anchor coordinate that holds a value (pb.x of solvers 1, 2 holds v0, pb.y
// of solver 3 holds sign1 * v1; the other anchor coordinates are constants), column adjoints first:
//   1: v0 = kb3 + pb.x, v1 = kb2, v2 = kb5          4: a = (kb0 kb1), v1 = kb2, b = (kb3 kb4), v2 = kb5
//   2: v0 = kb2 + pb.x, v1 = s1*kb4, v2 = s2*kb5    5: a = (kb0 kb1), b = (kb2 kb3), v1 = s1*kb4, v2 = s2*kb5
//   3: v0 = kb2, sd1 = kb8 + pb.y, v1 = s1*sd1, v2 = s2*kb9
//   6: a = (kb0 kb1), v1 = kb2, b = (kb3 .. kb6), v2 = s2*kb7
//   7: a = (kb0 .. kb3), v1 = s1*kb4, b = (kb5 .. kb8), v2 = s2*kb9
//   8: a = (kb10/2.0 - kb0, kb11/2.0 - kb1, kb10/2.0 + kb0, kb11/2.0 + kb1), b = (kb7 kb8), v0 = kb2,
//      v2 = s2*kb9
// sa(role, q, x) receives the adjoint of coordinate q of role a (0) or b (1), va(q, x) that of vq.
// Written out rather than derived from gather_row: the restatement in the test suite pins these
// addition orders and signed zeros, which a mechanical transpose of the recipe would change in
// cases 1, 2, 3 and 8.
template <class SA, class VA>
__device__ __forceinline__ void gather_row_transpose(const gcs_b200_program_row& row, const double* kb, double anchor, SA&& sa, VA&& va)
{
    const double s1 = row.sign[1], s2 = row.sign[2];
    switch (row.solver) {
    case 1: va(0, kb[3] + anchor), va(1, kb[2]), va(2, kb[5]); break;
    case 4:
        sa(0, 0, kb[0]), sa(0, 1, kb[1]), va(1, kb[2]), sa(1, 0, kb[3]), sa(1, 1, kb[4]), va(2, kb[5]);
        break;
    case 2: va(0, kb[2] + anchor), va(1, s1 * kb[4]), va(2, s2 * kb[5]); break;
    case 5:
        sa(0, 0, kb[0]), sa(0, 1, kb[1]), sa(1, 0, kb[2]), sa(1, 1, kb[3]), va(1, s1 * kb[4]), va(2, s2 * kb[5]);
        break;
    case 6:
        sa(0, 0, kb[0]), sa(0, 1, kb[1]), va(1, kb[2]);
        sa(1, 0, kb[3]), sa(1, 1, kb[4]), sa(1, 2, kb[5]), sa(1, 3, kb[6]), va(2, s2 * kb[7]);
        break;
    case 7:
        sa(0, 0, kb[0]), sa(0, 1, kb[1]), sa(0, 2, kb[2]), sa(0, 3, kb[3]), va(1, s1 * kb[4]);
        sa(1, 0, kb[5]), sa(1, 1, kb[6]), sa(1, 2, kb[7]), sa(1, 3, kb[8]), va(2, s2 * kb[9]);
        break;
    case 3: va(0, kb[2]), va(1, s1 * (kb[8] + anchor)), va(2, s2 * kb[9]); break;
    case 8: {
        const double mx = kb[10] / 2.0, my = kb[11] / 2.0;
        sa(0, 0, mx - kb[0]), sa(0, 1, my - kb[1]), sa(0, 2, mx + kb[0]), sa(0, 3, my + kb[1]);
        sa(1, 0, kb[7]), sa(1, 1, kb[8]), va(0, kb[2]), va(2, s2 * kb[9]);
        break;
    }
    }
}

// value vq of a row, from a table whose entries are `stride` doubles apart (0 where it reads none)
__device__ __forceinline__ double row_value(const gcs_b200_program_row& row, int q, const double* val, long long stride)
{
    return row.value[q] >= 0 ? val[row.value[q] * stride] : 0.0;
}

// gather_row's two sides.  Both take what the row reads (its slots a, b and v0 .. v2) once, before
// the switch: with the accessors reading row.elem / row.value at every use, the compiler reloads
// them, and the gather kernel takes a quarter more instructions.
struct GatherColumns {  // instance j: anchors into its positions, columns into the kind batch
    double* pa;
    double* pb;
    double v[3];
    const double* canvas;
    double* cols;
    long long cap, i;
    __device__ __forceinline__ double& slot(int role, int q) { return (role ? pb : pa)[q]; }
    __device__ __forceinline__ double value(int q) const { return v[q]; }
    __device__ __forceinline__ double cst(int c) const { return canvas[c]; }
    __device__ __forceinline__ void in(int col, double x) { cols[col * cap + i] = x; }
};

struct GatherTangents {  // their tangents along one direction, coordinates T apart; columns into kd
    double* pa;
    double* pb;
    double v[3];
    long long T;
    double kd[13];
    __device__ __forceinline__ double& slot(int role, int q) { return (role ? pb : pa)[q * T]; }
    __device__ __forceinline__ double value(int q) const { return v[q]; }
    __device__ __forceinline__ double cst(int) const { return 0.0; }
    __device__ __forceinline__ void in(int col, double x) { kd[col] = x; }
};

__global__ void __launch_bounds__(kThreads) program_gather_kernel(const WaveArgs w)
{
    Where at;
    if (!locate(w, at)) return;
    const gcs_b200_program_row& row = w.rows[at.r];
    double* const pos = w.pos + at.j * w.n_slots * 4;
    const double* const val = w.val + at.j * w.n_values;
    GatherColumns s { pos + 4 * (long long)row.elem[0], pos + 4 * (long long)row.elem[1],
        { row_value(row, 0, val, 1), row_value(row, 1, val, 1), row_value(row, 2, val, 1) }, row.canvas, w.cols[at.k],
        w.cap[at.k], at.i };
    w.code[at.k][at.i] = (uint8_t)row.code;
    gather_row(row, s);
}

// The scatter's test: the row's chosen run converged, so its output is a root.  Also gives the
// chosen seed and n, the kind's sub-systems in the launch.
__device__ __forceinline__ bool chosen_root(const WaveArgs& w, const Where& at, unsigned& root, long long& n)
{
    n = (w.seg[at.k + 1] - w.seg[at.k]) * w.K;
    root = w.root[at.k][at.i];
    if (root >= 2) return false;
    return w.conv[at.k][root * n + at.i] != 0;
}

__global__ void __launch_bounds__(kThreads) program_scatter_kernel(const WaveArgs w)
{
    Where at;
    if (!locate(w, at)) return;
    const gcs_b200_program_row& row = w.rows[at.r];
    const int nin = in_cols(at.k + 1), nout = out_cols(at.k + 1);
    const double* const c = w.cols[at.k];
    const long long cap = w.cap[at.k], i = at.i;
    double* const dst = w.pos + at.j * w.n_slots * 4 + 4 * (long long)row.elem[2];
    for (int q = 0; q < nout; ++q) dst[q] = c[(nin + q) * cap + i];
    unsigned root;
    long long n;
    if (w.nonconverged && !chosen_root(w, at, root, n)) atomicAdd(w.nonconverged + at.j, 1u);
}

// The linearisation of a converged row at its chosen root (chosen_root): its input columns, and the
// unknown there, the output point (K1, K3, K4) or the chosen seed's normal (K2, K5; candidate planes
// [2][2][n]).
template <int KIND>
__device__ __forceinline__ gcsk::RowTangent<KIND> linearisation(std::integral_constant<int, KIND>, const WaveArgs& w, const Where& at,
    unsigned root, long long n)
{
    constexpr int nin = gcsk::Sys<KIND>::kCols;
    const double* const c = w.cols[at.k];
    const long long cap = w.cap[at.k];
    double k[nin];
#pragma unroll
    for (int q = 0; q < nin; ++q) k[q] = c[q * cap + at.i];
    double ux, uy;
    if constexpr (KIND == GCS_KIND_SDD || KIND == GCS_KIND_ANG) {
        ux = w.cand[at.k][(root * 2 + 0) * n + at.i], uy = w.cand[at.k][(root * 2 + 1) * n + at.i];
    } else {
        ux = c[nin * cap + at.i], uy = c[(nin + 1) * cap + at.i];
    }
    gcsk::RowTangent<KIND> lin;
    lin.init(k, ux, uy);
    return lin;
}

__global__ void __launch_bounds__(kThreads) program_tangent_kernel(const WaveArgs w)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= w.seg[kKinds] * w.K * w.T) return;
    const long long T = w.T, s = g / T;
    Where at;
    place(w, s, at);
    const gcs_b200_program_row& row = w.rows[at.r];
    double* const dpos = w.dpos + at.j * w.n_slots * 4 * T + (g - s * T);
    const double* const dval = w.dval + at.j * w.n_values * T + (g - s * T);
    GatherTangents d { dpos + 4 * (long long)row.elem[0] * T, dpos + 4 * (long long)row.elem[1] * T,
        { row_value(row, 0, dval, T), row_value(row, 1, dval, T), row_value(row, 2, dval, T) }, T, {} };
    gather_row(row, d);
    const int kind = at.k + 1;
    unsigned root;
    long long n;
    double out[4];
    if (!chosen_root(w, at, root, n)) {
        // not a root, so the implicit function theorem does not apply
        out[0] = out[1] = out[2] = out[3] = __longlong_as_double(0x7ff8000000000000LL);
    } else {
        with_kind(kind, [&](auto K) { linearisation(K, w, at, root, n).apply(d.kd, out); });
    }
    double* const dst = dpos + 4 * (long long)row.elem[2] * T;
    for (int q = 0; q < out_cols(kind); ++q) dst[q * T] = out[q];
}

// One wave of the adjoint sweep, over the batches a recorded run kept.  The transpose of the
// scatter, the row's linearisation and the gather of program_tangent_kernel, in reverse:
//   1. ob = the adjoints of the target's written coordinates, which are then zeroed; for solvers
//      1-3 also the anchors the gather wrote (all zeroed, the one that holds a value kept);
//   2. a row whose chosen run did not converge has no derivative: a non-zero (or NaN) ob sets the
//      (instance, cotangent) flag and the row contributes kb = 0; otherwise kb = row_adjoint(ob);
//   3. gather_row_transpose, written to the contribution buffer (program_adjoint_reduce_kernel
//      adds them up).
__global__ void __launch_bounds__(kThreads) program_adjoint_kernel(const WaveArgs w)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= w.seg[kKinds] * w.K * w.T) return;
    const long long T = w.T, KT = w.K * T, s = g / T, t = g - s * T;
    Where at;
    place(w, s, at);
    const gcs_b200_program_row& row = w.rows[at.r];
    double* const apos = w.apos + at.j * w.n_slots * 4 * T + t;
    auto ap = [&](int slot, int q) -> double& { return apos[(4 * (long long)slot + q) * T]; };
    const int a = row.elem[0], b = row.elem[1], tgt = row.elem[2];
    const int kind = at.k + 1, nout = out_cols(kind);
    double ob[4] = {};
    for (int q = 0; q < nout; ++q) ob[q] = ap(tgt, q), ap(tgt, q) = 0.0;
    double anchor = 0.0;
    if (row.solver <= 3) {
        anchor = row.solver == 3 ? ap(b, 1) : ap(b, 0);
        for (int q = 0; q < (row.solver == 3 ? 4 : 2); ++q) ap(a, q) = 0.0;
        ap(b, 0) = 0.0, ap(b, 1) = 0.0;
    }
    unsigned root;
    long long n;
    double kb[13] = {};
    if (!chosen_root(w, at, root, n)) {
        bool touched = false;
        for (int q = 0; q < nout; ++q) touched |= !(ob[q] == 0.0);
        if (touched) w.flag[at.j * T + t] = 1;
    } else {
        with_kind(kind, [&](auto K) { gcsk::row_adjoint(linearisation(K, w, at, root, n), ob, kb); });
    }
    const long long jt = at.j * T + t;
    double* const sc = w.scon + at.r * 8 * KT + jt;  // [role][coordinate]
    double* const vc = w.vcon + at.r * 3 * KT + jt;  // [q]
    gather_row_transpose(row, kb, anchor, [&](int role, int q, double v) { sc[(role * 4 + q) * KT] = v; },
        [&](int q, double v) { vc[q * KT] = v; });
}

// reader lists of one wave: slot entries first (target slot, coordinates read), then value entries
struct AdjEntry {
    int32_t target;
    int32_t ncoord;  // 2 (point) or 4 (line) for a slot entry, 0 for a value entry
};

struct ReduceArgs {
    const AdjEntry* ent;        // the wave's entries
    const long long* begin;     // [n_ent + 1] into `readers`
    const long long* readers;   // slot entry: row * 2 + role; value entry: row * 3 + q (rows relative to the wave)
    long long n_ent, K, T;
    double* apos;               // [K][n_slots][4][T]
    double* aval;               // [K][n_values][T]
    const double* scon;
    const double* vcon;
    long long n_slots, n_values;
    const uint8_t* flag;        // [K][T] of the sweep (program_adjoint_flag_kernel)
};

// one thread per (entry, instance, cotangent): the entry's contributions added to its table entry
// one at a time, in the reader list's ascending (row, role) order
__global__ void __launch_bounds__(kThreads) program_adjoint_reduce_kernel(const ReduceArgs r)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long KT = r.K * r.T;
    if (g >= r.n_ent * KT) return;
    const long long e = g / KT, jt = g - e * KT, j = jt / r.T, t = jt - j * r.T;
    const AdjEntry en = r.ent[e];
    const long long lo = r.begin[e], hi = r.begin[e + 1];
    if (en.ncoord > 0) {
        double* const tab = r.apos + (j * r.n_slots + en.target) * 4 * r.T + t;
        for (int c = 0; c < en.ncoord; ++c) {
            double acc = tab[c * r.T];
            for (long long i = lo; i < hi; ++i) acc = acc + r.scon[(r.readers[i] * 4 + c) * KT + jt];
            tab[c * r.T] = acc;
        }
    } else {
        double* const tab = r.aval + (j * r.n_values + en.target) * r.T + t;
        double acc = *tab;
        for (long long i = lo; i < hi; ++i) acc = acc + r.vcon[r.readers[i] * KT + jt];
        *tab = acc;
    }
}

// the NaN rule, after wave 0: adj_values[k][:][t] = NaN where the (k, t) flag is set
__global__ void __launch_bounds__(kThreads) program_adjoint_flag_kernel(const ReduceArgs r)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= r.K * r.n_values * r.T) return;
    const long long j = g / (r.n_values * r.T), t = g % r.T;
    if (r.flag[j * r.T + t]) r.aval[g] = __longlong_as_double(0x7ff8000000000000LL);
}

int validate_desc(const gcs_b200_program_desc* d)
{
    if (!d) return failf(GCS_E_INVALID, "null program descriptor");
    if (d->n_waves < 0 || d->n_slots < 0 || d->n_values < 0 || d->n_rows < 0)
        return failf(GCS_E_INVALID, "negative count in the program descriptor");
    if (!d->offsets) return failf(GCS_E_INVALID, "null offsets");
    if ((d->n_rows > 0 && !d->rows) || (d->n_slots > 0 && (!d->slot_is_line || !d->initial)) || (d->n_values > 0 && !d->value_is_angle))
        return failf(GCS_E_INVALID, "null table in the program descriptor");
    const long long nseg = (long long)d->n_waves * kKinds;
    if (d->offsets[0] != 0) return failf(GCS_E_INVALID, "offsets[0] is %lld, not 0", (long long)d->offsets[0]);
    for (long long s = 0; s < nseg; ++s)
        if (d->offsets[s + 1] < d->offsets[s])
            return failf(GCS_E_INVALID, "offsets decrease at segment %lld (%lld after %lld)", s, (long long)d->offsets[s + 1], (long long)d->offsets[s]);
    if (d->offsets[nseg] != d->n_rows)
        return failf(GCS_E_INVALID, "offsets end at %lld, not at n_rows = %lld", (long long)d->offsets[nseg], (long long)d->n_rows);
    for (int s = 0; s < d->n_slots; ++s)
        if (d->slot_is_line[s] > 1) return failf(GCS_E_INVALID, "slot %d: type %d is neither point (0) nor line (1)", s, d->slot_is_line[s]);
    for (long long s = 0; s < nseg; ++s) {
        const int kind = (int)(s % kKinds) + 1;
        for (long long r = d->offsets[s]; r < d->offsets[s + 1]; ++r) {
            const gcs_b200_program_row& row = d->rows[r];
            if (row.solver < 1 || row.solver > 8) return failf(GCS_E_INVALID, "row %lld: unknown solver id %d", r, row.solver);
            if (kKindOfSolver[row.solver] != kind)
                return failf(GCS_E_INVALID, "row %lld: solver %d (kind %d) in a kind-%d segment", r, row.solver, kKindOfSolver[row.solver], kind);
            if (row.code < 0 || row.code > 255) return failf(GCS_E_INVALID, "row %lld: code %d out of range", r, row.code);
            for (int q = 0; q < 3; ++q) {
                const int e = row.elem[q];
                if (e < 0 || e >= d->n_slots) return failf(GCS_E_INVALID, "row %lld: element slot %d out of range (%d slots)", r, e, d->n_slots);
                if ((d->slot_is_line[e] != 0) != kRoleIsLine[row.solver][q])
                    return failf(GCS_E_INVALID, "row %lld: slot %d of role %c has the wrong element type for solver %d", r, e, 'a' + q, row.solver);
                const int v = row.value[q];
                if (!kReads[row.solver][q]) {
                    if (v != -1) return failf(GCS_E_INVALID, "row %lld: solver %d reads no v%d, value slot must be -1 (got %d)", r, row.solver, q, v);
                    continue;
                }
                if (v < 0 || v >= d->n_values) return failf(GCS_E_INVALID, "row %lld: value slot %d out of range (%d values)", r, v, d->n_values);
                const bool cosine = q == 0 && (row.solver == 3 || row.solver == 8);
                if ((d->value_is_angle[v] != 0) != cosine)
                    return failf(GCS_E_INVALID, "row %lld: value slot %d is %s an angle slot, v%d of solver %d needs %s", r, v,
                        d->value_is_angle[v] ? "" : "not", q, row.solver, cosine ? "one" : "a distance");
            }
            if (row.elem[0] == row.elem[1] || row.elem[0] == row.elem[2] || row.elem[1] == row.elem[2])
                return failf(GCS_E_INVALID, "row %lld: the three roles need three distinct slots", r);
        }
    }
    // The footprint rule of the wave plan (makePlan, host/src/b200/leaf_batch.cpp): within one wave
    // no slot is written by two rows, and no slot written by one row is read by another.  The rows
    // of a wave run concurrently, so otherwise the scatter's writes race, or a zero-fixed row's
    // anchors (written by the gather) race with another row's gather reading them.  Writes: a, b, c
    // of solvers 1-3, c of 4-8; reads: a, b of 4-8.  Per slot, the last wave that touched it, the
    // row that did and whether it wrote.
    std::vector<int> wave_of((size_t)d->n_slots, -1);
    std::vector<long long> row_of((size_t)d->n_slots);
    std::vector<char> wrote((size_t)d->n_slots);
    for (int wave = 0; wave < d->n_waves; ++wave) {
        for (long long r = d->offsets[(long long)wave * kKinds]; r < d->offsets[(long long)(wave + 1) * kKinds]; ++r) {
            const gcs_b200_program_row& row = d->rows[r];
            const bool zero_fixed = row.solver <= 3;
            for (int q = 0; q < 3; ++q) {
                const size_t e = (size_t)row.elem[q];
                const bool writes = zero_fixed || q == 2;
                if (wave_of[e] == wave && (writes || wrote[e]))
                    return failf(GCS_E_INVALID, "wave %d: slot %d is %s by row %lld and %s by row %lld; rows of one wave run concurrently", wave,
                        (int)e, wrote[e] ? "written" : "read", row_of[e], writes ? "written" : "read", r);
                if (wave_of[e] != wave || writes) wave_of[e] = wave, row_of[e] = r, wrote[e] = writes;
            }
        }
    }
    return GCS_OK;
}

// A device buffer that only grows.
template <class T>
struct DeviceBuffer {
    T* ptr = nullptr;
    size_t bytes = 0;  // allocated

    // device current; makes the buffer at least `need` bytes long.  The old buffer is freed once
    // `st`, whose work in flight may still use it, is done.  A failed allocation leaves the buffer
    // empty and fails with GCS_E_NOMEM, naming what the buffer is for (`what`, printf-style).
    int grow(size_t need, cudaStream_t st, const char* what, ...)
    {
        if (need <= bytes) return GCS_OK;
        if (ptr) {
            PROG_TRY(cudaStreamSynchronize(st));
            PROG_TRY(cudaFree(ptr));
            ptr = nullptr, bytes = 0;
        }
        if (cudaMalloc(&ptr, need) != cudaSuccess) {
            cudaGetLastError();
            ptr = nullptr;
            char buf[300];
            va_list ap;
            va_start(ap, what);
            vsnprintf(buf, sizeof(buf), what, ap);
            va_end(ap);
            return failf(GCS_E_NOMEM, "cudaMalloc(%zu) for %s failed", need, buf);
        }
        bytes = need;
        return GCS_OK;
    }
};

}  // namespace

struct gcs_b200_program {
    int device = 0;
    int n_waves = 0, n_slots = 0, n_values = 0;
    long long n_rows = 0;
    std::vector<long long> offsets;
    long long max_rows[kKinds] = {};  // most rows of a kind in one wave
    gcs_b200_program_row* rows = nullptr;
    double* initial = nullptr;
    cudaStream_t stream = nullptr;  // uploads and the _host entry points
    // the kind batches of plain and tangent runs, reused by every wave
    DeviceBuffer<unsigned char> scratch;
    // tables of the _host entry points: gcs_b200_program_run_host, and the tangent tables of
    // gcs_b200_program_run_tangents_host
    DeviceBuffer<double> values, positions;
    DeviceBuffer<uint32_t> counts;
    DeviceBuffer<double> dvalues, dpositions;
    // reader lists of the adjoint sweep, built at create time: the entries of wave w are
    // [ent_off[w], ent_off[w+1]) of `ent` (slot entries, then value entries), the readers of entry e
    // are readers[begin[e] .. begin[e+1])
    std::vector<long long> ent_off;
    AdjEntry* ent = nullptr;
    long long* begin = nullptr;
    long long* readers = nullptr;
    long long max_wave_rows = 0;
    // the tape of the last recorded run (every wave's kind batches) and its instance count (0: none)
    DeviceBuffer<unsigned char> tape;
    long long recorded_k = 0;
    // working tables of the sweep
    DeviceBuffer<double> apos;     // [K][n_slots][4][T]
    DeviceBuffer<double> contrib;  // [max_wave_rows][11][K][T]: slot, then value contributions
    DeviceBuffer<uint8_t> flags;   // [K][T]
    DeviceBuffer<double> avalues;  // [K][n_values][T] of gcs_b200_program_adjoints_host
    cudaEvent_t ev[4] = {};
};

namespace {

size_t align256(size_t v) { return (v + 255) / 256 * 256; }

// sub-systems a kind's columns are spaced for: K instances of the kind's largest wave, in multiples
// of 32 so that every column starts 256-byte aligned like the library's other device batches
long long kind_cap(const gcs_b200_program* p, int kind, long long K) { return (p->max_rows[kind - 1] * K + 31) / 32 * 32; }

bool has_cand(int kind, bool tangents) { return tangents && (kind == GCS_KIND_SDD || kind == GCS_KIND_ANG); }

// input and output columns, then code, root and the two convergence planes, then (tangent runs, K2
// and K5) the candidate planes
size_t kind_bytes(int kind, long long cap, bool tangents)
{
    return align256((size_t)(in_cols(kind) + out_cols(kind)) * cap * sizeof(double)) + 4 * align256((size_t)cap)
        + (has_cand(kind, tangents) ? align256((size_t)4 * cap * sizeof(double)) : 0);
}

// the kind batches with `cap[k]` sub-systems of kind k + 1
size_t batches_bytes(const long long cap[kKinds], bool cand)
{
    size_t bytes = 0;
    for (int k = 1; k <= kKinds; ++k) bytes += kind_bytes(k, cap[k - 1], cand);
    return bytes;
}

struct CurrentDevice {
    int prev = -1;
    explicit CurrentDevice(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) cudaGetLastError(), prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~CurrentDevice()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// the kind batches of one wave (or of the scratch) laid out from `at` with `cap[k]` sub-systems of
// kind k + 1
void bind_batches(WaveArgs& w, unsigned char* at, const long long cap[kKinds], bool cand)
{
    for (int k = 1; k <= kKinds; ++k) {
        w.cols[k - 1] = reinterpret_cast<double*>(at);
        w.cap[k - 1] = cap[k - 1];
        unsigned char* flags = at + align256((size_t)(in_cols(k) + out_cols(k)) * cap[k - 1] * sizeof(double));
        w.code[k - 1] = flags, w.root[k - 1] = flags + align256((size_t)cap[k - 1]), w.conv[k - 1] = flags + 2 * align256((size_t)cap[k - 1]);
        w.cand[k - 1] = has_cand(k, cand) ? reinterpret_cast<double*>(flags + 4 * align256((size_t)cap[k - 1])) : nullptr;
        at += kind_bytes(k, cap[k - 1], cand);
    }
}

// the tape's sub-system counts of wave `wave`: the wave's own rows x K, in multiples of 32
void tape_caps(const gcs_b200_program* p, int wave, long long K, long long cap[kKinds])
{
    const long long* off = p->offsets.data() + (size_t)wave * kKinds;
    for (int k = 0; k < kKinds; ++k) cap[k] = ((off[k + 1] - off[k]) * K + 31) / 32 * 32;
}

// The tape of a recorded run of K instances: the byte offset of every wave's kind batches (candidate
// planes included), then the tape's size.
std::vector<size_t> tape_layout(const gcs_b200_program* p, long long K)
{
    std::vector<size_t> at(1, 0);
    for (int wave = 0; wave < p->n_waves; ++wave) {
        long long cap[kKinds];
        tape_caps(p, wave, K, cap);
        at.push_back(at.back() + batches_bytes(cap, true));
    }
    return at;
}

// w's rows and segments for wave `wave`; with a tape layout (tape_layout of w.K), also its batches
// on the tape
void bind_wave(const gcs_b200_program* p, WaveArgs& w, int wave, const std::vector<size_t>* tape_at = nullptr)
{
    const long long* off = p->offsets.data() + (size_t)wave * kKinds;
    w.rows = p->rows + off[0];
    for (int k = 0; k <= kKinds; ++k) w.seg[k] = off[k] - off[0];
    if (tape_at) {
        long long cap[kKinds];
        tape_caps(p, wave, w.K, cap);
        bind_batches(w, p->tape.ptr + (*tape_at)[(size_t)wave], cap, true);
    }
}

// Launches `kernel` on `st` over `threads` threads (nothing when there are none) and counts the
// launch.  A grid beyond 31 bits fails, naming the work (`what`, printf-style).
template <class A>
int launch(void (*kernel)(A), long long threads, cudaStream_t st, const A& args, const char* what, ...)
{
    if (threads == 0) return GCS_OK;
    const long long grid = (threads + kThreads - 1) / kThreads;
    if (grid > 0x7fffffffLL) {
        char buf[300];
        va_list ap;
        va_start(ap, what);
        vsnprintf(buf, sizeof(buf), what, ap);
        va_end(ap);
        return failf(GCS_E_INVALID, "%s are too many for one launch", buf);
    }
    kernel<<<(unsigned)grid, kThreads, 0, st>>>(args);
    gcsk::api_count_launch();
    PROG_TRY(cudaGetLastError());
    return GCS_OK;
}

// T = 0: a plain run.  T > 0: also the tangents along T directions (dvalues / dpositions).
// recorded: every wave's batches at their own place of the tape (T = 0 only)
int run_on(gcs_b200_program* p, long long K, const double* values, double* positions, uint32_t* nonconverged, int variant,
    cudaStream_t st, long long T = 0, const double* dvalues = nullptr, double* dpositions = nullptr, bool recorded = false)
{
    WaveArgs w;
    memset(&w, 0, sizeof(w));
    w.K = K;
    w.pos = positions, w.val = values, w.n_slots = p->n_slots, w.n_values = p->n_values;
    w.nonconverged = nonconverged;
    w.T = T, w.dpos = dpositions, w.dval = dvalues;
    std::vector<size_t> tape_at;
    if (recorded) {
        p->recorded_k = 0;  // until this run is enqueued whole
        tape_at = tape_layout(p, K);
        PROG_RC(p->tape.grow(tape_at.back(), st, "the tape of a recorded run of %lld instances", K));
    } else {
        // K instances of every kind's largest wave
        long long cap[kKinds];
        for (int k = 1; k <= kKinds; ++k) cap[k - 1] = kind_cap(p, k, K);
        PROG_RC(p->scratch.grow(batches_bytes(cap, T > 0), st, "the kind batches of %lld instances", K));
        bind_batches(w, p->scratch.ptr, cap, T > 0);
    }
    // every instance starts from the initial positions: one copy, then doubling copies
    const size_t table = (size_t)p->n_slots * 4 * sizeof(double);
    if (table) {
        PROG_TRY(cudaMemcpyAsync(positions, p->initial, table, cudaMemcpyDeviceToDevice, st));
        for (long long have = 1; have < K;) {
            const long long n = have < K - have ? have : K - have;
            PROG_TRY(cudaMemcpyAsync(reinterpret_cast<unsigned char*>(positions) + (size_t)have * table, positions, (size_t)n * table,
                cudaMemcpyDeviceToDevice, st));
            have += n;
        }
    }
    if (nonconverged) PROG_TRY(cudaMemsetAsync(nonconverged, 0, (size_t)K * sizeof(uint32_t), st));
    // every slot's tangent is 0 before the first wave: the initial positions are constants
    if (T > 0 && table) PROG_TRY(cudaMemsetAsync(dpositions, 0, (size_t)K * T * table, st));
    for (int wave = 0; wave < p->n_waves; ++wave) {
        bind_wave(p, w, wave, recorded ? &tape_at : nullptr);
        const long long subs = w.seg[kKinds] * K;
        if (subs == 0) continue;
        PROG_RC(launch(program_gather_kernel, subs, st, w, "wave %d: %lld sub-systems", wave, subs));
        gcs_b200_batch batch[kKinds];
        const gcs_b200_batch* list[kKinds];
        int count = 0;
        for (int k = 1; k <= kKinds; ++k) {
            const long long n = (w.seg[k] - w.seg[k - 1]) * K;
            if (n == 0) continue;
            gcs_b200_batch& b = batch[count];
            memset(&b, 0, sizeof(b));
            b.kind = k, b.n_seeds = 2, b.n = n, b.mem = GCS_MEM_DEVICE, b.variant = variant;
            const long long cap = w.cap[k - 1];
            for (int c = 0; c < in_cols(k); ++c) b.in[c] = w.cols[k - 1] + c * cap;
            for (int c = 0; c < out_cols(k); ++c) b.out[c] = w.cols[k - 1] + (in_cols(k) + c) * cap;
            b.code = w.code[k - 1], b.root_index = w.root[k - 1], b.converged = w.conv[k - 1], b.cand = w.cand[k - 1];
            list[count++] = &b;
        }
        PROG_RC(gcs_b200_solve_many(list, count, p->device, st));
        PROG_RC(launch(program_scatter_kernel, subs, st, w, "wave %d: %lld sub-systems", wave, subs));
        if (T > 0)
            PROG_RC(launch(program_tangent_kernel, subs * T, st, w, "wave %d: %lld sub-systems x %lld directions", wave, subs, T));
    }
    if (recorded) p->recorded_k = K;
    return GCS_OK;
}

// device current; the sweep's working tables for the recorded K x T cotangents
int ensure_adjoint_tables(gcs_b200_program* p, long long T, cudaStream_t st)
{
    const long long K = p->recorded_k, KT = K * T;
    const size_t pbytes = (size_t)KT * p->n_slots * 4 * sizeof(double), cbytes = (size_t)KT * p->max_wave_rows * 11 * sizeof(double);
    const size_t vbytes = (size_t)KT * p->n_values * sizeof(double);
    const char* what = "the %s of %lld instances x %lld cotangents";
    PROG_RC(p->apos.grow(pbytes, st, what, "slot adjoints", K, T));
    PROG_RC(p->contrib.grow(cbytes, st, what, "adjoint contributions", K, T));
    PROG_RC(p->flags.grow((size_t)KT, st, what, "NaN flags", K, T));
    return p->avalues.grow(vbytes, st, what, "value adjoints", K, T);
}

// device current, checks done, p->apos holds the cotangents of the recorded run's positions: the
// sweep, waves from last to first, into adj_values [K][n_values][T]
int sweep_on(gcs_b200_program* p, long long T, double* adj_values, cudaStream_t st)
{
    const long long K = p->recorded_k, KT = K * T;
    if (p->n_values) PROG_TRY(cudaMemsetAsync(adj_values, 0, (size_t)KT * p->n_values * sizeof(double), st));
    PROG_TRY(cudaMemsetAsync(p->flags.ptr, 0, (size_t)KT, st));
    const std::vector<size_t> tape_at = tape_layout(p, K);
    WaveArgs w;
    memset(&w, 0, sizeof(w));
    w.K = K, w.T = T, w.n_slots = p->n_slots, w.n_values = p->n_values;
    w.apos = p->apos.ptr, w.flag = p->flags.ptr;
    w.scon = p->contrib.ptr, w.vcon = p->contrib.ptr + (size_t)p->max_wave_rows * 8 * KT;
    ReduceArgs r;
    memset(&r, 0, sizeof(r));
    r.K = K, r.T = T, r.apos = p->apos.ptr, r.aval = adj_values, r.scon = w.scon, r.vcon = w.vcon;
    r.n_slots = p->n_slots, r.n_values = p->n_values, r.flag = p->flags.ptr;
    for (int wave = p->n_waves - 1; wave >= 0; --wave) {
        bind_wave(p, w, wave, &tape_at);
        const long long subs = w.seg[kKinds] * K;
        if (subs == 0) continue;
        r.ent = p->ent + p->ent_off[(size_t)wave];
        r.begin = p->begin + p->ent_off[(size_t)wave];
        r.readers = p->readers;
        r.n_ent = p->ent_off[(size_t)wave + 1] - p->ent_off[(size_t)wave];
        const char* what = "wave %d: %lld sub-systems x %lld cotangents";
        PROG_RC(launch(program_adjoint_kernel, subs * T, st, w, what, wave, subs, T));
        PROG_RC(launch(program_adjoint_reduce_kernel, r.n_ent * KT, st, r, what, wave, subs, T));
    }
    return launch(program_adjoint_flag_kernel, KT * p->n_values, st, r, "%lld value adjoints", KT * p->n_values);
}

// the checks that need no program come first; a null table is refused unless the program has
// nothing to put in it
int check_adjoints(const gcs_b200_program* p, int T, const double* adj_positions, const double* adj_values)
{
    if (T < 1) return failf(GCS_E_INVALID, "n_cotangents must be >= 1 (got %d)", T);
    if ((!adj_positions && !(p && p->n_slots == 0)) || (!adj_values && !(p && p->n_values == 0)))
        return failf(GCS_E_INVALID, "null adjoint table (adj_positions or adj_values)");
    if (!p) return failf(GCS_E_INVALID, "null program");
    if (p->recorded_k < 1) return failf(GCS_E_INVALID, "no recorded run: call gcs_b200_program_run_recorded first");
    return GCS_OK;
}

int check_run(const gcs_b200_program* p, long long K, const double* values, const double* positions, int variant)
{
    if (!p) return failf(GCS_E_INVALID, "null program");
    if (K < 1) return failf(GCS_E_INVALID, "n_instances must be >= 1 (got %lld)", K);
    if ((p->n_values > 0 && !values) || (p->n_slots > 0 && !positions)) return failf(GCS_E_INVALID, "null value or position table");
    if (variant < GCS_VARIANT_DEFAULT || variant > GCS_VARIANT_CONTRACTED_LINEAR) return failf(GCS_E_INVALID, "unknown variant %d", variant);
    return GCS_OK;
}

// the checks that need no program come first; a null tangent table is refused unless the program
// has nothing to put in it
int check_tangent_run(const gcs_b200_program* p, long long K, const double* values, const double* positions, int T,
    const double* dvalues, const double* dpositions, int variant)
{
    if (T < 1) return failf(GCS_E_INVALID, "n_tangents must be >= 1 (got %d)", T);
    if (variant < GCS_VARIANT_DEFAULT || variant > GCS_VARIANT_CONTRACTED_LINEAR) return failf(GCS_E_INVALID, "unknown variant %d", variant);
    if ((!dvalues && !(p && p->n_values == 0)) || (!dpositions && !(p && p->n_slots == 0)))
        return failf(GCS_E_INVALID, "null tangent table (dvalues or dpositions)");
    return check_run(p, K, values, positions, variant);
}

// one copy of the _host entry points; none when `bytes` is 0
struct Copy {
    void* dst;
    const void* src;
    size_t bytes;
};

// Device current, checks done: a _host entry point on the program's stream.  The uploads, work(st),
// the downloads, then a synchronise; ms[0 .. 2] (unless null) the upload, device and download times.
template <class Work>
int on_host(gcs_b200_program* p, std::initializer_list<Copy> up, Work&& work, std::initializer_list<Copy> down, float ms[3])
{
    const cudaStream_t st = p->stream;
    PROG_TRY(cudaEventRecord(p->ev[0], st));
    for (const Copy& c : up)
        if (c.bytes) PROG_TRY(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyHostToDevice, st));
    PROG_TRY(cudaEventRecord(p->ev[1], st));
    const int rc = work(st);
    if (rc != GCS_OK) {
        cudaStreamSynchronize(st);
        return rc;
    }
    PROG_TRY(cudaEventRecord(p->ev[2], st));
    for (const Copy& c : down)
        if (c.bytes) PROG_TRY(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, st));
    PROG_TRY(cudaEventRecord(p->ev[3], st));
    PROG_TRY(cudaStreamSynchronize(st));
    if (ms)
        for (int q = 0; q < 3; ++q) PROG_TRY(cudaEventElapsedTime(&ms[q], p->ev[q], p->ev[q + 1]));
    return GCS_OK;
}

// device current, checks done
int run_host(gcs_b200_program* p, long long K, const double* values, double* positions, uint32_t* nonconverged, int variant,
    float ms[3], long long T = 0, const double* dvalues = nullptr, double* dpositions = nullptr, bool recorded = false)
{
    const size_t vbytes = (size_t)K * p->n_values * sizeof(double), pbytes = (size_t)K * p->n_slots * 4 * sizeof(double);
    const size_t cbytes = (size_t)K * sizeof(uint32_t);
    const cudaStream_t st = p->stream;
    PROG_RC(p->values.grow(vbytes, st, "the values of %lld instances", K));
    PROG_RC(p->positions.grow(pbytes, st, "the positions of %lld instances", K));
    PROG_RC(p->counts.grow(cbytes, st, "the nonconverged counts of %lld instances", K));
    PROG_RC(p->dvalues.grow(vbytes * T, st, "the value tangents of %lld instances x %lld directions", K, T));
    PROG_RC(p->dpositions.grow(pbytes * T, st, "the position tangents of %lld instances x %lld directions", K, T));
    return on_host(p, { { p->values.ptr, values, vbytes }, { p->dvalues.ptr, dvalues, vbytes * T } },
        [&](cudaStream_t s) {
            return run_on(p, K, p->values.ptr, p->positions.ptr, nonconverged ? p->counts.ptr : nullptr, variant, s, T, p->dvalues.ptr,
                p->dpositions.ptr, recorded);
        },
        { { positions, p->positions.ptr, pbytes }, { dpositions, p->dpositions.ptr, pbytes * T },
            { nonconverged, p->counts.ptr, nonconverged ? cbytes : 0 } },
        ms);
}

}  // namespace

extern "C" {

int gcs_b200_program_create(const gcs_b200_program_desc* d, int device, gcs_b200_program** out)
{
    if (!out) return failf(GCS_E_INVALID, "null output handle");
    *out = nullptr;
    int rc = validate_desc(d);
    if (rc != GCS_OK) return rc;
    const int ndev = gcs_b200_device_count();
    if (ndev <= 0) return failf(GCS_E_NO_DEVICE, "no CUDA device; this library has no CPU fallback");
    if (device < 0 || device >= ndev) return failf(GCS_E_NO_DEVICE, "device %d out of range (%d present)", device, ndev);
    CurrentDevice cur(device);
    auto* p = new gcs_b200_program();
    p->device = device, p->n_waves = d->n_waves, p->n_slots = d->n_slots, p->n_values = d->n_values, p->n_rows = d->n_rows;
    p->offsets.assign(d->offsets, d->offsets + (size_t)d->n_waves * kKinds + 1);
    for (int w = 0; w < d->n_waves; ++w)
        for (int k = 0; k < kKinds; ++k) {
            const long long rows = p->offsets[(size_t)w * kKinds + k + 1] - p->offsets[(size_t)w * kKinds + k];
            if (rows > p->max_rows[k]) p->max_rows[k] = rows;
        }
    auto bail = [&](int code) {
        gcs_b200_program_destroy(p);
        return code;
    };
    if (cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(failf(GCS_E_CUDA, "stream creation failed"));
    for (auto& e : p->ev)
        if (cudaEventCreate(&e) != cudaSuccess) return bail(failf(GCS_E_CUDA, "event creation failed"));
    const size_t row_bytes = (size_t)d->n_rows * sizeof(gcs_b200_program_row), init_bytes = (size_t)d->n_slots * 4 * sizeof(double);
    if ((row_bytes && cudaMalloc(&p->rows, row_bytes) != cudaSuccess) || (init_bytes && cudaMalloc(&p->initial, init_bytes) != cudaSuccess)) {
        cudaGetLastError();
        return bail(failf(GCS_E_NOMEM, "cudaMalloc for a program of %lld rows and %d slots failed", (long long)d->n_rows, d->n_slots));
    }
    // The reader lists of the adjoint sweep.  Per wave, every slot read (roles a, b of solvers 4-8)
    // and every value read gets one entry, slots first; its readers, (row, role) for a slot and (row,
    // q) for a value with rows relative to the wave, are listed in ascending order.
    std::vector<AdjEntry> ent;
    std::vector<long long> begin(1, 0), readers;
    {
        std::vector<long long> slot_ent((size_t)d->n_slots, -1), value_ent((size_t)d->n_values, -1);
        std::vector<std::vector<long long>> lists;
        p->ent_off.assign(1, 0);
        for (int wave = 0; wave < d->n_waves; ++wave) {
            const long long lo = d->offsets[(long long)wave * kKinds], hi = d->offsets[(long long)(wave + 1) * kKinds];
            if (hi - lo > p->max_wave_rows) p->max_wave_rows = hi - lo;
            const size_t first = ent.size();
            lists.clear();
            for (int pass = 0; pass < 2; ++pass)  // slots, then values
                for (long long r = lo; r < hi; ++r) {
                    const gcs_b200_program_row& row = d->rows[r];
                    for (int q = 0; q < 3; ++q) {
                        const bool slot_read = pass == 0 && q < 2 && row.solver >= 4;
                        const bool value_read = pass == 1 && row.value[q] >= 0;
                        if (!slot_read && !value_read) continue;
                        const int target = slot_read ? row.elem[q] : row.value[q];
                        long long& e = (slot_read ? slot_ent : value_ent)[(size_t)target];
                        if (e < 0) {
                            e = (long long)lists.size();
                            lists.emplace_back();
                            ent.push_back({ target, slot_read ? (kRoleIsLine[row.solver][q] ? 4 : 2) : 0 });
                        }
                        lists[(size_t)e].push_back(slot_read ? (r - lo) * 2 + q : (r - lo) * 3 + q);
                    }
                }
            for (size_t e = first; e < ent.size(); ++e) {
                const std::vector<long long>& l = lists[e - first];
                readers.insert(readers.end(), l.begin(), l.end());
                begin.push_back((long long)readers.size());
                (ent[e].ncoord ? slot_ent : value_ent)[(size_t)ent[e].target] = -1;
            }
            p->ent_off.push_back((long long)ent.size());
        }
    }
    const size_t ent_bytes = ent.size() * sizeof(AdjEntry), begin_bytes = begin.size() * sizeof(long long);
    const size_t reader_bytes = readers.size() * sizeof(long long);
    if ((ent_bytes && cudaMalloc(&p->ent, ent_bytes) != cudaSuccess) || cudaMalloc(&p->begin, begin_bytes) != cudaSuccess
        || (reader_bytes && cudaMalloc(&p->readers, reader_bytes) != cudaSuccess)) {
        cudaGetLastError();
        return bail(failf(GCS_E_NOMEM, "cudaMalloc for the reader lists of %zu entries failed", ent.size()));
    }
    if ((row_bytes && cudaMemcpyAsync(p->rows, d->rows, row_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || (init_bytes && cudaMemcpyAsync(p->initial, d->initial, init_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || (ent_bytes && cudaMemcpyAsync(p->ent, ent.data(), ent_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || cudaMemcpyAsync(p->begin, begin.data(), begin_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess
        || (reader_bytes && cudaMemcpyAsync(p->readers, readers.data(), reader_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || cudaStreamSynchronize(p->stream) != cudaSuccess)
        return bail(failf(GCS_E_CUDA, "program upload failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = p;
    return GCS_OK;
}

int gcs_b200_program_run(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged, int variant,
    void* stream)
{
    PROG_RC(check_run(p, K, values, positions, variant));
    CurrentDevice cur(p->device);
    return run_on(p, K, values, positions, nonconverged, variant, static_cast<cudaStream_t>(stream));
}

int gcs_b200_program_run_host(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int variant, float ms[3])
{
    PROG_RC(check_run(p, K, values, positions, variant));
    CurrentDevice cur(p->device);
    return run_host(p, K, values, positions, nonconverged, variant, ms);
}

int gcs_b200_program_run_tangents(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int32_t T, const double* dvalues, double* dpositions, int variant, void* stream)
{
    PROG_RC(check_tangent_run(p, K, values, positions, T, dvalues, dpositions, variant));
    CurrentDevice cur(p->device);
    return run_on(p, K, values, positions, nonconverged, variant, static_cast<cudaStream_t>(stream), T, dvalues, dpositions);
}

int gcs_b200_program_run_tangents_host(gcs_b200_program* p, int64_t K, const double* values, double* positions,
    uint32_t* nonconverged, int32_t T, const double* dvalues, double* dpositions, int variant, float ms[3])
{
    PROG_RC(check_tangent_run(p, K, values, positions, T, dvalues, dpositions, variant));
    CurrentDevice cur(p->device);
    return run_host(p, K, values, positions, nonconverged, variant, ms, T, dvalues, dpositions);
}

int gcs_b200_program_run_recorded(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int variant, void* stream)
{
    PROG_RC(check_run(p, K, values, positions, variant));
    CurrentDevice cur(p->device);
    return run_on(p, K, values, positions, nonconverged, variant, static_cast<cudaStream_t>(stream), 0, nullptr, nullptr, true);
}

int gcs_b200_program_run_recorded_host(gcs_b200_program* p, int64_t K, const double* values, double* positions,
    uint32_t* nonconverged, int variant, float ms[3])
{
    PROG_RC(check_run(p, K, values, positions, variant));
    CurrentDevice cur(p->device);
    return run_host(p, K, values, positions, nonconverged, variant, ms, 0, nullptr, nullptr, true);
}

int gcs_b200_program_adjoints(gcs_b200_program* p, int32_t T, const double* adj_positions, double* adj_values, void* stream)
{
    PROG_RC(check_adjoints(p, T, adj_positions, adj_values));
    CurrentDevice cur(p->device);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    PROG_RC(ensure_adjoint_tables(p, T, st));
    const size_t pbytes = (size_t)p->recorded_k * T * p->n_slots * 4 * sizeof(double);
    if (pbytes) PROG_TRY(cudaMemcpyAsync(p->apos.ptr, adj_positions, pbytes, cudaMemcpyDeviceToDevice, st));
    return sweep_on(p, T, adj_values, st);
}

int gcs_b200_program_adjoints_host(gcs_b200_program* p, int32_t T, const double* adj_positions, double* adj_values, float ms[3])
{
    PROG_RC(check_adjoints(p, T, adj_positions, adj_values));
    CurrentDevice cur(p->device);
    PROG_RC(ensure_adjoint_tables(p, T, p->stream));
    const size_t pbytes = (size_t)p->recorded_k * T * p->n_slots * 4 * sizeof(double);
    const size_t vbytes = (size_t)p->recorded_k * T * p->n_values * sizeof(double);
    return on_host(p, { { p->apos.ptr, adj_positions, pbytes } }, [&](cudaStream_t st) { return sweep_on(p, T, p->avalues.ptr, st); },
        { { adj_values, p->avalues.ptr, vbytes } }, ms);
}

void gcs_b200_program_destroy(gcs_b200_program* p)
{
    if (!p) return;
    {
        CurrentDevice cur(p->device);
        if (p->stream) cudaStreamSynchronize(p->stream), cudaStreamDestroy(p->stream);
        for (auto e : p->ev)
            if (e) cudaEventDestroy(e);
        cudaFree(p->rows), cudaFree(p->initial), cudaFree(p->scratch.ptr);
        cudaFree(p->values.ptr), cudaFree(p->positions.ptr), cudaFree(p->counts.ptr);
        cudaFree(p->dvalues.ptr), cudaFree(p->dpositions.ptr);
        cudaFree(p->ent), cudaFree(p->begin), cudaFree(p->readers), cudaFree(p->tape.ptr);
        cudaFree(p->apos.ptr), cudaFree(p->contrib.ptr), cudaFree(p->flags.ptr), cudaFree(p->avalues.ptr);
        cudaGetLastError();
    }
    delete p;
}

}  // extern "C"
