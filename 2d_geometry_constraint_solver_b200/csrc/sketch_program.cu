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
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <type_traits>
#include <vector>

#include "../../include/gcs_b200.h"
#include "api_common.cuh"
#include "newton_adjoint.cuh"

using gcsk::DeviceScope;
using gcsk::fail;
using gcsk::in_cols;
using gcsk::out_cols;
using gcsk::with_kind;

namespace {

constexpr int kKinds = GCS_KIND_COUNT;
constexpr int kThreads = 256;

// Gcs::B200::kindOf / the roles' element types / the values each solver reads, by solver id
constexpr int kKindOfSolver[9] = { 0, GCS_KIND_PP, GCS_KIND_SDD, GCS_KIND_ANG, GCS_KIND_PP, GCS_KIND_SDD, GCS_KIND_PPL,
    GCS_KIND_PLL, GCS_KIND_ANG };
constexpr bool kRoleIsLine[9][3] = { {}, { 0, 0, 0 }, { 0, 0, 1 }, { 1, 0, 1 }, { 0, 0, 0 }, { 0, 0, 1 }, { 0, 1, 0 },
    { 1, 1, 0 }, { 1, 0, 1 } };
constexpr bool kReads[9][3] = { {}, { 1, 1, 1 }, { 1, 1, 1 }, { 1, 1, 1 }, { 0, 1, 1 }, { 0, 1, 1 }, { 0, 1, 1 },
    { 0, 1, 1 }, { 1, 0, 1 } };

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

// ---- fused runs (gcs_b200_program_run_fused): every wave in one cooperative launch ----
// One thread per (row, instance) of a wave does what the wave path spreads over the gather, the kind
// batch's solve, the scatter and the tangent kernel, with the columns in registers instead of a kind
// batch: gather_row, then newton_pair_kernel's body (same device functions, same operations in the
// same order, so the same bits as every bit-identical mapping), then the scatter's writes and count,
// then the tangents along every direction.  A grid barrier separates the waves.
constexpr int kFusedThreads = 128;

struct FusedArgs {
    const gcs_b200_program_row* rows;
    const long long* offsets;  // device copy of the descriptor's offsets
    int n_waves;
    long long K, n_slots, n_values, T;
    const double* initial;     // [n_slots][4]
    // Other blocks write positions and dpositions during the launch (earlier waves' targets, which
    // later waves read): they are read with plain loads, never __ldg, and are not `const __restrict__`.
    // The grid barrier between waves orders those writes before the reads.
    double* pos;               // [K][n_slots][4]
    double* dpos;              // [K][n_slots][4][T]
    const double* val;         // [K][n_values]
    const double* dval;        // [K][n_values][T]
    uint32_t* nonconverged;    // [K] or null
};

// kKindOfSolver on the device
__device__ __forceinline__ int kind_of_solver(int solver)
{
    switch (solver) {
    case 1: case 4: return GCS_KIND_PP;
    case 2: case 5: return GCS_KIND_SDD;
    case 6: return GCS_KIND_PPL;
    case 7: return GCS_KIND_PLL;
    default: return GCS_KIND_ANG;
    }
}

// gather_row's side for a fused run: anchors into the positions, columns into registers
struct GatherRegisters {
    double* pa;
    double* pb;
    double v[3];
    const double* canvas;
    double k[13];
    __device__ __forceinline__ double& slot(int role, int q) { return (role ? pb : pa)[q]; }
    __device__ __forceinline__ double value(int q) const { return v[q]; }
    __device__ __forceinline__ double cst(int c) const { return canvas[c]; }
    __device__ __forceinline__ void in(int col, double x) { k[col] = x; }
};

// Row `row` (of kind KIND) for instance j.  Out of line per kind, so that the kernel holds one
// kind's registers at a time rather than the union of all five.
template <int KIND>
__device__ __noinline__ void fused_row(const FusedArgs& f, const gcs_b200_program_row& row, long long j)
{
    using S = gcsk::Sys<KIND>;
    double* const pos = f.pos + j * f.n_slots * 4;
    const double* const val = f.val + j * f.n_values;
    GatherRegisters g { pos + 4 * (long long)row.elem[0], pos + 4 * (long long)row.elem[1],
        { row_value(row, 0, val, 1), row_value(row, 1, val, 1), row_value(row, 2, val, 1) }, row.canvas, {} };
    gather_row(row, g);
    // newton_pair_kernel
    S sys;
    sys.load(g.k);
    double cx[2], cy[2];
    if constexpr (S::kGuessFromCols) {
        gcsk::column_seed<KIND>(g.k, 0, cx[0], cy[0]);
        gcsk::column_seed<KIND>(g.k, 1, cx[1], cy[1]);
    } else {
        gcsk::default_seed(0, cx[0], cy[0]);
        gcsk::default_seed(1, cx[1], cy[1]);
    }
    gcsk::FastConsts fc;
    fc.init((double)(f.K >> 62));  // 0.0, opaque to the compiler
    bool cva = fabs(0.0 - cx[0]) < fc.tol && fabs(0.0 - cy[0]) < fc.tol;
    bool cvb = fabs(0.0 - cx[1]) < fc.tol && fabs(0.0 - cy[1]) < fc.tol;
    int ita = 0, itb = 0;
    gcsk::newton_run2<KIND>(sys, sys, fc, cx[0], cy[0], ita, cva, !cva, cx[1], cy[1], itb, cvb, !cvb);
    double out[4];
    const int root = gcsk::select_and_finish<KIND, 2>(g.k, (uint8_t)row.code, cx, cy, out);
    // program_scatter_kernel, with chosen_root's test
    double* const dst = pos + 4 * (long long)row.elem[2];
#pragma unroll
    for (int q = 0; q < S::kOut; ++q) dst[q] = out[q];
    const bool converged = root ? cvb : cva;
    if (f.nonconverged && !converged) atomicAdd(f.nonconverged + j, 1u);
    if (f.T == 0) return;
    // program_tangent_kernel, one direction after the other; the unknown at the root is the output
    // point (K1, K3, K4) or the chosen seed's normal (K2, K5), which is the chosen candidate either way
    const long long T = f.T;
    double* const dpos = f.dpos + j * f.n_slots * 4 * T;
    const double* const dval = f.dval + j * f.n_values * T;
    gcsk::RowTangent<KIND> lin;
    if (converged) lin.init(g.k, root ? cx[1] : cx[0], root ? cy[1] : cy[0]);
#pragma unroll 1
    for (long long t = 0; t < T; ++t) {
        GatherTangents d { dpos + 4 * (long long)row.elem[0] * T + t, dpos + 4 * (long long)row.elem[1] * T + t,
            { row_value(row, 0, dval + t, T), row_value(row, 1, dval + t, T), row_value(row, 2, dval + t, T) }, T, {} };
        gather_row(row, d);
        double dout[4];
        if (!converged) {
            // not a root, so the implicit function theorem does not apply
            dout[0] = dout[1] = dout[2] = dout[3] = __longlong_as_double(0x7ff8000000000000LL);
        } else {
            lin.apply(d.kd, dout);
        }
        double* const ddst = dpos + 4 * (long long)row.elem[2] * T + t;
#pragma unroll
        for (int q = 0; q < S::kOut; ++q) ddst[q * T] = dout[q];
    }
}

// A persistent grid, launched cooperatively (launch_cooperative) with at most as many blocks as
// can be co-resident.  Every thread reaches every grid.sync(): there is no early return, the loops
// are grid-stride, and the wave bounds come from the device copy of the offsets, the same for every
// thread.
__global__ void __launch_bounds__(kFusedThreads) program_fused_kernel(const __grid_constant__ FusedArgs f)
{
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const long long first = (long long)blockIdx.x * blockDim.x + threadIdx.x, step = (long long)gridDim.x * blockDim.x;
    // what run_on's copies and memsets do: every instance starts from the initial positions (copied
    // as bits), the counts and every slot's tangent from 0
    const long long table = f.n_slots * 4;
    const long long* const init = reinterpret_cast<const long long*>(f.initial);
    long long* const pos = reinterpret_cast<long long*>(f.pos);
    for (long long q = first; q < f.K * table; q += step) pos[q] = init[q % table];
    if (f.nonconverged)
        for (long long q = first; q < f.K; q += step) f.nonconverged[q] = 0;
    for (long long q = first; q < f.K * table * f.T; q += step) f.dpos[q] = 0.0;
    grid.sync();
    for (int wave = 0; wave < f.n_waves; ++wave) {
        const long long lo = f.offsets[wave * kKinds], hi = f.offsets[(wave + 1) * kKinds];
        if (hi == lo) continue;  // the same for every thread: no barrier for an empty wave
        // sub-system s = r * K + j as place() orders them
        for (long long s = first; s < (hi - lo) * f.K; s += step) {
            const long long r = s / f.K, j = s - r * f.K;
            const gcs_b200_program_row& row = f.rows[lo + r];
            with_kind(kind_of_solver(row.solver), [&](auto K) { fused_row<decltype(K)::value>(f, row, j); });
        }
        grid.sync();
    }
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

// ---- fitting values to targets (gcs_b200_program_fit) ----
// Per instance the working state is one row of `work`, `stride` = 3 n^2 + 5 n + 3 doubles (n = n_free):
// x, xt (trial), x0 (the caller's start), g, gt [n], A, At [n][n] (upper triangle used), L [n][n]
// (Cholesky factor, lower), c, ct, failed.  The trial's (xt, At, gt, ct, failed) come from the
// tangent run at xt and program_fit_normal_kernel.
constexpr int kFitPoll = 4;  // gcs_b200_program_fit_host reads the running count every kFitPoll iterations

struct FitArgs {
    long long K, n, n_obs, n_values, n_slots, stride;
    const double* lo;          // [n] box, intersected with [-1, 1] for an angle slot
    const double* hi;
    const double* w;           // [n_obs]
    const int32_t* free;       // [n] value slots
    const int32_t* obs;        // [n_obs] slot * 4 + coordinate
    double* val;               // [K][n_values], the runs' value table
    double* dval;              // [K][n_values][n]: the selector
    const double* pos;         // [K][n_slots][4] of the last tangent run
    const double* dpos;        // [K][n_slots][4][n]
    const uint32_t* nc;        // [K]
    const double* target;      // [K][n_obs]
    double* work;              // [K][stride]
    gcs_b200_fit_result* res;  // [K]
    uint32_t* running;         // [max_iterations + 1]: instances still running after iteration it
    int it, last, max_it;
    double lambda0, cost_tol, ftol, xtol, gtol;
};

struct FitState {
    double *x, *xt, *x0, *g, *gt, *A, *At, *L, *c;  // c[0] = c, c[1] = ct, c[2] = failed
    __device__ FitState(const FitArgs& f, long long k)
    {
        const long long n = f.n;
        x = f.work + k * f.stride, xt = x + n, x0 = xt + n, g = x0 + n, gt = g + n, A = gt + n, At = A + n * n, L = At + n * n;
        c = L + n * n;
    }
};

// x clamped into [lo, hi]; NaN stays NaN
__device__ __forceinline__ double clamp_box(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }

// One thread per max(K x n_values x n, max_iterations + 1): the selector dvalues[k][v][t] = (v ==
// free[t]); for the first K x n threads, x0 = the caller's value, x = xt = clamp_box(x0) written back
// into the value table; for the first K, a RUNNING result with lambda0; the running counts zeroed.
__global__ void __launch_bounds__(kThreads) program_fit_start_kernel(const FitArgs f)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n = f.n;
    if (g < f.K * f.n_values * n) f.dval[g] = (g / n) % f.n_values == f.free[g % n] ? 1.0 : 0.0;
    if (g < f.K * n) {
        const long long k = g / n, i = g % n;
        FitState s(f, k);
        double& v = f.val[k * f.n_values + f.free[i]];
        s.x0[i] = v;
        s.x[i] = s.xt[i] = v = clamp_box(v, f.lo[i], f.hi[i]);
    }
    if (g < f.K) {
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
        f.res[g] = gcs_b200_fit_result { GCS_FIT_RUNNING, 0, nan, nan, f.lambda0 };
    }
    if (g <= f.max_it) f.running[g] = 0;
}

// One thread per (instance k, entry e), e in [0, P + n] with P = n (n + 1) / 2: e < P is A_ij (i <= j,
// row-major over the upper triangle), P <= e < P + n is g_{e-P}, e = P + n is c and the failure flag.
// With r_o = p_o - target_o and J_oi = dpos[k][obs_o][i], every sum runs over o = 0 .. n_obs-1, one
// term at a time from 0.0:
//   A_ij = A_ij + (w_o * J_oi) * J_oj,   g_i = g_i + (w_o * J_oi) * r_o,   c = c + (w_o * r_o) * r_o
// failed: nonconverged[k] > 0, or some observed p_o or J_oi is not finite.
__global__ void __launch_bounds__(kThreads) program_fit_normal_kernel(const FitArgs f)
{
    const long long n = f.n, P = n * (n + 1) / 2, E = P + n + 1;
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= f.K * E) return;
    const long long k = g / E, e = g - k * E;
    FitState s(f, k);
    const double* const pos = f.pos + k * f.n_slots * 4;
    const double* const dpos = f.dpos + k * f.n_slots * 4 * n;
    const double* const tgt = f.target + k * f.n_obs;
    if (e < P) {
        long long i = 0, r = e;
        while (r >= n - i) r -= n - i, ++i;
        const long long j = i + r;
        double a = 0.0;
        for (long long o = 0; o < f.n_obs; ++o) {
            const double* const J = dpos + f.obs[o] * n;
            a = a + (f.w[o] * J[i]) * J[j];
        }
        s.At[i * n + j] = a;
    } else if (e < P + n) {
        const long long i = e - P;
        double a = 0.0;
        for (long long o = 0; o < f.n_obs; ++o) a = a + (f.w[o] * dpos[f.obs[o] * n + i]) * (pos[f.obs[o]] - tgt[o]);
        s.gt[i] = a;
    } else {
        double c = 0.0;
        bool failed = f.nc[k] > 0;
        for (long long o = 0; o < f.n_obs; ++o) {
            const double p = pos[f.obs[o]], r = p - tgt[o];
            c = c + (f.w[o] * r) * r;
            failed |= !isfinite(p);
            for (long long i = 0; i < n; ++i) failed |= !isfinite(dpos[f.obs[o] * n + i]);
        }
        s.c[1] = c, s.c[2] = failed ? 1.0 : 0.0;
    }
}

// L L^T = A + lambda D (A upper, row-major), D_jj = max(A_jj, floor), column by column:
//   s = A_jj + lambda * D_jj, then s = s - L_jk * L_jk for k = 0 .. j-1; a pivot s that is not > 0
//   fails; L_jj = sqrt(s); for i > j: s = A_ji, s = s - L_ik * L_jk for k = 0 .. j-1, L_ij = s / L_jj
__device__ __forceinline__ bool fit_cholesky(const double* A, double lambda, double floor, double* L, long long n)
{
    for (long long j = 0; j < n; ++j) {
        const double ajj = A[j * n + j];
        double s = ajj + lambda * (ajj > floor ? ajj : floor);
        for (long long q = 0; q < j; ++q) s = s - L[j * n + q] * L[j * n + q];
        if (!(s > 0.0)) return false;
        const double d = sqrt(s);
        L[j * n + j] = d;
        for (long long i = j + 1; i < n; ++i) {
            double t = A[j * n + i];
            for (long long q = 0; q < j; ++q) t = t - L[i * n + q] * L[j * n + q];
            L[i * n + j] = t / d;
        }
    }
    return true;
}

// One thread per instance; a finished instance returns at once (frozen).  In order:
//   1. iterations += 1.  Iteration 0: a failed trial is START_FAILED (x0 back into the values, done);
//      otherwise accept.  Later: accept when !failed and ct < c.  Accept: x, g, A, c <- xt, gt, At, ct
//      and, after iteration 0, lambda = max(lambda / 10, 1e-12); then gi = max_i |g_i| (ascending i,
//      `a > gi ? a : gi` from 0.0), COST if c <= cost_tol, else GTOL if gi <= gtol, else (after
//      iteration 0) FTOL if c_old - c <= ftol * c_old.  Reject: lambda = 10 * max(lambda, 1e-12),
//      STALLED if lambda > 1e16.
//   2. Still running: floor = 1e-12 * max_j A_jj (as gi, from 0.0); fit_cholesky, and while it fails
//      lambda = 10 * max(lambda, 1e-12), STALLED once lambda > 1e16.
//   3. Still running: y_i = (-g_i - sum_{q < i} L_iq y_q) / L_ii (ascending i; the sum as s = s -
//      L_iq * y_q from s = -g_i), then d_i = (y_i - sum_{q > i} L_qi d_q) / L_ii (descending i, q
//      ascending); xt_i = clamp_box(x_i + d_i); XTOL if max_i |xt_i - x_i| <= xtol * (max_i |x_i| +
//      xtol) (both maxima as gi).
//   4. The values get xt while running, x once finished or after the last iteration.
__global__ void __launch_bounds__(kThreads) program_fit_update_kernel(const FitArgs f)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= f.K) return;
    gcs_b200_fit_result& res = f.res[k];
    if (res.status != GCS_FIT_RUNNING) return;
    const long long n = f.n;
    FitState s(f, k);
    double* const val = f.val + k * f.n_values;
    res.iterations += 1;
    const bool failed = s.c[2] != 0.0;
    if (f.it == 0 && failed) {
        for (long long i = 0; i < n; ++i) val[f.free[i]] = s.x0[i];
        res.status = GCS_FIT_START_FAILED;
        return;
    }
    int status = GCS_FIT_RUNNING;
    double lambda = res.lambda;
    const auto reject = [&] {
        lambda = 10.0 * (lambda > 1e-12 ? lambda : 1e-12);
        if (lambda > 1e16) status = GCS_FIT_STALLED;
    };
    if (!failed && (f.it == 0 || s.c[1] < s.c[0])) {
        const double c_old = s.c[0], c = s.c[1];
        for (long long i = 0; i < n; ++i) s.x[i] = s.xt[i], s.g[i] = s.gt[i];
        for (long long q = 0; q < n * n; ++q) s.A[q] = s.At[q];
        s.c[0] = c;
        if (f.it > 0) lambda = lambda / 10.0 > 1e-12 ? lambda / 10.0 : 1e-12;
        double gi = 0.0;
        for (long long i = 0; i < n; ++i) {
            const double a = fabs(s.g[i]);
            gi = a > gi ? a : gi;
        }
        if (c <= f.cost_tol) status = GCS_FIT_COST;
        else if (gi <= f.gtol) status = GCS_FIT_GTOL;
        else if (f.it > 0 && c_old - c <= f.ftol * c_old) status = GCS_FIT_FTOL;
        res.cost = c, res.grad_inf = gi;
    } else {
        reject();
    }
    if (status == GCS_FIT_RUNNING) {
        double amax = 0.0;
        for (long long j = 0; j < n; ++j) amax = s.A[j * n + j] > amax ? s.A[j * n + j] : amax;
        const double floor = 1e-12 * amax;
        while (status == GCS_FIT_RUNNING && !fit_cholesky(s.A, lambda, floor, s.L, n)) reject();
    }
    if (status == GCS_FIT_RUNNING) {
        double* const d = s.xt;  // y, then d, then the trial
        for (long long i = 0; i < n; ++i) {
            double t = -s.g[i];
            for (long long q = 0; q < i; ++q) t = t - s.L[i * n + q] * d[q];
            d[i] = t / s.L[i * n + i];
        }
        for (long long i = n - 1; i >= 0; --i) {
            double t = d[i];
            for (long long q = i + 1; q < n; ++q) t = t - s.L[q * n + i] * d[q];
            d[i] = t / s.L[i * n + i];
        }
        double step = 0.0, xmax = 0.0;
        for (long long i = 0; i < n; ++i) {
            d[i] = clamp_box(s.x[i] + d[i], f.lo[i], f.hi[i]);
            const double a = fabs(d[i] - s.x[i]), b = fabs(s.x[i]);
            step = a > step ? a : step;
            xmax = b > xmax ? b : xmax;
        }
        if (step <= f.xtol * (xmax + f.xtol)) status = GCS_FIT_XTOL;
    }
    res.status = status, res.lambda = lambda;
    const double* const next = status == GCS_FIT_RUNNING && !f.last ? s.xt : s.x;
    for (long long i = 0; i < n; ++i) val[f.free[i]] = next[i];
    if (status == GCS_FIT_RUNNING) atomicAdd(f.running + f.it, 1u);
}

int validate_desc(const gcs_b200_program_desc* d)
{
    if (!d) return fail(GCS_E_INVALID, "null program descriptor");
    if (d->n_waves < 0 || d->n_slots < 0 || d->n_values < 0 || d->n_rows < 0)
        return fail(GCS_E_INVALID, "negative count in the program descriptor");
    if (!d->offsets) return fail(GCS_E_INVALID, "null offsets");
    if ((d->n_rows > 0 && !d->rows) || (d->n_slots > 0 && (!d->slot_is_line || !d->initial)) || (d->n_values > 0 && !d->value_is_angle))
        return fail(GCS_E_INVALID, "null table in the program descriptor");
    const long long nseg = (long long)d->n_waves * kKinds;
    if (d->offsets[0] != 0) return fail(GCS_E_INVALID, "offsets[0] is %lld, not 0", (long long)d->offsets[0]);
    for (long long s = 0; s < nseg; ++s)
        if (d->offsets[s + 1] < d->offsets[s])
            return fail(GCS_E_INVALID, "offsets decrease at segment %lld (%lld after %lld)", s, (long long)d->offsets[s + 1], (long long)d->offsets[s]);
    if (d->offsets[nseg] != d->n_rows)
        return fail(GCS_E_INVALID, "offsets end at %lld, not at n_rows = %lld", (long long)d->offsets[nseg], (long long)d->n_rows);
    for (int s = 0; s < d->n_slots; ++s)
        if (d->slot_is_line[s] > 1) return fail(GCS_E_INVALID, "slot %d: type %d is neither point (0) nor line (1)", s, d->slot_is_line[s]);
    for (long long s = 0; s < nseg; ++s) {
        const int kind = (int)(s % kKinds) + 1;
        for (long long r = d->offsets[s]; r < d->offsets[s + 1]; ++r) {
            const gcs_b200_program_row& row = d->rows[r];
            if (row.solver < 1 || row.solver > 8) return fail(GCS_E_INVALID, "row %lld: unknown solver id %d", r, row.solver);
            if (kKindOfSolver[row.solver] != kind)
                return fail(GCS_E_INVALID, "row %lld: solver %d (kind %d) in a kind-%d segment", r, row.solver, kKindOfSolver[row.solver], kind);
            if (row.code < 0 || row.code > 255) return fail(GCS_E_INVALID, "row %lld: code %d out of range", r, row.code);
            for (int q = 0; q < 3; ++q) {
                const int e = row.elem[q];
                if (e < 0 || e >= d->n_slots) return fail(GCS_E_INVALID, "row %lld: element slot %d out of range (%d slots)", r, e, d->n_slots);
                if ((d->slot_is_line[e] != 0) != kRoleIsLine[row.solver][q])
                    return fail(GCS_E_INVALID, "row %lld: slot %d of role %c has the wrong element type for solver %d", r, e, 'a' + q, row.solver);
                const int v = row.value[q];
                if (!kReads[row.solver][q]) {
                    if (v != -1) return fail(GCS_E_INVALID, "row %lld: solver %d reads no v%d, value slot must be -1 (got %d)", r, row.solver, q, v);
                    continue;
                }
                if (v < 0 || v >= d->n_values) return fail(GCS_E_INVALID, "row %lld: value slot %d out of range (%d values)", r, v, d->n_values);
                const bool cosine = q == 0 && (row.solver == 3 || row.solver == 8);
                if ((d->value_is_angle[v] != 0) != cosine)
                    return fail(GCS_E_INVALID, "row %lld: value slot %d is %s an angle slot, v%d of solver %d needs %s", r, v,
                        d->value_is_angle[v] ? "" : "not", q, row.solver, cosine ? "one" : "a distance");
            }
            if (row.elem[0] == row.elem[1] || row.elem[0] == row.elem[2] || row.elem[1] == row.elem[2])
                return fail(GCS_E_INVALID, "row %lld: the three roles need three distinct slots", r);
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
                    return fail(GCS_E_INVALID, "wave %d: slot %d is %s by row %lld and %s by row %lld; rows of one wave run concurrently", wave,
                        (int)e, wrote[e] ? "written" : "read", row_of[e], writes ? "written" : "read", r);
                if (wave_of[e] != wave || writes) wave_of[e] = wave, row_of[e] = r, wrote[e] = writes;
            }
        }
    }
    return GCS_OK;
}

// gcs_b200_fit_check's checks, against a program's counts and slot and value types
int validate_fit(const gcs_b200_fit_desc* f, int n_slots, int n_values, const uint8_t* slot_is_line, const uint8_t* value_is_angle)
{
    if (!f) return fail(GCS_E_INVALID, "null fit descriptor");
    if (f->n_free < 1 || f->n_free > 32) return fail(GCS_E_INVALID, "n_free must be in 1..32 (got %d)", f->n_free);
    if (f->n_obs < 1) return fail(GCS_E_INVALID, "n_obs must be >= 1 (got %d)", f->n_obs);
    if (!f->free_values || !f->obs_slots || !f->obs_coords) return fail(GCS_E_INVALID, "null table in the fit descriptor");
    for (int i = 0; i < f->n_free; ++i) {
        const int v = f->free_values[i];
        if (v < 0 || v >= n_values) return fail(GCS_E_INVALID, "free value %d: value slot %d out of range (%d values)", i, v, n_values);
        for (int j = 0; j < i; ++j)
            if (f->free_values[j] == v) return fail(GCS_E_INVALID, "free value %d: value slot %d is already free value %d", i, v, j);
        const double lo = f->lower ? f->lower[i] : -INFINITY, hi = f->upper ? f->upper[i] : INFINITY;
        if (std::isnan(lo) || std::isnan(hi)) return fail(GCS_E_INVALID, "free value %d: NaN bound", i);
        if (lo > hi) return fail(GCS_E_INVALID, "free value %d: lower bound %g above upper bound %g", i, lo, hi);
        if (value_is_angle[v] && (lo > 1.0 || hi < -1.0))
            return fail(GCS_E_INVALID, "free value %d: the box [%g, %g] of an angle slot (a cosine) does not meet [-1, 1]", i, lo, hi);
    }
    for (int o = 0; o < f->n_obs; ++o) {
        const int s = f->obs_slots[o], c = f->obs_coords[o];
        if (s < 0 || s >= n_slots) return fail(GCS_E_INVALID, "observation %d: slot %d out of range (%d slots)", o, s, n_slots);
        const int ncoord = slot_is_line[s] ? 4 : 2;
        if (c < 0 || c >= ncoord)
            return fail(GCS_E_INVALID, "observation %d: coordinate %d of a %s slot (0..%d)", o, c, slot_is_line[s] ? "line" : "point", ncoord - 1);
        if (f->weights && !(std::isfinite(f->weights[o]) && f->weights[o] > 0.0))
            return fail(GCS_E_INVALID, "observation %d: weight %g is not finite and positive", o, f->weights[o]);
    }
    if (f->max_iterations < 0) return fail(GCS_E_INVALID, "max_iterations must be >= 0 (got %d)", f->max_iterations);
    const struct {
        const char* name;
        double v;
    } tol[] = { { "lambda0", f->lambda0 }, { "cost_tol", f->cost_tol }, { "ftol", f->ftol }, { "xtol", f->xtol }, { "gtol", f->gtol } };
    for (const auto& t : tol)
        if (!(std::isfinite(t.v) && t.v >= 0.0)) return fail(GCS_E_INVALID, "%s must be finite and >= 0 (got %g)", t.name, t.v);
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
            CUDA_TRY(cudaStreamSynchronize(st));
            CUDA_TRY(cudaFree(ptr));
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
            return fail(GCS_E_NOMEM, "cudaMalloc(%zu) for %s failed", need, buf);
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
    // fused runs: the device copy of `offsets`, and the co-resident blocks of program_fused_kernel on
    // the program's device (0 until the first fused run asks)
    long long* offsets_dev = nullptr;
    long long fused_capacity = 0;
    // the kind batches of plain and tangent runs, reused by every wave
    DeviceBuffer<unsigned char> scratch;
    // tables of the _host entry points, and the counts and tangent tables of _host runs and of fits
    // (grow_tables)
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
    // fits: host copies of the element and value types (for the descriptor checks); the working
    // state, descriptor tables and running counts (fit_on); targets and results of
    // gcs_b200_program_fit_host
    std::vector<uint8_t> slot_is_line, value_is_angle;
    DeviceBuffer<unsigned char> fit_state;
    DeviceBuffer<double> fit_targets;
    DeviceBuffer<gcs_b200_fit_result> fit_results;
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

// Launches `kernel` on `st` over `threads` threads, nothing when there are none.  too_many(): the
// failure when they need a grid beyond 31 bits.
template <class A, class TooMany>
int launch(void (*kernel)(A), long long threads, cudaStream_t st, const A& args, TooMany&& too_many)
{
    if (threads == 0) return GCS_OK;
    return gcsk::launch_kernel(kernel, (threads + kThreads - 1) / kThreads, kThreads, 0, st, too_many, args);
}

// how a run goes: wave by wave through the kind batches (gcs_b200_program_run[_tangents]), the same
// keeping every wave's batches on the tape (gcs_b200_program_run_recorded), or in one cooperative
// launch (gcs_b200_program_run_fused)
enum class RunKind { waves, recorded, fused };

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
        RC_TRY(p->tape.grow(tape_at.back(), st, "the tape of a recorded run of %lld instances", K));
    } else {
        // K instances of every kind's largest wave
        long long cap[kKinds];
        for (int k = 1; k <= kKinds; ++k) cap[k - 1] = kind_cap(p, k, K);
        RC_TRY(p->scratch.grow(batches_bytes(cap, T > 0), st, "the kind batches of %lld instances", K));
        bind_batches(w, p->scratch.ptr, cap, T > 0);
    }
    // every instance starts from the initial positions: one copy, then doubling copies
    const size_t table = (size_t)p->n_slots * 4 * sizeof(double);
    if (table) {
        CUDA_TRY(cudaMemcpyAsync(positions, p->initial, table, cudaMemcpyDeviceToDevice, st));
        for (long long have = 1; have < K;) {
            const long long n = have < K - have ? have : K - have;
            CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<unsigned char*>(positions) + (size_t)have * table, positions, (size_t)n * table,
                cudaMemcpyDeviceToDevice, st));
            have += n;
        }
    }
    if (nonconverged) CUDA_TRY(cudaMemsetAsync(nonconverged, 0, (size_t)K * sizeof(uint32_t), st));
    // every slot's tangent is 0 before the first wave: the initial positions are constants
    if (T > 0 && table) CUDA_TRY(cudaMemsetAsync(dpositions, 0, (size_t)K * T * table, st));
    for (int wave = 0; wave < p->n_waves; ++wave) {
        bind_wave(p, w, wave, recorded ? &tape_at : nullptr);
        const long long subs = w.seg[kKinds] * K;
        if (subs == 0) continue;
        const auto too_many = [&] { return fail(GCS_E_INVALID, "wave %d: %lld sub-systems are too many for one launch", wave, subs); };
        RC_TRY(launch(program_gather_kernel, subs, st, w, too_many));
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
        RC_TRY(gcs_b200_solve_many(list, count, p->device, st));
        RC_TRY(launch(program_scatter_kernel, subs, st, w, too_many));
        if (T > 0)
            RC_TRY(launch(program_tangent_kernel, subs * T, st, w, [&] {
                return fail(GCS_E_INVALID, "wave %d: %lld sub-systems x %lld directions are too many for one launch", wave, subs, T);
            }));
    }
    if (recorded) p->recorded_k = K;
    return GCS_OK;
}

// Device current, checks done: a fused run (T = 0: plain) on `st`, one cooperative launch.  The grid:
// as many blocks as the largest wave's rows x K sub-systems fill, at most as many as can be
// co-resident on the device, at least one.
int fused_on(gcs_b200_program* p, long long K, const double* values, double* positions, uint32_t* nonconverged, cudaStream_t st,
    long long T, const double* dvalues, double* dpositions)
{
    if (p->fused_capacity == 0) {
        int per_sm = 0, sms = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, program_fused_kernel, kFusedThreads, 0));
        CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, p->device));
        p->fused_capacity = (long long)per_sm * sms;
    }
    const long long need = (p->max_wave_rows * K + kFusedThreads - 1) / kFusedThreads;
    long long grid = need < p->fused_capacity ? need : p->fused_capacity;
    if (grid < 1) grid = 1;
    FusedArgs f;
    memset(&f, 0, sizeof(f));
    f.rows = p->rows, f.offsets = p->offsets_dev, f.n_waves = p->n_waves;
    f.K = K, f.n_slots = p->n_slots, f.n_values = p->n_values, f.T = T;
    f.initial = p->initial, f.pos = positions, f.dpos = dpositions, f.val = values, f.dval = dvalues, f.nonconverged = nonconverged;
    return gcsk::launch_cooperative(program_fused_kernel, (unsigned)grid, kFusedThreads, 0, st, f);
}

// device current; the sweep's working tables for the recorded K x T cotangents
int ensure_adjoint_tables(gcs_b200_program* p, long long T, cudaStream_t st)
{
    const long long K = p->recorded_k, KT = K * T;
    const size_t pbytes = (size_t)KT * p->n_slots * 4 * sizeof(double), cbytes = (size_t)KT * p->max_wave_rows * 11 * sizeof(double);
    const size_t vbytes = (size_t)KT * p->n_values * sizeof(double);
    const char* what = "the %s of %lld instances x %lld cotangents";
    RC_TRY(p->apos.grow(pbytes, st, what, "slot adjoints", K, T));
    RC_TRY(p->contrib.grow(cbytes, st, what, "adjoint contributions", K, T));
    RC_TRY(p->flags.grow((size_t)KT, st, what, "NaN flags", K, T));
    return p->avalues.grow(vbytes, st, what, "value adjoints", K, T);
}

// device current, checks done, p->apos holds the cotangents of the recorded run's positions: the
// sweep, waves from last to first, into adj_values [K][n_values][T]
int sweep_on(gcs_b200_program* p, long long T, double* adj_values, cudaStream_t st)
{
    const long long K = p->recorded_k, KT = K * T;
    if (p->n_values) CUDA_TRY(cudaMemsetAsync(adj_values, 0, (size_t)KT * p->n_values * sizeof(double), st));
    CUDA_TRY(cudaMemsetAsync(p->flags.ptr, 0, (size_t)KT, st));
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
        const auto too_many = [&] {
            return fail(GCS_E_INVALID, "wave %d: %lld sub-systems x %lld cotangents are too many for one launch", wave, subs, T);
        };
        RC_TRY(launch(program_adjoint_kernel, subs * T, st, w, too_many));
        RC_TRY(launch(program_adjoint_reduce_kernel, r.n_ent * KT, st, r, too_many));
    }
    return launch(program_adjoint_flag_kernel, KT * p->n_values, st, r,
        [&] { return fail(GCS_E_INVALID, "%lld value adjoints are too many for one launch", KT * p->n_values); });
}

// the checks that need no program come first; a null table is refused unless the program has
// nothing to put in it
int check_adjoints(const gcs_b200_program* p, int T, const double* adj_positions, const double* adj_values)
{
    if (T < 1) return fail(GCS_E_INVALID, "n_cotangents must be >= 1 (got %d)", T);
    if ((!adj_positions && !(p && p->n_slots == 0)) || (!adj_values && !(p && p->n_values == 0)))
        return fail(GCS_E_INVALID, "null adjoint table (adj_positions or adj_values)");
    if (!p) return fail(GCS_E_INVALID, "null program");
    if (p->recorded_k < 1) return fail(GCS_E_INVALID, "no recorded run: call gcs_b200_program_run_recorded first");
    return GCS_OK;
}

int check_run(const gcs_b200_program* p, long long K, const double* values, const double* positions, int variant)
{
    if (!p) return fail(GCS_E_INVALID, "null program");
    if (K < 1) return fail(GCS_E_INVALID, "n_instances must be >= 1 (got %lld)", K);
    if ((p->n_values > 0 && !values) || (p->n_slots > 0 && !positions)) return fail(GCS_E_INVALID, "null value or position table");
    if (variant < GCS_VARIANT_DEFAULT || variant > GCS_VARIANT_CONTRACTED_LINEAR) return fail(GCS_E_INVALID, "unknown variant %d", variant);
    return GCS_OK;
}

// the checks that need no program come first; a null tangent table is refused unless the program
// has nothing to put in it
int check_tangent_run(const gcs_b200_program* p, long long K, const double* values, const double* positions, int T,
    const double* dvalues, const double* dpositions, int variant)
{
    if (T < 1) return fail(GCS_E_INVALID, "n_tangents must be >= 1 (got %d)", T);
    if (variant < GCS_VARIANT_DEFAULT || variant > GCS_VARIANT_CONTRACTED_LINEAR) return fail(GCS_E_INVALID, "unknown variant %d", variant);
    if ((!dvalues && !(p && p->n_values == 0)) || (!dpositions && !(p && p->n_slots == 0)))
        return fail(GCS_E_INVALID, "null tangent table (dvalues or dpositions)");
    return check_run(p, K, values, positions, variant);
}

// a fused run's checks: n_tangents >= 0, then a plain run's (T = 0) or a tangent run's
int check_fused_run(const gcs_b200_program* p, long long K, const double* values, const double* positions, int T, const double* dvalues,
    const double* dpositions)
{
    if (T < 0) return fail(GCS_E_INVALID, "n_tangents must be >= 0 (got %d)", T);
    if (T == 0) return check_run(p, K, values, positions, GCS_VARIANT_DEFAULT);
    return check_tangent_run(p, K, values, positions, T, dvalues, dpositions, GCS_VARIANT_DEFAULT);
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
    CUDA_TRY(cudaEventRecord(p->ev[0], st));
    for (const Copy& c : up)
        if (c.bytes) CUDA_TRY(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaEventRecord(p->ev[1], st));
    const int rc = work(st);
    if (rc != GCS_OK) {
        cudaStreamSynchronize(st);
        return rc;
    }
    CUDA_TRY(cudaEventRecord(p->ev[2], st));
    for (const Copy& c : down)
        if (c.bytes) CUDA_TRY(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(p->ev[3], st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (ms)
        for (int q = 0; q < 3; ++q) CUDA_TRY(cudaEventElapsedTime(&ms[q], p->ev[q], p->ev[q + 1]));
    return GCS_OK;
}

// device current: the counts and tangent tables for K instances and T directions of the runs the
// program drives itself (_host runs, fits); host: also the _host entry points' values and positions
int grow_tables(gcs_b200_program* p, long long K, long long T, bool host, cudaStream_t st)
{
    const size_t vbytes = (size_t)K * p->n_values * sizeof(double), pbytes = (size_t)K * p->n_slots * 4 * sizeof(double);
    if (host) {
        RC_TRY(p->values.grow(vbytes, st, "the values of %lld instances", K));
        RC_TRY(p->positions.grow(pbytes, st, "the positions of %lld instances", K));
    }
    RC_TRY(p->counts.grow((size_t)K * sizeof(uint32_t), st, "the nonconverged counts of %lld instances", K));
    RC_TRY(p->dvalues.grow(vbytes * T, st, "the value tangents of %lld instances x %lld directions", K, T));
    return p->dpositions.grow(pbytes * T, st, "the position tangents of %lld instances x %lld directions", K, T);
}

// device current, checks done
int run_host(gcs_b200_program* p, long long K, const double* values, double* positions, uint32_t* nonconverged, int variant,
    float ms[3], long long T = 0, const double* dvalues = nullptr, double* dpositions = nullptr, RunKind how = RunKind::waves)
{
    const size_t vbytes = (size_t)K * p->n_values * sizeof(double), pbytes = (size_t)K * p->n_slots * 4 * sizeof(double);
    const size_t cbytes = (size_t)K * sizeof(uint32_t);
    RC_TRY(grow_tables(p, K, T, true, p->stream));
    return on_host(p, { { p->values.ptr, values, vbytes }, { p->dvalues.ptr, dvalues, vbytes * T } },
        [&](cudaStream_t s) {
            uint32_t* const counts = nonconverged ? p->counts.ptr : nullptr;
            if (how == RunKind::fused) return fused_on(p, K, p->values.ptr, p->positions.ptr, counts, s, T, p->dvalues.ptr, p->dpositions.ptr);
            return run_on(p, K, p->values.ptr, p->positions.ptr, counts, variant, s, T, p->dvalues.ptr, p->dpositions.ptr,
                how == RunKind::recorded);
        },
        { { positions, p->positions.ptr, pbytes }, { dpositions, p->dpositions.ptr, pbytes * T },
            { nonconverged, p->counts.ptr, nonconverged ? cbytes : 0 } },
        ms);
}

int check_fit(const gcs_b200_program* p, const gcs_b200_fit_desc* fit, long long K, const double* values, const double* targets,
    const double* positions, const gcs_b200_fit_result* results, int variant)
{
    RC_TRY(check_run(p, K, values, positions, variant));
    if (!targets || !results) return fail(GCS_E_INVALID, "null target or result table");
    return validate_fit(fit, p->n_slots, p->n_values, p->slot_is_line.data(), p->value_is_angle.data());
}

// Device current, checks done, grow_tables(K, n_free): the fit on `st` (gcs_b200_program_fit).  poll:
// read the running count back every kFitPoll iterations and stop when it is 0 (gcs_b200_program_fit_host).
int fit_on(gcs_b200_program* p, const gcs_b200_fit_desc* fit, long long K, double* values, const double* targets, double* positions,
    uint32_t* nonconverged, gcs_b200_fit_result* results, int variant, cudaStream_t st, bool poll)
{
    const long long n = fit->n_free, n_obs = fit->n_obs, nv = p->n_values, ns = p->n_slots;
    // the descriptor's tables: lo, hi [n], w [n_obs] (doubles), then free [n], obs [n_obs] (int32)
    std::vector<double> dbl((size_t)(2 * n + n_obs));
    std::vector<int32_t> idx((size_t)(n + n_obs));
    for (long long i = 0; i < n; ++i) {
        const bool angle = p->value_is_angle[(size_t)fit->free_values[i]] != 0;
        double lo = fit->lower ? fit->lower[i] : -INFINITY, hi = fit->upper ? fit->upper[i] : INFINITY;
        if (angle) lo = lo > -1.0 ? lo : -1.0, hi = hi < 1.0 ? hi : 1.0;
        dbl[(size_t)i] = lo, dbl[(size_t)(n + i)] = hi;
        idx[(size_t)i] = fit->free_values[i];
    }
    for (long long o = 0; o < n_obs; ++o) {
        dbl[(size_t)(2 * n + o)] = fit->weights ? fit->weights[o] : 1.0;
        idx[(size_t)(n + o)] = fit->obs_slots[o] * 4 + fit->obs_coords[o];
    }
    // one allocation: the working state, the descriptor's tables, the running counts
    const long long stride = 3 * n * n + 5 * n + 3;
    const size_t wbytes = (size_t)(K * stride) * sizeof(double), dbytes = dbl.size() * sizeof(double), ibytes = idx.size() * sizeof(int32_t);
    RC_TRY(p->fit_state.grow(wbytes + dbytes + ibytes + (size_t)(fit->max_iterations + 1) * sizeof(uint32_t), st,
        "the working state of a fit of %lld instances", K));
    unsigned char* const at = p->fit_state.ptr;
    CUDA_TRY(cudaMemcpyAsync(at + wbytes, dbl.data(), dbytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(at + wbytes + dbytes, idx.data(), ibytes, cudaMemcpyHostToDevice, st));
    FitArgs f;
    memset(&f, 0, sizeof(f));
    f.K = K, f.n = n, f.n_obs = n_obs, f.n_values = nv, f.n_slots = ns, f.stride = stride;
    f.work = reinterpret_cast<double*>(at), f.lo = f.work + K * stride, f.hi = f.lo + n, f.w = f.lo + 2 * n;
    f.free = reinterpret_cast<const int32_t*>(at + wbytes + dbytes), f.obs = f.free + n;
    f.running = reinterpret_cast<uint32_t*>(at + wbytes + dbytes + ibytes);
    f.val = values, f.dval = p->dvalues.ptr, f.pos = positions, f.dpos = p->dpositions.ptr, f.nc = p->counts.ptr;
    f.target = targets, f.res = results;
    f.max_it = fit->max_iterations;
    f.lambda0 = fit->lambda0, f.cost_tol = fit->cost_tol, f.ftol = fit->ftol, f.xtol = fit->xtol, f.gtol = fit->gtol;
    const auto too_many = [&] { return fail(GCS_E_INVALID, "a fit of %lld instances x %lld free values is too large for one launch", K, n); };
    const long long start = K * nv * n > f.max_it + 1 ? K * nv * n : f.max_it + 1;
    RC_TRY(launch(program_fit_start_kernel, start, st, f, too_many));
    for (int it = 0; it <= f.max_it; ++it) {
        RC_TRY(run_on(p, K, values, positions, p->counts.ptr, variant, st, n, p->dvalues.ptr, p->dpositions.ptr));
        f.it = it, f.last = it == f.max_it;
        RC_TRY(launch(program_fit_normal_kernel, K * (n * (n + 1) / 2 + n + 1), st, f, too_many));
        RC_TRY(launch(program_fit_update_kernel, K, st, f, too_many));
        if (poll && !f.last && it % kFitPoll == kFitPoll - 1) {
            uint32_t running = 0;
            CUDA_TRY(cudaMemcpyAsync(&running, f.running + it, sizeof(running), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (running == 0) break;  // every instance frozen: the values hold the results
        }
    }
    return run_on(p, K, values, positions, nonconverged, variant, st);
}

}  // namespace

extern "C" {

int gcs_b200_program_create(const gcs_b200_program_desc* d, int device, gcs_b200_program** out)
{
    if (!out) return fail(GCS_E_INVALID, "null output handle");
    *out = nullptr;
    int rc = validate_desc(d);
    if (rc != GCS_OK) return rc;
    const int ndev = gcs_b200_device_count();
    if (ndev <= 0) return fail(GCS_E_NO_DEVICE, "no CUDA device; this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(GCS_E_NO_DEVICE, "device %d out of range (%d present)", device, ndev);
    DeviceScope on(device);
    RC_TRY(on.rc);
    auto* p = new gcs_b200_program();
    p->device = device, p->n_waves = d->n_waves, p->n_slots = d->n_slots, p->n_values = d->n_values, p->n_rows = d->n_rows;
    p->offsets.assign(d->offsets, d->offsets + (size_t)d->n_waves * kKinds + 1);
    p->slot_is_line.assign(d->slot_is_line, d->slot_is_line + d->n_slots);
    p->value_is_angle.assign(d->value_is_angle, d->value_is_angle + d->n_values);
    for (int w = 0; w < d->n_waves; ++w)
        for (int k = 0; k < kKinds; ++k) {
            const long long rows = p->offsets[(size_t)w * kKinds + k + 1] - p->offsets[(size_t)w * kKinds + k];
            if (rows > p->max_rows[k]) p->max_rows[k] = rows;
        }
    auto bail = [&](int code) {
        gcs_b200_program_destroy(p);
        return code;
    };
    if (cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(GCS_E_CUDA, "stream creation failed"));
    for (auto& e : p->ev)
        if (cudaEventCreate(&e) != cudaSuccess) return bail(fail(GCS_E_CUDA, "event creation failed"));
    const size_t row_bytes = (size_t)d->n_rows * sizeof(gcs_b200_program_row), init_bytes = (size_t)d->n_slots * 4 * sizeof(double);
    const size_t off_bytes = p->offsets.size() * sizeof(long long);
    if ((row_bytes && cudaMalloc(&p->rows, row_bytes) != cudaSuccess) || (init_bytes && cudaMalloc(&p->initial, init_bytes) != cudaSuccess)
        || cudaMalloc(&p->offsets_dev, off_bytes) != cudaSuccess) {
        cudaGetLastError();
        return bail(fail(GCS_E_NOMEM, "cudaMalloc for a program of %lld rows and %d slots failed", (long long)d->n_rows, d->n_slots));
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
        return bail(fail(GCS_E_NOMEM, "cudaMalloc for the reader lists of %zu entries failed", ent.size()));
    }
    if ((row_bytes && cudaMemcpyAsync(p->rows, d->rows, row_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || (init_bytes && cudaMemcpyAsync(p->initial, d->initial, init_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || cudaMemcpyAsync(p->offsets_dev, p->offsets.data(), off_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess
        || (ent_bytes && cudaMemcpyAsync(p->ent, ent.data(), ent_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || cudaMemcpyAsync(p->begin, begin.data(), begin_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess
        || (reader_bytes && cudaMemcpyAsync(p->readers, readers.data(), reader_bytes, cudaMemcpyHostToDevice, p->stream) != cudaSuccess)
        || cudaStreamSynchronize(p->stream) != cudaSuccess)
        return bail(fail(GCS_E_CUDA, "program upload failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = p;
    return GCS_OK;
}

int gcs_b200_program_run(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged, int variant,
    void* stream)
{
    RC_TRY(check_run(p, K, values, positions, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_on(p, K, values, positions, nonconverged, variant, static_cast<cudaStream_t>(stream));
}

int gcs_b200_program_run_host(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int variant, float ms[3])
{
    RC_TRY(check_run(p, K, values, positions, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_host(p, K, values, positions, nonconverged, variant, ms);
}

int gcs_b200_program_run_tangents(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int32_t T, const double* dvalues, double* dpositions, int variant, void* stream)
{
    RC_TRY(check_tangent_run(p, K, values, positions, T, dvalues, dpositions, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_on(p, K, values, positions, nonconverged, variant, static_cast<cudaStream_t>(stream), T, dvalues, dpositions);
}

int gcs_b200_program_run_tangents_host(gcs_b200_program* p, int64_t K, const double* values, double* positions,
    uint32_t* nonconverged, int32_t T, const double* dvalues, double* dpositions, int variant, float ms[3])
{
    RC_TRY(check_tangent_run(p, K, values, positions, T, dvalues, dpositions, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_host(p, K, values, positions, nonconverged, variant, ms, T, dvalues, dpositions);
}

int gcs_b200_program_run_recorded(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int variant, void* stream)
{
    RC_TRY(check_run(p, K, values, positions, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_on(p, K, values, positions, nonconverged, variant, static_cast<cudaStream_t>(stream), 0, nullptr, nullptr, true);
}

int gcs_b200_program_run_recorded_host(gcs_b200_program* p, int64_t K, const double* values, double* positions,
    uint32_t* nonconverged, int variant, float ms[3])
{
    RC_TRY(check_run(p, K, values, positions, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_host(p, K, values, positions, nonconverged, variant, ms, 0, nullptr, nullptr, RunKind::recorded);
}

int gcs_b200_program_run_fused(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int32_t T, const double* dvalues, double* dpositions, void* stream)
{
    RC_TRY(check_fused_run(p, K, values, positions, T, dvalues, dpositions));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return fused_on(p, K, values, positions, nonconverged, static_cast<cudaStream_t>(stream), T, dvalues, dpositions);
}

int gcs_b200_program_run_fused_host(gcs_b200_program* p, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int32_t T, const double* dvalues, double* dpositions, float ms[3])
{
    RC_TRY(check_fused_run(p, K, values, positions, T, dvalues, dpositions));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    return run_host(p, K, values, positions, nonconverged, GCS_VARIANT_DEFAULT, ms, T, dvalues, dpositions, RunKind::fused);
}

int gcs_b200_program_adjoints(gcs_b200_program* p, int32_t T, const double* adj_positions, double* adj_values, void* stream)
{
    RC_TRY(check_adjoints(p, T, adj_positions, adj_values));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    RC_TRY(ensure_adjoint_tables(p, T, st));
    const size_t pbytes = (size_t)p->recorded_k * T * p->n_slots * 4 * sizeof(double);
    if (pbytes) CUDA_TRY(cudaMemcpyAsync(p->apos.ptr, adj_positions, pbytes, cudaMemcpyDeviceToDevice, st));
    return sweep_on(p, T, adj_values, st);
}

int gcs_b200_program_adjoints_host(gcs_b200_program* p, int32_t T, const double* adj_positions, double* adj_values, float ms[3])
{
    RC_TRY(check_adjoints(p, T, adj_positions, adj_values));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    RC_TRY(ensure_adjoint_tables(p, T, p->stream));
    const size_t pbytes = (size_t)p->recorded_k * T * p->n_slots * 4 * sizeof(double);
    const size_t vbytes = (size_t)p->recorded_k * T * p->n_values * sizeof(double);
    return on_host(p, { { p->apos.ptr, adj_positions, pbytes } }, [&](cudaStream_t st) { return sweep_on(p, T, p->avalues.ptr, st); },
        { { adj_values, p->avalues.ptr, vbytes } }, ms);
}

int gcs_b200_program_fit(gcs_b200_program* p, const gcs_b200_fit_desc* fit, int64_t K, double* values, const double* targets,
    double* positions, uint32_t* nonconverged, gcs_b200_fit_result* results, int variant, void* stream)
{
    RC_TRY(check_fit(p, fit, K, values, targets, positions, results, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    RC_TRY(grow_tables(p, K, fit->n_free, false, st));
    return fit_on(p, fit, K, values, targets, positions, nonconverged, results, variant, st, false);
}

int gcs_b200_program_fit_host(gcs_b200_program* p, const gcs_b200_fit_desc* fit, int64_t K, double* values, const double* targets,
    double* positions, uint32_t* nonconverged, gcs_b200_fit_result* results, int variant, float ms[3])
{
    RC_TRY(check_fit(p, fit, K, values, targets, positions, results, variant));
    DeviceScope on(p->device);
    RC_TRY(on.rc);
    const size_t vbytes = (size_t)K * p->n_values * sizeof(double), pbytes = (size_t)K * p->n_slots * 4 * sizeof(double);
    const size_t cbytes = (size_t)K * sizeof(uint32_t), tbytes = (size_t)K * fit->n_obs * sizeof(double);
    const size_t rbytes = (size_t)K * sizeof(gcs_b200_fit_result);
    const cudaStream_t st = p->stream;
    RC_TRY(grow_tables(p, K, fit->n_free, true, st));
    RC_TRY(p->fit_targets.grow(tbytes, st, "the targets of %lld instances", (long long)K));
    RC_TRY(p->fit_results.grow(rbytes, st, "the fit results of %lld instances", (long long)K));
    return on_host(p, { { p->values.ptr, values, vbytes }, { p->fit_targets.ptr, targets, tbytes } },
        [&](cudaStream_t s) {
            return fit_on(p, fit, K, p->values.ptr, p->fit_targets.ptr, p->positions.ptr, nonconverged ? p->counts.ptr : nullptr,
                p->fit_results.ptr, variant, s, true);
        },
        { { values, p->values.ptr, vbytes }, { positions, p->positions.ptr, pbytes }, { nonconverged, p->counts.ptr, nonconverged ? cbytes : 0 },
            { results, p->fit_results.ptr, rbytes } },
        ms);
}

int gcs_b200_fit_check(const gcs_b200_program_desc* d, const gcs_b200_fit_desc* fit)
{
    RC_TRY(validate_desc(d));
    return validate_fit(fit, d->n_slots, d->n_values, d->slot_is_line, d->value_is_angle);
}

void gcs_b200_program_destroy(gcs_b200_program* p)
{
    if (!p) return;
    {
        DeviceScope on(p->device);  // released whether or not the switch succeeded
        if (p->stream) cudaStreamSynchronize(p->stream), cudaStreamDestroy(p->stream);
        for (auto e : p->ev)
            if (e) cudaEventDestroy(e);
        cudaFree(p->rows), cudaFree(p->initial), cudaFree(p->offsets_dev), cudaFree(p->scratch.ptr);
        cudaFree(p->values.ptr), cudaFree(p->positions.ptr), cudaFree(p->counts.ptr);
        cudaFree(p->dvalues.ptr), cudaFree(p->dpositions.ptr);
        cudaFree(p->ent), cudaFree(p->begin), cudaFree(p->readers), cudaFree(p->tape.ptr);
        cudaFree(p->apos.ptr), cudaFree(p->contrib.ptr), cudaFree(p->flags.ptr), cudaFree(p->avalues.ptr);
        cudaFree(p->fit_state.ptr), cudaFree(p->fit_targets.ptr), cudaFree(p->fit_results.ptr);
        cudaGetLastError();
    }
    delete p;
}

}  // extern "C"
