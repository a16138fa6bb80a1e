/*
 * gcs_b200.h — C ABI of the B200-native batched Newton-Raphson sub-system solver.
 *
 * This is the drop-in boundary for ONE path of the reference
 * (SolyomBalint/2D_geometry_constraint_solver): the 2-unknown Newton-Raphson root finder
 *   src/constraint_solver/src/solving/equations/newton_raphson.hpp:41-102   (solve2D)
 * fed by the equation primitives
 *   src/constraint_solver/src/solving/equations/equation_primitives.hpp:23-199
 * and followed by the root-selection heuristics
 *   src/constraint_solver/src/solving/solvers/heuristics.hpp:22-335
 * and the line write-back helper `reconstructLineEndpoints`
 *   src/constraint_solver/src/solving/solvers/point_line_solvers.cpp:74-106.
 *
 * The reference has no FFI of its own (it is one C++ shared library); this header is what a
 * binding for that path binds.  One "solve" = one `solve2D` call (all seeds) + the heuristic that
 * picks the root (+ line reconstruction where the unknown is a line).  The host packer (the C++
 * layer in 2d_geometry_constraint_solver_b200/host, mirroring the reference's eight
 * `Solvers::*::solve` functions) turns matched 3-element components into the
 * structure-of-arrays batches described below.
 *
 * Conventions
 *   - plain C, no exceptions, every entry point returns 0 on success or a negative GCS_E_* code;
 *     `gcs_b200_last_error()` returns a thread-local message for the last failure.
 *   - all pointers are caller-owned; the library retains nothing after a call returns, except
 *     the internal per-device staging arena used by the host-buffer entry points.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     GCS_E_NO_DEVICE.
 *   - arithmetic is IEEE-754 binary64; the default kernels (GCS_VARIANT_DEFAULT .. GCS_VARIANT_PAIR)
 *     use no contraction and reproduce the reference's roundings, the opt-in GCS_VARIANT_CONTRACTED*
 *     kernels use fused multiply-adds under the tolerance contract stated at their definition;
 *     constants below equal the reference's (newton_raphson.hpp:17, :20, :105-107;
 *     heuristics.hpp:173, :209).
 */
#ifndef GCS_B200_H
#define GCS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define GCS_B200_API
#else
#define GCS_B200_API __attribute__((visibility("default")))
#endif

/* ---- constants of the path (reference file:line in the comment) ---- */
#define GCS_CONVERGENCE_THRESHOLD 0.00001 /* newton_raphson.hpp:17 */
#define GCS_MAXIMUM_ITERATIONS 1000       /* newton_raphson.hpp:20 */
#define GCS_DEFAULT_GUESS 20000.0         /* newton_raphson.hpp:105-107: (+g,+g), (-g,-g) */
#define GCS_PARALLEL_EPSILON 1e-10        /* heuristics.hpp:173 */
#define GCS_COLLINEAR_EPSILON 1e-8        /* heuristics.hpp:209 */

/* ---- error codes ---- */
#define GCS_OK 0
#define GCS_E_INVALID (-1)   /* bad descriptor (kind, n_seeds, null column, ...) */
#define GCS_E_NO_DEVICE (-2) /* no CUDA device / device index out of range */
#define GCS_E_CUDA (-3)      /* a CUDA runtime call failed; see gcs_b200_last_error() */
#define GCS_E_NOT_INIT (-4)
#define GCS_E_NOMEM (-5)

/* ---- equation-pair kinds (what the kernels are specialised on) ----
 * K1 PP   : point-to-point distance x2                 (equation_primitives.hpp:23-28)
 *           used by ZeroFixedPointsTriangleSolver / TwoFixedPointsDistanceSolver
 *           (point_point_solvers.cpp:56-65, :136-145); selection pickByTriangleOrientation.
 * K2 SDD  : lineNormalSignedDistanceDiff + unitNormalConstraint (equation_primitives.hpp:176-199)
 *           used by ZeroFixedPPLTriangleSolver / TwoFixedPointsLineSolver
 *           (point_line_solvers.cpp:205-222, :349-367); selection pickLineBySignedDistances;
 *           output = line endpoints via reconstructLineEndpoints.
 * K3 PPL  : pointToPointDistance + pointToLineDistance (equation_primitives.hpp:23-28, :70-76)
 *           used by FixedPointAndLineFreePointSolver (point_line_solvers.cpp:500-512);
 *           selection pickByTriangleOrientationWithFallback with perpendicular feet.
 * K4 PLL  : pointToLineDistance x2, used by TwoFixedLinesFreePointSolver
 *           (point_line_solvers.cpp:636-649); selection via line intersection (:656-682).
 * K5 ANG  : lineNormalAngleConstraint + unitNormalConstraint (equation_primitives.hpp:141-149,
 *           :196-199), used by ZeroFixedLLPAngleTriangleSolver / FixedLineAndPointFreeLineSolver
 *           (line_angle_solvers.cpp:293-311, :483-501); selection
 *           pickLineNormalByAngleOrientation; output = line endpoints.
 */
#define GCS_KIND_PP 1
#define GCS_KIND_SDD 2
#define GCS_KIND_PPL 3
#define GCS_KIND_PLL 4
#define GCS_KIND_ANG 5
#define GCS_KIND_COUNT 5

/* Input columns (each `const double[n]`, SoA, 16-byte aligned base recommended).
 * "solver space" = coordinates already solved by earlier components; "canvas" = the sketch.
 *
 * K1 PP (6):  0 ax  1 ay  2 ra  3 bx  4 by  5 rb
 *     fixed point A, |free-A|, fixed point B, |free-B|.
 * K2 SDD (9): 0 p1x 1 p1y 2 p2x 3 p2y 4 s1 5 s2 6 gnx 7 gny 8 canvas_len
 *     fixed points P1,P2 (solver space), signed distances s_i = signOf(canvas side)*d_i,
 *     canvas unit normal of the free line (guess 0; guess 1 is its negation),
 *     canvas length of the free line.
 * K3 PPL (10): 0 px 1 py 2 r 3 xa 4 ya 5 xb 6 yb 7 s 8 cfx 9 cfy
 *     fixed point + distance, fixed line endpoints (solver space), signed line distance,
 *     canvas position of the free point (read only when GCS_CODE_COLLINEAR is set).
 * K4 PLL (12): 0 xa1 1 ya1 2 xb1 3 yb1 4 s1  5 xa2 6 ya2 7 xb2 8 yb2 9 s2  10 cfx 11 cfy
 * K5 ANG (13): 0 fdx 1 fdy 2 cosA 3 gnx 4 gny 5 cfdx 6 cfdy 7 px 8 py 9 s 10 r2x 11 r2y
 *              12 canvas_len
 *     fixed line direction (solver space), cos(angle), canvas unit normal of the free line,
 *     canvas direction of the fixed line, the constraining point (solver space) and its signed
 *     distance to the free line, second reference point for reconstruction, canvas length.
 *
 * Anchored shapes.  The zero-fixed solvers place their first elements at the origin / on the x
 * axis (point_point_solvers.cpp:48-50, point_line_solvers.cpp:179-181,
 * line_angle_solvers.cpp:249-274), which makes some columns identically zero.  Such a column may
 * be passed as NULL: it is read as all zeros (same arithmetic, same results), needs no buffer and
 * is never copied to the device.  Allowed (gcs_b200_column_may_be_null): K1 ax, ay, by (0, 1, 4);
 * K2 p1x, p1y, p2y (0, 1, 3); K5 fdy, px, r2x, r2y (1, 7, 10, 11).  Any other NULL input column is
 * GCS_E_INVALID.
 */
#define GCS_MAX_IN_COLS 13
#define GCS_MAX_OUT_COLS 4
#define GCS_MAX_SEEDS 8

/* Orientation code column (`const uint8_t[n]`): the canvas-side facts the heuristics need,
 * reduced by the packer to a few bits ("orientation signs" of the north-star batch layout).
 *   bits 1:0  sign0 + 1, sign0 in {-1,0,+1} (three-valued sign(x) = (x>0)-(x<0))
 *             K1: sign(triangleOrientation(canvasA, canvasB, canvasFree))   heuristics.hpp:52
 *             K2: sign(canvas signed distance of P1 to the line)            heuristics.hpp:261
 *             K3/K4: sign(canvas reference-triangle orientation)            heuristics.hpp:220-223
 *             K5: sign(canvasFixedDir x canvasFreeDir) after flipOrientation heuristics.hpp:310-312
 *   bits 3:2  sign1 + 1 (K2 only: canvas signed distance of P2)             heuristics.hpp:262
 *   bit  4    GCS_CODE_COLLINEAR: |canvasOri| < 1e-8 -> nearest-to-canvas   heuristics.hpp:212-217
 *   bit  5    GCS_CODE_CANVAS_PARALLEL (K4): the canvas lines do not intersect,
 *             point_line_solvers.cpp:674-682
 */
#define GCS_CODE_SIGN0(code) ((int)((code) & 3) - 1)
#define GCS_CODE_SIGN1(code) ((int)(((code) >> 2) & 3) - 1)
#define GCS_CODE_COLLINEAR 0x10
#define GCS_CODE_CANVAS_PARALLEL 0x20
#define GCS_MAKE_CODE(sign0, sign1, flags) \
    ((uint8_t)((((sign0) + 1) & 3) | ((((sign1) + 1) & 3) << 2) | (flags)))

/* where the column pointers of a batch live */
#define GCS_MEM_HOST 0
#define GCS_MEM_DEVICE 1

/* kernel selection.  Variants 0-4 produce bit-identical results (same device functions, same
 * operation order per Newton run); they differ in how runs are mapped to lanes.
 * DEFAULT = SORTED for launches of at least 2^18 runs (n * n_seeds), STATIC below; K4 from 2^17
 * runs: SEQ. */
#define GCS_VARIANT_DEFAULT 0
#define GCS_VARIANT_STATIC 1 /* one lane per (sub-system, seed), static mapping */
#define GCS_VARIANT_REFILL 2 /* persistent CTAs, TMA-staged tiles, warp-level lane refill */
#define GCS_VARIANT_SORTED 3 /* CTA tiles; runs sorted by predicted update count, one lane finishes one run */
#define GCS_VARIANT_PAIR 4 /* one lane per sub-system, its two seeds iterated in lockstep (2 seeds only; else static) */
/* Tolerance-class arithmetic (csrc/newton_relaxed.cuh): the update from the seed as a closed-form
 * 2x2 solve on fused multiply-adds, the updates after it as the scalar Newton map along the line
 * every equation pair of the path contains (the radical line for K1); K4, a linear pair, is solved
 * in closed form with its iteration counts certified (CONTRACTED_LINEAR).  Contract: iteration counts, convergence flags and root indices equal to every
 * other variant's; coordinates within 1e-9 relative (the north star's tolerance) instead of bit
 * for bit.  The discrete half of the contract rests on guards (runs and selections whose decisions
 * could depend on the arithmetic are detected and redone with the literal device functions) whose
 * sufficiency is an error-analysis argument plus evidence - tests/test_gpu_relaxed.py,
 * tests/test_gpu_soak.py and the soaks of profiles/ (> 1e8 sub-systems without a difference on the
 * final arithmetic; earlier soaks did find two holes, which is why the carry term exists and why the
 * line constants are formed from cancellation-free factors) - NOT a machine-checked proof.
 * Opt-in: DEFAULT never resolves to it, and the host mirror stays on the bit-identical kernels.
 * CONTRACTED = CONTRACTED_STATIC (measured fastest at every size) except the 8-seed K1, which takes
 * CONTRACTED_SEQ, and K4, which takes CONTRACTED_LINEAR; CONTRACTED_SORTED runs the closed-form
 * 2x2 solve for every update on the sorted tiles (its runs are handed from lane to lane mid-way). */
#define GCS_VARIANT_CONTRACTED 5
#define GCS_VARIANT_CONTRACTED_STATIC 6
#define GCS_VARIANT_CONTRACTED_SORTED 7
#define GCS_VARIANT_CONTRACTED_SEQ 8 /* contracted arithmetic, one lane per sub-system, seeds one after the other */
#define GCS_VARIANT_SEQ 9            /* bit-identical arithmetic in the same mapping */
/* K4 only (a linear pair): the solution in closed form, every seed's two decisions certified instead
 * of iterated, uncertified sub-systems redone literally; any other kind resolves as CONTRACTED */
#define GCS_VARIANT_CONTRACTED_LINEAR 10

typedef struct gcs_b200_batch {
    int32_t kind;    /* GCS_KIND_* */
    int32_t n_seeds; /* 2 = reference semantics; 8 = multi-start (kinds with default guesses) */
    int64_t n;       /* sub-systems in this batch */
    int32_t mem;     /* GCS_MEM_HOST or GCS_MEM_DEVICE for every pointer below */
    int32_t variant; /* GCS_VARIANT_* */
    const double* in[GCS_MAX_IN_COLS]; /* kind-specific input columns, each length n */
    const uint8_t* code;               /* [n] orientation codes */
    const double* guesses;             /* NULL = kind default; else [n_seeds][2][n] */
    double* out[GCS_MAX_OUT_COLS];     /* point kinds: x,y ; line kinds: p1x,p1y,p2x,p2y */
    double* cand;                      /* optional [n_seeds][2][n]: every seed's end point */
    int16_t* iters;                    /* optional [n_seeds][n]: updates applied per seed */
    uint8_t* converged;                /* optional [n_seeds][n]: 1 iff loop left via break */
    uint8_t* root_index;               /* optional [n]: index of the candidate chosen */
} gcs_b200_batch;

/* number of input / output columns of a kind (0 for an unknown kind) */
GCS_B200_API int gcs_b200_kind_in_cols(int kind);
GCS_B200_API int gcs_b200_kind_out_cols(int kind);
/* 1 if input column `col` of `kind` may be NULL (an anchor column, read as zeros), else 0 */
GCS_B200_API int gcs_b200_column_may_be_null(int kind, int col);

/* library / device management */
GCS_B200_API int gcs_b200_device_count(void);
GCS_B200_API int gcs_b200_init(int device_count, const int* devices); /* NULL = 0..count-1 */
GCS_B200_API void gcs_b200_shutdown(void);
GCS_B200_API const char* gcs_b200_last_error(void);
GCS_B200_API const char* gcs_b200_version(void);

/* Solve one batch on one device, asynchronously on `cuda_stream` (a cudaStream_t, NULL = the
 * default stream).  batch->mem must be GCS_MEM_DEVICE.  Replaces a loop of
 * `Equations::solve2D` + `pickBy*` calls (newton_raphson.hpp:41-102, heuristics.hpp). */
GCS_B200_API int gcs_b200_solve(const gcs_b200_batch* batch, int device, void* cuda_stream);

/* Several device-resident batches as ONE job (e.g. one batch per equation kind of a dependency
 * wave, or the K1 + K5 halves of a cluster batch): stream-ordered on `cuda_stream` as a whole -
 * everything enqueued before the call precedes every launch, everything enqueued after it follows
 * all of them - while inside the job the launches run concurrently on internal streams, so that one
 * kernel's ramp-up, drain and literal re-runs are covered by its neighbours.  The batches must not
 * alias each other's outputs. */
GCS_B200_API int gcs_b200_solve_many(const gcs_b200_batch* const* batches, int count, int device, void* cuda_stream);

/* Same with HOST buffers: copies inputs H2D, solves, copies outputs D2H and synchronises.
 * This is the call the host-side solver mirror makes. */
GCS_B200_API int gcs_b200_solve_host(const gcs_b200_batch* batch, int device);

/* The same without the final synchronisation: the batch is cut into index ranges that move up,
 * are solved and move down on three streams (pinned host buffers overlap fully); several batches
 * can be queued back to back, e.g. one per equation kind of a dependency wave.  Inputs must stay
 * valid and outputs are undefined until gcs_b200_wait(device) returns. */
GCS_B200_API int gcs_b200_solve_host_async(const gcs_b200_batch* batch, int device);
GCS_B200_API int gcs_b200_wait(int device);
/* Only the sub-systems [first, first + count) of the batch, on `device`, asynchronously: the
 * unit gcs_b200_solve_sharded is made of (a caller can place index ranges on devices its own way).
 * The range's results land in rows first .. first+count-1 of the batch's arrays; the per-seed
 * planes keep the full batch's pitch n. */
GCS_B200_API int gcs_b200_solve_host_range_async(const gcs_b200_batch* batch, int device, int64_t first, int64_t count);

/* Host buffers, sharded by batch index over the first n_dev devices of the last gcs_b200_init
 * call, in the order given there (without an init call: ordinals 0..n_dev-1; n_dev <= 0: all of
 * them): device g takes the contiguous range [g*n/G, (g+1)*n/G).  No collective: every device
 * runs its own upload / solve / download pipeline and writes its range of the caller's arrays
 * (explicit guesses and cand planes included).  Synchronous. */
GCS_B200_API int gcs_b200_solve_sharded(const gcs_b200_batch* batch, int n_dev);

/* number of kernel launches issued by this process so far (bench bookkeeping) */
GCS_B200_API int64_t gcs_b200_launch_count(void);
/* name of the kernel a batch of this kind / seed count / variant is solved by (thread-local string) */
GCS_B200_API const char* gcs_b200_kernel_name(int kind, int n_seeds, int variant);
/* the variant GCS_VARIANT_DEFAULT resolves to for a K1 launch of n sub-systems x n_seeds seeds */
GCS_B200_API int gcs_b200_default_variant(int64_t n, int n_seeds);
/* the kernel mapping `variant` (GCS_VARIANT_DEFAULT / GCS_VARIANT_CONTRACTED / an explicit one)
 * resolves to for a launch of n sub-systems of `kind` x n_seeds seeds */
GCS_B200_API int gcs_b200_resolve_variant(int variant, int kind, int64_t n, int n_seeds);

/* GCS_VARIANT_CONTRACTED*: cumulative number of Newton runs on `device` that the guards handed to
 * the literal code since the last call with reset != 0: out[0] run-level guards (conditioning,
 * convergence band, update cap), out[1] root-selection guard.  Diagnostic; synchronises the device. */
GCS_B200_API int gcs_b200_contracted_stats(int device, uint64_t out[2], int reset);
/* the same by reason: out[0] conditioning floor (G1), [1] root selection (G5), [2] |det| bounce (G2),
 * [3] convergence band undecided (G3), [4] update cap (G4), [5] non-finite / huge update (G4),
 * [6], [7] reserved (0) */
GCS_B200_API int gcs_b200_contracted_stats_ex(int device, uint64_t out[8], int reset);

/* Test hook: while set (dev_buf != NULL, capacity > 0), every gcs_b200_solve launch of a
 * GCS_VARIANT_CONTRACTED[_STATIC] batch on `device` with n * n_seeds <= capacity also writes, per
 * Newton run ([n_seeds][n] bytes at dev_buf), how the run was decided: 0 closed form, first-level
 * tests only; 1 closed form, second-level margin test consulted; 2 closed form, careful mode;
 * 3 redone literally by a run-level guard; 4 redone literally by the selection guard.
 * tests/test_gpu_margins.py checks the runs the guards accepted against the CPU checker's own
 * record of how close the literal trajectory came to each decision boundary. */
GCS_B200_API int gcs_b200_debug_path_buffer(int device, uint8_t* dev_buf, int64_t capacity);

/* FP64 pipe micro-benchmarks used as roofline denominators (seconds-scale, device `device`):
 *   what = 0: dependent-free DFMA throughput, returns TFLOP/s counting FMA = 2 flops
 *   what = 1: DADD/DMUL mix throughput (1 flop per instruction), TFLOP/s
 *   what = 2: DFMA dependent-issue latency in SM clocks
 * Returns a negative GCS_E_* code as a double on failure. */
GCS_B200_API double gcs_b200_fp64_probe(int device, int what);

/* Copy-only probe of the host link on `device` (the ceiling of the host-buffer entry points for
 * the same byte counts): `bytes_up` host->device and `bytes_down` device->host, each as `pieces`
 * equal copies from / to pinned (write_combined != 0: write-combined) host memory, on the
 * library's two copy streams.  out[0] = H2D alone GB/s, out[1] = D2H alone GB/s, out[2] / out[3] =
 * best / median milliseconds over `reps` for both directions issued together. */
GCS_B200_API int gcs_b200_pcie_probe(int device, size_t bytes_up, size_t bytes_down, int pieces, int write_combined,
    int reps, double out[4]);

/* Page-locked host memory for batch columns: the host-buffer entry points move pinned buffers at
 * PCIe rate and asynchronously, pageable ones through the driver's staging copies.  Returns NULL
 * when no CUDA device is available (callers may then fall back to ordinary memory: only the
 * transfer gets slower).  Free with gcs_b200_host_free.  (A C++ host such as the reference has no
 * other way to get pinned memory without linking the CUDA runtime itself.) */
GCS_B200_API void* gcs_b200_host_alloc(size_t bytes);
/* flags: GCS_HOST_WRITE_COMBINED = write-combined pinned memory for INPUT columns the host only
 * ever writes front to back (uncached for host reads; no cache snooping on the way to the device) */
#define GCS_HOST_WRITE_COMBINED 1
GCS_B200_API void* gcs_b200_host_alloc_ex(size_t bytes, int flags);
GCS_B200_API void gcs_b200_host_free(void* p);

/* On-device synthetic instance generator for the parametric sweep (BASELINE config 5) and the
 * 1M-cluster configs: fills K1 columns for indices [first, first+n) with the counter-based
 * splitmix64 stream documented in DESIGN.md.  All pointers are device pointers. */
GCS_B200_API int gcs_b200_synth_pp(int device, void* cuda_stream, uint64_t seed, int64_t first,
    int64_t n, int perturb_of, double* const cols[6], uint8_t* code);

/* ---- sketch programs (csrc/sketch_program.cu) ----
 * The wave plan of a decomposed sketch as device-resident row recipes, run for K instances of the
 * sketch's constraint values: topology and canvas are fixed, only the values vary per instance.  A
 * run enqueues, per wave, one gather launch (writes the kind batches' input columns from the
 * position and value tables, and the zero-fixed anchors into the position table), the kind batches
 * through gcs_b200_solve_many (rows_k x K sub-systems each, 2 seeds), and one scatter launch (every
 * row's output into its target slot), with no host synchronisation between waves. */
typedef struct gcs_b200_program_row {
    int32_t solver;   /* Gcs::B200::SolverId, 1..8 */
    int32_t elem[3];  /* element slots of roles a, b, c (c receives the result) */
    int32_t value[3]; /* value slots of v0, v1, v2; -1 where the solver reads none */
    int32_t code;     /* orientation code of the row (GCS_MAKE_CODE) */
    double sign[3];   /* signOf(canvas side) factor of v0..v2 (1 where the value is not signed) */
    /* canvas constants: solvers 2, 5: gnx gny canvas_len; 6, 7: cfx cfy; 3, 8: gnx gny cfdx cfdy
     * canvas_len, and for 3 also fdx fdy x1 x2 (direction and endpoints (x1,0), (x2,0) of the
     * anchored line) */
    double canvas[9];
} gcs_b200_program_row;

typedef struct gcs_b200_program_desc {
    int32_t n_waves;
    int32_t n_slots;
    int32_t n_values;
    int32_t reserved;
    int64_t n_rows;
    const gcs_b200_program_row* rows; /* [n_rows], wave-major, kind-minor */
    const int64_t* offsets;           /* [n_waves * GCS_KIND_COUNT + 1]: rows of (wave w, kind k) are
                                         offsets[w*5 + k-1] .. offsets[w*5 + k]; offsets[0] = 0,
                                         non-decreasing, last = n_rows */
    const uint8_t* slot_is_line;      /* [n_slots]: 0 point, 1 line */
    const double* initial;            /* [n_slots][4]: positions before the first wave (point: x, y, -, -) */
    const uint8_t* value_is_angle;    /* [n_values]: 1 = the slot holds cos(angle) (read as v0 of solvers 3, 8 only) */
} gcs_b200_program_desc;

typedef struct gcs_b200_program gcs_b200_program;

/* Validates the descriptor (before any device call: slots, value slots, offsets, solver ids, the
 * kind of every row's segment, role types, and that the rows of one wave, which run concurrently,
 * have disjoint footprints: no slot written by two rows of a wave, none written by one row and read
 * by another; writes are roles a, b, c of solvers 1-3 and c of solvers 4-8, reads a, b of solvers
 * 4-8; shared reads are fine) and uploads it to `device`.  Host pointers; nothing of them is kept.
 * GCS_E_INVALID with a message for a malformed descriptor, GCS_E_NO_DEVICE without a device. */
GCS_B200_API int gcs_b200_program_create(const gcs_b200_program_desc* desc, int device, gcs_b200_program** out);
/* Runs K = n_instances >= 1 instances, stream-ordered on `cuda_stream`; every pointer is a device
 * pointer.  values [K][n_values] (angle slots hold cos(angle)); positions [K][n_slots][4] is
 * written from the program's initial positions first, so no state carries over between runs;
 * nonconverged [K] (may be NULL): per instance, the rows whose chosen Newton run did not converge.
 * Runs of one program must not overlap (they share its batch buffers): order them on one stream.
 * Launches per run: at most n_waves * (2 + kinds present), independent of K. */
GCS_B200_API int gcs_b200_program_run(gcs_b200_program* prog, int64_t n_instances, const double* values, double* positions,
    uint32_t* nonconverged, int variant, void* cuda_stream);
/* The same with host buffers (pinned ones move asynchronously): values up, run, positions and
 * counts down on the program's own stream, then synchronises.  ms (may be NULL) receives the
 * device time of upload, run and download. */
GCS_B200_API int gcs_b200_program_run_host(gcs_b200_program* prog, int64_t n_instances, const double* values, double* positions,
    uint32_t* nonconverged, int variant, float ms[3]);
/* Tangent runs: gcs_b200_program_run, plus the directional derivatives of every position with
 * respect to the values (forward mode).  For each instance k and T = n_tangents >= 1 directions
 * dvalues[k][:][t]:
 *     dpositions[k][s][c][t] = sum_v d positions[k][s][c] / d values[k][v] * dvalues[k][v][t]
 * Layouts are instance-major with the direction innermost: dvalues [K][n_values][T], dpositions
 * [K][n_slots][4][T].  With dvalues[k] the identity (T = n_values), dpositions[k] read as
 * [n_slots * 4][T] is the full Jacobian of instance k.  An angle slot holds cos(angle), so its
 * dvalues entry is d(cos(angle)).
 * Every slot's tangent is 0 before the first wave (the initial positions are constants).  A row
 * whose chosen Newton run did not converge (what `nonconverged` counts) is not a root, and the
 * tangents of its target are NaN; they propagate to whatever depends on it.  A converged row's
 * tangent is the implicit-function-theorem one, a 2x2 solve with the Jacobian at its root
 * (csrc/newton_tangent.cuh states the operation order); a singular Jacobian gives what the IEEE
 * division gives.  Root choice is piecewise constant and contributes nothing.
 * Positions, nonconverged and the kernels that solve them are those of gcs_b200_program_run; the
 * run adds one launch per wave.  Checked before any device call: n_tangents >= 1, dvalues non-null
 * when n_values > 0, dpositions non-null when n_slots > 0, and what gcs_b200_program_run checks. */
GCS_B200_API int gcs_b200_program_run_tangents(gcs_b200_program* prog, int64_t n_instances, const double* values,
    double* positions, uint32_t* nonconverged, int32_t n_tangents, const double* dvalues, double* dpositions,
    int variant, void* cuda_stream);
/* The same with host buffers, as gcs_b200_program_run_host (dvalues go up with the values, dpositions
 * come down with the positions). */
GCS_B200_API int gcs_b200_program_run_tangents_host(gcs_b200_program* prog, int64_t n_instances, const double* values,
    double* positions, uint32_t* nonconverged, int32_t n_tangents, const double* dvalues, double* dpositions,
    int variant, float ms[3]);
/* Recorded runs: gcs_b200_program_run, plus a tape that the adjoint sweep below reads.  Every (wave,
 * kind) batch gets its own place in one program-owned tape allocation (input and output columns,
 * code, root and convergence planes, and the candidate planes of K2 / K5), each starting at a
 * multiple of 32 sub-systems, instead of one set of batches reused by every wave.  Positions,
 * nonconverged, the kernels that solve them and the launch count are those of gcs_b200_program_run.
 * The tape takes about  sum over waves and kinds of rows x K x (8 x (in + out columns) + 4, + 32 for
 * K2 / K5)  bytes: it grows with n_rows x K, not with the largest wave as a plain run's batches do.
 * It is kept until the next recorded run replaces it; plain and tangent runs leave it alone. */
GCS_B200_API int gcs_b200_program_run_recorded(gcs_b200_program* prog, int64_t n_instances, const double* values, double* positions,
    uint32_t* nonconverged, int variant, void* cuda_stream);
/* The same with host buffers, as gcs_b200_program_run_host. */
GCS_B200_API int gcs_b200_program_run_recorded_host(gcs_b200_program* prog, int64_t n_instances, const double* values,
    double* positions, uint32_t* nonconverged, int variant, float ms[3]);
/* Adjoints (reverse mode) of the program's last recorded run, with that run's K: for each instance k
 * and T = n_cotangents >= 1 cotangents adj_positions[k][:][:][t] (a weight on every position
 * coordinate),
 *     adj_values[k][v][t] = sum_{s,c} adj_positions[k][s][c][t] * d positions[k][s][c] / d values[k][v]
 * the transpose of the Jacobian whose columns gcs_b200_program_run_tangents computes.  Layouts are
 * instance-major with the cotangent innermost: adj_positions [K][n_slots][4][T] (device, read, not
 * changed), adj_values [K][n_values][T] (device, fully written).  An angle slot holds cos(angle), so
 * its adjoint is with respect to cos(angle).
 * Order of summation (deterministic: independent of K, the stream and the schedule): a working copy
 * of adj_positions is swept over the waves from last to first.  Per wave, each row takes the adjoints
 * of the slot coordinates it wrote (its target, and for solvers 1-3 the anchors) and zeroes them,
 * maps them through the transpose of its linearisation and of the gather (csrc/newton_adjoint.cuh,
 * csrc/sketch_program.cu state the operation order), and every slot and value entry the wave read
 * then receives its rows' contributions in ascending (row, role) order, each added to the running
 * entry one at a time.  What is left in the working table after wave 0 belongs to the initial
 * positions, which are constants, and is dropped.
 * Rows without a root: a row whose chosen Newton run did not converge has no derivative.  If its
 * output adjoint for (k, t) is not all zero (NaN counts as non-zero), adj_values[k][:][t] is NaN
 * entirely (forward mode gives NaN for every value it depends on); if it is all zero, the row
 * contributes nothing.
 * Stream-ordered on `cuda_stream` and must come after its recorded run there (the tape is read on the
 * device); does not synchronise.  Launches: at most 2 per non-empty wave + 1.  Memory: working tables
 * of K x T x (n_slots x 32 + n_values x 8 + rows of the largest wave x 88 + 1) bytes.  Checked before
 * any device call: a null program, n_cotangents >= 1, adj_positions non-null when n_slots > 0,
 * adj_values non-null when n_values > 0, and that the program has a recorded run. */
GCS_B200_API int gcs_b200_program_adjoints(gcs_b200_program* prog, int32_t n_cotangents, const double* adj_positions,
    double* adj_values, void* cuda_stream);
/* The same with host buffers: adj_positions up, the sweep, adj_values down on the program's own
 * stream, then synchronises; ms (may be NULL) receives the device time of the three. */
GCS_B200_API int gcs_b200_program_adjoints_host(gcs_b200_program* prog, int32_t n_cotangents, const double* adj_positions,
    double* adj_values, float ms[3]);
GCS_B200_API void gcs_b200_program_destroy(gcs_b200_program* prog);

/* Test hook: on-device self check of the hand-written division / square root / 2x2 QR fast paths
 * against the generic IEEE code (csrc/selftest.cu).  Fills counts[8]:
 *   [0] divisions on the fast path, [1] of those differing from a/b,
 *   [2] square roots on the fast path, [3] of those differing from sqrt(a),
 *   [4] 2x2 systems accepted by the fast solver, [5] of those differing from the generic solver,
 *   [6] systems tried, [7] operand pairs tried.   [1], [3], [5] must be 0. */
GCS_B200_API int gcs_b200_selftest(int device, uint64_t seed, int64_t n, uint64_t counts[8]);

#ifdef __cplusplus
}
#endif

#endif /* GCS_B200_H */
