/*
 * mtg_b200.h -- C-ABI of the B200-native batched linear min-derivative solver.
 *
 * Drop-in boundary for ONE path of ethz-asl/mav_trajectory_generation:
 * PolynomialOptimization<N>::solveLinear() and the per-segment assembly feeding it.
 * The reference has no FFI layer; what these entry points replace is the body of the
 * following members (paths under mav_trajectory_generation/include/mav_trajectory_generation/):
 *
 *   mtg_solve_linear_batch_*      impl/polynomial_optimization_linear_impl.h:338-379 solveLinear()
 *                                 + :285-305 updateSegmentTimes() (A^-1, Q per segment)
 *                                 + :307-336 constructR()
 *                                 + :262-283 updateSegmentsFromCompactConstraints()
 *   mtg_coeffs_from_constraints_* impl/...linear_impl.h:499-508 setFreeConstraints()
 *                                 -> :262-283 updateSegmentsFromCompactConstraints()
 *   mtg_compute_cost_batch_*      impl/...linear_impl.h:123-140 computeCost()
 *   mtg_problem_layout            impl/...linear_impl.h:181-260 setupConstraintReorderingMatrix()
 *                                 (the 0/1 matrix C as one column index per row; host only)
 *
 * Conventions
 *   - plain C, no torch / Eigen / STL types cross this boundary; every buffer is caller-owned.
 *   - all arithmetic fp64; polynomial coefficients in INCREASING powers
 *     (polynomial_optimization_linear.h:43-44).
 *   - a "problem" is a constraint TOPOLOGY shared by the whole batch: N coefficients,
 *     derivative_to_optimize r, K segments, D dimensions, and which derivatives each of the
 *     K+1 vertices fixes.  Per trajectory only the segment times and the fixed constraint
 *     VALUES differ (the reference re-uses one factorisation for all D for the same reason,
 *     linear_impl.h:369-375).
 *   - d_fixed / d_free use the reference's compact ordering: constraints sorted by
 *     (vertex, derivative) (polynomial_optimization_linear.h:287-295), i.e. exactly
 *     getFixedConstraints()/getFreeConstraints() (polynomial_optimization_linear.h:194-206).
 *   - nothing here aborts or throws: argument errors return a negative code
 *     (the reference CHECK-aborts, e.g. linear_impl.h:60,76,289,297); per-trajectory numeric
 *     trouble is reported in status[] and never stops the batch.
 *   - a handle is bound to one CUDA device and is single-caller (the reference object is not
 *     thread-safe either); use one handle per host thread / per GPU.
 *   - there is NO CPU fallback: every compute entry point launches sm_100a kernels or fails.
 */
#ifndef MTG_B200_H_
#define MTG_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MTG_MAX_N 12 /* Polynomial::kMaxN, polynomial.h:44 */

/* return codes */
#define MTG_OK 0
#define MTG_ERR_BAD_ARG (-1)      /* null pointer, odd N, r out of [0, N/2-1], K < 1, D < 1 ... */
#define MTG_ERR_CUDA (-2)         /* CUDA runtime error; see mtg_last_error() */
#define MTG_ERR_NO_DEVICE (-3)    /* no sm_100 device / extension cannot run */
#define MTG_ERR_ALLOC (-4)

/* per-trajectory status bits (status[b] == 0 means solved) */
#define MTG_STATUS_BAD_TIME 1     /* some segment time <= 0 or NaN (reference: CHECK_GT, linear_impl.h:297) */
#define MTG_STATUS_NOT_SPD 2      /* non-positive / NaN pivot in the R_pp factorisation */

/* which kernel family a problem is routed to (introspection for tests / profiles) */
#define MTG_KERNEL_WAYPOINT 1     /* specialised block-tridiagonal Cholesky kernels, waypoint topology */
#define MTG_KERNEL_GENERIC 2      /* arbitrary per-vertex masks: masked block-tridiagonal Cholesky */
#define MTG_KERNEL_NOFREE 3       /* n_free == 0: back-substitution only (linear_impl.h:343-349) */

typedef struct mtg_handle mtg_handle;

typedef struct mtg_problem {
  int32_t N; /* coefficients per polynomial, even, 2..12   (template parameter _N, linear.h:45-51) */
  int32_t r; /* derivative_to_optimize in [0, N/2-1]        (setupFromVertices arg, linear.h:67-69) */
  int32_t K; /* number of segments (= vertices - 1) >= 1 */
  int32_t D; /* dimensions >= 1 */
  /* fixed_mask[(K+1)*(N/2)], row-major [vertex][derivative]: 1 = the vertex has a constraint on
   * that derivative (Vertex::hasConstraint, vertex.h:84), 0 = free.  NULL selects the
   * createRandomVertices / "waypoint" topology (vertex.cpp:27-82): first and last vertex fix
   * derivatives 0..N/2-1, interior vertices fix position only. */
  const uint8_t* fixed_mask;
} mtg_problem;

typedef struct mtg_layout {
  int32_t n_all;    /* K*N          getNumberAllConstraints()   */
  int32_t n_fixed;  /*              getNumberFixedConstraints() */
  int32_t n_free;   /*              getNumberFreeConstraints()  */
  int32_t kernel;   /* MTG_KERNEL_* this problem is routed to   */
} mtg_layout;

/* ---- lifecycle ------------------------------------------------------------------------- */
int mtg_create(int device, mtg_handle** out);
void mtg_destroy(mtg_handle* h);
/* last error text of this handle (or of the last failed mtg_create when h == NULL) */
const char* mtg_last_error(const mtg_handle* h);
/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
int64_t mtg_launch_count(const mtg_handle* h);
/* 1 when the visible device of the handle is compute capability 10.x */
int mtg_device_is_sm100(const mtg_handle* h);

/* tuning knobs (results are identical to rounding; used by tests and profiles)
 *   MTG_OPT_WAYPOINT_VARIANT: 0 = default (6 where it applies, else 4 for K <= 8, 3 while the factor fits on chip at
 *                                 two CTAs per SM, 5 beyond),
 *                             1 = one thread per trajectory, 2 = twisted (state in shared memory),
 *                             3 = twisted with the sweep state in tensor memory + TMA tensor stores,
 *                             4 = persistent version of 3 with deep input prefetch,
 *                             5 = chunked (checkpoint + recompute) kernel, any K (default for K too large for 3),
 *                             6 = 4 with the inputs moved by TMA bulk copies (B % 16 == 0, 16-byte aligned inputs, K
 *                                 small enough for an input tile beside the state: K <= 16 at N = 10, D = 3). */
#define MTG_OPT_WAYPOINT_VARIANT 1
#define MTG_OPT_RING_DEPTH 2      /* reserved (the persistent kernel is built with a 3-deep input ring) */
#define MTG_OPT_CTAS_PER_SM 3     /* variant 4 only: cap on resident CTAs per SM, 0 = as many as fit, 9 = one CTA per tile */
#define MTG_OPT_STAGGER_US 4      /* reserved (accepted, no effect: the start-time stagger experiment was removed, DESIGN.md 4) */
#define MTG_OPT_CHUNK_BLOCKS 6    /* chunked (large-K) kernel: resident vertex blocks per lane, 0 = auto */
#define MTG_OPT_GENERIC_VARIANT 7 /* arbitrary masks: 0 = masked block kernel (default), 1 = banded kernel in global scratch */
#define MTG_OPT_MELLINGER_UNFUSED 8 /* 1 = batched Mellinger gradient through expand + solve + cost kernels */
#define MTG_OPT_TMA_INPUTS 9      /* 0 = never, 1 = the TMA-input kernel (v5) where two input tiles fit (double buffered),
                                    2 (default) = also where only one fits (single buffered) */
#define MTG_OPT_EARLY_REFILL 10   /* TMA-input kernel with one tile buffer: 0 = the buffer is refilled with the next tile two
                                   * outward-sweep steps before the tile ends (default), -1 = while the last segment is emitted */
#define MTG_OPT_V5_STATIC_SHAPE 11 /* TMA-input kernel: 0 = the instantiation compiled for the problem's K (K = 16 and 8 at
                                    * N = 10, r = 4, D = 3; K = 4 at N = 8, r = 3, D = 3) where the launch layout is the one
                                    * it was built for (default), -1 = always the run-time-shape kernel; bitwise identical */
#define MTG_OPT_DYNAMIC_TILES 5   /* persistent kernel: warps draw tiles from a global counter: 0 = auto, 1 = always, 2 = never */
int mtg_set_option(mtg_handle* h, int key, int value);

/* ---- host-only layout: the constraint reordering (linear_impl.h:181-260) ---------------- */
/* slot_col (nullable) receives K*N entries: row i*N+s of C (segment i, slot s; s < N/2 is
 * derivative s at the segment start, s >= N/2 derivative s-N/2 at its end) has its single 1 in
 * column slot_col[i*N+s]; columns [0,n_fixed) are d_fixed, [n_fixed, n_fixed+n_free) are d_free. */
int mtg_problem_layout(const mtg_problem* p, mtg_layout* out, int32_t* slot_col);

/* ---- the hot path, DEVICE pointers, asynchronous on `stream` (a cudaStream_t, may be 0) --- */
/* seg_times [B][K], d_fixed [B][D][n_fixed]  ->  coeffs [B][K][D][N]
 * optional: d_free [B][D][n_free], status [B] (int32). */
int mtg_solve_linear_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                               const double* d_fixed, double* coeffs, double* d_free, int32_t* status,
                               void* stream);

/* SURVEY.md 8f-1 ("next" row): time allocation + constraint packing fused into the solve, for the
 * createRandomVertices topology.  positions [B][K+1][D]; segment times are computed on the device as
 * estimateSegmentTimesNfabian(v_max, a_max, magic) (reference src/vertex.cpp:255-272; pass magic = 6.5
 * for the reference default), start/end derivatives 1..N/2-1 are zero (Vertex::makeStartOrEnd,
 * src/vertex.cpp:147-153).  coeffs [B][K][D][N]; seg_times_out [B][K] and status are optional.
 * Reads 8*(K+1)*D bytes per trajectory instead of 8*(K + D*n_fixed). */
int mtg_solve_waypoints_nfabian_batch_f64(mtg_handle* h, int32_t N, int32_t r, int32_t K, int32_t D, int64_t B,
                                          const double* positions, double v_max, double a_max, double magic,
                                          double* coeffs, double* seg_times_out, int32_t* status, void* stream);

/* updateSegmentsFromCompactConstraints for given d_free (setFreeConstraints path). */
int mtg_coeffs_from_constraints_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B,
                                          const double* seg_times, const double* d_fixed,
                                          const double* d_free, double* coeffs, void* stream);

/* computeCost(): cost[b] = 0.5 * sum_{segments, dims} c^T Q(T) c. */
int mtg_compute_cost_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                               const double* coeffs, double* cost, void* stream);

/* SURVEY.md 8f-2 ("next" row): the nonlinear time optimiser's numerical gradient, batched.
 * PolynomialOptimizationNonLinear::getCostAndGradientMellinger (reference
 * impl/polynomial_optimization_nonlinear_impl.h:286-364): cost[b] = computeCost() at seg_times[b], grad[b][n] =
 * (cost with +0.1 s on segment n and -0.1/(K-1) s on the others, clamped at 0.1 s, re-solved) - cost) / 0.1.
 * The K+1 solves of every trajectory run as ONE cost-only launch over the expanded batch: the perturbed times are
 * generated inside the kernel and the cost 0.5 d^T H d is accumulated from the solved end-point derivatives, so no
 * perturbed input and no coefficient is ever written (shapes without a fused kernel take expand + solve + cost
 * kernels).  cost may be NULL. */
int mtg_cost_gradient_mellinger_batch_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                          const double* d_fixed, double* cost, double* grad, void* stream);

/* SURVEY.md 8f-3 ("next" row): batched Trajectory::evaluate on a uniform grid t_s = t_start + s*dt,
 * s < n_samples (reference src/trajectory.cpp:48-79 conventions per sample: a time on a vertex belongs to the
 * segment on its right, t == total time is the end of the last segment, beyond the end yields zeros;
 * Horner form of Polynomial::evaluate, polynomial.h:134-149).  coeffs [B][K][D][N] -> out [B][n_samples][D]. */
int mtg_evaluate_batch_f64(mtg_handle* h, int32_t N, int32_t K, int32_t D, int64_t B, const double* seg_times,
                           const double* coeffs, int32_t derivative, double t_start, double dt, int32_t n_samples,
                           double* out, void* stream);

/* SURVEY.md 8f-3: batched Trajectory::evaluateRange (reference src/trajectory.cpp:81-141) -- and with
 * derivs = {0,1,2,3,4} the sample set of sampleTrajectoryInRange (src/trajectory_sampling.cpp:45-110) -- for B
 * trajectories at once.  The reference's sequential walk is replayed exactly (running time_in_segment += dt; the
 * sample clock starts at the start of the segment that contains t_start; a sample on a segment end belongs to the
 * left segment; the walk ends after the last segment), and every sample is Polynomial::evaluate's arithmetic
 * (separate multiply and add), so samples are bit-identical to an x86 build of the reference.
 *   out            [B][max_samples][n_derivs][D]   (rows >= n_samples[b] are zero)
 *   n_samples      [B]  number of samples the reference would produce (may exceed max_samples: only the first
 *                       max_samples are stored); -1 when t_start lies beyond the trajectory (reference: LOG(ERROR),
 *                       empty result)
 *   sampling_times [B][max_samples] or NULL: the reference's `sampling_times` output
 * derivs is a HOST array of n_derivs (<= 8) derivative orders. */
int mtg_evaluate_range_batch_f64(mtg_handle* h, int32_t N, int32_t K, int32_t D, int64_t B, const double* seg_times,
                                 const double* coeffs, double t_start, double t_end, double dt, int32_t n_derivs,
                                 const int32_t* derivs, int32_t max_samples, double* out, int32_t* n_samples,
                                 double* sampling_times, void* stream);

/* ---- the hot path, HOST pointers (what PolynomialOptimization<N>::solveLinear() calls) ---- */
/* Same contract with host buffers; H2D, kernels and D2H are pipelined over internal streams and
 * the call returns when the results are in the host buffers.  Pinned buffers (mtg_host_alloc)
 * make the copies asynchronous; pageable buffers work but serialise. */
int mtg_solve_linear_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                    const double* d_fixed, double* coeffs, double* d_free,
                                    int32_t* status);
int mtg_solve_waypoints_nfabian_batch_host_f64(mtg_handle* h, int32_t N, int32_t r, int32_t K, int32_t D, int64_t B,
                                               const double* positions, double v_max, double a_max, double magic,
                                               double* coeffs, double* seg_times_out, int32_t* status);
int mtg_coeffs_from_constraints_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B,
                                               const double* seg_times, const double* d_fixed,
                                               const double* d_free, double* coeffs);
int mtg_compute_cost_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                    const double* coeffs, double* cost);

/* host-pointer variants of the two widened entry points (single stream: copy in, kernels, copy out) */
int mtg_cost_gradient_mellinger_batch_host_f64(mtg_handle* h, const mtg_problem* p, int64_t B, const double* seg_times,
                                               const double* d_fixed, double* cost, double* grad);
int mtg_evaluate_range_batch_host_f64(mtg_handle* h, int32_t N, int32_t K, int32_t D, int64_t B, const double* seg_times,
                                      const double* coeffs, double t_start, double t_end, double dt, int32_t n_derivs,
                                      const int32_t* derivs, int32_t max_samples, double* out, int32_t* n_samples,
                                      double* sampling_times);

/* ---- memory helpers (so host code above the ABI needs no CUDA headers) -------------------- */
void* mtg_host_alloc(mtg_handle* h, uint64_t bytes);   /* pinned */
void mtg_host_free(mtg_handle* h, void* ptr);
void* mtg_device_alloc(mtg_handle* h, uint64_t bytes);
void mtg_device_free(mtg_handle* h, void* ptr);
int mtg_memcpy_h2d(mtg_handle* h, void* dst, const void* src, uint64_t bytes, void* stream);
int mtg_memcpy_d2h(mtg_handle* h, void* dst, const void* src, uint64_t bytes, void* stream);
int mtg_memcpy_d2d(mtg_handle* h, void* dst, const void* src, uint64_t bytes, void* stream);  /* incl. peer memory */
int mtg_stream_synchronize(mtg_handle* h, void* stream);

/* ---- NVLink peer memory between the one-process-per-GPU ranks of a job ----------------------------------------
 * The owner exports a device buffer (64-byte CUDA IPC handle + offset of `ptr` inside its allocation), another
 * rank imports it with ITS device current, which makes the buffer directly addressable by the kernels of that
 * rank: handing a slice of the root's coefficient buffer to mtg_solve_linear_batch_f64 as `coeffs` makes the solve
 * kernels store their results over NVLink straight into their final place -- the gather of BASELINE config C5
 * fused into the solve (mav_trajectory_generation_b200/sharding.py:peer_solve_into_root). */
int mtg_ipc_export(mtg_handle* h, const void* ptr, uint8_t handle_out[64], uint64_t* offset_out);
int mtg_ipc_import(mtg_handle* h, const uint8_t handle[64], uint64_t offset, void** ptr_out, void** base_out);
int mtg_ipc_close(mtg_handle* h, void* base);

/* library version (major*10000 + minor*100 + patch) */
int mtg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MTG_B200_H_ */
