/*
 * dhqr.h — C-ABI of libdhqr.so: B200-native (sm_100a) blocked Householder QR behind
 * DistributedHouseholderQR.jl's qr! / \ entry points.
 *
 * The reference (pure Julia) has no FFI of its own; each entry point below names the Julia
 * method it replaces (S:n = src/DistributedHouseholderQR.jl:n of the reference).  A Julia shim
 * (distributedhouseholderqr.jl_b200/julia/DistributedHouseholderQRB200.jl, see INTEGRATION.md)
 * ccall's these with CuPtr{Float64}; the Python host package binds them with ctypes.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / CUDA.jl types in any signature.
 *   - every function returns int: 0 = ok; < 0 = -(1-based index of the offending argument),
 *     LAPACK-info style; > 0 = CUDA/NCCL failure (text via dhqr_last_error()).
 *   - matrices are column-major double with leading dimension lda >= m (Julia Matrix /
 *     localpart(DArray)).  Device pointers unless the name says _host_.
 *   - stream-ordered: work is enqueued on the caller's cudaStream_t (passed as void*; NULL =
 *     legacy default stream).  Synchronisation points, all of them: (i) the _host_ entry points block
 *     until their result is in host memory; (ii) dhqr_qr_f64 with the default blocked path synchronises
 *     the stream ONCE before returning whenever a panel went through the speculative 128-column chain
 *     (option "wide_panel", on by default: its conditioning guards are evaluated on the device and a
 *     refused panel is redone by the 32-column chain); (iii) with nranks > 1 every qr / apply_qt /
 *     backsolve call exchanges the column partition first (one small all-gather + stream sync);
 *     (iv) workspace growth (first call, or a larger problem than any before) allocates device memory.
 *     Everything else returns without synchronising.
 *   - no pointer to caller memory is retained after return; workspace lives in the handle.
 *   - a handle is not thread-safe and its calls share one workspace: one handle per host thread, and
 *     consecutive calls on one handle must be on the same stream or ordered by the caller (events);
 *     the library does not order calls that arrive on different streams (the reference is not
 *     re-entrant either: Polyester @batch, S:203-206).
 *   - SPMD for multi-GPU: every rank (one process per GPU) makes the same call with its own
 *     column block (col0 = first global column, 0-based = the reference's LocalColumnBlock.dj, S:34).
 *   - storage format on return == the reference's (S:127-135): Householder vectors scaled to
 *     |v|^2 = 2 in the lower trapezoid INCLUDING the diagonal, R's strict upper triangle above
 *     it, diag(R) in alpha.
 */
#ifndef DHQR_H
#define DHQR_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dhqr_context *dhqr_handle;

#define DHQR_VERSION 100 /* 0.1.0 */
#define DHQR_NCCL_UNIQUE_ID_BYTES 128

/* ---- library / handle -------------------------------------------------------------------- */
int dhqr_version(void);
/* Text of the last error raised on the calling thread ("" if none). */
const char *dhqr_last_error(void);

/* Single-GPU handle on CUDA device `device` (replaces nothing in the reference: the Julia
 * package keeps no state; the handle owns workspace and the grid-barrier words). */
int dhqr_create(dhqr_handle *h, int device);
/* Multi-GPU handle: rank `rank` of `nranks`, NCCL communicator built from `unique_id`
 * (DHQR_NCCL_UNIQUE_ID_BYTES bytes from dhqr_nccl_unique_id() on rank 0, shipped by the host:
 * torch.distributed in Python, Distributed.jl in Julia).  Replaces the reference's use of
 * Distributed/SharedArrays (S:116-118, S:141-143, S:227-229, S:260-267, S:302, S:318). */
int dhqr_create_dist(dhqr_handle *h, int device, const void *unique_id, int rank, int nranks);
int dhqr_nccl_unique_id(void *out_unique_id);
int dhqr_destroy(dhqr_handle h);
/* Tunables (dhqr_set_option / dhqr_get_option):
 *   "nb"          outer panel width, multiple of 32 in [32,128] (default 128)
 *   "lookahead"   1 (default): panel chain on a high-priority stream ahead of the bulk update; 0: one stream, serial
 *   "wide_panel"  1 (default): full, 32-aligned outer panels of width 128 are factored by the 128-column chain
 *                 (CholeskyQR2 + Householder reconstruction on the whole panel: 3 grid-wide reductions per 128 columns,
 *                 no cooperative launch); refused panels and all other panels use the 32-column chain below
 *   "wide_kappa"  guard of the 128-column chain (default 1000, >= 1): a panel whose first Cholesky factor has
 *                 ||D R1^{-1}||_F above it is refused and redone by the 32-column chain
 *   "panel_fast"  1 (default): inner panels by CholeskyQR2 + Householder reconstruction with on-device fallback
 *                 to the column-by-column kernel; 0: always column by column
 *   "qt_vec"      1 (default): Q'b / Qb with ONE right-hand side as a GEMV sweep (T' of every panel computed first, then two
 *                 HBM-bound launches per panel that read the reflectors in place); 0: the GEMM-shaped block update, as for nrhs > 1
 *   "host_chunk"  columns per upload chunk of dhqr_qr_host_f64 (default 512, a multiple of 128; 0: one upload, no overlap);
 *                 "host_h2d_gbs" (50), "host_tflops" (27), "host_chain_us" (300): what its join-step planner assumes about the
 *                 host link, the device and a step of the schedule on a narrow window; "host_first" (0 = three panels): columns
 *                 of the first, exposed upload; "host_trace" 1: stage timeline on stderr.  A wrong assumption costs idle time,
 *                 never correctness
 *   "sync"        1: cudaStreamSynchronize + error check after every kernel launch (debugging; implies serial)
 *   "profile"     1: CUDA-event bracket per launch (implies serial), read with dhqr_profile_get
 *   read-only:    "sms", "rank", "nranks", "panels_fast", "panels_fallback" (inner panels taken by either path),
 *                 "wide_panels" (outer panels factored by the 128-column chain), "wide_redone" (restarts after a refusal)
 * Any other key is refused with -2. */
int dhqr_set_option(dhqr_handle h, const char *key, int64_t value);
int dhqr_get_option(dhqr_handle h, const char *key, int64_t *value);
/* Number of kernel launches enqueued by this handle since creation (bench.py: gpu_launches). */
int dhqr_launch_count(dhqr_handle h, int64_t *count);
/* Per-kernel-class timing with CUDA events on the launching stream (option "profile" = 1 turns the
 * brackets on; the reference keeps the same kind of accumulators as t1a/t1b/t2, S:126-146, S:291).
 * dhqr_profile_get returns slot `index` (0.. until -2): class name, accumulated milliseconds, launch
 * count and algorithmic work (flops for the GEMM classes, bytes for the panel).  Blocks on the events. */
int dhqr_profile_reset(dhqr_handle h);
int dhqr_profile_get(dhqr_handle h, int index, char *name, int name_len, double *ms, int64_t *count,
                     double *work);

/* ---- qr!  (S:311-315 -> householder! S:113-120 -> _householder! S:122-148 -> _householder_inner!
 *            S:198-213 with partialdot S:42-49 and hotloop! S:156-160) --------------------------
 * Factor the m x n_global matrix whose columns [col0, col0+n_local) are stored in dA_local
 * (m x n_local, lda).  In place.  d_alpha (length n_global) receives diag(R) on every rank.
 * nb: 0 = handle default (blocked, compact-WY trailing update on the fp64 tensor pipe);
 *     1 = unblocked column-by-column path (BASELINE config 2);
 *     otherwise a multiple of 32 in [32,128]. */
int dhqr_qr_f64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                double *dA_local, int64_t lda, double *d_alpha, int nb, void *stream);

/* ---- \  (S:317-321 -> solve_householder! S:284-294) ---------------------------------------- */
/* b <- Q'b  (_solve_householder1! S:226-242 / S:215-224).  d_b: m x nrhs, ldb >= m, in place;
 * identical on every rank on entry and on return. */
int dhqr_apply_qt_f64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                      const double *dA_local, int64_t lda, double *d_b, int64_t ldb, int nrhs,
                      void *stream);
/* b <- Q b = H_1 ... H_n b: the inverse of the sweep above (not in the reference, which never forms Q; SURVEY 8f-3:
 * exposes the factorisation as an operator, e.g. to form Q explicitly or to compute residuals b - A x = Q [0; (Q'b)[n:]]). */
int dhqr_apply_q_f64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                     const double *dA_local, int64_t lda, double *d_b, int64_t ldb, int nrhs, void *stream);
/* b[0:n] <- R^{-1} b[0:n]  (_solve_householder2! S:256-282 / S:244-254), R = triu(A,1)+diag(alpha). */
int dhqr_backsolve_f64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                       const double *dA_local, int64_t lda, const double *d_alpha, double *d_b,
                       int64_t ldb, int nrhs, void *stream);
/* Both phases (solve_householder! S:284-294): x = d_b[0:n_global, :] on return. */
int dhqr_solve_f64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                   const double *dA_local, int64_t lda, const double *d_alpha, double *d_b,
                   int64_t ldb, int nrhs, void *stream);

/* ---- ComplexF64 (the reference's second element type: test/runtests.jl:43; alphafactor(::Complex) S:9, the conjugating
 * partialdot S:51-59, the complex hotloop! S:162-196).  Matrices and vectors are interleaved (re, im) doubles = Julia
 * ComplexF64 / C double _Complex; lda, ldb count COMPLEX elements; alpha is complex (length n).  Same storage format:
 * v scaled to |v|^2 = 2 in the lower trapezoid including the diagonal, H_j = I - v_j v_j^H, diag(R) in alpha.
 * Single GPU: col0 must be 0 and n_local == n_global.  Stream-ordered, no synchronisation. */
int dhqr_qr_c64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local, void *dA_local,
                int64_t lda, void *d_alpha, void *stream);
int dhqr_apply_qt_c64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                      const void *dA_local, int64_t lda, void *d_b, int64_t ldb, int nrhs, void *stream);
int dhqr_backsolve_c64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                       const void *dA_local, int64_t lda, const void *d_alpha, void *d_b, int64_t ldb,
                       int nrhs, void *stream);
int dhqr_solve_c64(dhqr_handle h, int64_t m, int64_t n_global, int64_t col0, int64_t n_local,
                   const void *dA_local, int64_t lda, const void *d_alpha, void *d_b, int64_t ldb, int nrhs,
                   void *stream);
/* partialdot(a, b, is, ::Type{<:Complex}) (S:51-59): *d_out = sum_{i in [i0,i1)} conj(a[i]) * b[i]. */
int dhqr_partialdot_c64(dhqr_handle h, const void *d_a, const void *d_b, int64_t i0, int64_t i1, void *d_out,
                        void *stream);

/* ---- host-buffer entry points (single GPU): the call a CPU-side user of qr! / \ makes -------
 * hA (m x n, lda) is copied to the device, factored, and copied back with alpha; blocks until
 * the result is in host memory.  With pinned host memory the call is a pipeline: the matrix goes up in
 * column chunks, the factorisation starts on the first one, every later chunk joins the trailing matrix
 * after a catch-up with the reflectors already finished, and finished panels travel back while later
 * ones are factored; only the first upload and the last download are exposed.  Same reflectors as
 * dhqr_qr_f64 on the resident matrix (every column receives every reflector once, in order). */
int dhqr_qr_host_f64(dhqr_handle h, int64_t m, int64_t n, double *hA, int64_t lda, double *h_alpha,
                     int nb);
/* The upload plan dhqr_qr_host_f64 would use for an m x n matrix with panels of nb columns (pure host logic, needs no device;
 * exposed for tests and for callers that want to size pinned staging buffers): chunk j = columns [bounds[j], bounds[j+1]),
 * j < *nchunks; join[j] = step of the look-ahead schedule at which it enters the trailing matrix (join[0] = 0: the first chunk is
 * the initial window).  Every boundary is a multiple of nb (the last is n); join is non-decreasing and never later than one step
 * before the panel chain reaches into the chunk (bounds[j] / nb - 3).  chunk, first, h2d_gbs, tflops, chain_us: the options
 * "host_chunk", "host_first", "host_h2d_gbs", "host_tflops", "host_chain_us".  cap = capacity of bounds (cap) and join (cap - 1). */
int dhqr_plan_host_upload(int64_t m, int64_t n, int nb, int chunk, int first, int h2d_gbs, int tflops, int chain_us, int cap,
                          int64_t *bounds, int *join, int *nchunks);
/* x = H \ b from a host-resident factorisation (hA, h_alpha) and host b (length m); x length n. */
int dhqr_ldiv_host_f64(dhqr_handle h, int64_t m, int64_t n, const double *hA, int64_t lda,
                       const double *h_alpha, const double *h_b, double *h_x);

/* ---- primitives exposed for parity tests ---------------------------------------------------- */
/* partialdot(a, b, is, ::Type{<:Real}) (S:42-49): *d_out = sum_{i in [i0,i1)} a[i]*b[i] (0-based). */
int dhqr_partialdot_f64(dhqr_handle h, const double *d_a, const double *d_b, int64_t i0, int64_t i1,
                        double *d_out, void *stream);
/* A[i,j] = U[0,1) from the counter-based generator keyed on (seed, i0+i, j0+j); bit-identical to
 * oracle/dhqr_oracle.c:dhqr_oracle_uniform (mirrors rand(T,m,n) at test/runtests.jl:45-46). */
int dhqr_fill_uniform_f64(dhqr_handle h, uint64_t seed, int64_t i0, int64_t j0, int64_t m, int64_t n,
                          double *dA, int64_t lda, void *stream);

/* ---- kernel-level hooks (unit tests of the individual CUDA kernels; not part of the drop-in) --
 * gemm_vta : Wext[nbp x (nbp+ncols)] = V' * [V | C]  (split over rows, partials reduced by ymake/tinv)
 * tinv     : Linv = (I + stril(V'V))^{-1}
 * ymake    : Y = -Linv * W
 * gemm_cvy : C += V * Y   on rows >= row_lo
 * All operate on the handle's internal V buffer, filled from (dV, ldv) by the call. */
int dhqr_k_block_reflector_f64(dhqr_handle h, int64_t rows, int nbp, const double *dV, int64_t ldv,
                               int64_t row_lo, int ncols, double *dC, int64_t ldc, double *d_linv_out,
                               void *stream);
/* Copy an internal workspace buffer ("wpart", "ybuf", "linv", "vbuf") to d_dst (debugging / tests). */
int dhqr_debug_copy_f64(dhqr_handle h, const char *which, double *d_dst, int64_t nelems, void *stream);
/* Panel kernel: factor the rows x ncols (ncols <= 32) panel at dP in place (reference recurrences
 * S:127-135 + S:208-209 restricted to the panel), alpha -> d_alpha[0:ncols]. */
int dhqr_k_panel_f64(dhqr_handle h, int64_t rows, int ncols, double *dP, int64_t ldp, double *d_alpha,
                     void *stream);

/* 128-column panel chain (CholeskyQR2 + Householder reconstruction, dhqr_wide.cuh): factor the rows x 128 panel at dP in
 * place (same output as 128 steps of S:127-135 + S:208-209 restricted to the panel), alpha -> d_alpha[0:128].
 * *refused = 1 when the on-device guards turned the panel down (dP is then untouched).  Synchronises `stream`. */
int dhqr_k_wide_panel_f64(dhqr_handle h, int64_t rows, double *dP, int64_t ldp, double *d_alpha, int *refused,
                          void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DHQR_H */
