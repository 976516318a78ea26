/*
 * b200lasso.h -- C ABI of libb200lasso.so: the B200 (sm_100a) implementation of the
 * lasso block proximal-gradient hot path of kingold5/convex_optimization.
 *
 * This is the drop-in boundary (SURVEY.md section 8(b)): plain pointers and sizes, int
 * status returns (0 = ok, non-zero = failure, text via b200l_last_error()), an opaque
 * context, no Python or torch types.  The Python mirror of the reference interface
 * (convex_optimization_b200/{gpu_calculation,lasso}.py) binds it with ctypes; see
 * INTEGRATION.md for the stub a maintainer of the reference would add.
 *
 * Every entry point names the reference interface (file:line under the reference
 * tree) it replaces.  There is no CPU fallback: every compute entry point fails when
 * no CUDA device is present.
 */
#ifndef B200LASSO_H
#define B200LASSO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200L_ABI_VERSION 1
#define B200L_NTRACE 16
#define B200L_NTTRACE 96

/* arithmetic type of A and of the inner products (vectors and line-search scalars are
 * always kept in double, SURVEY.md section 7 "keep line-search scalars in f64") */
#define B200L_F32 0
#define B200L_F64 1

/* device layout of A.  ROWMAJOR is the reference's GPU layout (BLOCK, N, w)
 * (gpu_calculation.py:172-173); TRANSPOSED is the pre-transposed (BLOCK, w, N) copy the
 * reference only sketched (gpu_calculation.py:94-113,174 and README:3). */
#define B200L_ROWMAJOR 0
#define B200L_TRANSPOSED 1

typedef struct b200l_ctx b200l_ctx;

/* -- diagnostics ------------------------------------------------------------------ */
const char *b200l_last_error(void);          /* text of the last failure on this thread */
int b200l_abi_version(void);
int b200l_device_count(int *count);          /* fails (non-zero) without a CUDA driver/GPU */
/* name, SM count, max opt-in shared memory per block, L2 bytes of `device` */
int b200l_device_info(int device, char *name, int name_len, int *sm_count,
                      int *smem_optin, int *l2_bytes);

/* -- context ----------------------------------------------------------------------
 * Replaces GPU_Calculation.__init__/init_cpu_array/init_gpu_array
 * (gpu_calculation.py:148-236): problem shape, block count, device buffers.
 * N rows, K columns, nblocks column blocks of width w = K / nblocks (K % nblocks == 0,
 * as the reference requires, cpu_calculation.py:27).  `ld` (out) is the padded leading
 * dimension, in elements, of one row of a device block: ROWMAJOR blocks are (N, ld) with
 * ld >= w, TRANSPOSED blocks are (w, ld) with ld >= N; rows start 16-byte aligned. */
int b200l_ctx_create(b200l_ctx **out, int dtype, int layout, int64_t N, int64_t K,
                     int32_t nblocks, int device);
int b200l_ctx_destroy(b200l_ctx *ctx);
int b200l_ctx_ld(const b200l_ctx *ctx, int64_t *ld);
/* stream all work of this context is issued on (a cudaStream_t; NULL = default stream) */
int b200l_ctx_set_stream(b200l_ctx *ctx, void *stream);
/* Device storage of A, owned by the caller (a torch CUDA tensor in the Python mirror;
 * the reference's A_b_gpu, gpu_calculation.py:224): nblocks contiguous blocks of
 * rows*ld elements of `dtype`, padding zero-filled, pointer 128-byte aligned. */
int b200l_ctx_bind_A(b200l_ctx *ctx, const void *A_dev);

/* -- legacy mat-vec entry points (host vectors, as the reference's methods) ---------
 * diag_ata  : column squared norms d_k, out[K] doubles, block-major
 *             (GPU_Calculation.diag_ATA gpu_calculation.py:246-261, kernel :116-137;
 *              cpu_calculation.py:35-42).
 * gemv_t    : g[w] = A_m^T r[N]   (mat_tMulVec_DiffSize gpu_calculation.py:264-277,
 *             kernel :20-55; fun_s12 cpu_calculation.py:30-31; cublasDgemv 'N' lasso.py:336).
 * gemv_n    : q[N] = A_m d[w]     (matMulVec_DiffSize gpu_calculation.py:280-292,
 *             kernel :58-91; fun_s22 cpu_calculation.py:45-46; cublasDgemv 'T' lasso.py:342).
 * Vectors are host doubles; the copies are inside the call, like the reference's. */
int b200l_diag_ata(b200l_ctx *ctx, double *out_host);
int b200l_gemv_t(b200l_ctx *ctx, int32_t m, const double *r_host, double *g_host);
int b200l_gemv_n(b200l_ctx *ctx, int32_t m, const double *d_host, double *q_host);
/* The same two mat-vecs on DEVICE vectors of doubles, queued on the context's stream without any
 * copy to or from the host and without synchronisation: what the reference's cuBLAS classes do
 * with cublasDgemv on gpuarrays (lasso.py:334-353, :404-419, :546-557).  r_dev: N entries,
 * g_dev: w entries; d_dev: w entries, q_dev: N entries. */
int b200l_gemv_t_dev(b200l_ctx *ctx, int32_t m, const double *r_dev, double *g_dev);
int b200l_gemv_n_dev(b200l_ctx *ctx, int32_t m, const double *d_dev, double *q_dev);
/* diag(A^T A) is computed once per bound matrix (one pass over A) and kept: b200l_diag_ata and
 * b200l_set_problem share it.  b200l_set_diag replaces it by the caller's values -- the d_ATA
 * argument of the solver classes (lasso.py:26-30), d_host[nblocks * w] doubles, block-major;
 * d_host = NULL goes back to the diagonal of the bound matrix. */
int b200l_set_diag(b200l_ctx *ctx, const double *d_host);

/* -- fused solver state -------------------------------------------------------------
 * The fused path keeps x (K), the running residual r = A x - b (N), d = diag(A^T A) and
 * 1/d on the device.  Replaces the host state of ClassLasso.run (lasso.py:210-219) and
 * the device state of ClassLassoCB_v2 (lasso.py:367-375,477-500).
 * set_problem : upload b (host, N doubles), compute d on the device (lasso.py:29-30),
 *               set x = 0 and r = -b (lasso.py:89-91,105).
 * set_x       : warm start (not in the reference; SURVEY.md section 8(f)1): x <- x0
 *               (host, K doubles), r <- A x0 - b.
 * get_x/get_r : copy x (K doubles) / r (N doubles) to the host. */
int b200l_set_problem(b200l_ctx *ctx, const double *b_host);
int b200l_reset(b200l_ctx *ctx);              /* x = 0, r = -b, stop counter = 0 */
int b200l_set_x(b200l_ctx *ctx, const double *x_host);
/* keep x and r, restart the stop counter and the cyclic block order (next mu of a path) */
int b200l_restart_counters(b200l_ctx *ctx);
int b200l_get_x(b200l_ctx *ctx, double *x_host);
int b200l_get_r(b200l_ctx *ctx, double *r_host);

/* -- the hot path -------------------------------------------------------------------
 * Runs up to `nsteps` iterations of the reference loop body (lasso.py:102-157 /
 * :228-278 / :508-599) in ONE persistent cooperative kernel: for each step
 *   m = order[step]                                            (lasso.py:104)
 *   g = A_m^T r ; u = d_m*x_m - g ; Bx = S_mu(u)/d_m ; D = Bx - x_m   (:107-119)
 *   q = A_m D ; gamma = clip(-(r.q + mu(|Bx|_1-|x_m|_1))/|q|^2, 0, 1)  (:121-136)
 *   err = |g - clip(g - x_m, -mu, mu)|_inf and the all-blocks stop rule (:138-150)
 *   x_m += gamma D ; r += gamma q                                (:153-155)
 * order_host : nsteps block indices, or NULL for the cyclic order (t % nblocks)
 *              continuing from the context's step counter.
 * err_bound  : < 0 disables the stop rule (the reference's non-float ERR_BOUND,
 *              lasso.py:74-77).
 * err_hist_host / time_hist_host : optional per-step outputs (nsteps doubles each):
 *              the error criterion of the step (err_iter, lasso.py:54-58) and seconds
 *              since kernel start at the end of the step (time_iter, lasso.py:60-62).
 * steps_done : loop bodies entered (the reference's t+1 at exit, lasso.py:64-68).
 * stopped    : 1 if the stop rule fired (the breaking step's update is NOT applied,
 *              lasso.py:141-153).
 * kernel_ms  : device time of the launch measured with CUDA events on the stream.
 * If steps_done, stopped, kernel_ms and both hist pointers are all NULL the call does
 * not synchronise. */
int b200l_run(b200l_ctx *ctx, const int32_t *order_host, int64_t nsteps, double mu,
              double err_bound, double *err_hist_host, double *time_hist_host,
              int64_t *steps_done, int32_t *stopped, double *kernel_ms);

/* launch geometry of the fused kernel for this context (for DESIGN/bench reporting) */
int b200l_run_config(b200l_ctx *ctx, int32_t *grid, int32_t *threads, int32_t *smem_bytes,
                     int32_t *tile_rows, int32_t *ring_slots, int32_t *tiles_per_slab);
/* tunables: ring slot bytes target (0 = default: 48 KiB when a block stays in L2 between the two
 * passes, else 64 KiB).  max_inflight_tiles must be 0: a CTA keeps as many bulk copies in flight as
 * its ring has slots, and any other value fails. */
int b200l_set_tuning(b200l_ctx *ctx, int32_t slot_bytes_target, int32_t max_inflight_tiles);

/* Diagnostics of the hot path.  run_traced runs `nsteps` unbounded steps (cyclic order,
 * like b200l_run with err_bound < 0) and returns, for every CTA and step,
 * B200L_NTRACE time stamps in ns since kernel start: [0] step start, [1] pass 1 (A_m^T r)
 * done, [2] partial gradient published, [3] my columns gathered, [4] partials combined,
 * [5] pending step resolved (gamma), [6] prox done / D published, [7] D gathered,
 * [8] pass 2 (A_m D) done, [9] line-search partials done, [10] first inbox fetch landed,
 * [11] inbox words thread 0 had to re-read from L2, [12] inbox tags checked and missing words
 * repaired, [13] barrier after that, [14] column sums done, [15] multi-GPU: the peers' rows of
 * this step summed.  trace_host holds
 * grid*nsteps*B200L_NTRACE uint64 (grid = b200l_run_config's grid, also returned in grid_out).
 * No counterpart in the reference (its only timer is lasso.py:234-236). */
int b200l_run_traced(b200l_ctx *ctx, int64_t nsteps, double mu, uint64_t *trace_host,
                     uint64_t *tile_trace_host, int32_t *grid_out, double *kernel_ms);
/* tile_trace_host (optional, grid*nsteps*B200L_NTTRACE uint64, absolute ns): per CTA and
 * step six groups of 16 stamps for the first 16 tiles of the slab: [0..15] pass-1 tile
 * arrived, [16..31] pass-1 tile consumed, [32..47] pass-2 tile arrived, [48..63] pass-2
 * tile consumed (consumer warp 0), [64..79] / [80..95] the producer issued the pass-1 /
 * pass-2 bulk copy of the tile. */
/* upper bound, in seconds, on any single cross-CTA wait inside the fused kernel (default
 * 5 s); when exceeded the kernel exits and b200l_run fails instead of hanging the device */
int b200l_set_wait_limit(b200l_ctx *ctx, double seconds);
/* diagnostics only: bit 0 skips the exchange waits, bit 1 the pass-1 arithmetic, bit 2 the
 * pass-2 arithmetic of the fused kernel, to time the remaining parts.  Results are invalid.
 * Bit 18 (262144) is the one flag with valid results: the step-wise mat-vecs then always use the
 * load-batch kernels instead of the TMA-streamed one (tests cover both).  flags with any other
 * bit set fail and leave the previous flags in place. */
int b200l_debug_flags(b200l_ctx *ctx, int32_t flags);

/* -- synthetic instances on the device (reference recipe: parameters.py:20-28) ---------
 * gen_gaussian fills the bound A with iid N(0,1) entries that are a pure function of
 * (seed, row, GLOBAL column): Philox4x32-10, counter (column/4, row, 0, "LASO"), key = seed,
 * Box-Muller on 24-bit uniforms.  rank/world say which column slice of every block this
 * context holds (local column j of block m = global column m*w*world + rank*w + j), so any
 * sharding yields the same matrix.  row_sumsq returns sum_k A_ik^2 over the LOCAL columns
 * (N doubles; sum over the ranks, then scale_rows with 1/sqrt makes unit-l2 rows, parameters.py:22-23).
 * No counterpart in the reference beyond the NumPy recipe. */
int b200l_gen_gaussian(b200l_ctx *ctx, uint64_t seed, int32_t rank, int32_t world);
int b200l_row_sumsq(b200l_ctx *ctx, double *out_host);
int b200l_scale_rows(b200l_ctx *ctx, const double *scale_host);

/* -- multi-GPU: one process per GPU ------------------------------------------------
 * Rank `rank` of `world` creates its context with the LOCAL column count (K/world): column
 * slice `rank` of every block, exactly the reference's P-way split of a block
 * (cpu_calculation.py:23-27 with P = world).  Each rank owns its x columns; the residual r
 * is replicated.  Inside the fused kernel the partial products A_{m,rank} D_rank are
 * summed over the ranks through peer memory (the reduce of lasso.py:126), in rank order, so
 * all ranks hold bitwise the same q, gamma and r.  mu and b must be identical on all ranks
 * and all ranks must call b200l_run with the same arguments.
 * comm_export : allocate this rank's inbox and return its CUDA IPC handle (64 bytes);
 * comm_connect: given the handles of all ranks (rank-major, handle_stride bytes apart,
 *               e.g. from an all-gather), map the peers' inboxes.
 * world = 1 (default) needs neither. */
#define B200L_MAX_WORLD 8
#define B200L_IPC_HANDLE_BYTES 64
int b200l_comm_export(b200l_ctx *ctx, int32_t rank, int32_t world, void *handle_out, int32_t handle_bytes);
int b200l_comm_connect(b200l_ctx *ctx, const void *all_handles, int32_t handle_stride);
int b200l_comm_destroy(b200l_ctx *ctx);
/* Teardown is collective and has two halves: every rank calls comm_close_peers (unmaps the
 * peers' inboxes), then a barrier over the ranks, then comm_destroy (frees its own inbox): an
 * exported allocation must not be freed while an importer still has it open. */
int b200l_comm_close_peers(b200l_ctx *ctx);
/* Inboxes provided by the caller instead of CUDA IPC (e.g. symmetric memory of the host
 * framework): comm_inbox_bytes gives the size one rank's inbox needs for this shape and world
 * size; comm_attach takes the addresses, in this process, of all ranks' inboxes (zero-filled,
 * peer_ptrs[rank] local) and, when not NULL, a multicast (NVLS) mapping of the same buffers --
 * the kernel then sends every row with ONE multimem store instead of world-1 peer stores.  The
 * caller keeps ownership of the memory; comm_destroy only forgets it. */
int b200l_comm_inbox_bytes(b200l_ctx *ctx, int32_t world, int64_t *bytes);
int b200l_comm_attach(b200l_ctx *ctx, int32_t rank, int32_t world, void *const *peer_ptrs, void *mc_ptr);

/* 0.5*|r|^2 + mu*|x|_1 from the device state (lasso.py:46-47 with the running residual) */
int b200l_objective(b200l_ctx *ctx, double mu, double *value);
/* the two terms separately: rss = |r|^2 and l1 = |x|_1 of THIS context.  With column shards on
 * several GPUs r is replicated but x is the local slice: the objective of the whole instance is
 * 0.5 * rss + mu * (sum of l1 over the ranks). */
int b200l_objective_terms(b200l_ctx *ctx, double *rss, double *l1);

#ifdef __cplusplus
}
#endif
#endif /* B200LASSO_H */
