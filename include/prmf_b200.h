/* prmf_b200.h -- C ABI of the B200-native PRMF hot path (libprmf_b200.so).
 *
 * The reference (gitter-lab/prmf) is pure Python and has no FFI; the boundary this library replaces is
 * the numeric body of `script/prmf_runner.py`:
 *     nmf_pathway                     :556-792   (driver; stays on the host, calls the entry points below)
 *     nmf_manifold_vec_update         :374-451   -> prmf_step
 *     nmf_manifold_vec_update_tradeoff:497-554   -> prmf_step (tradeoff >= 0)
 *     nmf_manifold_vec_obj            :336-372   -> prmf_step (objective parts per inner step)
 *     normalize_laplacian             :56-65     -> prmf_set_pathways (derived once, on the device)
 *     score_latent_pathway_match_global :115-127 , restrict :129-194 (scores)   -> prmf_scores
 *     force_distinct_lapls            :209-258   (edge weights)                 -> prmf_scores
 *     find_mins                       :37-54                                    -> prmf_scores (quad_raw)
 *
 * Conventions: every call returns 0 on success and a negative code on failure (the text is available
 * from prmf_last_error); plain pointers and sizes only; the caller owns every host pointer for the
 * duration of the call; the library owns all device memory until prmf_destroy.  A handle is bound to
 * one GPU and one host thread.  Matrices are C-order (row-major) IEEE fp64.  There is no CPU fallback:
 * without a CUDA device prmf_create fails.
 */
#ifndef PRMF_B200_H
#define PRMF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct prmf_handle prmf_handle;

#define PRMF_OK              0
#define PRMF_ERR_ARG        -1
#define PRMF_ERR_CUDA       -2
#define PRMF_ERR_STATE      -3
#define PRMF_ERR_NCCL       -4
#define PRMF_ERR_NOMEM      -5
#define PRMF_ERR_TIMEOUT    -6   /* a bounded device-side wait expired (lost launch, dead peer rank); the handle refuses further steps */

#define PRMF_OBJ_STRIDE      8   /* doubles per inner step written by prmf_step (see below) */
#define PRMF_UNIQUE_ID_BYTES 128

/* ABI version of this header (bumped on any signature change). */
int prmf_abi_version(void);

/* Create a solver handle on GPU `device` for a row block of `m_local` samples (of `m_global` in the
 * whole job), `n` genes and `k` latent factors.  `stream` is a cudaStream_t to run on (e.g. torch's
 * current stream) or NULL for a private stream.  Replaces the array allocations of
 * nmf_pathway (prmf_runner.py:647-655). */
int prmf_create(prmf_handle** out, int device, int64_t m_local, int64_t m_global, int64_t n, int k,
                void* stream);
int prmf_destroy(prmf_handle* h);

/* Storage / arithmetic mode of the X streams.  PRMF_X_F64 (prmf_create) is the parity mode: X in fp64, DFMA.
 * PRMF_X_TF32 (opt-in; BASELINE config 5, "dense-enough contraction for the tensor-core path") keeps X and X^T
 * in HBM as fp32 rounded to tf32 and runs X.V (:420) and X^T.U (:424) on the tcgen05 tensor cores with fp32
 * accumulation in TMEM; U, V, the updates, the objective and the reductions over ranks stay fp64.  Not bit-parity
 * with the reference: the tests state its tolerance.
 * PRMF_X_F32 (opt-in) keeps X and X^T in HBM as exact fp32 values (half the bytes of PRMF_X_F64) and streams them
 * through the same fp64 DFMA kernels, widening each element exactly before its first use.  Given X32, an f32 handle
 * returns bit for bit what a PRMF_X_F64 handle returns given X32 widened to fp64.  Single rank only: m_local must
 * equal m_global, and prmf_comm_init / prmf_p2p_attach return PRMF_ERR_STATE. */
#define PRMF_X_F64  0
#define PRMF_X_TF32 1
#define PRMF_X_F32  2
int prmf_create_ex(prmf_handle** out, int device, int64_t m_local, int64_t m_global, int64_t n, int k,
                   void* stream, int x_dtype);
int prmf_x_dtype(const prmf_handle* h);

/* Last error text of `h` (or of the last failed prmf_create when h is NULL). */
const char* prmf_last_error(const prmf_handle* h);

/* Upload this rank's row block of X (host pointer, `ld` doubles between rows) and compute the local
 * sum of squares.  prmf_set_X_device takes a DEVICE pointer instead (copied into the library's padded
 * layout on the handle's stream).  X argument of nmf_pathway / nmf_manifold_vec_update (:556,:374). */
int prmf_set_X(prmf_handle* h, const double* X_host, int64_t ld);
int prmf_set_X_device(prmf_handle* h, const double* X_dev, int64_t ld);
/* PRMF_X_TF32 and PRMF_X_F32 handles only: fp32 source (host pointer, or device pointer when on_device != 0), `ld`
 * floats between rows, stored exactly (PRMF_X_F32) or rounded to tf32.  The fp64 entry points above also work in
 * those modes: the values are rounded on the device, to tf32 or to the nearest fp32 value. */
int prmf_set_X_f32(prmf_handle* h, const float* X, int64_t ld, int on_device);

/* Global ||X||_F^2 (all-reduced when a communicator is attached); `np.linalg.norm(X)` at :640. */
int prmf_get_normX_sq(prmf_handle* h, double* out);

/* All P pathways packed block-diagonally over LOCAL support indices (replaces the per-pathway n x n
 * scipy W, D, L matrices and support lists built at prmf_runner.py:673-696):
 *   path_ptr[P+1]     offsets into support_idx / rows              (path_ptr[P] = S)
 *   support_idx[S]    gene index (0..n-1) of every support node, pathway after pathway
 *   row_ptr[S+1]      offsets into col_local / w                   (row_ptr[S] = E)
 *   col_local[E]      neighbour as an index INTO THE SAME PATHWAY's support (0..s_p-1)
 *   w[E]              symmetric edge weights (each undirected edge appears in both rows; a self loop once)
 * The library derives degrees, diag(L) and diag(L)^-1/2 (normalize_laplacian, :56-65). */
int prmf_set_pathways(prmf_handle* h, int32_t P, const int64_t* path_ptr, const int32_t* support_idx,
                      const int64_t* row_ptr, const int32_t* col_local, const double* w);

/* Initial / current factors.  U is this rank's m_local x k block, V is n x k (replicated).  Either
 * pointer may be NULL to skip it.  U_init / V_init of nmf_pathway (:650-655) and its return value.
 * The library tracks U and V separately: calls that read one fail with PRMF_ERR_STATE until it has been set (again,
 * after prmf_nnls_x). */
int prmf_set_UV(prmf_handle* h, const double* U_local, const double* V);
int prmf_get_UV(prmf_handle* h, double* U_local, double* V);

/* Active pathway of every factor for the following inner steps: k_to_lapl_ind of :717-730 /
 * map_k_to_lapls :260-270. */
int prmf_set_active(prmf_handle* h, const int32_t* pathway_of_factor);

/* `n_steps` inner multiplicative updates (nmf_manifold_vec_update, :419-449) with the objective of
 * every step (nmf_manifold_vec_obj, :336-372).  tradeoff < 0 keeps gamma/delta fixed; tradeoff in [0,1]
 * feeds gamma = delta = (1-t)*recon/(t*manifold) back after every step on the device (:542-548).
 * obj_parts (host, n_steps x PRMF_OBJ_STRIDE): recon, manifold, ignore, fro, obj, gamma, delta, recon^2
 * (gamma/delta are the values the step was computed with).  gamma_delta_out (host, 2 doubles or NULL):
 * gamma, delta to use for the next step.  All steps are enqueued without host synchronisation; the
 * call returns after one synchronisation at the end.  With a communicator attached every step includes
 * the all-reduce of X^T U, U^T U and sum(U^2) over ranks. */
int prmf_step(prmf_handle* h, int n_steps, double gamma, double delta, double tradeoff,
              double* obj_parts, double* gamma_delta_out);

/* Enqueue-only variant for timing: no synchronisation, results stay on the device until
 * prmf_step_collect copies the last `n_steps` rows. */
int prmf_step_async(prmf_handle* h, int n_steps, double gamma, double delta, double tradeoff);
int prmf_step_collect(prmf_handle* h, int n_steps, double* obj_parts, double* gamma_delta_out);

/* Factor x pathway tables from the current V (each k x P, row-major, host pointers, any may be NULL):
 *   mass[k][p]      = sum_{i in supp_p} vhat_i^2          (score_mass^2, :123; vhat = v_k/||v_k||)
 *   quad_norm[k][p] = vhat^T Lhat_p vhat                  (1 - score_manifold, :124; objective :350)
 *   quad_raw[k][p]  = v_k^T L_p v_k                       (force_distinct_lapls :232; find_mins :49) */
int prmf_scores(prmf_handle* h, double* mass, double* quad_norm, double* quad_raw);

/* End of a block of inner steps in one call (nmf_pathway :739-768): the score tables of the current V (when
 * want_scores != 0; same three tables as prmf_scores, any may be NULL), the objective rows of the last `n_steps`
 * steps enqueued by prmf_step_async and gamma/delta, with ONE host wait.  With prefetch != 0 the library enqueues,
 * before the host waits, the part of the NEXT inner step that does not depend on the active pathways (the X.V
 * pass and the U update, :420-422): the GPU keeps streaming X while the host runs restrict / the multinomial
 * draws.  The next prmf_step / prmf_step_async continues from there; prmf_get_UV, prmf_snapshot_best and the
 * objective calls still see the U of the finished block; prmf_set_UV, prmf_restore_best and prmf_set_X discard
 * the speculative work.  Results are identical with and without prefetch. */
int prmf_block_end(prmf_handle* h, int n_steps, double* obj_parts, double* gamma_delta_out, int want_scores,
                   double* mass, double* quad_norm, double* quad_raw, int prefetch);

/* Best-iterate bookkeeping of nmf_pathway (:745-750, :778-782) without host traffic. */
int prmf_snapshot_best(prmf_handle* h);
int prmf_restore_best(prmf_handle* h);

/* Exact residual ||X - U V^T||_F^2 by one extra pass over X (verification of the pass-free identity
 * used inside prmf_step; all-reduced when a communicator is attached). */
int prmf_residual_sq(prmf_handle* h, double* out);

/* Objective of the CURRENT X, U, V and active set as a standalone call (nmf_manifold_vec_obj, :336-372), with the
 * residual taken by an explicit pass over X as the reference does.  out: PRMF_OBJ_STRIDE doubles, same layout as
 * a row of prmf_step's obj_parts. */
int prmf_objective(prmf_handle* h, double gamma, double delta, double* out);

/* ---- multi-GPU (one handle per rank / process) ------------------------------------------------------
 * prmf_nccl_load dlopens the NCCL the host process already uses (path of libnccl.so.2, or NULL to look
 * it up); rank 0 calls prmf_comm_unique_id and ships the 128 bytes to the other ranks (any transport,
 * e.g. torch.distributed.broadcast); every rank calls prmf_comm_init.  Afterwards prmf_set_X reduces
 * ||X||^2 and prmf_step all-reduces the packed [X^T U | U^T U | sum U^2] buffer every inner step. */
int prmf_nccl_load(const char* libnccl_path);
int prmf_comm_unique_id(uint8_t* id_out /* PRMF_UNIQUE_ID_BYTES */);
int prmf_comm_init(prmf_handle* h, int rank, int nranks, const uint8_t* id);

/* The per-step sum over ranks through NVLink / CUDA-IPC peer memory instead of NCCL.  Every rank exports a CUDA IPC
 * handle of its exchange buffer (PRMF_IPC_HANDLE_BYTES), the handles are gathered by the host (any transport) and every
 * rank attaches all of them; then all ranks call the collective prmf_p2p_finalize, which agrees on the variant:
 *   - k <= 10, every rank able to run the persistent step kernel with the same split of the genes (the default):
 *     the sum is part of the pass-2 tail of that kernel -- every thread block pushes the local sums of its share of
 *     genes into every rank's receive slots as self-validating {32 value bits | 32 sequence bits} word pairs (one
 *     16-byte store each, no fence, no flag), polls the same entries of all ranks in its own memory, adds them in rank
 *     order and updates its rows of V.  No collective launch; bitwise identical on all ranks.
 *   - otherwise: the packed buffers of all ranks are pulled with P2P loads inside the V-update kernel (flag barrier in
 *     peer memory), or inside the pass-2 kernel with PRMF_XCHG=1.
 * Needs one process per rank on one node with peer access (or several ranks sharing one device: IPC works there too).
 * prmf_comm_init is OPTIONAL for the first variant: without a communicator the set-up reductions (||X||^2, the
 * agreement itself) are summed over the same peer buffers; configurations that need the other variants then fail with
 * PRMF_ERR_STATE.  All device-side waits on peers are bounded (PRMF_ERR_TIMEOUT). */
#define PRMF_IPC_HANDLE_BYTES 64
int prmf_p2p_export(prmf_handle* h, uint8_t* handle_out);
int prmf_p2p_attach(prmf_handle* h, int rank, int nranks, const uint8_t* handles /* nranks x 64 bytes */);
int prmf_p2p_finalize(prmf_handle* h);

/* How the per-step sum over ranks is done: 0 one rank, 1 ncclAllReduce, 2 NVLink peer loads inside the V-update
 * kernel, 3 NVLink peer loads inside the pass-2 X-stream kernel, 4 NVLink peer stores (push) inside the persistent
 * step kernel (the default for k <= 10 when every rank can take it; agreed in prmf_p2p_finalize). */
int prmf_exchange_mode(const prmf_handle* h);

/* ---- introspection used by bench.py and the tests ---------------------------------------------------*/
/* Number of kernel launches issued by this handle so far. */
int64_t prmf_launch_count(const prmf_handle* h);
/* Device time (ms, CUDA events on the handle's stream) per phase of the inner step, accumulated since the
 * last call with reset != 0, and the number of timed occurrences of each.  Phases (PRMF_N_PHASES):
 * 0 pass 1 (X.V), 1 U update, 2 pass 2 (X^T.U), 3 partial sums + all-reduce, 4 V update, 5 objective. */
#define PRMF_N_PHASES 6
int prmf_kernel_times(prmf_handle* h, int reset, double* phase_ms, int64_t* phase_count);
/* Enable (1) / disable (0) per-kernel event timing inside prmf_step (off by default). */
int prmf_set_profiling(prmf_handle* h, int on);
/* A_local (m_local x k, row-major, host) = X_local . V for the current V: the pass-1 X stream of the inner step
 * (prmf_runner.py:420) on its own.  It is the dense product of the steps around the path as well: the ridge transfer
 * of a fitted V to new samples (reference script/transfer_learning.R:108, B^T = Y^T Z (Z^T Z + l I)^-1) needs exactly
 * Y^T Z.  Sharded handles return their own row block. */
int prmf_project(prmf_handle* h, double* A_local);
/* X^T . U for the current U (n x k, row-major): the pass-2 stream of the inner step on its own.  The current U is the
 * one last given to prmf_set_UV, or the result of the steps since.  With U = ones it gives the column sums of X.
 * Single-rank handles only; PRMF_ERR_STATE as well when U was never set or prmf_nnls_x has used it since. */
int prmf_project_t(prmf_handle* h, double* B_out);
/* For every column c of B: x_c = argmin_{x >= 0} || op(X) x - b_c ||_2 with op(X) = X^T (transpose != 0; b: n, x: m)
 * or X (transpose == 0; b: m, x: n) -- scipy.optimize.nnls(op(X), b_c) for all k columns at once, sharing each pass
 * over X (Lawson & Hanson's active-set method, the duals A^T (b - A x) from the X streams of the inner step).
 * B_host / x_out row-major (rows x k), rnorm_out[k] = || op(X) x_c - b_c ||, status_out[k]: 1 converged, -1 maxiter
 * reached (counted as scipy counts, default 3 * #unknowns when maxiter <= 0), -2 the passive set outgrew the device
 * capacity (min(#equations, #unknowns, 1024) columns), -3 the Gram matrix of the passive columns lost positive
 * definiteness.  iter_out[k] (may be NULL): the iterations of each problem as scipy counts them (one per outer
 * iteration, including the last one that finds the optimum, and one per step back).  A problem with status -2 or -3 leaves a message in prmf_last_error; the call still returns PRMF_OK.
 * Repeated calls return bitwise-identical results.  Needs X; fp64 or f32, single-rank handles only (PRMF_ERR_STATE otherwise).
 * U and V of the handle are unset afterwards: calls that read them fail with PRMF_ERR_STATE until prmf_set_UV gives
 * them again. */
int prmf_nnls_x(prmf_handle* h, int transpose, const double* B_host, int maxiter, double* x_out, double* rnorm_out,
                int32_t* status_out, int32_t* iter_out);
/* The library keeps the two large buffers of a destroyed handle (X and its transposed copy) for the next handle of the
 * same shape on the same device (allocating and freeing multi-GB buffers dominates a short solve otherwise); at most
 * 4 buffers / 24 GB are held.  PRMF_POOL=0 (environment) disables the cache; this call frees what is held. */
int prmf_release_pool(void);
/* Fault injection for the tests of the bounded device waits (SURVEY section 5: a lost launch or a dead peer must come
 * back as an error code, not as a hang).  kind 1: the next persistent step launch waits for a thread-block arrival
 * that never happens; kind 2: it waits for a peer-exchange flag that never comes.  The waits expire after
 * PRMF_SPIN_TIMEOUT_MS (environment, default 10 000 ms) and the step returns PRMF_ERR_TIMEOUT. */
int prmf_debug_inject_fault(prmf_handle* h, int kind);
/* The cudaStream_t the handle launches on. */
void* prmf_stream(const prmf_handle* h);

/* ---- "next" row of the scope table: the step before the path --------------------------------------------
 * GPU version of `X = quantile_transform(X)` (script/prmf_runner.py:1019-1020; sklearn defaults: uniform output,
 * n_quantiles = min(1000, m), axis 0).  X_dev / out_dev are DEVICE pointers (m x n, row-major, leading dimensions
 * ld / ld_out; out may alias X).  The caller supplies what numpy derives on the host so the device mirrors it
 * exactly: references (np.linspace(0,1,nq)), and for q = (references*100)/100 the order-statistic indices
 * lo = floor((ms-1) q), hi = min(lo+1, ms-1) and weights g = (ms-1) q - lo.  rows_dev (ms row indices, or NULL
 * with ms == m) is sklearn's row subsample used for fitting the quantiles.  quantiles_out_host (n x nq,
 * gene-major) may be NULL.  Fails on NaN input. */
int prmf_quantile_transform(int device, void* stream, const double* X_dev, int64_t m, int64_t n, int64_t ld,
                            const int64_t* rows_dev, int64_t ms, int nq, const double* refs_host,
                            const int64_t* lo_host, const int64_t* hi_host, const double* g_host, double* out_dev,
                            int64_t ld_out, double* quantiles_out_host);
const char* prmf_preprocess_last_error(void);

/* ---- "next" row of the scope table: the step after the path ----------------------------------------------
 * GPU version of `measure_cv_performance(V, X_test)` (prmf/__init__.py:768-798; script/prmf_runner.py:1074-1079):
 * for every held-out sample x_i (row of X_host, mt x n, `ld` doubles between rows) solve
 * u_i = argmin_{u >= 0} ||x_i - V u|| (V_host: n x k, k <= 128) for the whole batch at once -- the reference loops
 * over scipy.optimize.nnls per sample.  Outputs (host, any may be NULL): U_out mt x k; rnorm_out[i] = ||x_i - V u_i||;
 * xnorm_sq_out[i] = ||x_i||^2; status_out[i] = 1 converged, -1 iteration limit (3 k, as scipy), -2 singular block. */
int prmf_nnls_rows(int device, const double* V_host, int64_t n, int k, const double* X_host, int64_t mt, int64_t ld,
                   double* U_out, double* rnorm_out, double* xnorm_sq_out, int32_t* status_out);
const char* prmf_cv_last_error(void);

/* ---- host-side helper (plain C++, no CUDA, no handle) ------------------------------------------------------
 * One factor of `restrict` (script/prmf_runner.py:159-171) from the rows of the score tables: scores_out[i] =
 * sqrt(mass_row[ids[i]]) + (1 - quad_row[ids[i]]) (:123-125), threshold = np.percentile(scores, 100 q) with linear
 * interpolation (q = 0.199 at :159), keep_out = the positions i with scores_out[i] strictly above it.  Returns their
 * number (0: all scores equal, the case in which the reference raises), negative on bad arguments.  Bit-identical
 * to the numpy expressions it replaces; the decision logic itself stays on the host as in the reference. */
int64_t prmf_host_restrict(const double* mass_row, const double* quad_row, const int64_t* ids, int64_t n, double q,
                           double* scores_out, int64_t* keep_out);
/* All factors of one `restrict` call (:129-194) in one crossing: factor f (row factor[f] of the k x P tables) has the
 * candidates ids[off[f] .. off[f+1]); its survivors and their scores are written, compacted, to kept_ids /
 * kept_scores at [kept_off[f], kept_off[f+1]).  Returns 0; -(f+1) when factor f keeps nothing; -1000000 on bad
 * arguments. */
int64_t prmf_host_restrict_batch(const double* mass, const double* quad, int64_t P, int32_t nf, const int32_t* factor,
                                 const int64_t* ids, const int64_t* off, double q, int64_t* kept_ids,
                                 double* kept_scores, int64_t* kept_off);

#ifdef __cplusplus
}
#endif
#endif /* PRMF_B200_H */
