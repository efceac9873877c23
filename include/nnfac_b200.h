/*
 * nnfac_b200 -- C ABI of the B200-native (sm_100a) factor-update path of nn-fac.
 *
 * The reference (ax-le/nn-fac v0.3.4) is pure Python/numpy and has no FFI: its
 * "plugin interface" for this path is a set of module functions.  Each entry
 * point below names the reference expression it replaces (paths relative to the
 * reference root).  A maintainer binds them with ctypes; see INTEGRATION.md.
 *
 * Conventions
 *   - every matrix pointer is a DEVICE pointer, row-major, with an explicit
 *     leading dimension (elements, not bytes);
 *   - dtype: NNFAC_F32 or NNFAC_F64 (all operands of one call share it);
 *   - stream: a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - return value: 0 on success, negative nnfac_status otherwise; the message
 *     is available from nnfac_last_error() (thread-local).  Nothing throws.
 *   - calls are asynchronous on `stream` unless stated otherwise.
 */
#ifndef NNFAC_B200_H
#define NNFAC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNFAC_ABI_VERSION 1

typedef enum { NNFAC_F32 = 0, NNFAC_F64 = 1 } nnfac_dtype;

typedef enum {
  NNFAC_OK = 0,
  NNFAC_ERR_ARG = -1,      /* invalid argument                                   */
  NNFAC_ERR_CUDA = -2,     /* CUDA runtime / driver error                        */
  NNFAC_ERR_UNSUPPORTED = -3, /* shape or option outside what this build covers  */
  NNFAC_ERR_ALLOC = -4
} nnfac_status;

/* flags of nnfac_hals_nnls */
#define NNFAC_HALS_NORMALIZE 1u /* nnls.py:179-185 */
#define NNFAC_HALS_NONZERO 2u   /* nnls.py:173-177 */
#define NNFAC_HALS_NO_TC 4u     /* fp32: skip the tensor-core sweep (its step operand is a bf16 hi/lo split); the CUDA-core sweeps
                                 * ignore this bit */

typedef struct nnfac_ctx nnfac_ctx; /* per-device workspace + launch limits; not thread-safe.  Scratch shared by several
                                     * kernels is guarded: a call on another stream than the last user of the same
                                     * scratch first waits for that user, so streams are ordered, never racing. */

int nnfac_abi_version(void);
const char* nnfac_last_error(void);
int nnfac_ctx_create(int device, nnfac_ctx** out);
int nnfac_ctx_destroy(nnfac_ctx* ctx);
int nnfac_ctx_sm_count(const nnfac_ctx* ctx);
/* Number of kernels this library has launched on behalf of `ctx` since creation. */
int64_t nnfac_ctx_launch_count(const nnfac_ctx* ctx);

/* ---------------------------------------------------------------------------------------------
 * Collective HALS solves (several GPUs of one node, one process per GPU; new -- the reference is single-process).
 * When the columns of one solve (nn_fac/update_rules/nnls.py:156-198) are spread over several GPUs, the stop test of
 * nnls.py:156 still sums the squared steps of ALL columns (nnls.py:170,195).  Each rank owns a small "board" in its
 * device memory; the sweep kernels of all ranks post their partial sums on every board over NVLink (peer-mapped memory)
 * once per sweep and take the same decision, so the sharded solve stops after exactly the sweeps of the unsharded one.
 *   1. every rank: nnfac_ctx_board_export(ctx, handle)          -> 64-byte CUDA IPC handle of its board
 *   2. exchange the handles between the ranks (any transport; the host layer uses torch.distributed.all_gather)
 *   3. every rank: nnfac_ctx_board_attach(ctx, world, rank, handles ( world x 64 bytes, in rank order ))
 *   4. nnfac_ctx_collective(ctx, 1, slice_lengths ( columns of every rank's slice )) before a solve that is one slice
 *      of a joint solve -- every rank must make the same sequence of such solves -- and (ctx, 0, NULL) after it.
 * 1 <= world <= 8 (a group of one runs the same protocol on its own board; its results equal the plain solve's).
 * Applies to the tensor-core sweep (fp32, rank <= 128: nnfac_nmf_plan_hals_solve, nnfac_hals_nnls).
 * -------------------------------------------------------------------------------------------*/
int nnfac_ctx_board_export(nnfac_ctx* ctx, void* handle_out);
int nnfac_ctx_board_attach(nnfac_ctx* ctx, int world, int rank, const void* handles);
int nnfac_ctx_collective(nnfac_ctx* ctx, int on, const int64_t* slice_lengths);
/* Variant of the tensor-core sweep's stop test (nnls.py:156): 0 = the total of a sweep is collected after three blocks of
 * the next sweep, 2 = after the WHOLE next sweep (one sweep of lag; one wasted sweep per solve, no exposed exchange) wherever
 * the shape allows, 1 = chosen per shape (default), -1 = back to the environment (NNFAC_SWEEP_LAG) / default.  Both variants
 * execute the same sweeps with the same sums; on one GPU their results are bit-identical. */
int nnfac_ctx_sweep_variant(nnfac_ctx* ctx, int mode);

/* ---------------------------------------------------------------------------------------------
 * Exchange steps of the column-sharded path over peer-mapped memory (new; csrc/peer_xchg.cu).  Every rank owns a region
 * [flags | stage | send] in device memory, exported with CUDA IPC and mapped by its peers like the boards above
 * (create -> export -> exchange handles -> attach).  The stage buffer (phase 0) is laid out
 * [tail block: r x tail_pitch | inbox: (world * splits) slabs of r_pad x chunk]: with nnfac_nmf_plan_set_push (below) the fused
 * pass of rank p writes the partial of every row tile straight into slab (p * splits + split) of the inbox of the rank that owns
 * those rows of U, over NVLink, from its own epilogue -- the reduce-scatter is part of the X pass -- and the tail block carries
 * the rank's own small partial sums (Gram of V, row sums of V).  After its post on phase 0 a rank finds every partial of its
 * rows in local memory.  The slice results go into the send buffer (phase 1, [r x pitch]: the slice, its Gram behind it); after
 * a second post nnfac_nmf_plan_set_factor_pulled reads all slices from the peers' send buffers while it builds the operand
 * planes (all-gather + install in one kernel).  The consumers wait for every rank's post themselves; every rank must make the
 * same sequence of calls.
 * -------------------------------------------------------------------------------------------*/
typedef struct nnfac_xchg nnfac_xchg;
int nnfac_xchg_create(nnfac_ctx* ctx, int64_t stage_floats, int64_t send_floats, nnfac_xchg** out);
int nnfac_xchg_export(nnfac_xchg* x, void* handle_out);
int nnfac_xchg_attach(nnfac_xchg* x, int world, int rank, const void* handles);
int nnfac_xchg_destroy(nnfac_xchg* x);
void* nnfac_xchg_ptr(nnfac_xchg* x, int which);                 /* local stage (0) / send (1) buffer */
int nnfac_xchg_post(nnfac_xchg* x, int phase, void* stream);    /* this rank's buffer `phase` is complete (stream-ordered) */
/* nnfac_xchg_post(x, 0) that first writes column `col` of the stage ([rows x pitch]) from tail_src[0 .. rows): the small partial
 * sums that travel with the post (row sums of V, mu.py:85-87, in column 0 of the tail block) without a copy kernel of their own. */
int nnfac_xchg_post_tail(nnfac_xchg* x, const float* tail_src, int rows, int64_t pitch, int64_t col, void* stream);
/* out[k][j] = sum over the ranks, in rank order, of element k * pitch + col + j of every rank's buffer `which` ([r x pitch];
 * k < r, j < tail): the partial Grams in the tail blocks (which = 0, pitch = tail_pitch, col = 0), the slices' Grams behind the
 * slices in the send buffers (which = 1, col = chunk).  Call after this rank's post on `which`; the kernel waits until every
 * rank has posted as often. */
int nnfac_xchg_pull_tail(nnfac_xchg* x, int which, float* out, int64_t ld_out, int r, int64_t pitch, int64_t col, int tail, void* stream);
/* The beta = 1 update (nn_fac/update_rules/mu.py:84-88) of this rank's rows of U from the inbox: waits for every rank's post on
 * phase 0, sums the slabs in slab order and the partial row sums of V (column 0 of every rank's tail block, nnfac_xchg_post_tail
 * with pitch = tail_pitch, col = 0), writes max(F[k][lo+c] * num / den[k], floor) for the rows [lo, lo + ncols) of U^T into this
 * rank's send buffer ([r x ld_send]).  F = the current U^T (r x ld_f). */
int nnfac_xchg_inbox_mu_apply(nnfac_xchg* x, int64_t inbox_off, int nslabs, int64_t slab_stride, int64_t chunk, int64_t tail_pitch,
                              const float* F, int64_t ld_f, int r, int64_t lo, int64_t ncols, double floor_value, int64_t ld_send,
                              void* stream);

/* ---------------------------------------------------------------------------------------------
 * HALS NNLS solver: replaces nn_fac/update_rules/nnls.py:156-198 (hals_nnls_acc sweep loop with
 * the deterministic stop rule, i.e. alpha = inf).  V (r x n) is updated IN PLACE; the caller
 * makes the copy that nnls.py:147 makes.  Rows k >= r of UtU/V are never touched
 * (tests/nnls_tests.py:40-47).
 *   sparsity : value subtracted in the numerator (0 = no sparsity term, nnls.py:162-167)
 *   result   : device double[4] = { eps, cnt, zero_diag_row (-1 if none, only with NONZERO), sweeps }
 * Any rank, any n, every option: fp32 without options up to rank 128 runs on the tensor-core sweep, rank <= 128 otherwise on
 * the register-resident CUDA-core sweep, everything else (rank > 128; normalize / nonzero on more columns than that kernel
 * keeps resident) on a general sweep that keeps nothing on chip (slow; may synchronise the stream every few sweeps to look at
 * its device-side stop flag unless the stream is being captured).
 * -------------------------------------------------------------------------------------------*/
int nnfac_hals_nnls(nnfac_ctx* ctx, int dtype, const void* UtM, int64_t ld_utm, const void* UtU,
                    int64_t ld_utu, void* V, int64_t ld_v, int r, int64_t n, int maxiter,
                    double delta, double sparsity, unsigned flags, double* result, void* stream);
/* Out-of-place fp32 variant: Vout = hals_nnls_acc(UtM, UtU, Vin), Vin is not modified (nnls.py:147 makes that copy).
 * Same rule and result vector; no normalize / nonzero. */
int nnfac_hals_solve_f32(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, const float* UtU, int64_t ld_utu,
                         const float* Vin, int64_t ld_vin, float* Vout, int64_t ld_vout, int r, int64_t n, int maxiter,
                         double delta, double sparsity, double* result, void* stream);
/* The same with the right-hand side given as the sum of nslabs slabs UtM + s * slab_stride ([r_pad x ld_utm] each,
 * slab_stride = r_pad * ld_utm): split-K partials of an X pass, or the inbox the peers' fused passes pushed their partials into
 * (nnfac_nmf_plan_set_push).  The tensor-core sweep adds the slabs itself, in slab order; shapes outside it first sum them
 * into scratch (r x n floats). */
int nnfac_hals_solve_slabs_f32(nnfac_ctx* ctx, const float* UtM, int64_t ld_utm, int nslabs, int64_t slab_stride, int r_pad,
                               float* scratch, const float* UtU, int64_t ld_utu, const float* Vin, int64_t ld_vin, float* Vout,
                               int64_t ld_vout, int r, int64_t n, int maxiter, double delta, double sparsity, double* result,
                               void* stream);

/* ---------------------------------------------------------------------------------------------
 * Strided, batched, K-blocked GEMM on CUDA cores (fp32 or fp64 accumulate in the operand type):
 *   C[b][i][j] = sum_{q<kb} sum_{k<K} A[b*sa_b + q*sa_q + i*sa_i + k*sa_k] * B[b*sb_b + q*sb_q + k*sb_k + j*sb_j]
 * written to C[b*sc_b + i*ldc + j].  Covers the dense call sites the reference hands to numpy:
 * Grams and cross products (nmf.py:407-408,432-433; ntf.py:442-445,449), K = U V (mu.py:82),
 * mode products (mu.py:141,159; ntd.py:672).  Deterministic (fixed summation order).
 * -------------------------------------------------------------------------------------------*/
int nnfac_gemm_strided(nnfac_ctx* ctx, int dtype, void* C, int64_t ldc, int64_t sc_b, const void* A,
                       int64_t sa_i, int64_t sa_k, int64_t sa_q, int64_t sa_b, const void* B,
                       int64_t sb_k, int64_t sb_j, int64_t sb_q, int64_t sb_b, int64_t M, int64_t N,
                       int64_t K, int64_t kb, int64_t batch, void* stream);

/* Gram of a rank-major factor: out (r x r) = F F^T with F (r x len) row-major -- V V^T (nmf.py:407) and U^T U
 * (nmf.py:432) when the factors are kept as V (r x n) and U^T (r x m).  Deterministic. */
int nnfac_gram(nnfac_ctx* ctx, int dtype, void* out, int64_t ld_out, const void* F, int64_t ld_f, int r,
               int64_t len, void* stream);

/* Multiplicative-update element-wise terms, mu.py:84-97 / mu.py:143-155:
 *   P = K^(beta-2) * X   and   Q = K^(beta-1)   (either output may be NULL; in-place on K allowed) */
int nnfac_mu_terms(nnfac_ctx* ctx, int dtype, double beta, const void* K, const void* X, void* P,
                   void* Q, int64_t count, void* stream);

/* F_out[i][k] = max(F_in[i][k] * (num[i][k] / den)^gamma, floor), mu.py:88,91,94,97,159.
 * den = den_mat[i][k] when den_vec is NULL; else the beta=1 row-sum form (mu.py:85-87):
 * den_vec[k] (vec_per_row = 0, F is m x r) or den_vec[i] (vec_per_row = 1, F is r x n). */
int nnfac_mu_apply(nnfac_ctx* ctx, int dtype, void* F_out, const void* F_in, const void* num,
                   const void* den_mat, const void* den_vec, int vec_per_row, int64_t rows,
                   int64_t cols, double gamma, double floor_value, void* stream);

/* out[0] = beta_divergence(A, B, beta) summed over `count` elements, beta_divergence.py:42-52.
 * fp64 accumulation, deterministic two-stage reduction. */
int nnfac_beta_divergence(nnfac_ctx* ctx, int dtype, double beta, const void* A, const void* B,
                          int64_t count, double* out, void* stream);

/* out[0] = sum (A - B)^2  (the Frobenius term of nmf.py:452); B may be NULL (-> sum A^2). */
int nnfac_sq_diff(nnfac_ctx* ctx, int dtype, const void* A, const void* B, int64_t count,
                  double* out, void* stream);

/* out[0] = sum A*B  (ntf.py:470 inner product) */
int nnfac_dot(nnfac_ctx* ctx, int dtype, const void* A, const void* B, int64_t count, double* out,
              void* stream);

/* out[i] = sum_j A[i][j]  (mu.py:86) */
int nnfac_row_sums(nnfac_ctx* ctx, int dtype, const void* A, int64_t lda, int64_t rows,
                   int64_t cols, void* out, void* stream);

/* out[0] = max_j sum_i |A[i][j]|  (numpy's matrix 1-norm used by nmf.py:452, ntf.py:466) */
int nnfac_norm1(nnfac_ctx* ctx, int dtype, const void* A, int64_t lda, int64_t rows, int64_t cols,
                double* out, void* stream);

/* out (cols x rows) = in (rows x cols)^T */
int nnfac_transpose(nnfac_ctx* ctx, int dtype, void* out, int64_t ld_out, const void* in,
                    int64_t ld_in, int64_t rows, int64_t cols, void* stream);

/* Khatri-Rao product of two factors (ntf.py:448): out[(i*J + j)][q] = A[i][q] * B[j][q]. */
int nnfac_khatri_rao(nnfac_ctx* ctx, int dtype, void* out, const void* A, int64_t I, const void* B,
                     int64_t J, int64_t r, void* stream);

/* out[i][j] = A[i][j] * B[i][j] (Hadamard of Grams, ntf.py:445); in place allowed. */
int nnfac_hadamard(nnfac_ctx* ctx, int dtype, void* out, const void* A, const void* B,
                   int64_t count, void* stream);
/* out = a X + b Y, element-wise (contiguous, `count` elements): the coupled right-hand side UtM + mu Vtarget of
 * nn_fac/update_rules/nnls.py:318 (hals_coupling_nnls_acc). */
int nnfac_axpby(nnfac_ctx* ctx, int dtype, void* out, double a, const void* X, double b, const void* Y, int64_t count,
                void* stream);

/* Row-wise L2 normalisation of the Tucker core unfolding (ntd.py:676-681), in place. */
/* One projected-gradient step on the Tucker core, ntd.py:607-617:  delta = min(step * (-MtX + P + sparse), core);
 * core -= delta; upd = ||delta||_2, with the loop state {upd_0, upd, cnt, done} kept on the device (double[4], start
 * {0, 1, 1, 0}): the step is a no-op once `done` is set (cnt > 300 or upd < delta * upd_0).  P = core x_n (F_n^T F_n). */
int nnfac_core_pg_step(nnfac_ctx* ctx, int dtype, void* core, const void* MtX, const void* P, int64_t count, double step,
                       double sparse, double delta, double* state, void* stream);
/* Same step with the step size and the sparsity coefficient read from the device: state = double[6] =
 * {upd_0, upd, cnt, done, step, sparse}.  No per-call host scalars besides delta, so a batch of steps captured into a CUDA
 * graph can be replayed for every outer iteration (the step size changes with the factors, ntd.py:590-594). */
int nnfac_core_pg_step_dev(nnfac_ctx* ctx, int dtype, void* core, const void* MtX, const void* P, int64_t count, double delta,
                           double* state, void* stream);
/* The same step for a 3-way core (r0 x r1 x r2, row-major, every rank <= 64) INCLUDING the product
 * P = core x_0 M0 x_1 M1 x_2 M2 of ntd.py:610 (M_n: r_n x r_n, row-major, the Grams F_n^T F_n): two kernels per step instead
 * of three generic GEMMs + the step.  Z: workspace of r0*r1*r2 elements.  dev_scalars != 0: step / sparse from state[4],
 * state[5] (state = double[6]) as in nnfac_core_pg_step_dev, else from the arguments (state = double[4]). */
int nnfac_core_pg_step3(nnfac_ctx* ctx, int dtype, void* core, const void* MtX, const void* M0, const void* M1, const void* M2,
                        int r0, int r1, int r2, void* Z, double step, double sparse, int dev_scalars, double delta, double* state,
                        void* stream);
int nnfac_normalize_rows(nnfac_ctx* ctx, int dtype, void* A, int64_t lda, int64_t rows,
                         int64_t cols, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NMF plan: the fp32 headline path (tcgen05 / TMA).  The data matrix X (m x n) is kept resident as
 * bf16 hi/lo planes (4 bytes per element, ~17 mantissa bits) in both orientations so that each of
 * the two X passes of an outer iteration (nmf.py:408 and nmf.py:433) streams K-major tiles.
 * Rank <= 128.  A plan is bound to one context and one stream at a time.
 * -------------------------------------------------------------------------------------------*/
typedef struct nnfac_nmf_plan nnfac_nmf_plan;
int nnfac_nmf_plan_create(nnfac_ctx* ctx, int64_t m, int64_t n, int r, nnfac_nmf_plan** out);
/* Same plan inside a caller-owned device workspace (256-byte aligned, >= nnfac_nmf_plan_bytes() bytes, e.g. a block of a
 * caching allocator): repeated factorisations of same-shaped data then never call cudaMalloc / cudaFree.  The workspace is
 * cleared on `stream` and must outlive the plan. */
int nnfac_nmf_plan_bytes(nnfac_ctx* ctx, int64_t m, int64_t n, int r, size_t* bytes);
int nnfac_nmf_plan_create_in(nnfac_ctx* ctx, int64_t m, int64_t n, int r, void* workspace, size_t workspace_bytes,
                             void* stream, nnfac_nmf_plan** out);
/* One-sided plans: sides = 1 keeps only the planes of X (passes over side 0), 2 only those of X^T (side 1), 3 both.  The
 * MTTKRP of a tensor unfolding (ntf.py:449) only ever reads side 0: half the memory.  A pass over an absent side is refused. */
int nnfac_nmf_plan_bytes_sided(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, size_t* bytes);
int nnfac_nmf_plan_create_sided(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, void* workspace, size_t workspace_bytes,
                                void* stream, nnfac_nmf_plan** out);
/* Plans with `planes` bf16 planes per value (every other create / bytes call means planes = 2):
 *   2: hi + lo, 16 significant bits, products of 3 MMAs;
 *   3: hi = RN(x), mid = RN(x - hi), lo = RN(x - hi - mid): hi + mid + lo == x for every finite fp32 x whose lo does not
 *      underflow (above 2^128 - 2^119, where RN(x) would overflow bf16, hi is rounded toward zero instead), products of the six terms down to order 2^-16 (fp32 accumulation).  Rank <= 64; 6 bytes per element and
 *      orientation.  Ingest (load_x*), set_factor, cross, fused (mode 1 after enable_f32, whose copies are then the caller's
 *      values), reduce and info cover it; mu_finish, hals_solve, set_factor_gathered / _pulled, set_krao*, set_push and views
 *      return NNFAC_ERR_UNSUPPORTED without writing anything (apply or solve on a copy, then set_factor). */
int nnfac_nmf_plan_bytes_planes(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, int planes, size_t* bytes);
int nnfac_nmf_plan_create_planes(nnfac_ctx* ctx, int64_t m, int64_t n, int r, int sides, int planes, void* workspace,
                                 size_t workspace_bytes, void* stream, nnfac_nmf_plan** out);
/* View plans: the unfolding of another mode of the C-order tensor whose mode-0 unfolding `base` holds (I_0 x rest, rest % 64 == 0),
 * addressed in place through TMA maps over the SAME planes -- the reference copies the tensor once per mode (ntf.py:309-311).
 * The tensor is read as (left, I, right); the view is the I x (left*right) unfolding of the middle axis: the last mode
 * (right == 1, I % 8 == 0) as an MN-major tensor-core operand, middle modes (right % 64 == 0) through a 3-D map.  A view supports
 * nnfac_nmf_plan_set_krao, nnfac_nmf_plan_cross(which = 0), _reduce and _info; NNFAC_ERR_UNSUPPORTED when the extents do not
 * allow it (the caller then builds a one-sided plan on a copy of that unfolding).  `base` must outlive the view. */
int nnfac_nmf_plan_view_bytes(nnfac_ctx* ctx, const nnfac_nmf_plan* base, int64_t left, int64_t I, int64_t right, int r, size_t* bytes);
int nnfac_nmf_plan_create_view(nnfac_ctx* ctx, const nnfac_nmf_plan* base, int64_t left, int64_t I, int64_t right, int r,
                               void* workspace, size_t workspace_bytes, void* stream, nnfac_nmf_plan** out);
int nnfac_nmf_plan_destroy(nnfac_nmf_plan* plan);
/* Ingest X (device fp32, row-major, leading dimension ldx >= n): one read of X, two plane writes. */
int nnfac_nmf_plan_load_x(nnfac_nmf_plan* plan, const float* X, int64_t ldx, void* stream);
/* The same ingest slab by slab (rows [row0, row0+rows) of X; Xrows points at row row0), so that a host can overlap the
 * upload of X with its ingest; call nnfac_nmf_plan_load_x_done once after the last slab. */
int nnfac_nmf_plan_load_x_rows(nnfac_nmf_plan* plan, const float* Xrows, int64_t ldx, int64_t row0, int64_t rows, void* stream);
int nnfac_nmf_plan_load_x_done(nnfac_nmf_plan* plan, void* stream);
/* Optional fp32 copies of X and X^T (= hi + lo of the planes; hi + mid + lo of a 3-plane plan, which needs them for mode 1) in a caller-owned, 256-byte aligned workspace: the beta = 1
 * fused pass then reads x from fp32 instead of reconstructing it from two bf16 planes (3 instructions per element fewer).
 * Call after the ingest; the workspace must outlive the plan. */
int nnfac_nmf_plan_f32_bytes(const nnfac_nmf_plan* plan, size_t* bytes);
int nnfac_nmf_plan_enable_f32(nnfac_nmf_plan* plan, void* workspace, size_t workspace_bytes, void* stream);
/* which = 0: out (r x m) = F X^T with F = V (r x n)      -- VMt, nmf.py:408
 * which = 1: out (r x n) = F X   with F = U^T (r x m)    -- UtM, nmf.py:433
 * F and out are device fp32, row-major.  Deterministic.  F == NULL: use the factor installed in the plan
 * (nnfac_nmf_plan_set_factor / nnfac_nmf_plan_mu_finish), whose operand planes already exist.  out == NULL: the split-K
 * partials stay in the plan for nnfac_nmf_plan_hals_solve(UtM = NULL) or nnfac_nmf_plan_reduce. */
int nnfac_nmf_plan_cross(nnfac_nmf_plan* plan, int which, const float* F, int64_t ldf, float* out,
                         int64_t ld_out, void* stream);
/* MTTKRP operand (ntf.py:448-449): the Khatri-Rao product of two rank-major factors At (r x I), Bt (r x J), I*J == n,
 * written straight into the operand planes that nnfac_nmf_plan_cross(which = 0, F = NULL) reads. */
int nnfac_nmf_plan_set_krao(nnfac_nmf_plan* plan, const float* At, int64_t lda, int64_t I, const float* Bt, int64_t ldb,
                            int64_t J, void* stream);
/* The same Khatri-Rao operand as the rank-contiguous planes of factor 1, for nnfac_nmf_plan_fused(plan, 0, 0, ...): with the
 * mode's own factor installed as factor 0 that pass yields the MTTKRP (ntf.py:449) and the direct residual
 * ||unfold(T, mode) - F krao^T||_F^2 of the CP model (instead of the cancelling ntf.py:470) in one pass over the tensor. */
int nnfac_nmf_plan_set_krao_rows(nnfac_nmf_plan* plan, const float* At, int64_t lda, int64_t I, const float* Bt, int64_t ldb,
                                 int64_t J, void* stream);
/* out (r x R of `side`) = sum of the split-K partials of the last X pass over `side` run with out == NULL. */
int nnfac_nmf_plan_reduce(nnfac_nmf_plan* plan, int side, float* out, int64_t ld_out, void* stream);
/* The same sum in the send layout of a reduce-scatter over `slabs` ranks (column-sharded U side, nn_fac/_fast.py):
 * out = [slabs][r][chunk + tail_cols]; column `row` of the result goes to out[row / chunk][k][row % chunk], and the small
 * matrix `tail` (r x tail_cols, the partial Gram; NULL with tail_cols = 0) is copied behind every chunk. */
int nnfac_nmf_plan_reduce_chunked(nnfac_nmf_plan* plan, int side, float* out, int64_t chunk, int slabs, const float* tail,
                                  int64_t ld_tail, int tail_cols, void* stream);
/* Install a factor into the plan (builds all of its bf16 operand planes):
 * which = 0: U, passed as U^T (r x m, row-major); which = 1: V (r x n). */
int nnfac_nmf_plan_set_factor(nnfac_nmf_plan* plan, int which, const float* Ft, int64_t ld, void* stream);
/* The same from the output of an all-gather of column slices, G = [slices][r][chunk] (slice s = columns
 * [s*chunk, (s+1)*chunk) of the factor); also writes the factor itself, rank-major, into Ft_out (r x len). */
int nnfac_nmf_plan_set_factor_gathered(nnfac_nmf_plan* plan, int which, const float* G, int64_t chunk, float* Ft_out,
                                       int64_t ld_out, void* stream);
/* The same straight from the peers' send buffers of an exchange region: slice s is read from rank s's send buffer
 * ([r x pitch]) over NVLink.  Call after this rank's nnfac_xchg_post(x, 1, stream): the kernel waits until every rank has
 * posted as often. */
int nnfac_nmf_plan_set_factor_pulled(nnfac_nmf_plan* plan, int which, const nnfac_xchg* x, int64_t chunk, int64_t pitch,
                                     float* Ft_out, int64_t ld_out, void* stream);
/* Column-sharded path, U side (new): from now on a fused pass over side 0 that keeps its partials (out = NULL) writes them into
 * the inbox of the rank that owns those rows of U -- x's stage buffer on that rank, inbox_off floats in, laid out
 * [world * splits][r_pad][chunk] (slab = source rank * splits + split; chunk = rows of U per rank, a multiple of 128) -- instead of
 * the plan's own buffer.  x = NULL switches it off.  slabs / slab_stride (optional) receive world * splits and r_pad * chunk. */
int nnfac_nmf_plan_set_push(nnfac_nmf_plan* plan, const nnfac_xchg* x, int64_t inbox_off, int64_t chunk, int* slabs,
                            int64_t* slab_stride);
/* out (r x n) = sum of nslabs slabs ([r_pad x ld] each, r_pad * ld floats apart) in slab order: the plain sum of the partials a
 * rank finds in its inbox (numerator of the beta = 2 update, mu.py:89-91). */
int nnfac_reduce_slabs_f32(nnfac_ctx* ctx, const float* slabs, int64_t ld, int nslabs, int r, int r_pad, int64_t n, float* out,
                           int64_t ld_out, void* stream);
/* HALS solve of factor `which` (nn_fac/update_rules/nnls.py:24-198, deterministic rule, no normalize / nonzero) whose
 * result F_out (r x len, may not alias F_in) is installed in the plan by the sweep kernel itself (no separate pass over
 * the factor).  result: double[4] = {eps, cnt, -1, sweeps}.  Returns NNFAC_ERR_UNSUPPORTED without an error text when
 * the shape is outside the tensor-core sweep (rank > 128, or more than 512 columns per SM at rank <= 64 / 256 at rank
 * <= 128): use nnfac_hals_nnls +
 * nnfac_nmf_plan_set_factor then.  UtM == NULL: the right-hand side is the sum of the split-K partials the last X pass
 * over side `which` left in the plan (the solve adds them in the reduction kernel's order). */
int nnfac_nmf_plan_hals_solve(nnfac_nmf_plan* plan, int which, const float* UtM, int64_t ld_utm, const float* UtU,
                              int64_t ld_utu, const float* F_in, int64_t ld_in, float* F_out, int64_t ld_out, int maxiter,
                              double delta, double sparsity, double* result, void* stream);
/* One fused X pass (mode 0: rank <= 128, mode 1: rank <= 64) over side 0 (rows of X) or side 1 (rows of X^T), using the installed
 * factors: the model tile U V is formed and consumed on chip, never written to HBM.
 *   mode 0: out (r x rows) = the HALS cross product of nmf.py:408 / :433, cost_out = ||X - U V||_F^2 (nmf.py:452)
 *   mode 1: out (r x rows) = the beta=1 MU numerator ((X / UV) V^T)^T of mu.py:84-88 (side 0) or its
 *           transposed twin for V (mu.py:27, side 1); cost_out = KL(X | U V) when want_cost != 0.
 * cost_out is a device double and may be NULL.  out may be NULL in mode 1 (see nnfac_nmf_plan_mu_finish). */
int nnfac_nmf_plan_fused(nnfac_nmf_plan* plan, int side, int mode, int want_cost, float* out, int64_t ld_out,
                         double* cost_out, void* stream);
/* beta = 1 multiplicative update of factor `which` (0: U as U^T, 1: V), mu.py:84-88, straight from the numerator
 * partials that the last mode-1 nnfac_nmf_plan_fused call over side `which` left in the plan when it was given
 * out = NULL:  F_out = max(F_in * num / den[k], floor_value), den = r row sums of the other factor (mu.py:85-87).
 * F_out is installed in the plan as nnfac_nmf_plan_set_factor would do.  One kernel. */
int nnfac_nmf_plan_mu_finish(nnfac_nmf_plan* plan, int which, const float* F_in, int64_t ld_in, const float* den,
                             double floor_value, float* F_out, int64_t ld_out, void* stream);
/* General-beta MU pass (beta >= 0 other than 1 and 2; mu.py:84-97) over side 0 or 1 with the installed factors, K = U V formed
 * and consumed on chip.  The split partials of the numerator (K^(beta-2) * X) V^T (side 0; its twin for V on side 1) stay in the
 * plan; those of the denominator K^(beta-1) V^T go to den_partial, a caller-owned device buffer of at least
 * nnfac_nmf_plan_fused_beta_bytes bytes.  cost_out (device double, may be NULL): the beta-divergence of X from U V when
 * want_cost != 0.  NNFAC_ERR_UNSUPPORTED for rank > 64, 3-plane plans, view plans, plans with the push exchange set, and
 * beta = 1 or 2 (nnfac_nmf_plan_fused). */
int nnfac_nmf_plan_fused_beta_bytes(const nnfac_nmf_plan* plan, size_t* bytes);
int nnfac_nmf_plan_fused_beta(nnfac_nmf_plan* plan, int side, double beta, int want_cost, float* den_partial, double* cost_out,
                              void* stream);
/* General-beta update of factor `which` from the two partial sets of the last nnfac_nmf_plan_fused_beta pass over side `which`
 * (both summed in the order of nnfac_nmf_plan_reduce): F_out = max(F_in * (num / den)^gamma, floor_value), gamma = the
 * exponent of beta_divergence.py:75-80; F_out is installed in the plan as nnfac_nmf_plan_set_factor would do.  One kernel. */
int nnfac_nmf_plan_mu_finish_beta(nnfac_nmf_plan* plan, int which, const float* F_in, int64_t ld_in, const float* den_partial,
                                  double gamma, double floor_value, float* F_out, int64_t ld_out, void* stream);
/* Work decomposition chosen for one side (for benchmarks / DESIGN.md); any pointer may be NULL. */
int nnfac_nmf_plan_info(const nnfac_nmf_plan* plan, int which, int* splits, int* stages_per_unit,
                        int* num_units, int* num_stages, int* grid);

/* ---------------------------------------------------------------------------------------------
 * Synthetic data for benchmarks and tests (not on the factorisation path): out[i][j] (+)= scale * u, u uniform in [0, 1),
 * a pure function of (seed, stream_id, row0 + i, col0 + j) -- Philox4x32-10, counter (row, column, stream, 0) -- so that
 * any shard of a matrix on any number of GPUs regenerates the same values (SURVEY.md 8(d)).  Device fp32, row-major.
 * -------------------------------------------------------------------------------------------*/
int nnfac_philox_uniform(nnfac_ctx* ctx, float* out, int64_t ld, int64_t rows, int64_t cols, int64_t row0, int64_t col0,
                         uint64_t seed, uint32_t stream_id, double scale, int accumulate, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NNFAC_B200_H */
