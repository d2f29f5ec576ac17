/*
 * matcouply_b200 — C ABI of the B200-native AO-ADMM engine (libmatcouply_b200.so).
 *
 * The reference (MarieRoald/matcouply, pure Python) has no FFI: its boundary is the Python call surface
 * `matcouply.decomposition.cmf_aoadmm` (decomposition.py:662) and the `ADMMPenalty` protocol (penalties.py:21).
 * This header is the seam underneath our Python mirror of that surface (`matcouply_b200/decomposition.py`,
 * `matcouply_b200/penalties.py`): every numerical step of the reference hot path maps onto one entry point below;
 * each entry cites the reference lines it replaces.  INTEGRATION.md shows the ctypes binding a maintainer would add
 * on the reference side.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in `_host`; the caller owns every buffer;
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), no hidden allocation, no host sync;
 *   - return value: 0 = B2_OK, otherwise an error code; `b2_last_error()` returns a thread-local message;
 *   - dtype: B2_F32 / B2_F64 for every floating-point buffer of a call (scalars in `double`);
 *   - matrices are dense row-major; "packed" means the vertical concatenation of the per-slice matrices
 *     (np.concatenate(list, axis=0)) addressed through `row_off[G+1]` (int64 prefix sum of the J_i);
 *   - reference symbols: I slices X_i (J_i x K), A (I x R), B_i (J_i x R), C (K x R); N = sum_i J_i.
 */
#ifndef MATCOUPLY_B200_H
#define MATCOUPLY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { B2_OK = 0, B2_ERR_INVALID = 1, B2_ERR_CUDA = 2 };
enum { B2_F32 = 0, B2_F64 = 1 };
enum { B2_VARIANT_AUTO = 0, B2_VARIANT_FMA = 1, B2_VARIANT_DMMA = 2 };

/* penalty kinds (penalties.py: Parafac2 :1018, Unimodality :983, L2Ball :844, L1Penalty :545, Box :511,
 * NonNegativity :488) */
enum { B2_PEN_NONNEG = 0, B2_PEN_BOX = 1, B2_PEN_L1 = 2, B2_PEN_L2BALL = 3, B2_PEN_UNIMODAL = 4, B2_PEN_PARAFAC2 = 5,
       /* column-coupled kinds finished by their own b2_prox_* call (penalties.py:595, :928, :750) */
       B2_PEN_GL2 = 6, B2_PEN_SIMPLEX = 7, B2_PEN_TV = 8,
       /* prox evaluated by the caller (user-defined ADMMPenalty subclass): the kernels only leave V = x + dual in `dual` */
       B2_PEN_HOST = 9,
       /* TemporalSmoothnessPenalty (mode 1 only): couples B_i to B_{i-1}; finished by b2_prox_temporal */
       B2_PEN_TEMPORAL = 10 };

/* how a row of an ADMM state matrix finds its group (slice) */
enum { B2_GROUP_SINGLE = 0 /* every row -> group 0 (C-mode) */,
       B2_GROUP_INDEXED = 1 /* group_of_row[row]     (B-mode) */,
       B2_GROUP_IDENTITY = 2 /* group = row           (A-mode) */ };

typedef struct {
    int32_t kind;           /* B2_PEN_* */
    int32_t non_negativity; /* L1 / L2Ball / Unimodality flag */
    double p0;              /* L1: reg_strength; Box: min_val; L2Ball: norm_bound */
    double p1;              /* Box: max_val */
    void* aux;              /* n x R auxiliary variable; PARAFAC2: the product P_i*Delta ("aux as matrix") */
    void* dual;             /* n x R scaled dual variable */
} b2_penalty_desc;

/* kernel-selection switches (process-wide; default 1 = on, except B2_OPT_XSTREAM_HYBRID which is off).  They only choose between equivalent kernels — tests flip
 * them to cross-check the tensor-core formulations against the scalar ones. */
enum { B2_OPT_PF2_ROWPASS_MMA = 0 /* row pass of b2_pf2_rowpass: 0 = shuffle kernel, 1 = DMMA tile kernel, 2 (default) = DMMA tile
                                     kernel + its steady-state specialisation (fp64, R % 4 == 0, deferred prox, PARAFAC2
                                     alone or with non-negativity) */,
       B2_OPT_POLAR_WARP = 1 /* polar step of b2_pf2_polar: 2 (default) = warp per slice, Jacobi in registers; 1 = warp per slice in shared memory; 0 = CTA per slice */,
       B2_OPT_ADMM_LOCAL_MMA = 2 /* DMMA formulation of b2_admm_local (CTA-per-slice path) */,
       B2_OPT_XSTREAM_HYBRID = 3 /* fp64 X-stream kernel variants: 0 (default) = padded DMMA column blocks, Y kernel with 12
                                    consumer warps from R = 17 on (fp64-pipe-bound ranks) and 8 below; 1 = DMMA blocks +
                                    DFMA remainder columns (R = 8b+1..4; measured 2-6 % slower than padding); 2 = Y kernel
                                    always with 12 consumer warps; 3 = always 8 */,
       B2_OPT_UNIMODAL_VARIANT = 4 /* b2_prox_unimodal: (column ring depth, shared-memory stack-cache depth, CTAs per
                                      SM) of the PAVA kernel: 0 = (8, 4, 4) round 1, 1 = (4, 8, 4), 2 = (8, 8, 4), 3 = (4, 16, 3),
                                      4 = (4, 8, 5), 5 = (4, 12, 4); 6 = variant 1 with the exact reciprocal-based division
                                      and 256-bit record loads / stores; 9 = 6 with merge + finalisation in one trip;
                                      10 / 11 = 9 with a compact copy of the prefix errors for the peak search (staged in
                                      shared memory / in registers) and one reciprocal per trip; 12 / 13 = 10 / 11 with 16
                                      loads in flight in the fill pass; 14 (default) / 15 = 11 / 10 with the fill as a
                                      second, streaming kernel (when every column has a scratch slot, else 11);
                                      same results, different speed */,
       B2_OPT_COUNT = 5 };
int b2_set_option(int option, int value);
int b2_get_option(int option);

const char* b2_last_error(void);
int b2_version(void);
int b2_device_sm_count(void);
/* number of CUDA kernels this library has launched so far in the calling process */
unsigned long long b2_launch_count(void);

/* ---- X-stream contractions (the HBM-bound hot kernels) ------------------------------------------------------
 * X: packed data, n_rows x K, row stride ldx elements (ldx*sizeof % 16 == 0, pad columns zero).
 * b2_xstream_y:  Y (n_rows x R) = X * C.              decomposition.py:242 (X_i (C*a_i) = (X_i C)*a_i), :148-152.
 * b2_xstream_z:  Z (K x R) = X^T * W, W n_rows x R (row stride ldw = b2_xstream_z_ldw(R, dtype, variant), pad columns
 *                zero), decomposition.py:312-315 with W_i = B_i * a_i.
 *                W must be allocated with n_rows rounded up to a multiple of 32 rows, zero tail.
 * ws: scratch of at least b2_xstream_workspace_bytes(K, R, dtype) bytes, 16-byte aligned.
 * variant: B2_VARIANT_FMA (fp32/fp64 FMA pipes) or B2_VARIANT_DMMA (fp64 tensor cores, DMMA.8x8x4); AUTO picks.
 * max_ctas: 0 = one CTA per SM. */
int b2_xstream_y(const void* X, long long n_rows, int K, int ldx, const void* C, int R, void* Y, int dtype, void* ws,
                 size_t ws_bytes, int variant, int max_ctas, void* stream);
int b2_xstream_z(const void* X, long long n_rows, int K, int ldx, const void* W, int ldw, int R, void* Z, int dtype,
                 void* ws, size_t ws_bytes, int variant, int max_ctas, void* stream);
int b2_xstream_z_ldw(int R, int dtype, int variant);
size_t b2_xstream_workspace_bytes(int K, int R, int dtype);
/* out[0] = sum(X**2) in double (decomposition.py:906, _root_sum_squared_list :347). ws >= 8*4*SMs bytes. */
int b2_sumsq(const void* X, long long n_rows, int K, int ldx, int dtype, double* out, void* ws, size_t ws_bytes,
             void* stream);

/* ---- single-read fused X-stream pass for slice-local CMF (SURVEY.md §8b `b2_xstream_fused_local`) ----------------
 * ONE pass over X per outer iteration for problems whose B-mode penalties are all row-local (NONNEG, BOX, L1;
 * n_pen <= 2), fp64: per slice g (rows row_off[g] .. row_off[g+1])
 *     Y_g = X_g C;  B_g <- n_inner ADMM iterations on rhs = Y_g * a_g with Minv_g, rho_g (decomposition.py:242, 259-289;
 *     aux/dual of `pens_host` updated in place);  G[g] = X_g^T B_g (K x R);  Z = sum_g G[g] diag(a_g) (K x R,
 *     decomposition.py:312-315);  BtB[g] = B_g^T B_g.
 * The A-update's diag(B_g^T X_g C_new) (decomposition.py:145-158) then comes from b2_slice_gdot(G, C_new) without
 * another pass over X.  The reference reads X three times per outer iteration (:242, :315, :148-152).
 * sched: device array [n_ctas x rounds] of slice ids (-1 = none): CTA c processes sched[c*rounds + 0 ..] in order;
 *   every slice must appear exactly once (the host balances rows per CTA); n_ctas <= b2_device_sm_count().
 * ws: >= b2_xstream_fused_workspace_bytes(K, R, n_ctas) bytes, 16-byte aligned.
 * b2_xstream_fused_local_supported: 1 when the kernel applies (fp64, K * ceil(R/8) <= 1024, C fits shared memory). */
int b2_xstream_fused_local_supported(int K, int R, int dtype, int n_pen);
size_t b2_xstream_fused_workspace_bytes(int K, int R, int n_ctas);
int b2_xstream_fused_local(const void* X, long long n_rows, int K, int ldx, const int64_t* row_off, int n_slices,
                           const int32_t* sched, int n_ctas, int rounds, const void* C, const void* A,
                           const void* rho, const void* Minv, const b2_penalty_desc* pens_host, int n_pen,
                           int n_inner, int R, void* B, void* Z, void* G, void* BtB, int dtype, void* ws,
                           size_t ws_bytes, void* stream);
/* rhs[g][c] = sum_k G[g][k][c] * C[k][c]  (= diag(B_g^T X_g C) from G[g] = X_g^T B_g), fp64 */
int b2_slice_gdot(const void* G, const void* C, int n_groups, int K, int R, void* rhs, int dtype, void* stream);

/* ---- small dense / batched per-slice math --------------------------------------------------------------------*/
/* G (R x R) = M^T M for a dense n x R matrix with row stride ld >= R (C^T C :138,:240 ; sum_i (B_i a_i)^T (B_i a_i)
 * :314). ws >= 16*R*R*SMs bytes. */
int b2_gram(const void* M, long long n, int R, int ld, void* G, int dtype, void* ws, size_t ws_bytes, void* stream);
/* lhs[g] = G o (a_g a_g^T), g < n_groups  (decomposition.py:243). */
int b2_scale_gram(const void* G, const void* A, int n_groups, int R, void* lhs, int dtype, void* stream);
/* rho[g] = 0.5 * trace(lhs[g]) * scale ; rho_max[0] = max_g rho[g]  (decomposition.py:162-165, 247-250, 319).
 * n_groups == 0 (empty shard): rho_max[0] = -inf, the identity of the MAX all-reduce that follows. */
int b2_rho_from_trace(const void* lhs, int n_groups, int R, double scale, void* rho, void* rho_max, int dtype,
                      void* stream);
/* If rho_max != NULL every rho[g] is first overwritten by rho_max[0] (constant_feasibility_penalty).
 * Minv[g] = inverse(lhs[g] + (rho[g]*n_reg + l2) * I) via Cholesky; replaces the SVD solve of :168-172, :252-256,
 * :320-321 (x (U/s) Uh == x lhs^-1 for symmetric positive definite lhs).  A matrix whose Cholesky pivot is <= 0 or
 * NaN (no penalty and no ridge on a rank-deficient Gram, or a negative l2) takes a Jacobi eigen-decomposition instead,
 * Minv = Q diag(1/lam) Q^T — what the reference's SVD route computes for ANY symmetric lhs — so there is no silent NaN. */
int b2_factor_batch(const void* lhs, int n_groups, int R, void* rho, const void* rho_max, int n_reg, double l2,
                    void* Minv, int dtype, void* stream);
/* Per slice g: rhs[g][r] = sum_j B[j][r]*Y[j][r] (= diag(B_i^T X_i C), :158) and
 * cross[g] = (B_g^T B_g) o CtC (:155).  rhs may be NULL; CtC may be NULL (then cross = B^T B, used for PARAFAC2). */
int b2_slice_cross(const void* B, const void* Y, const int64_t* row_off, int n_groups, int R, const void* CtC,
                   void* cross, void* rhs, int dtype, void* stream);
/* W[row][0:R] = B[row] o A[group_of_row[row]]  (B_i * a_i, :313); W has row stride ldw >= R. */
int b2_rowscale(const void* B, const void* A, const int32_t* group_of_row, long long n, int R, void* W, int ldw,
                int dtype, void* stream);

/* ---- fused ADMM step ------------------------------------------------------------------------------------------
 * For every row:  s = rhs[row] o rhs_scale[g] + rho[g] * sum_p (aux_p[row] - dual_p[row])      (:261-273,:328-331,:179-195)
 *                 x[row] = s * Minv[g]
 *   then per penalty p:  v = x[row] + dual_p[row]
 *        elementwise kinds (NONNEG, BOX, L1):  aux_p[row] = prox(v, rho[g]); dual_p[row] = v - aux_p[row]   (:275-285)
 *        column-coupled kinds (L2BALL, UNIMODAL, PARAFAC2): dual_p[row] = v  (finished by the b2_prox_* / b2_pf2_* calls)
 * rhs_scale (n_groups x R) may be NULL. group_of_row is used when group_mode == B2_GROUP_INDEXED. */
int b2_admm_solve(long long n, int R, const void* rhs, const void* rhs_scale, int group_mode,
                  const int32_t* group_of_row, const void* rho, const void* Minv, const b2_penalty_desc* pens_host,
                  int n_pen, void* x, int dtype, void* stream);

/* Whole inner ADMM loop in one pass for modes whose penalties are all row-local (NONNEG, BOX, L1; n_pen <= 2):
 * `n_inner` iterations of the update above with the row state held in registers (decomposition.py:259-289, 325-342,
 * 176-217).  If w_out != NULL also writes w_out[row][0:R] = x[row] o rhs_scale[g] (row stride ldw) — the scaled
 * factor B_i * a_i consumed by b2_xstream_z.  With group_mode INDEXED and row_off != NULL (or group_mode SINGLE) the
 * kernel runs one CTA per group with Minv_g staged in shared memory; BtB_out (optional, INDEXED + row_off only)
 * receives B_g^T B_g of the new x. */
int b2_admm_local(long long n, int R, const void* rhs, const void* rhs_scale, int group_mode,
                  const int32_t* group_of_row, const int64_t* row_off, int n_groups, const void* rho, const void* Minv,
                  const b2_penalty_desc* pens_host, int n_pen, int n_inner, void* x, void* w_out, int ldw,
                  void* BtB_out, int dtype, void* stream);

/* ---- column-coupled proximal operators (V arrives in `dual`, see b2_admm_solve) --------------------------------*/
/* L2Ball (penalties.py:920-925): per group and column  aux = clip(V)*bound/max(||clip(V)_col||, bound); dual = V - aux.
 * phase 0: everything.  Row-sharded groups (mode 0 over several ranks): phase 1 only writes the local column sums of
 * squares to colsq_io (n_groups x R doubles), the caller all-reduces them, phase 2 scales with the reduced sums. */
int b2_prox_l2ball(void* aux, void* dual, const int64_t* row_off, int n_groups, int R, double bound, int non_negativity,
                   double* colsq_io, int phase, int dtype, void* stream);
/* Self-test of the exact integer-divisor division the unimodal kernel uses (reciprocal + two Markstein corrections)
 * against the IEEE division: n pseudo-random numerators x divisors 1..max_cnt; *mismatches_dev (device, 8 bytes)
 * receives the number of differing results (must be 0). */
int b2_selftest_div_count(long long n, unsigned long long seed, int max_cnt, unsigned long long* mismatches_dev,
                          void* stream);
/* Unimodality (penalties.py:1014-1015 -> _unimodal_regression.py:24-141): per group and column aux = unimodal
 * regression of V (PAVA prefix/suffix isotonic fits, `<=` pooling, first strict minimum peak); dual = V - aux.
 * peaks (may be NULL): n_groups x R int32 peak indices t*.  ws >= b2_unimodal_workspace_bytes(). fp64 arithmetic. */
int b2_prox_unimodal(void* aux, void* dual, const int64_t* row_off, int n_groups, int R, int max_rows,
                     int non_negativity, int32_t* peaks, int dtype, void* ws, size_t ws_bytes, void* stream);
size_t b2_unimodal_workspace_bytes(int n_groups, int R, int max_rows);

/* PARAFAC2 (penalties.py:1224-1250).  With V_i = B_i + dual_i (in `dual`) and S_i = V_i^T V_i (b2_slice_cross):
 *   b2_pf2_polar:  W_i such that P_i = V_i W_i = polar(V_i Delta^T)   (R x R Jacobi eigen-decomposition of
 *                  Delta S_i Delta^T instead of the J_i x R SVD of :1234-1235), and
 *                  num_part[g] = rho_i W_i^T S_i = rho_i P_i^T V_i (summand of :1244).
 *                  Qstore (optional, n_groups x R x R doubles) receives the eigenvectors; with warm != 0 the Jacobi
 *                  sweeps start from the eigenvectors stored by the previous call (same result, fewer sweeps).
 *   b2_pf2_delta:  Delta_new = sum_g num_part[g] / sum_g rho[g]  in fixed order (:1240-1245); also writes the
 *                  un-normalised sums to `sums` (R*R + 1 values: numerator, then sum rho) for a cross-rank all-reduce;
 *                  with `sums_in` != NULL it only normalises those (already reduced) sums.
 *   b2_pf2_apply:  pd[row] = V[row] W_g Delta_new (= P_i Delta) ; dual[row] = V[row] - pd[row] (:282-285);
 *                  optionally basis[row] = V[row] W_g (= P_i). */
int b2_pf2_polar(const void* S, const void* Delta, const void* rho, int n_groups, int R, void* Wmat, void* num_part,
                 void* Qstore, int warm, int dtype, void* stream);
/* Fused row pass of one B-mode inner iteration when pens[0] is PARAFAC2 (one CTA per slice).  `deferred` is a bit set:
 *   bit 0 set:     pens[0].dual holds the pre-image V of the previous prox; P Delta = V (W_g Delta) and
 *                  dual = V - P Delta are formed on the fly (pens[0].aux is not read);
 *   bit 0 clear:   pens[0].aux = P Delta and pens[0].dual are read as stored;
 *   bit 1 set:     the ELEMENTWISE companions (NONNEG, BOX, L1) arrive as ONE array: their dual slot holds the previous
 *                  prox argument T = x + dual, from which aux = prox(T) and dual = T - aux are recomputed (aux not read);
 *   bit 2 set:     ... and leave as one array: only T' = x + dual is stored (dual slot), aux is not written.
 *                  A B-update runs its first pass with bits 1, 2 = (0, 1), the middle passes (1, 1), the last (1, 0), so
 *                  explicit (aux, dual) exist before and after it (bit-identical to passing them through every pass).
 *   x = (rho_g * sum_p (aux_p - dual_p) + Y o a_g) Minv_g ; pens[0].dual <- V' = x + dual_pf2 ; S_out[g] = V'^T V' ;
 *   other penalties: elementwise kinds are finished (aux = prox, dual update), column-coupled kinds get dual <- x + dual.
 * x / w_out (= x o a_g, row stride ldw) / BtB_out[g] = x_g^T x_g are written only when non-NULL (last inner iteration).
 * comp_stats_part (optional, 3 * n_groups doubles; last pass = x non-NULL, exactly one companion): per slice
 *   [sum (aux_1 - x)^2, sum x^2, sum |x|] of the companion, the terms of its feasibility gap and penalty value
 *   (decomposition.py:406-415, penalties.py:589-592), taken while aux and x are in registers instead of a further pass
 *   over both arrays; reduce them with b2_group_stats_sum.  Only the steady-state kernel serves it — ask
 *   b2_pf2_rowpass_fused_stats_supported(R, dtype, n_pen, kind of pens[1], deferred) first; in that case bit 2 may also
 *   stay set on the last pass (the companion is kept as ONE array T across outer iterations: aux = prox(T), dual = T - aux). */
int b2_pf2_rowpass(const int64_t* row_off, int n_groups, int R, const void* Y, const void* A, const void* rho,
                   const void* Minv, const b2_penalty_desc* pens_host, int n_pen, int deferred, const void* Wmat,
                   const void* Delta, void* x, void* w_out, int ldw, void* S_out, void* BtB_out,
                   double* comp_stats_part, int dtype, void* stream);
int b2_pf2_rowpass_fused_stats_supported(int R, int dtype, int n_pen, int companion_kind, int deferred);
/* out[0:3] = sum over groups of part[3 g + 0:3], fixed order (per-slice partials of b2_pf2_rowpass / b2_pf2_gap). */
int b2_group_stats_sum(const double* part, int n_groups, double* out, void* stream);

/* ---- per-slice Gram bookkeeping shared by the C- and A-updates (decomposition.py:155, 158, 312-314) ---------------
 * b2_slice_gram:        BtB[g] = B_g^T B_g                       (DMMA, one CTA per slice)
 * b2_slice_coldot:      rhs[g][c] = sum_j B[j][c] * Y[j][c]      (= diag(B_g^T X_g C))
 * b2_weighted_gram_sum: out = sum_g (a_g a_g^T) o BtB[g]         (= sum_i (B_i a_i)^T (B_i a_i)), fixed order
 * b2_hadamard_bcast:    cross[g] = BtB[g] o CtC */
int b2_slice_gram(const void* B, const int64_t* row_off, int n_groups, int R, void* BtB, int dtype, void* stream);
int b2_slice_coldot(const void* B, const void* Y, const int64_t* row_off, int n_groups, int R, void* rhs, int dtype,
                    void* stream);
int b2_weighted_gram_sum(const void* BtB, const void* A, int n_groups, int R, void* out, int dtype, void* stream);
int b2_hadamard_bcast(const void* BtB, const void* CtC, int n_groups, int R, void* cross, int dtype, void* stream);
int b2_pf2_delta(const void* num_part, const void* rho, int n_groups, int R, void* Delta_new, void* sums,
                 const void* sums_in, int dtype, void* stream);
int b2_pf2_apply(void* pd, void* dual, void* basis, const void* Wmat, const void* Delta_new,
                 const int32_t* group_of_row, long long n, int R, int dtype, void* stream);
/* Feasibility-gap terms of the PARAFAC2 penalty from the deferred state, nothing materialised
 * (decomposition.py:406-415 with penalties.py:1287-1304):  out[0] = sum_i ||V_i W_i Delta - x_i||^2 (= ||P_i Delta - B_i||^2),
 * out[1] = sum ||x||^2, out[2] = sum |x|.  ws >= 3 * n_groups doubles. */
int b2_pf2_gap(const void* V, const void* x, const int64_t* row_off, int n_groups, int R, const void* Wmat,
               const void* Delta, double* out, int dtype, void* ws, size_t ws_bytes, void* stream);

/* ---- fused reductions for feasibility gaps / loss (decomposition.py:351-452, 617-627; penalties.py:589-592) ------
 * out[0] = sum((x-y)^2), out[1] = sum(x^2), out[2] = sum(|x|) over n elements (y may be NULL -> out[0] = 0). double. */
int b2_reduce_stats(const void* x, const void* y, long long n, double* out, int dtype, void* ws, size_t ws_bytes,
                    void* stream);
/* out[0] = sum_i rhs_i . a_i ; out[1] = sum_i a_i^T cross_i a_i   (decomposition.py:446-449). */
int b2_fit_terms(const void* rhs, const void* cross, const void* A, int n_groups, int R, double* out, int dtype,
                 void* ws, size_t ws_bytes, void* stream);

/* ---- standalone elementwise prox (ADMMPenalty.factor_matrix_update for NONNEG/BOX/L1 with a scalar rho) ---------*/
int b2_prox_elementwise(const void* v, void* out, long long n, int kind, int non_negativity, double p0, double p1,
                        double rho, int dtype, void* stream);

/* UnitSimplex (penalties.py:953-980): per group and column, aux = max(V - mu, 0) with the multiplier mu found by the
 * reference's bisection (bracket of :957-964, scipy.optimize.bisect's loop and tolerances); dual = V - aux.
 * max_rows = the largest group (sizes the shared-memory staging). */
int b2_prox_simplex(void* aux, void* dual, const int64_t* row_off, int n_groups, int max_rows, int R, int dtype,
                    void* stream);
/* TotalVariationPenalty (penalties.py:819-827): per group g and column, aux = soft_threshold(TV-denoise(V, 2 reg /
 * rho_g), l1 / rho_g) with Condat's direct algorithm (the un-vendored condat_tv dependency's algorithm); dual = V - aux.
 * rho: device array, rho[g * rho_stride] (stride 0 = one value for all groups). */
int b2_prox_tv(void* aux, void* dual, const int64_t* row_off, int n_groups, int R, const void* rho, int rho_stride,
               double reg_strength, double l1_strength, int dtype, void* stream);
/* out[0] = sum_g sum_cols sum_k |x_g[k+1] - x_g[k]|  (:832); part: n_groups doubles of scratch. */
int b2_tv_norm(const void* x, const int64_t* row_off, int n_groups, int R, double* out, double* part, int dtype,
               void* stream);
/* GeneralizedL2Penalty (penalties.py:724-730): every group has J rows; aux_g = U diag((rho_g/2) / (s + rho_g/2)) U^T V_g
 * with the J x J eigenvectors U and eigenvalues s of the norm matrix; dual = V - aux.  tmp: n_groups*J*R elements. */
int b2_prox_gl2(void* aux, void* dual, int n_groups, int J, int R, const void* U, const void* s, const void* rho,
                int rho_stride, void* tmp, int dtype, void* stream);
/* out[0] = sum_g trace(x_g^T M x_g) (:732-733), M symmetric J x J.  tmp: n_groups*J*R elements, part: 256 doubles. */
int b2_quadform(const void* M, const void* x, int n_groups, int J, int R, double* out, void* tmp, double* part,
                int dtype, void* stream);

/* Parafac2(update_basis_matrices=False) (penalties.py:1231-1248): the basis matrices P (packed n x R) stay fixed.
 * phase 1: num_part[g] = rho_g P_g^T V_g (V in `dual`), the summand b2_pf2_delta reduces;
 * phase 2: pd = P Delta, dual = V - pd. */
int b2_pf2_fixed_basis(void* pd, void* dual, const void* P, const void* Delta, const int64_t* row_off, int n_groups,
                       long long n, int R, const void* rho, double* num_part, int phase, int dtype, void* stream);

/* ---- TemporalSmoothnessPenalty: lam * sum_{i>=1} ||B_i - B_{i-1}||_F^2 over the slice order (DESIGN.md §11) -------
 * n_slices slices of equal height, packed one after the other: element (i, p) at i * n_pos + p with n_pos = J * R.
 * For every position p:  (diag(rho) + 2 lam L) z = rho o v,  L the path-graph Laplacian of the slices; V arrives in
 * `dual`, the call leaves aux = z and dual = V - aux (as stored).  rho: device array in the data's dtype,
 * rho[i * rho_stride] (stride 0 = one value for all slices).  fp32 data is solved in fp64.  Partition solve in
 * chunks of 32 slices; bit-reproducible (fixed order, no atomics).  ws: >= b2_prox_temporal_workspace_bytes(n_slices,
 * n_pos, world) bytes, 8-byte aligned; its content must survive from stage 1 to stage 2.
 * stage 0: the whole system (single GPU; world = 1, has_left = has_right = 0, xch may be NULL).
 * Sharded runs (slices [lo, lo + n_slices) of a larger problem on this rank; has_left / has_right: the problem has
 * slices before / after them):
 *   stage 1: solve the local block with zero outer boundaries and write row `rank` of xch (world x (2 n_pos + 4)
 *            doubles, zero-filled by the caller): [first-slice values (n_pos), last-slice values (n_pos), the first /
 *            last entries of T_loc^-1 (2 lam e_first), of T_loc^-1 (2 lam e_last)]; aux / dual untouched.
 *   (caller: sum-all-reduce xch over the ranks; ranks without slices contribute a zero row)
 *   stage 2: solve the 2 x world reduced system (identically on every rank) and finish aux / dual. */
int b2_prox_temporal(void* aux, void* dual, long long n_slices, long long n_pos, const void* rho, int rho_stride,
                     double lam, int stage, int has_left, int has_right, double* xch, int world, int rank, int dtype,
                     void* ws, size_t ws_bytes, void* stream);
size_t b2_prox_temporal_workspace_bytes(long long n_slices, long long n_pos, int world);
/* The same solve with one thread per position running Thomas over all n_slices slices (the forward sweep is parked
 * in aux, in the data's dtype): the latency-bound baseline the partition solve is measured and tested against.
 * ws as for stage 0 of b2_prox_temporal. */
int b2_prox_temporal_serial(void* aux, void* dual, long long n_slices, long long n_pos, const void* rho,
                            int rho_stride, double lam, int dtype, void* ws, size_t ws_bytes, void* stream);
/* out[0] = lam * sum_i ||x_i - x_{i-1}||^2 over the local pairs; part: n_slices doubles of scratch (per-pair partials,
 * summed in a fixed order).  Sharded: xch = world x (n_pos + 1) doubles, all-reduced, row r = [last slice of rank r,
 * 1 if rank r holds slices]; the pair (last slice of the nearest earlier rank with slices, x_0) is added, so that
 * every pair is counted on exactly one rank.  xch NULL: no such pair. */
int b2_temporal_norm(const void* x, long long n_slices, long long n_pos, double lam, const double* xch, int rank,
                     double* out, double* part, int dtype, void* stream);

/* ---- masked fitting (missing entries, EM refill after every outer iteration; DESIGN.md §10) --------------------
 * Missing-entry refill.  For every packed row n (slice g = group_of_row[n]) and every missing column k in
 * miss_col[miss_row_ptr[n] .. miss_row_ptr[n+1]) (int64 row pointer of n_rows+1 entries, int32 columns < K):
 *   xhat = sum_r B[n][r] A[g][r] C[k][r];   d = xhat - X[n][k]   (X[n][k] = the fill the iteration just used)
 *   out[0] += (X[n][k] - xhat)^2      missing-entry part of ||F - X_hat||^2
 *   out[1] += xhat^2 - X[n][k]^2      change of ||F||^2
 *   Y[n][:] += d * C[k][:]             keeps Y = F C valid (Y may be NULL)
 *   X[n][k]  = xhat
 * X: n_rows x K with row stride ldx; A (I x R), B and Y (n_rows x R), C (K x R) dense.  fp32 / fp64 like the engine;
 * sums in double, reduced in a fixed order (no atomics on the sums: runs are bit-reproducible, as everywhere else in
 * this library).  ws: >= b2_mask_refill_workspace_bytes(n_rows) bytes. */
int b2_mask_refill(void* X, long long n_rows, int K, int ldx, const int64_t* miss_row_ptr, const int32_t* miss_col,
                   const int32_t* group_of_row, const void* A, const void* B, const void* C, int R, void* Y,
                   double* out, int dtype, void* ws, size_t ws_bytes, void* stream);
size_t b2_mask_refill_workspace_bytes(long long n_rows);

/* ---- initial state: device-side continuation of a NumPy RandomState (MT19937) stream ----------------------------
 * out[0:n] = the next n doubles `np.random.RandomState.random_sample` / `uniform(0, 1)` would return for the generator
 * whose state is state_io (device, 625 uint32: the 624 key words and the position, as in RandomState.get_state());
 * state_io is advanced so the host generator can continue the stream (decomposition.py:31-39, 78-89;
 * penalties.py:125-147, 239-261 draw everything from one RandomState). */
int b2_mt19937_uniform(void* state_io, double* out, long long n, void* stream);
/* HOST function (state_io is a HOST pointer, no CUDA call): advance the same 625-word state by n_words 32-bit outputs
 * (2 per double) in O(1) of n_words — MT19937 jump-ahead, t^J mod the characteristic polynomial applied by Horner's
 * rule.  Lets a rank of a sharded run skip the rows of other ranks in the reference's single RandomState stream
 * (decomposition.py:31-39, 78-89) instead of walking them; bit-identical to drawing and discarding. */
int b2_mt19937_jump_host(unsigned* state_io, unsigned long long n_words);

/* ---- measurement helpers (bench.py / DESIGN.md roofline denominators) -------------------------------------------
 * kind 0: fp64 FMA pipe, 1: DMMA.8x8x4, 2: fp32 FMA, 3: DMMA + DFMA interleaved (pipe overlap probe). Runs `iters` dependent-chain-free iterations on every SM and
 * writes the number of floating-point operations issued to flops_host. Time it with CUDA events around the call. */
int b2_microbench_flops(int kind, int iters, double* flops_host, void* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MATCOUPLY_B200_H */
