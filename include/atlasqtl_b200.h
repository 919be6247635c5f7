/*
 * atlasqtl_b200 -- C ABI of the B200-native CAVI sweep hot path of atlasqtl.
 *
 * This is the drop-in boundary for the reference's R <-> native interface of that path:
 *
 *   reference interface replaced                                   file:line (under /root/reference)
 *   ------------------------------------------------------------   ---------------------------------
 *   .Call `_atlasqtl_coreDualLoop` (15 SEXP args), R closure       src/RcppExports.cpp:17-38,
 *       coreDualLoop(cp_X, cp_Y_X, gam_vb, log_Phi..., c)          R/RcppExports.R:4-6,
 *       called once per VB iteration                               R/atlasqtl_global_local_core.R:167-170
 *   the Gram / cross-product set-up that feeds it                  R/atlasqtl_global_local_core.R:40-42,112-115
 *   the p x q / n x q reductions around it (update_nu/rho/eta/     R/update_vb.R:19-31,116-118,127-157,217-234
 *       kappa_vb_, update_m2_beta_, update_Z_ row/col sums)
 *   log_Phi / log_1_min_Phi tables                                 R/atlasqtl_global_local_core.R:61-63,293-295
 *   ELBO term B (e_beta_gamma_)                                    R/elbo.R:10-34
 *
 * The reference's dual-form argument list (p x p Gram matrix) cannot exist at the sizes this library
 * targets, so the state (X, residual Y - X beta, gam_vb, mu_beta_vb, tables) lives on the device
 * between calls and the per-iteration entry points exchange only p-, q- and scalar-sized objects
 * (SURVEY.md section 8b).  INTEGRATION.md shows the `.Call` shim and the patched R call site.
 *
 * Conventions
 *   - every function returns 0 on success, a negative AQ_E* code on failure; aq_last_error() gives
 *     the message of the last failure on the calling thread.  No C++ exception or CUDA sticky error
 *     crosses this boundary.
 *   - all matrices are column-major double (R layout); index vectors are int32, 0-based, exactly as
 *     the reference passes them (R/atlasqtl_global_local_core.R:162-163).
 *   - pointers are HOST pointers unless the name ends in _dev.
 *   - one context = one GPU = one contiguous slab of q_local traits (traits are independent inside
 *     a sweep, src/coreLoop.cpp:58-85).  X is replicated per context.
 *   - calls on one context must come from one host thread at a time; the library never calls back.
 */
#ifndef ATLASQTL_B200_H_
#define ATLASQTL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AQ_OK 0
#define AQ_EINVAL (-1)   /* bad argument (NULL, dimension, permutation out of range, ...) */
#define AQ_ECUDA (-2)    /* CUDA runtime failure */
#define AQ_ENOMEM (-3)   /* device allocation failed */
#define AQ_ESTATE (-4)   /* call order violated (e.g. sweep before set_state / refresh_tables) */
#define AQ_EUNSUPPORTED (-5) /* shape outside what this build of the kernels covers */

typedef struct aq_ctx aq_ctx;

const char* aq_last_error(void);
int aq_version(void);

/* Number of SMs, free / total bytes of the device; a cheap "is there a usable GPU" probe. */
int aq_device_info(int device, int* sm_count, int64_t* free_bytes, int64_t* total_bytes);

/*
 * Create a context on `device` and upload the data.
 *   X  n x p  standardised predictors (post-conditions of R/prepare_atlasqtl.R:57-72)
 *   Y  n x q_local  centred responses of this slab (R/prepare_atlasqtl.R:83)
 * Replaces cp_X <- crossprod(X); cp_Y_X <- crossprod(Y, X); Y_norm_sq (R/atlasqtl_global_local_core.R:40-42):
 * the library keeps X (tiled in sweep order) and the residual instead.
 */
int aq_create(aq_ctx** out, int device, int n, int p, int q_local, const double* X, const double* Y);
int aq_destroy(aq_ctx* ctx);

/*
 * Pre-processing on the device: what prepare_data_ does to X and Y before the core sees them
 * (R/prepare_atlasqtl.R:57-83 with rm_constant_ / rm_collinear_, R/utils.R:276-343), without ever holding more than the
 * kept, standardised columns in fp64:
 *   X <- scale(X)                                  centre, divide by the n-1 standard deviation       (:57)
 *   rm_constant_                                   columns that scale() turned into NaN                (:59-62)
 *   rm_collinear_: duplicated(X, MARGIN = 2)       exact duplicates (of the standardised values), the first one is kept (:68-69)
 *   Y <- scale(Y, center = TRUE, scale = FALSE)    column means over the observed (non-NaN) entries    (:83)
 * aq_prep_x takes the raw n x p_raw predictors (column-major doubles); aq_prep_geno takes packed genotype calls: column j
 * starts at geno + j * bytes_per_col, sample i is bits 2 (i % 4) .. 2 (i % 4) + 1 of byte i / 4, values 0 / 1 / 2 (3 is an
 * error: X may not have missing values, check_structure_ R/prepare_atlasqtl.R:18).  p_kept (may be NULL) = columns left.
 * aq_prep_result (any pointer may be NULL, all of length p_raw): status 0 kept / 1 constant / 2 duplicate, dup_of = the
 * raw index of the kept column a duplicate equals (-1 otherwise; the names of rmvd_coll_x, R/utils.R:327-333), and the
 * column mean and n-1 standard deviation used (0 for a constant column).
 * aq_create_prepared: as aq_create on the prep's device with p = p_kept, X standardised on the fly from the raw input,
 * Y_raw (n x q_local, NaN = missing) centred on the device, missing entries set to 0; n_obs (may be NULL, length q_local)
 * = observed entries per trait.  A Y with missing entries still needs aq_set_missing.  The prep can serve several
 * contexts (one per trait slab) and may be destroyed once they exist.
 * aq_get_x / aq_get_y: the n x p standardised predictors / n x q_local centred responses a context holds (host, column-major).
 */
typedef struct aq_prep aq_prep;
int aq_prep_x(aq_prep** out, int device, int n, int p_raw, const double* X_raw, int* p_kept);
int aq_prep_geno(aq_prep** out, int device, int n, int p_raw, const uint8_t* geno, int64_t bytes_per_col, int* p_kept);
int aq_prep_result(const aq_prep* prep, uint8_t* status, int32_t* dup_of, double* mean, double* sd);
int aq_prep_dims(const aq_prep* prep, int* n, int* p_raw, int* p_kept);   /* any pointer may be NULL */
int aq_prep_destroy(aq_prep* prep);
int64_t aq_prep_launch_count(const aq_prep* prep);
int aq_create_prepared(aq_ctx** out, const aq_prep* prep, int q_local, const double* Y_raw, double* n_obs);
int aq_get_x(aq_ctx* ctx, double* X);
int aq_get_y(aq_ctx* ctx, double* Y);
/*
 * Free the context's untiled copy of X ([p][n] doubles: 20 GB at n = 5000, p = 500k).  The sweep reads the tiled images
 * only; the untiled copy serves re-tiling for a new shuffled_ind (aq_set_order), the missing-response kernel and aq_get_x,
 * which return AQ_ESTATE afterwards.  For runs with the reference's fixed identity order (R/atlasqtl_global_local_core.R:162)
 * and no missing responses X is then held once.
 */
int aq_release_x(aq_ctx* ctx);

/* Dimensions and padded leading dimensions of the device layout (for callers that pass _dev pointers). */
int aq_dims(const aq_ctx* ctx, int* n, int* p, int* q_local, int* p_pad, int* q_pad);

/*
 * Visiting order of the SNPs for subsequent sweeps: shuffled_ind of coreDualLoop
 * (src/coreLoop.cpp:64-65; the reference default is 0:(p-1), R/atlasqtl_global_local_core.R:162).
 * Must be a permutation of 0..p-1.  NULL selects the identity.  Re-tiles X and its block Gram band
 * when the order changes; a no-op otherwise.
 */
int aq_set_order(aq_ctx* ctx, const int32_t* shuffled_ind);

/*
 * Load the variational state gam_vb, mu_beta_vb (p x q_local) and derive beta_vb = gam_vb * mu_beta_vb
 * and the residual Y - X beta_vb on the device (replaces update_beta_vb_, update_cp_X_Xbeta_,
 * R/atlasqtl_global_local_core.R:112-115).  Also returns the per-trait sums of aq_sweep (any may be NULL).
 */
int aq_set_state(aq_ctx* ctx, const double* gam_vb, const double* mu_beta_vb,
                 double* colsum_gam, double* colsum_gam_mu2, double* colsum_beta2, double* resid_sq);

/* Copy the state back in R layout (any pointer may be NULL): the in-place outputs of coreDualLoop. */
int aq_get_state(aq_ctx* ctx, double* gam_vb, double* mu_beta_vb, double* beta_vb);

/*
 * Asynchronous hand-off of the state for checkpoints (checkpoint_, R/utils.R:571-627: gam_vb / beta_vb every 100
 * iterations) and outputs.  aq_snapshot copies gam_vb and mu_beta_vb device-to-device in stream order (milliseconds),
 * so the sweeps issued afterwards do not disturb it; aq_snapshot_fetch transposes and downloads THAT copy on a second
 * stream (same outputs as aq_get_state, any may be NULL) and returns once the host buffers are filled.  It touches the
 * snapshot only, so it may be called from another host thread while the context's owner keeps sweeping -- the one
 * exception to the one-thread-at-a-time rule.  One snapshot at a time: aq_snapshot waits for a fetch in flight.
 */
int aq_snapshot(aq_ctx* ctx);
int aq_snapshot_fetch(aq_ctx* ctx, double* gam_vb, double* mu_beta_vb, double* beta_vb);

/* Residual Y - X beta_vb (n x q_local), mainly for tests: X'(Y - residual) is the reference's cp_betaX_X. */
int aq_get_residual(aq_ctx* ctx, double* resid);

/*
 * The three tables of the last aq_refresh_tables, p x q_local each in R layout (column-major), mainly for tests that pin
 * the table pass entry by entry: D = log(1 - Phi(u)) - log Phi(u) at u = theta_j + zeta_k (the log-odds the sweep
 * reads), W = imr1 - imr0 and I0 = imr0 at U = sqrt(c_next) u (U = u when c_next is 1).  Any pointer may be NULL.
 * AQ_ESTATE before the first aq_refresh_tables.
 */
int aq_get_tables(aq_ctx* ctx, double* D, double* W, double* I0);

/*
 * Streaming p x q_local pass after theta_vb / zeta_vb changed
 * (replaces R/atlasqtl_global_local_core.R:61-63 and :293-295):
 *   D    = log(1 - Phi(theta_j + zeta_k)) - log Phi(theta_j + zeta_k)      (the only way the sweep uses the tables)
 *   W    = imr1 - imr0,  I0 = imr0 at U = sqrt(c_next) (theta_j + zeta_k)  (inv_mills_ratio_, R/utils.R:172-191)
 * c_next is the temperature of the NEXT sweep (its update_Z_ evaluates the CDFs at sqrt(c) (theta + zeta),
 * R/update_vb.R:219-224).  If elbo_b_part != NULL it also returns the p x q part of ELBO term B
 * (R/elbo.R:19-26):  sum_jk [ gam lp + (1-gam) lq - gam log(gam+eps) - (1-gam) log(1-gam+eps) ]
 * with the post-update lp / lq and the current gam_vb.
 */
int aq_refresh_tables(aq_ctx* ctx, const double* theta_vb, const double* zeta_vb, double c_next,
                      double* elbo_b_part);

/*
 * One Gauss-Seidel sweep over all SNPs x the slab's traits: coreDualLoop (src/coreLoop.cpp:38-86) in
 * sample space, blocked over SNPs, in the order of aq_set_order.
 *   in : c, log_sig2_inv_vb, and per-trait tau_vb, log_tau_vb, sig2_beta_vb (length q_local)
 *   out (length q_local, any may be NULL), all evaluated on the post-sweep state:
 *     colsum_gam      colSums(gam_vb)                               (update_eta_vb_, update_nu_vb_)
 *     colsum_gam_mu2  colSums(gam_vb * mu_beta_vb^2); colSums(m2_beta) = this + sig2_beta_vb * colsum_gam
 *     colsum_beta2    colSums(beta_vb^2)                            (update_kappa_vb_)
 *     resid_sq        colSums((Y - X beta_vb)^2) = Y_norm_sq - 2 colSums(beta*t(cp_Y_X)) + colSums(cp_X_Xbeta*beta)
 *     colsum_zpart    sum_j [gam_jk W_jk + I0_jk]; colSums(Z)_k = colsum_zpart_k / sqrt(c) + sum(theta) + p zeta_k
 */
int aq_sweep(aq_ctx* ctx, double c, double log_sig2_inv_vb, const double* tau_vb, const double* log_tau_vb,
             const double* sig2_beta_vb, double* colsum_gam, double* colsum_gam_mu2, double* colsum_beta2,
             double* resid_sq, double* colsum_zpart);

/*
 * rowsum_zpart_j = sum_k [gam_jk W_jk + I0_jk] over this slab (length p);
 * rowSums(Z)_j = (sum over slabs) / sqrt(c) + q theta_j + sum(zeta)   (update_theta_vb_, R/update_vb.R:179).
 * The _dev variant leaves the result in device memory (length p_pad doubles, first p valid) so that the
 * caller can all-reduce it across slabs (NCCL) without a host round trip.
 */
int aq_rowsums_zpart(aq_ctx* ctx, double* rowsum_zpart);
int aq_rowsums_zpart_dev(aq_ctx* ctx, double** rowsum_zpart_dev);

/*
 * Missing responses: the reference's second native entry, `.Call _atlasqtl_coreDualMisLoop` (16 SEXP args,
 * src/RcppExports.cpp:41-63; src/coreLoop.cpp:91-138) and its set-up (R/atlasqtl_global_local_core.R:19-33).
 *
 * aq_set_missing: mis_pat is the reference's n x q_local matrix ifelse(is.na(Y), 0, 1).  The Y handed to aq_create
 * may hold anything in the missing positions; they are zeroed here (:22).  Replaces X_norm_sq <- crossprod(X^2,
 * mis_pat) and the list cp_X_rm of q p x p matrices (:23-32): in sample space the per-trait Gram cp_X - cp_X_rm[[k]]
 * is X' diag(mis_k) X, i.e. a residual kept at zero in the missing rows.  n_obs (may be NULL) returns colSums(mis_pat)
 * (update_eta_vb_, R/update_vb.R:131; e_y_, R/elbo.R:141).  n <= 2048 in this build.
 * After this call the context must be driven through aq_set_state_mis / aq_sweep_mis; all other entry points
 * (aq_set_order, aq_refresh_tables, aq_rowsums_zpart, aq_get_state, aq_get_residual) are shared.
 *
 * aq_set_state_mis: as aq_set_state, with r_k = mis_k o (y_k - X beta_k); xn = X_norm_sq.  Extra per-trait sums
 * (any may be NULL): colsum_xn_gam = sum_j xn gam, colsum_xn_gam_mu2 = sum_j xn gam mu^2, colsum_xn_beta2 = sum_j xn
 * beta^2 -- with them update_kappa_vb_'s missing-value branch (R/update_vb.R:149-154) is
 *   kappa_vb = c (kappa + (resid_sq + sig2_inv colSums(m2) + colSums(xn m2) - colsum_xn_beta2) / 2).
 *
 * aq_sweep_mis: one sweep of coreDualMisLoop in the order of aq_set_order, with the p x q
 * sig2_beta_vb(j,k) = 1 / (c (xn(j,k) + sig2_inv_vb) tau_vb[k]) of update_sig2_beta_vb_ (R/update_vb.R:47) formed on
 * the fly.  Outputs (length q_local, any may be NULL) on the post-sweep state:
 *   colsum_gam, colsum_gam_mu2, resid_sq, colsum_zpart       as aq_sweep
 *   colsum_sig2b_gam      sum_j sig2_beta_jk gam;   colSums(m2_beta) = colsum_gam_mu2 + colsum_sig2b_gam
 *   colsum_xn_gam_mu2, colsum_xn_sig2b_gam                    colSums(xn m2_beta) is their sum
 *   colsum_xn_beta2       sum_j xn beta^2
 *   colsum_gam_logsig2b   sum_j gam log sig2_beta_jk           (e_beta_gamma_, R/elbo.R:28-30)
 */
int aq_set_missing(aq_ctx* ctx, const double* mis_pat, double* n_obs);
int aq_set_state_mis(aq_ctx* ctx, const double* gam_vb, const double* mu_beta_vb, double* colsum_gam,
                     double* colsum_gam_mu2, double* colsum_beta2, double* resid_sq, double* colsum_xn_gam,
                     double* colsum_xn_gam_mu2, double* colsum_xn_beta2);
int aq_sweep_mis(aq_ctx* ctx, double c, double log_sig2_inv_vb, double sig2_inv_vb, const double* tau_vb,
                 const double* log_tau_vb, double* colsum_gam, double* colsum_gam_mu2, double* colsum_sig2b_gam,
                 double* colsum_xn_gam_mu2, double* colsum_xn_sig2b_gam, double* colsum_xn_beta2, double* resid_sq,
                 double* colsum_zpart, double* colsum_gam_logsig2b);

/*
 * Selection sets without downloading the p x q PPI matrix (post-processing of the path's output:
 * `assign_bFDR` R/summarise_output.R:207-223 and the threshold sets of `summary` :99-106).  With e = 1 - gam_vb:
 *   aq_ppi_count_sum   count = #{(j,k): e <= t}, sum = sum of those e  (over this slab; deterministic reductions)
 *   aq_ppi_next_above  the smallest e > t (+Inf if none)
 *   aq_ppi_collect     the pairs with  lo < e <= hi  (mode 0)  or  gam_vb > lo  (mode 1)  as (j, k_local, gam_vb) triples in
 *                      arbitrary order; n_found is the number of matching pairs, of which min(n_found, capacity) were written
 * The running mean of the sorted e is non-decreasing, so {bFDR < thres} is a prefix of the sorted order: a bisection on t
 * with aq_ppi_count_sum finds it (atlasqtl_b200/summarise.py::select_bFDR_device; sums over slabs / GPUs add up).
 */
int aq_ppi_count_sum(aq_ctx* ctx, double t, double* count, double* sum);
int aq_ppi_next_above(aq_ctx* ctx, double t, double* next);
int aq_ppi_collect(aq_ctx* ctx, int mode, double lo, double hi, int64_t capacity, int32_t* out_j, int32_t* out_k,
                   double* out_gam, int64_t* n_found);

/* Count of kernel launches issued through this context so far (bench.py's gpu_launches). */
int64_t aq_launch_count(const aq_ctx* ctx);

/* Device time of the last aq_sweep's main kernel in milliseconds (CUDA events on the context's stream). */
int aq_last_sweep_ms(const aq_ctx* ctx, float* ms);
/* Same for the last launch of kernel group `which`: 0 sweep, 1 row sums (aq_rowsums_zpart), 2 tables (+ ELBO part). */
int aq_last_ms(const aq_ctx* ctx, int which, float* ms);

/* Block until everything queued on the context's stream has finished. */
int aq_sync(aq_ctx* ctx);

/*
 * Drop-in for the reference's stateless entry point at sizes where its p x p inputs exist:
 * same 15 arguments, same in-place outputs (gam_vb, m1_beta, cp_betaX_X, mu_beta_vb) as
 * coreDualLoop (src/coreLoop.cpp:38-52), plus the dimensions an R matrix carries in its dim attribute.
 * Needs X'X = cp_X to be factorised on every call, so it is a compatibility / parity entry, not the fast path.
 */
int aq_coreDualLoop(int device, int p, int q, const double* cp_X, const double* cp_Y_X, double* gam_vb,
                    const double* log_Phi_theta_plus_zeta, const double* log_1_min_Phi_theta_plus_zeta,
                    double log_sig2_inv_vb, const double* log_tau_vb, double* m1_beta, double* cp_betaX_X,
                    double* mu_beta_vb, const double* sig2_beta_vb, const double* tau_vb,
                    const int32_t* shuffled_ind, int n_ind, const int32_t* sample_q, int n_q, double c);


/*
 * Same for the missing-response entry point: the 16 arguments of coreDualMisLoop (src/coreLoop.cpp:91-106; .Call glue
 * src/RcppExports.cpp:41-63).  cp_X_rm is the R list of q p x p matrices crossprod(X[missing rows of trait k, ])
 * (R/atlasqtl_global_local_core.R:25-32) as an array of q pointers; sig2_beta_vb is p x q.  In-place outputs as above.
 * Every trait needs its own factorisation of cp_X - cp_X_rm[[k]]: compatibility / parity entry for small p and q.
 */
int aq_coreDualMisLoop(int device, int p, int q, const double* cp_X, const double* const* cp_X_rm, const double* cp_Y_X,
                       double* gam_vb, const double* log_Phi_theta_plus_zeta,
                       const double* log_1_min_Phi_theta_plus_zeta, double log_sig2_inv_vb, const double* log_tau_vb,
                       double* m1_beta, double* cp_betaX_X, double* mu_beta_vb, const double* sig2_beta_vb,
                       const double* tau_vb, const int32_t* shuffled_ind, int n_ind, const int32_t* sample_q, int n_q,
                       double c);

/*
 * How the last aq_sweep spread its trait tiles over the GPU: traits per tile, tiles, tiles a round of the persistent
 * grid processes (SMs or schedulable clusters), and the number of SNP segments every tile was cut into (1 = each CTA
 * sweeps all SNPs of its tiles; > 1 = segmented sweep, see DESIGN.md section 4.1).  Any pointer may be NULL.
 */
int aq_sweep_plan(const aq_ctx* ctx, int* traits_per_tile, int* ntiles, int* groups, int* nseg);

/*
 * Test hook: out[i] = the sweep's annealed logistic 1 / (1 + exp(x[i])) evaluated ON THE DEVICE with the very routine
 * the chain warp uses (== exp(-logOnePlusExp(x)), src/coreLoop.cpp:28-33, :75-77), so that its range handling
 * (|x| > 700, NaN) can be checked directly.  variant: 0 = two-constant argument reduction (tensor-bound 16-trait tiles),
 * 1 = the shorter dependency chain the chain-bound configurations use.  x, out: host arrays of length n.
 */
int aq_test_logistic(int device, int variant, const double* x, double* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* ATLASQTL_B200_H_ */
