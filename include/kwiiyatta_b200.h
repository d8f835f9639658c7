/* kwiiyatta_b200 -- C ABI of the B200-native alignment + spectral-mapping hot path.
 *
 * Drop-in boundary for Iselix/kwiiyatta (reference paths relative to /root/reference):
 *   - kw_dtw_*        replaces the call  fastdtw.fastdtw(x_feature, y_feature, dist=2, radius=radius)
 *                     at kwiiyatta/vocoder/align.py:71 (and fastdtw.dtw), batched over pairs;
 *   - kw_gmm_*        replaces  GaussianMixture(...).fit(dataarray)  at kwiiyatta/converter/gmm.py:20-26;
 *   - kw_convert_*    replaces  MLPG(self.gmm, windows, diff).transform(feature)  at
 *                     kwiiyatta/converter/gmm.py:28-34;
 *   - kw_delta_*      replaces  delta_features(feature, DELTA_WINDOWS)  at kwiiyatta/converter/delta.py:30,46.
 *
 * Conventions
 *   - plain C types only; every "dev" pointer is a CUDA device pointer owned by the caller;
 *   - "host" pointers are ordinary host memory, read before the call returns;
 *   - every entry point is stream-ordered on `stream` (a cudaStream_t passed as void*), spawns no
 *     threads, keeps no global state, and never frees or allocates caller-visible memory;
 *   - return value: 0 = OK, negative = kw_status below; kw_last_error() gives a message for the
 *     calling thread;
 *   - all matrices are row-major float64 unless stated otherwise.
 */
#ifndef KWIIYATTA_B200_H_
#define KWIIYATTA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum kw_status {
    KW_OK = 0,
    KW_ERR_INVALID = -1,      /* bad argument (maps to ValueError in the Python shim)          */
    KW_ERR_WORKSPACE = -2,    /* workspace too small                                            */
    KW_ERR_UNSUPPORTED = -3,  /* feature not built (maps to NotImplementedError)                */
    KW_ERR_CUDA = -4,         /* a CUDA runtime call failed                                     */
    KW_ERR_NO_DEVICE = -5     /* no usable sm_100 device                                        */
};

/* ABI version of this header; bumped on any signature change. */
int kw_abi_version(void);
/* Message describing the last failing call on this thread ("" if none). */
const char* kw_last_error(void);
/* Device properties the host-side roofline arithmetic needs. Any pointer may be NULL. */
int kw_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, int* clock_khz);

/* ------------------------------------------------------------------------------------------
 * DTW / FastDTW  (kwiiyatta/vocoder/align.py:71; fastdtw==0.3.2 semantics)
 *
 * A batch holds n_pairs independent (x, y) problems.  x_dev is the row-major concatenation of
 * all x sequences, shape (sum tx, feat_dim); y_dev likewise.  tx_host / ty_host are HOST arrays.
 *   radius  >= 1 : FastDTW with that radius;  radius < 0 : exhaustive DTW (fastdtw.dtw).
 *   p_norm  : 1 or 2 -- local distance (sum |d|) or sqrt(sum d^2)  (dist=1 / dist=2).
 *   precision : 0 = fp64 exact (paths bit-exact to the oracle), 1 = fp32 local distances
 *               (direct differences and sqrt in fp32, DP sums in fp64; path cost within 1e-6
 *               relative of the fp64 result, paths may differ on near-ties).
 *   tie_mode  : which of fastdtw 0.3.2's two back-ends decides between equal candidates:
 *               0 = pure Python (fastdtw.py: candidates compared after the local distance is
 *               added, first minimum in the order (i-1,j), (i,j-1), (i-1,j-1));
 *               1 = Cython (_fastdtw.pyx as recalled in SURVEY.md 8a: predecessors compared
 *               before the addition, the diagonal wins ties, then (i,j-1), then (i-1,j)).
 *               The two give the same path whenever margin_dev (below) is above rounding.
 * Outputs (device):
 *   cost_dev[n_pairs]            accumulated distance D[tx][ty];
 *   path_dev                     int32 (i, j) pairs; pair p owns the region of (tx[p]+ty[p]) points
 *                                starting at point index  sum_{q<p} (tx[q]+ty[q]);  the path occupies
 *                                the LAST path_len[p] points of its region, in forward order;
 *   path_begin_dev[n_pairs]      index (within the region) of the first path point;
 *   path_len_dev[n_pairs]        number of path points;
 *   cells_dev[n_pairs]           window cells evaluated, summed over resolution levels (may be NULL).
 *   margin_dev[2 * n_pairs]      (may be NULL; precision 0 only) smallest decision margin on the
 *                                returned path: at every cell of the path, the runner-up minus
 *                                the winner among the values the cell rule compared (+inf where
 *                                only one predecessor exists).  [2p] = finest level (the returned
 *                                path itself), [2p+1] = minimum over all resolution levels (the
 *                                coarser paths only shape the search window).  A margin far above
 *                                the rounding of the sums (1e-13 relative) means the path does not
 *                                depend on the tie order or on the last bit of a local distance.
 * ------------------------------------------------------------------------------------------ */
size_t kw_dtw_workspace_bytes(int n_pairs, const int32_t* tx_host, const int32_t* ty_host,
                              int feat_dim, int radius);

int kw_dtw_batch(int n_pairs, const double* x_dev, const double* y_dev,
                 const int32_t* tx_host, const int32_t* ty_host, int feat_dim,
                 int radius, int p_norm, int precision, int tie_mode,
                 double* cost_dev, int32_t* path_dev, int32_t* path_begin_dev,
                 int32_t* path_len_dev, int64_t* cells_dev, double* margin_dev,
                 void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Delta features  (nnmnkwii.preprocessing.delta_features with kwiiyatta's DELTA_WINDOWS,
 * kwiiyatta/converter/delta.py:8-12,30,46).  n_utts utterances concatenated; off_dev[n_utts+1]
 * are frame offsets (int64).  in (sum T, dim) -> out (sum T, 3*dim) = [static, delta, delta2],
 * zero-padded at each utterance's edges.
 * ------------------------------------------------------------------------------------------ */
int kw_delta_features(int n_utts, const int64_t* off_dev, int64_t total_frames, int dim,
                      const double* in_dev, double* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Joint full-covariance GMM EM  (sklearn GaussianMixture.fit as configured at
 * kwiiyatta/converter/gmm.py:9-26).  One EM iteration = kw_gmm_estep + kw_gmm_mstep_accumulate
 * (+ the caller's all-reduce of `stats` across ranks) + kw_gmm_mstep_finalize.
 *
 * Model buffers (device): weights (K), means (K, D), covariances (K, D, D),
 *   prec_chol (K, D, D) upper-triangular L with Sigma^-1 = L L^T (sklearn precisions_cholesky_),
 *   aux (K, D + 2): per component [ b = mu L (D values), log|L| (sum log diag), log w ].
 * stats layout (device, float64): K blocks of (1 + D + D*D): [ n_k, sum r (x-c_k), sum r (x-c_k)(x-c_k)^T ]
 *   followed by 2 scalars [ sum_n log p(x_n), n_frames ].  Length kw_gmm_stats_len(K, D).
 *   c_k is the centre the statistics were accumulated around (centres_dev, (K, D)); the
 *   finaliser undoes it, so any centre gives the same parameters up to rounding.
 * precision: 0 = fp64 (CUDA-core DFMA), 1 = split-fp16 tcgen05 tensor-core contractions.
 * ------------------------------------------------------------------------------------------ */
size_t kw_gmm_stats_len(int n_components, int dim);
/* Length (in doubles) of the responsibilities buffer: component-major, K rows of
 * round_up(n_frames, 128) frames each; resp[k * npad + n] is r_nk.  Pad frames are never read. */
size_t kw_gmm_resp_len(int64_t n_frames, int n_components);
size_t kw_gmm_workspace_bytes(int64_t n_frames, int n_components, int dim, int precision);

/* precision 1 only (no-op otherwise): centre, scale, split into fp16 hi/lo and tile the frames
 * into the workspace.  Call once per (x_dev, workspace) before kw_gmm_estep /
 * kw_gmm_mstep_accumulate with precision 1; those calls read the packed frames from the SAME
 * workspace and must be given the same n_frames, n_components and dim. */
int kw_gmm_pack_frames(int64_t n_frames, const double* x_dev, int n_components, int dim,
                       int precision, void* workspace_dev, size_t workspace_bytes, void* stream);

/* E-step: resp_dev (kw_gmm_resp_len doubles, component-major) responsibilities, sum of log p(x) accumulated into
 * stats[K*(1+D+D*D)] and n_frames into the next slot.
 * resp_form: 0 = resp_dev receives the responsibilities r_nk.  1 (precision 1 only; ignored with
 * precision 0) = the form an EM iteration wants: resp_dev keeps the weighted log-probabilities
 * log(w_k N(x_n | k)), and what the tensor-core M-step consumes (per component and 64-frame tile:
 * has-weight flag, fp32 weights, tile weight) goes straight to the workspace -- the K x N matrix
 * of responsibilities is never written or re-read.  Follow with kw_gmm_mstep_accumulate(precision 1,
 * resp_form 1) on the same workspace, or turn resp_dev into responsibilities in place with
 * kw_gmm_normalize_resp. */
int kw_gmm_estep(int64_t n_frames, const double* x_dev, int n_components, int dim,
                 const double* means_dev, const double* prec_chol_dev, const double* aux_dev,
                 double* resp_dev, double* stats_dev, int precision, int resp_form,
                 void* workspace_dev, size_t workspace_bytes, void* stream);

/* resp_dev as left by kw_gmm_estep(precision 1, resp_form 1) -> responsibilities, in place. */
int kw_gmm_normalize_resp(int64_t n_frames, int n_components, int dim, double* resp_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* Hard assignment argmax_k of the weighted log-probability (sklearn predict; with identity
 * precisions and equal weights this is the k-means assignment step).  labels_dev[n_frames] int32.
 * With precision 1 every frame whose tensor-core runner-up lies within 0.05 nat of its best is
 * re-evaluated in fp64: the two of them, or all components when a third one is within 0.05 nat as
 * well.  The labels therefore equal the fp64 argmax (the lowest index on equal fp64 values). */
int kw_gmm_hard_labels(int64_t n_frames, const double* x_dev, int n_components, int dim,
                       const double* means_dev, const double* prec_chol_dev, const double* aux_dev,
                       int32_t* labels_dev, int precision,
                       void* workspace_dev, size_t workspace_bytes, void* stream);

/* M-step sufficient statistics around centres_dev (K, D) from resp_dev.  Weight that cannot
 * matter is skipped, so the cost follows the sparsity of the posterior: precision 0 drops frames
 * with r_nk <= 1e-16 (below the rounding of n_k); precision 1 drops, per component, the 64-frame
 * tiles in which every r_nk <= 1e-8 (orders below the rounding of its split-fp16 contraction).
 * The summation order is fixed (bitwise reproducible).
 * resp_form: 0 = resp_dev holds responsibilities; 1 = use what kw_gmm_estep(precision 1,
 * resp_form 1) left in this workspace, resp_dev is not read (precision 1 only,
 * KW_ERR_UNSUPPORTED with precision 0). */
int kw_gmm_mstep_accumulate(int64_t n_frames, const double* x_dev, int n_components, int dim,
                            const double* resp_dev, const double* centres_dev,
                            double* stats_dev, int precision, int resp_form,
                            void* workspace_dev, size_t workspace_bytes, void* stream);

/* Parameters from (all-reduced) statistics.  weight_norm: 0 -> n_k / sum_k n_k (M-step),
 * 1 -> n_k / n_frames (GaussianMixture._initialize).  info_dev[K] receives 0 or the 1-based
 * index of the first non-positive Cholesky pivot. */
int kw_gmm_mstep_finalize(int n_components, int dim, double reg_covar, int weight_norm,
                          const double* stats_dev, const double* centres_dev,
                          double* weights_dev, double* means_dev, double* covariances_dev,
                          double* prec_chol_dev, double* aux_dev, int32_t* info_dev,
                          void* stream);

/* prec_chol / aux from given covariances (precisions_cholesky_ of an existing model). */
int kw_gmm_precision_cholesky(int n_components, int dim, const double* weights_dev,
                              const double* means_dev, const double* covariances_dev,
                              double* prec_chol_dev, double* aux_dev, int32_t* info_dev,
                              void* stream);

/* ------------------------------------------------------------------------------------------
 * Joint GMM with diagonal covariance blocks  (GaussianMixture(covariance_type='diagonal_blocks')).
 * D = 2 Dh is even, 2 <= D <= 144.  Each Dh x Dh block Sxx, Sxy, Syx, Syy of a covariance is
 * diagonal, so the model is one 2 x 2 Gaussian per component and feature pair (x_d, y_d) with
 * y_d = z[Dh + d].  FP64 on the CUDA cores; the summation order is fixed (bitwise reproducible).
 * One EM iteration = kw_gmm_db_estep + kw_gmm_db_mstep_accumulate (+ the caller's all-reduce of
 * `stats`) + kw_gmm_db_mstep_finalize, as for the full model.
 *
 * Compact model buffers (device, float64):
 *   weights (K), means (K, D) as for the full model;
 *   covariances (K, Dh, 3): per pair [ S_xx[d][d], S_xy[d][d], S_yy[d][d] ] (reg_covar included);
 *   factors (K, Dh, 3): per pair [ a, b, c ] of the upper factor U = [[a, b], [0, c]] with
 *     Sigma_d^-1 = U U^T.  In sklearn's (K, D, D) precisions_cholesky_ these are the entries
 *     (d, d), (d, Dh + d) and (Dh + d, Dh + d); every other entry is zero;
 *   aux (K, 2): [ log|U_k| (sum of log a + log c over the pairs), log w_k ].
 * stats layout: K blocks of (1 + D + 3 Dh): [ n_k, sum r (z - c_k), per pair sum r u^2,
 *   sum r u v, sum r v^2 ] with u = x_d - c_k[d], v = y_d - c_k[Dh + d], followed by the same
 *   2 scalars as the full model [ sum_n log p(x_n), n_frames ].  Length kw_gmm_db_stats_len.
 * Responsibilities: the full model's layout (kw_gmm_resp_len).
 * Every entry point checks all its arguments before it queues any work: n_frames >= 0,
 * n_components >= 1, the dimension, reg_covar >= 0, weight_norm, NULL buffers and the workspace
 * size (KW_ERR_INVALID / KW_ERR_WORKSPACE).
 * ------------------------------------------------------------------------------------------ */
size_t kw_gmm_db_stats_len(int n_components, int dim);
size_t kw_gmm_db_workspace_bytes(int64_t n_frames, int n_components, int dim);

/* E-step: responsibilities into resp_dev, {sum_n log p(x_n), n_frames} into the stats tail, and
 * (when lse_frame_dev is not NULL) each frame's log-normaliser logsumexp_k log(w_k N(x_n | k)). */
int kw_gmm_db_estep(int64_t n_frames, const double* x_dev, int n_components, int dim,
                    const double* means_dev, const double* factors_dev, const double* aux_dev,
                    double* resp_dev, double* stats_dev, double* lse_frame_dev,
                    void* workspace_dev, size_t workspace_bytes, void* stream);

/* M-step statistics around centres_dev (K, D) from responsibilities; frames with r_nk <= 1e-16
 * are skipped, as in the full model's FP64 M-step. */
int kw_gmm_db_mstep_accumulate(int64_t n_frames, const double* x_dev, int n_components, int dim,
                               const double* resp_dev, const double* centres_dev,
                               double* stats_dev, void* workspace_dev, size_t workspace_bytes,
                               void* stream);

/* Parameters from (all-reduced) statistics; weight_norm and info_dev as kw_gmm_mstep_finalize
 * (the pivot index counts in the expanded D x D matrix). */
int kw_gmm_db_mstep_finalize(int n_components, int dim, double reg_covar, int weight_norm,
                             const double* stats_dev, const double* centres_dev,
                             double* weights_dev, double* means_dev, double* covariances_dev,
                             double* factors_dev, double* aux_dev, int32_t* info_dev,
                             void* stream);

/* factors / aux from given compact covariances and weights. */
int kw_gmm_db_precision_cholesky(int n_components, int dim, const double* weights_dev,
                                 const double* covariances_dev, double* factors_dev,
                                 double* aux_dev, int32_t* info_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Conversion: posterior + conditional Gaussian + MLPG  (nnmnkwii MLPG.transform,
 * kwiiyatta/converter/gmm.py:28-34).  dim_half = D/2 (72), static_dim = dim_half/3 (24).
 *
 * kw_convert_prepare slices a joint model (optionally with the diff rewrite) into the
 * `prepared` block (device, float64, length kw_convert_prepared_len):
 *   [ px_prec_chol (K,Dh,Dh) | px_aux (K,Dh+2) | A^T (K,Dh,Dh) with A = Syx Sxx^-1 |
 *     offset (K,Dh) = mu_y - A mu_x | var (K,Dh) diagonal conditional variance |
 *     scratch (K,Dh,Dh) | mu_x (K,Dh) | mu_y (K,Dh) ]
 * kw_convert_batch converts n_utts utterances concatenated in src_dev (sum T, Dh) with int64
 * frame offsets off_dev[n_utts+1]; out_dev is (sum T, static_dim); mix_dev (sum T) int32 receives
 * the hard mixture sequence (may be NULL).
 * ------------------------------------------------------------------------------------------ */
size_t kw_convert_prepared_len(int n_components, int dim_half);
int kw_convert_prepare(int n_components, int dim_half, int diff, const double* weights_dev,
                       const double* means_dev, const double* covariances_dev,
                       double* prepared_dev, int32_t* info_dev, void* stream);
size_t kw_convert_workspace_bytes(int64_t total_frames, int n_components, int dim_half,
                                  int precision);
int kw_convert_batch(int n_utts, const int64_t* off_dev, int64_t total_frames, int max_frames,
                     const double* src_dev, int n_components, int dim_half,
                     const double* prepared_dev, double* out_dev, int32_t* mix_dev,
                     int precision, void* workspace_dev, size_t workspace_bytes, void* stream);

/* Global variance (GV; Toda, Black & Tokuda, IEEE TASLP 15(8), 2007; oracle/gv_ref.py).
 *
 * kw_gv_estimate: for the columns [col0, col0 + ncols) of the row-major (total_rows, ld) device
 * matrix x_dev, cut into n_utts utterances by int64 row offsets off_dev[n_utts + 1]:
 *   utt_var_dev (n_utts, ncols)  v = (1/T) sum_t (x_t - mean)^2 per utterance (0 where T = 0);
 *   mean_dev, var_dev (ncols)    mu_v and sigma^2_v = population variance of v, over the
 *                                utterances with T >= 1, sigma^2_v floored at 1e-12;
 *   sums_dev (2 ncols + 1)       [ sum v | sum v^2 | number of utterances ] (may be NULL), to be
 *                                summed over ranks and turned into mu_v, sigma^2_v by
 *                                kw_gv_from_sums (sigma^2_v = sum v^2 / n - mu_v^2, floored).
 * Every sum has a fixed order: the results are bitwise reproducible.
 *
 * kw_convert_gv_batch: kw_convert_batch followed by GV-considered generation per (utterance,
 * static dim): variance scaling of the ML trajectory to mu_v (gv_iter = 0 stops there: the GV
 * postfilter), then gv_iter steps of step-controlled diagonal-Newton ascent on
 *   F(y) = w_traj (-1/2 y^T R y + y^T r) - w_gv 1/2 (v(y) - mu_v)^2 / sigma^2_v
 * (R y = r the MLPG normal equations; w_traj > 0, w_gv >= 0).  gv_mean_dev / gv_var_dev
 * (static_dim) are mu_v and sigma^2_v.  Diff mode (a `prepared` block made with diff = 1):
 * static_src_dev points at the source static features, row stride static_ld (usually src_dev
 * itself, static_ld = dim_half); GV then applies to source + output.  NULL = plain conversion.
 * f_dev (n_utts, static_dim) receives the final F (of source + output in diff mode),
 * accepted_dev (n_utts, static_dim) the number of accepted steps; either may be NULL.
 * max_frames sizes the shared-memory staging (utterances above min(max_frames, 1024) frames are
 * iterated in global memory).  Workspace: kw_convert_gv_workspace_bytes.
 * ------------------------------------------------------------------------------------------ */
int kw_gv_estimate(int n_utts, const int64_t* off_dev, int64_t total_rows, int ld, int col0,
                   int ncols, const double* x_dev, double* utt_var_dev, double* sums_dev,
                   double* mean_dev, double* var_dev, void* stream);
int kw_gv_from_sums(int ncols, const double* sums_dev, double* mean_dev, double* var_dev,
                    void* stream);
size_t kw_convert_gv_workspace_bytes(int64_t total_frames, int n_components, int dim_half,
                                     int precision);
int kw_convert_gv_batch(int n_utts, const int64_t* off_dev, int64_t total_frames, int max_frames,
                        const double* src_dev, int n_components, int dim_half,
                        const double* prepared_dev, const double* gv_mean_dev,
                        const double* gv_var_dev, int gv_iter, double w_traj, double w_gv,
                        const double* static_src_dev, int static_ld, double* out_dev,
                        int32_t* mix_dev, double* f_dev, int32_t* accepted_dev, int precision,
                        void* workspace_dev, size_t workspace_bytes, void* stream);

/* Maximum-likelihood conversion over all mixture sequences (EM trajectory estimation; Toda, Black
 * & Tokuda, IEEE TASLP 15(8), 2007; oracle/mlpg_em_ref.py).  kw_convert_em_batch starts from the
 * kw_convert_batch output y0 and runs em_iter (>= 1) EM iterations on
 *   L(y) = sum_t log sum_m w_m N(x_t; mu_x, S_xx) N((W y)_t; E_{m,t}, diag D_m)
 * per utterance: E-step = the GMM E-step at dimension 2 * dim_half on [x_t ; (W y)_t] (precision
 * 0: FP64, 1: tensor cores); M-step = the MLPG system (W^T P W) y = W^T q with per-frame
 * P_t = sum_m gamma D_m^-1 and q_t = sum_m gamma D_m^-1 E_{m,t}, where posteriors gamma <= 1e-14
 * contribute nothing.  No iteration decreases L (up to rounding).  Diff mode is the same
 * iteration on a `prepared` block made with diff = 1.  out_dev (sum T, static_dim) receives y;
 * loglik_dev (n_utts, em_iter + 1), may be NULL, receives L(y_k) for k = 0 .. em_iter (the last
 * entry costs one more E-step), each summed in a fixed order.  Bitwise reproducible.  Needs
 * dim_half a multiple of 3 and 2 * dim_half <= 144.  Workspace: kw_convert_em_workspace_bytes. */
size_t kw_convert_em_workspace_bytes(int64_t total_frames, int n_components, int dim_half,
                                     int precision);
int kw_convert_em_batch(int n_utts, const int64_t* off_dev, int64_t total_frames,
                        const double* src_dev, int n_components, int dim_half,
                        const double* prepared_dev, int em_iter, double* out_dev,
                        double* loglik_dev, int precision, void* workspace_dev,
                        size_t workspace_bytes, void* stream);

/* Full conditional covariance (the ML trajectory of Toda, Black & Tokuda, IEEE TASLP 15(8), 2007;
 * oracle/mlpg_full_ref.py).  The hard-sequence conversion of kw_convert_batch with the full
 * conditional covariance Sigma_m = S_yy - A_m S_xy of each mixture (after the diff rewrite) in place
 * of the diagonal table `var`: y = argmax sum_t log N((W y)_t; E_{m_t,t}, Sigma_{m_t}), the
 * block-pentadiagonal SPD system R y = r with static_dim x static_dim blocks (static dimensions
 * coupled), solved per utterance by a block Cholesky factorisation.
 *
 * kw_convert_fullcov_prepare derives the `fullcov` block (device, float64, length
 * kw_convert_fullcov_prepared_len) from the covariances and a `prepared` block made by
 * kw_convert_prepare with the same dim_half and diff (neither is changed):
 *   [ G (K, 6, sd, sd): the six distinct blocks sum_{w,v} c[w][a+1] c[v][b+1] P^(w,v) of
 *     P = Sigma^-1 | B^T (K,Dh,Dh), B = P A | h (K,Dh) = P offset ]
 * Sigma and its factorisation live in a workspace of kw_convert_fullcov_prepare_workspace_bytes
 * that the call no longer needs once it has completed on `stream`.  info_dev (K) int32 is
 * non-zero where Sigma_k is not positive definite.  dim_half a multiple of 3 and <= 80.
 * kw_convert_fullcov_batch takes kw_convert_batch's arguments plus that block and writes the same
 * outputs (mix_dev may be NULL); max_frames is unused, as in kw_convert_batch, and bounds
 * nothing.  Workspace (kw_convert_fullcov_workspace_bytes): the block
 * factors kept between the forward and the backward sweep, 8 (3 sd^2 + sd) bytes per frame
 * (14 KB at sd = 24, where the diagonal path's band takes 768 B), plus what kw_convert_batch
 * needs besides its band. */
size_t kw_convert_fullcov_prepared_len(int n_components, int dim_half);
size_t kw_convert_fullcov_prepare_workspace_bytes(int n_components, int dim_half);
int kw_convert_fullcov_prepare(int n_components, int dim_half, int diff,
                               const double* covariances_dev, const double* prepared_dev,
                               double* fullcov_dev, int32_t* info_dev, void* workspace_dev,
                               size_t workspace_bytes, void* stream);
size_t kw_convert_fullcov_workspace_bytes(int64_t total_frames, int n_components, int dim_half,
                                          int precision);
int kw_convert_fullcov_batch(int n_utts, const int64_t* off_dev, int64_t total_frames,
                             int max_frames, const double* src_dev, int n_components,
                             int dim_half, const double* prepared_dev, const double* fullcov_dev,
                             double* out_dev, int32_t* mix_dev, int precision,
                             void* workspace_dev, size_t workspace_bytes, void* stream);

/* Low-delay conversion (fixed-lag MLPG; Muramatsu et al., Interspeech 2008;
 * oracle/mlpg_stream_ref.py) over n_slots concurrent streams, each one utterance arriving one
 * static frame (static_dim = dim_half / 3 values, mel-cepstrum without c0) per call.  Static j of
 * a stream completes its source vector x_{j-1} = [x~, delta, delta^2] (zero padded at the start
 * and, when the stream ends, at the end), and with it the hard mixture, conditional mean and
 * diagonal variance of frame j-1: n = j frames are known.  The frame emitted with static j is
 * y^(n)[n-1-delay], where y^(n) is kw_convert_batch's MLPG solution of frames [0, n) alone; so
 * frame s comes out delay + 1 frames after its static went in.  Ending a stream of T statics
 * emits its last min(T, delay + 1) frames from y^(T), the offline solution; with delay >= T-1 the
 * whole output equals kw_convert_batch's.  Per call and slot the cost is one E-step row, one
 * conditional mean and O(delay) per static dimension.
 *
 * The state of n_slots streams (device, float64, length kw_convert_stream_state_len) holds per
 * slot the frame count, the last two statics, the last two frames' precision terms and a ring of
 * delay + 2 Cholesky factor rows per static dimension: 8 (14 + 4 (delay + 2)) static_dim + 8 bytes.
 * kw_convert_stream_init empties every slot.  A state serves the n_slots, dim_half and delay it
 * was made for, and one `prepared` block (diff mode comes from that block).
 *
 * kw_convert_stream_push delivers one static per slot for the m (0 <= m <= n_slots) distinct
 * slots in the HOST array slots_host: static_dev (m, static_dim).  out_dev (m, static_dim)
 * receives the emitted frames and frame_dev (m) int64 their indices in their streams, -1 (and a
 * zero row) where a stream has not yet gone delay + 1 statics past its first.
 * kw_convert_stream_end ends the streams of the m slots, which are empty afterwards: out_dev
 * (m, delay + 1, static_dim) receives the last count_dev[i] (m, int64) frames of row i in order,
 * zero rows after them (an empty slot emits 0 frames).
 * Both check every argument before they queue any work, and a rejected call changes neither
 * the workspace nor the state: slots in [0, n_slots) and distinct, delay in [0, 8192],
 * dim_half a multiple of 3 and <= 80, precision 0 (FP64 E-step) or 1 (tensor cores, labels
 * re-checked in FP64 near ties), and a workspace of kw_convert_stream_workspace_bytes for m rows
 * (which does not depend on delay). */
size_t kw_convert_stream_state_len(int n_slots, int dim_half, int delay);
int kw_convert_stream_init(int n_slots, int dim_half, int delay, double* state_dev, void* stream);
size_t kw_convert_stream_workspace_bytes(int m, int n_components, int dim_half, int delay,
                                         int precision);
int kw_convert_stream_push(int n_slots, int delay, int m, const int32_t* slots_host,
                           const double* static_dev, int n_components, int dim_half,
                           const double* prepared_dev, double* state_dev, double* out_dev,
                           int64_t* frame_dev, int precision, void* workspace_dev,
                           size_t workspace_bytes, void* stream);
int kw_convert_stream_end(int n_slots, int delay, int m, const int32_t* slots_host,
                          int n_components, int dim_half, const double* prepared_dev,
                          double* state_dev, double* out_dev, int64_t* count_dev, int precision,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* Soft-posterior mapping without MLPG (nnmnkwii MLPGBase.transform; the mlpg=False branch of
 * kwiiyatta/converter/gmm.py:30-31): out (total, dim_half) = sum_m p(m|x) (mu_y + S_yx S_xx^-1 (x - mu_x)).
 * `prepared_dev` comes from kw_convert_prepare with the same dim_half. */
size_t kw_convert_soft_workspace_bytes(int64_t total_frames, int n_components, int dim_half);
int kw_convert_soft_batch(int64_t total_frames, const double* src_dev, int n_components,
                          int dim_half, const double* prepared_dev, double* out_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-array assembly on the device: from mel-cepstra to the (N, 2*3*order) matrix
 * GaussianMixture.fit receives, without the joint frames visiting the host (SURVEY.md 8f row 2).
 *
 * kw_dtw_features   make_feature (kwiiyatta/vocoder/align.py:20-58) for n_utts utterances
 *                   concatenated in mcep_dev (total_frames, width = order + 1), int64 frame offsets
 *                   off_dev[n_utts + 1]:  out (total_frames, width + 1) = [power flag, voicing flag,
 *                   mcep[1:]].  voiced_dev: one byte per frame (NULL = no voicing flag);
 *                   power_mode 0: power_weight where c0 >= threshold_dev[utt] (the caller computes
 *                   the per-utterance threshold: max / median / min of c0 -/+ the offset, or the
 *                   fixed value), 1: raw c0, 2: zero.
 * kw_path_select    strict filter (align.py:73-94, with the :78 quirk: x's VOICING flag is tested
 *                   against y's POWER flag) and pad trim (align.py:139-145) of the paths
 *                   kw_dtw_batch produced, in place: pair p's selected points end up at the FRONT
 *                   of its path region, selected_len_dev[p] of them.  region_off_dev[p] = point
 *                   index of pair p's region; xoff/yoff_dev[p] = first frame of pair p in the
 *                   concatenated feature matrices; tx/ty_dev: (padded) lengths.
 * kw_joint_frames   gather + drop c0 + delta features over the aligned sequence + hstack
 *                   (vocoder/abc/feature.py:170-194, converter/mcep.py:33, converter/delta.py:30,
 *                   converter/dataset.py:68): out (total_rows, 2 * (3 or 1) * order), row offsets
 *                   out_off_dev[n_pairs + 1] = prefix sums of selected_len; zero_flag_dev[row] = 1
 *                   where the row's absolute sum is not above 1e-7 (remove_zeros_frames,
 *                   converter/dataset.py:70: the caller drops those rows).
 * ------------------------------------------------------------------------------------------ */
int kw_dtw_features(int n_utts, const int64_t* off_dev, int64_t total_frames, int width,
                    const double* mcep_dev, const uint8_t* voiced_dev,
                    const double* threshold_dev, int power_mode, double power_weight,
                    double vuv_weight, double* out_dev, void* stream);
int kw_path_select(int n_pairs, const int64_t* region_off_dev, const int32_t* path_begin_dev,
                   const int32_t* path_len_dev, const int32_t* tx_dev, const int32_t* ty_dev,
                   const int64_t* xoff_dev, const int64_t* yoff_dev, const double* xfeat_dev,
                   const double* yfeat_dev, int feat_dim, int strict, int check_power,
                   int check_vuv, int trim, int pad_len, int32_t* path_dev,
                   int32_t* selected_len_dev, void* stream);
int kw_joint_frames(int n_pairs, const int64_t* out_off_dev, int64_t total_rows,
                    const int64_t* region_off_dev, const int32_t* path_dev,
                    const int64_t* xoff_dev, const int64_t* yoff_dev, const double* xmcep_dev,
                    const double* ymcep_dev, int width, int use_delta, double* out_dev,
                    uint8_t* zero_flag_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Hand-off to the MLSA differential filter: mel-cepstrum -> MLSA filter coefficients,
 * pysptk.mc2b(mc, alpha) as called at kwiiyatta/filter/mlsa.py:24-29 on the converted
 * (difference) mel-cepstra: b[M] = mc[M], b[m] = mc[m] - alpha b[m+1].  mc_dev and b_dev are
 * (total_frames, width) with width = order + 1; zero_power != 0 treats column 0 of the input as
 * zero (mlsa.py:23 removes the power coefficient first).  In place (b_dev == mc_dev) is allowed.
 * ------------------------------------------------------------------------------------------ */
int kw_mc2b(int64_t total_frames, int width, double alpha, int zero_power,
            const double* mc_dev, double* b_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KWIIYATTA_B200_H_ */
