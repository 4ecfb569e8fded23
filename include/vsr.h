/* vsr.h -- C ABI of the B200 refinement engine (libvsr.so).
 *
 * Drop-in boundary for the post-decode refinement path of ViSymRe
 * (aidalee123/Vision-SR).  The reference has no native code: the calls replaced are
 * Python-level, cited per entry point below (paths relative to the reference root).
 * Every entry point returns 0 on success, a negative VSR_E* code otherwise;
 * vsr_last_error() gives the text.  Unless marked "host", pointers are caller-owned
 * DEVICE memory (e.g. torch data_ptr()) and work is enqueued on the caller's
 * cudaStream_t (passed as void*; NULL = default stream) without host
 * synchronisation.  One handle per device; a handle is not thread-safe and owns one
 * scratch workspace, so calls on one handle must be stream-ordered with each other.
 *
 * The ISA of the skeleton programs is in vision-sr_b200/csrc/vsr_isa.h.
 */
#ifndef VSR_H_
#define VSR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSR_ABI_VERSION 1

enum {
  VSR_OK = 0,
  VSR_EINVAL = -1,   /* bad argument */
  VSR_ECUDA = -2,    /* CUDA runtime error (text in vsr_last_error) */
  VSR_ENOMEM = -3,
  VSR_ESTATE = -4,   /* points or programs not uploaded yet */
  VSR_ELIMIT = -5    /* program exceeds a static limit of the ISA */
};

typedef struct vsr_handle vsr_handle;

/* Options of one fit call.  Defaults (vsr_fit_opts_default) are scipy's, which the
 * reference inherits by calling minimize(..., method='BFGS') with no options
 * (src/visymre/architectures/bfgs.py:115, :179). */
typedef struct vsr_fit_opts {
  double gtol;           /* 1e-5 */
  double c1;             /* 1e-4 */
  double c2;             /* 0.9 */
  double xrtol;          /* 0 */
  double fd_eps;         /* 1.4901161193847656e-08 */
  double penalty;        /* 1e6: value of a non-finite loss (bfgs.py:106-112) */
  double loss_scale;     /* 1 for MSE, 1/mean(y) for NMSE (bfgs.py:84-92) */
  double stop_time;      /* seconds per restart before the loss turns into `penalty`
                            (TimedFun, bfgs.py:23-36); 1e9 = never */
  int32_t maxiter_per_k; /* 200 */
  int32_t grad_mode;     /* VSR_GRAD_DUAL (0) or VSR_GRAD_FD (1, scipy-parity mode) */
  int32_t eval_dtype;    /* VSR_F64 (0) or VSR_F32 (1): arithmetic of the optimiser's sweeps */
  int32_t score_dtype;   /* dtype of the final per-restart MSE (bfgs.py:126-132 scores in
                            X's dtype) */
  int32_t warps_per_run; /* 0 = choose from N and the number of runs */
  int32_t reserved;
} vsr_fit_opts;

int vsr_abi_version(void);
void vsr_fit_opts_default(vsr_fit_opts* o);

/* Creates the engine on CUDA device `device`.  Fails with VSR_ECUDA when there is no
 * usable device: there is no CPU fallback. */
int vsr_create(int device, vsr_handle** out);
void vsr_destroy(vsr_handle* h);
const char* vsr_last_error(const vsr_handle* h); /* h may be NULL: last create error */

/* Points.  Replaces the per-candidate pickling of (X_cpu, y_cpu) into worker
 * processes (src/visymre/architectures/model.py:457-458, :483, :490-491) and the
 * N x 10 sympy substitutions of bfgs.py:77-83.  X is column-major: column j (variable
 * x_{j+1}) starts at X + j*ldx elements; y has N elements.  `dtype` selects one of two
 * slots (VSR_F64 / VSR_F32) so a handle can hold the same points in both precisions.
 * vsr_set_points keeps the caller's device pointers (no copy); vsr_upload_points copies
 * HOST arrays into memory the handle owns. */
int vsr_set_points(vsr_handle* h, const void* X_dev, const void* y_dev, int64_t n_points,
                   int64_t ldx, int32_t n_vars, int32_t dtype);
int vsr_upload_points(vsr_handle* h, const void* X_host, const void* y_host, int64_t n_points,
                      int64_t ldx, int32_t n_vars, int32_t dtype, void* stream);

/* Per-point weights of the points in slot `dtype` (w_i > 0, finite, n_points = the slot's N).  Caller-owned
 * device memory, kept like vsr_set_points' pointers; NULL clears.  vsr_set_points / vsr_upload_points of that
 * slot clear it.  Read by vsr_fit (optimiser sweeps and the per-restart final MSE), vsr_eval (loss and
 * gradient) and vsr_gram (the F64 slot's weights: out_rss = sum w r^2, out_jtj = J^T W J).  Not read by
 * vsr_score (the drivers' unweighted R^2) or vsr_predict (reads neither y nor w).  With weights, the loss of
 * a fit and of vsr_eval is loss_scale * (1/N) sum_i w_i (f(x_i; c) - y_i)^2; w_i = 1 gives the unweighted
 * results bit for bit.  The elements are of the slot's type, like y.  VSR_EINVAL: n_points is not the
 * slot's N; VSR_ESTATE: the slot has no points. */
int vsr_set_weights(vsr_handle* h, const void* w_dev, int64_t n_points, int32_t dtype);

/* Robust loss of the points in slot `dtype`: `loss` is a VsrLoss (vsr_isa.h), scipy.optimize.least_squares'
 * `loss`, and f_scale its `f_scale` (C).  With z_i = w_i r_i^2 / C^2 (w_i = 1 without weights) every point
 * contributes cost_i = C^2 rho(z_i) instead of w_i r_i^2, and rho'(z_i) w_i r_i df/dc instead of
 * w_i r_i df/dc.  vsr_set_points / vsr_upload_points of that slot reset it to VSR_LOSS_LINEAR.  Read by
 * vsr_fit (optimiser sweeps from the eval slot, per-restart score from the score slot), vsr_eval (loss and
 * gradient) and vsr_gram (the F64 slot's loss); not by vsr_score or vsr_predict.  A residual that is nan or
 * +-inf contributes the linear terms; a z that overflows from a finite residual contributes scipy's rho(inf)
 * (C^2 pi / 2 for arctan, +inf otherwise) and no gradient.  VSR_LOSS_LINEAR launches today's kernels, and
 * huber with every z <= 1 gives the linear results bit for bit.  VSR_EINVAL: unknown loss, or f_scale^2 or
 * 1 / f_scale^2 not a finite normal double; VSR_ESTATE: the slot has no points. */
int vsr_set_loss(vsr_handle* h, int32_t loss, double f_scale, int32_t dtype);

/* Programs.  Replaces sp.lambdify of the N-term loss, once per restart (bfgs.py:104)
 * and of the fitted expression (bfgs.py:128).  HOST arrays: instruction words of all
 * C programs back to back, insn_off[C+1], literal pools back to back, imm_off[C+1],
 * and the number of constants k[C] of each program.  The handle copies them to the
 * device (asynchronously on `stream`; the host arrays may be reused on return). */
int vsr_upload_programs(vsr_handle* h, const uint64_t* insns, const int32_t* insn_off,
                        const double* imms, const int32_t* imm_off, const int32_t* k,
                        int32_t n_programs, void* stream);

/* Batched evaluation of n_pairs (program, constants) pairs over all points:
 *   out_loss[p]    = mean_i (f_{prog[p]}(x_i; consts[row[p]]) - y_i)^2   (may be nan/inf)
 *   out_grad[p][j] = d out_loss[p] / d c_j      (only when out_grad != NULL)
 * Replaces the lambdified loss evaluation (bfgs.py:106-112) and the per-restart score
 * (bfgs.py:120-132).  prog_idx[n_pairs] and const_row[n_pairs] are HOST int32 arrays
 * (const_row may be NULL = identity); consts[.][kstride] and out_grad[n_pairs][kstride]
 * are f64 device arrays; `dtype` picks the point slot and the arithmetic.  Pairs whose
 * program has more than VSR_MAX_DUAL constants get nan gradients.  With weights (vsr_set_weights) the
 * mean is of w_i r_i^2, with a robust loss (vsr_set_loss) of C^2 rho(z_i), and the gradient follows. */
int vsr_eval(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row,
             int32_t n_pairs, const double* consts, int32_t kstride, int32_t dtype,
             double* out_loss, double* out_grad, void* stream);

/* Driver-side scoring.  Replaces the block every driver runs after each fitfunc call
 * (scripts/Feynman_test.py:81-97, and the same lines in the other *_test.py): re-lambdify the
 * winner, predict on the FULL train / test set (1e5-1e6 rows), np.nan_to_num the prediction,
 * r2_score it.  Same arguments as vsr_eval, value only:
 *   out_mse[p] = mean_i (nan_to_num(f_{prog[p]}(x_i; consts[row[p]])) - y_i)^2
 * with numpy's rule (nan -> 0, +-inf -> +-largest finite value of the dtype); the caller
 * turns it into R^2 = 1 - out_mse / var(y) (src/visymre/scoring.py). */
int vsr_score(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row,
              int32_t n_pairs, const double* consts, int32_t kstride, int32_t dtype,
              double* out_mse, void* stream);

/* Gauss-Newton statistics of n_pairs (program, constants) pairs over all points, fp64:
 *   out_rss[p]          = sum_i (f(x_i; c) - y_i)^2
 *   out_jtj[p][a][b]    = sum_i df(x_i)/dc_a * df(x_i)/dc_b   (a, b < k; full symmetric,
 *                          row stride kstride; entries with a or b >= k are not written)
 * Same pair arguments as vsr_eval.  Programs with k > VSR_MAX_DUAL: jtj rows nan.
 * What a covariance of fitted constants is built from (sigma^2 (J^T J)^-1, as
 * scipy.optimize.curve_fit's pcov); the reference has no counterpart.  Always reads the VSR_F64
 * point slot.  Non-finite values propagate: a point where f is not real makes both outputs nan.
 * The result of a pair does not depend on the other pairs of the call, bit for bit.  With the F64
 * slot's weights out_rss = sum w r^2 and out_jtj = J^T W J; with its robust loss (vsr_set_loss)
 * out_rss = sum C^2 rho(z_i) and out_jtj = J^T W S J, S = diag(max(rho' + 2 z rho'', 2^-52)): the
 * statistics of least_squares' scaled Jacobian that curve_fit's pcov uses. */
int vsr_gram(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row, int32_t n_pairs,
             const double* consts, int32_t kstride, double* out_rss, double* out_jtj, void* stream);

/* Per-point values, and optionally delta-method variances, of n_pairs (program, constants) pairs
 * over all points of the `dtype` slot:
 *   out_value[p][i] = f_{prog[p]}(x_i; consts[row[p]])                       (nan / inf allowed)
 *   out_var[p][i]   = g_i^T cov[row[p]] g_i,  g_i = d f / d c at x_i        (f64 arithmetic)
 * cov [rows][kstride][kstride] f64 device, entries a, b < k read; cov == NULL <=> out_var == NULL.
 * Outputs are f64 device arrays with row stride ld_out >= n_points.  y is not read.
 * Programs with k > VSR_MAX_DUAL: out_var row nan.  A pair's outputs do not depend on the other
 * pairs of the call, bit for bit. */
int vsr_predict(vsr_handle* h, const int32_t* prog_idx, const int32_t* const_row, int32_t n_pairs,
                const double* consts, int32_t kstride, const double* cov, int32_t dtype,
                double* out_value, double* out_var, int64_t ld_out, void* stream);

/* Multi-restart BFGS for n_runs (program, restart) runs; run r of the list fits program
 * run_prog[r] from x0[run_slot[r]] and writes every output at row run_slot[r]
 * (slots let a rank fit a shard of a C x R problem in place).  run_prog and run_slot
 * are HOST int32 arrays; everything else is device memory.  Replaces
 * scipy.optimize.minimize(safe_loss, x0, method='BFGS') (bfgs.py:115, :179), restart
 * seeding being an INPUT (bfgs.py:103 draws from an unseeded global RNG).
 *   x0, out_consts, out_lastx : [n_slots][kstride] f64   (out_lastx = last point the
 *                               objective saw = what the reference records, bfgs.py:116)
 *   out_loss      [n_slots] f64  objective at out_consts (scaled, penalty applied)
 *   out_final_mse [n_slots] f64  plain MSE at out_lastx in score_dtype (nan allowed); the mean of
 *                               w r^2 with weights, of C^2 rho(z) with a robust loss on the score slot
 * The sweeps read the eval slot's weights and robust loss (vsr_set_weights, vsr_set_loss).
 *   out_info      [n_slots][4] int32: status (VsrFitStatus), nit, nfev, reserved
 * Programs with k == 0 are not optimised: status VSR_FIT_NOT_RUN, final MSE only. */
int vsr_fit(vsr_handle* h, const int32_t* run_prog, const int32_t* run_slot, int32_t n_runs,
            const double* x0, int32_t kstride, const vsr_fit_opts* opts, double* out_consts,
            double* out_lastx, double* out_loss, double* out_final_mse, int32_t* out_info,
            void* stream);

/* The same fit with HOST buffers end to end: uploads x0 and the run list, fits,
 * copies every output back and synchronises the stream.  This is the call the
 * reference-side binding makes (INTEGRATION.md). */
int vsr_fit_host(vsr_handle* h, const int32_t* run_prog, const int32_t* run_slot,
                 int32_t n_runs, int32_t n_slots, const double* x0, int32_t kstride,
                 const vsr_fit_opts* opts, double* out_consts, double* out_lastx,
                 double* out_loss, double* out_final_mse, int32_t* out_info, void* stream);

/* Constraint mask of the beam search (SURVEY 8f row 1).  Replaces the per-step, per-beam host
 * loop of Model.fitfunc2 (src/visymre/architectures/model.py:385-411) and the Python stack walk
 * _analyze_prefix_tree_context (model.py:522-560).  Token sets are bit masks over token ids
 * (< 64); ids that do not exist are -1.
 *   generated [beam][ld] int64 device: the beams' token ids, cur_len of them valid
 *   beam_scores [beam] f32 device: beams below -1e8 get an all-zero row (model.py:387)
 *   out_mask [beam][n_words] f32 device: 0 or -inf, to be ADDED to the log-probabilities
 * Stateless: needs no handle. */
typedef struct vsr_beam_rules {
  uint64_t arity1, arity2;   /* unary / binary operator ids */
  uint64_t transcendental;   /* model.py: transcendental_ids (no nesting of these) */
  uint64_t all_ops;          /* forbidden once the open slots fill the remaining length */
  uint64_t masked_vars;      /* variables absent from the data (model.py: masked_var_ids) */
  int32_t pow_id, c_id, start_id, finish_id, pad_id;
  int32_t length_eq;         /* cfg.length_eq */
} vsr_beam_rules;
int vsr_beam_mask(const int64_t* generated_dev, int64_t ld, int32_t beam, int32_t cur_len,
                  const float* beam_scores_dev, const vsr_beam_rules* rules, int32_t n_words,
                  float* out_mask_dev, void* stream);

/* The same mask, INCREMENTALLY: the decode loop appends one token per beam per step, so the walk's
 * state (the open frames of the prefix tree) is kept on the device and a step consumes one token per
 * beam: O(open frames) instead of O(cur_len) per beam per step.  The caller owns the state arrays
 * (it re-orders their rows when the beam search re-orders the beams) and initialises a fresh beam to
 * depth = 1, op[0] = -1, missing[0] = 1, cons[0] = 0, pos = 0.
 *   op, missing [beam][max_depth] int8; cons [beam][max_depth] uint64; depth, pos [beam] int32
 *   tokens [beam] int64: the token appended to every beam at this step
 *   out_mask [beam][n_words]: the mask for the NEXT token (what vsr_beam_mask gives for the prefix
 *   extended by `tokens`); rows of beams with a score below -1e8 are all zero */
int vsr_beam_mask_step(int8_t* op_dev, int8_t* missing_dev, uint64_t* cons_dev, int32_t* depth_dev,
                       int32_t* pos_dev, int32_t max_depth, const int64_t* tokens_dev, int32_t beam,
                       const float* beam_scores_dev, const vsr_beam_rules* rules, int32_t n_words,
                       float* out_mask_dev, void* stream);

/* Number of kernels this handle has launched since creation (bench.py reports it). */
int64_t vsr_launch_count(const vsr_handle* h);

/* Measurement hooks (bench.py): with profiling on, vsr_fit brackets its fit-kernel
 * launches and its scoring launches with CUDA events on the caller's stream.
 * vsr_read_profile synchronises on those events, returns the accumulated
 *   out[0] fit-kernel milliseconds   out[1] number of fit-kernel launches
 *   out[2] scoring milliseconds      out[3] number of scoring launches
 * and resets the accumulators. */
int vsr_set_profiling(vsr_handle* h, int32_t on);
/* Optional: a device int64 buffer [n_slots][8]; the fit kernel then records, per run, the
 * SM cycles its leader thread spent in each phase of the pass loop (optimiser logic,
 * barriers, sweep, reductions) and the number of passes.  NULL switches it off. */
int vsr_set_phase_buffer(vsr_handle* h, void* dev_i64_nslots_by_8);
int vsr_read_profile(vsr_handle* h, double out[4]);
/* Measurement hook: overrides the launch geometry of vsr_fit -- cluster size, threads per CTA, runs
 * in flight per cluster ("seats") and optimiser warps of the leader CTA (< 0: none); 0 keeps the
 * built-in choice of that item.  The environment variable VSR_GEOMETRY="cluster:threads:seats:opt"
 * is read ONCE, by vsr_create, as the initial value. */
int vsr_set_geometry(vsr_handle* h, int32_t cluster, int32_t threads, int32_t seats, int32_t opt_warps);

#ifdef __cplusplus
}
#endif
#endif /* VSR_H_ */
