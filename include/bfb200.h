/*
 * bfb200.h -- C ABI of libbfb200.so, the B200 (sm_100a) implementation of BayesFast's hot path:
 * PolyModel surrogate fit + value/gradient evaluation inside lock-step NUTS/HMC.
 *
 * The reference (h3jia/bayesfast) is pure Python + Cython and has no FFI seam of its own; its seams are
 * Python duck types (SURVEY.md section 8b).  Each entry point below names the reference interface it
 * replaces (paths relative to the reference root); bayesfast_b200/_cabi.py is the ctypes binding and
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes, no exceptions; every function returns 0 on success and a
 * negative code on failure, with a message available from bfb_last_error() (thread-local).
 * All floating point data is IEEE double; matrices are row-major.  "loc" arguments say where caller
 * buffers live: BFB_HOST (pageable or pinned host memory) or BFB_DEVICE (device memory of the handle's GPU).
 * A handle owns one CUDA stream; calls on one handle are not thread-safe, different handles are independent.
 * There is no CPU fallback: if no CUDA device is usable bfb_create fails.
 */
#ifndef BFB200_H
#define BFB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BFB_HOST 0
#define BFB_DEVICE 1

#define BFB_OK 0
#define BFB_ERR_CUDA (-1)
#define BFB_ERR_ARG (-2)
#define BFB_ERR_STATE (-3)
#define BFB_ERR_NUMERIC (-4)

enum { BFB_LINEAR = 1, BFB_QUADRATIC = 2, BFB_CUBIC_2 = 3, BFB_CUBIC_3 = 4 };
enum { BFB_NUTS = 0, BFB_HMC = 1 };

typedef struct bfb_context *bfb_handle;

const char *bfb_last_error(void);
int bfb_version(void);
int bfb_device_count(void);

int bfb_create(int device, bfb_handle *out);
int bfb_destroy(bfb_handle h);
/* Use an existing CUDA stream (e.g. torch.cuda.current_stream().cuda_stream) instead of the handle's own. */
int bfb_set_stream(bfb_handle h, void *cuda_stream);
int bfb_synchronize(bfb_handle h);

/* ------------------------------------------------------------------------------------------------
 * Model: replaces the state of bayesfast.modules.poly.PolyModel (configs[i]._coef, _mu, _hess, _alpha,
 * _f_mu; poly.py:19-158, 262-292), the ModuleBase input rescale (core/module.py:47-96, 221-227) and,
 * for the sampler, the surrogate-only bayesfast.core.density.Density (decay: density.py:740-746, 796-811;
 * variable transform: transforms/_constraint.pyx).
 * Coefficients are passed PACKED, i.e. as the lstsq solution slices of poly.py:572-587: per config and per
 * output of that config, in config order: linear n_in+1 | quadratic n_in(n_in+1)/2 (k<=l) |
 * cubic-2 n_in^2 (k,l) | cubic-3 C(n_in,3) (k<l<p)  -- the column order of _poly.pyx:143-177.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n, m, n_config;
    const int32_t *cfg_order;     /* [n_config] BFB_LINEAR.. */
    const int32_t *cfg_n_in;      /* [n_config] */
    const int32_t *cfg_n_out;     /* [n_config] */
    const int64_t *cfg_in_mask;   /* concatenated, sorted unique per config */
    const int64_t *cfg_out_mask;  /* concatenated */
    const double *cfg_coef;       /* concatenated packed coefficients, [config][output-in-config][packed] */
    int32_t use_bound;            /* PolyModel._use_bound and not _all_linear */
    const double *mu;             /* [n] */
    const double *hess;           /* [n,n] */
    double alpha;
    const double *f_mu;           /* [m] */
    int32_t use_scales;           /* module-level input_scales */
    const double *s0, *sdiff;     /* [n] */
    int32_t use_decay;
    const double *d_mu, *d_hess;  /* [n], [n,n] */
    double d_alpha2, d_gamma;
    int32_t use_transform;        /* Density.input_scales is not None */
    const double *ranges;         /* [n,2] */
    const uint8_t *hard_bounds;   /* [n,2] */
} bfb_model_desc;

int bfb_set_model(bfb_handle h, const bfb_model_desc *desc);

/* PolyModel.fun_and_jac for C points (module rescale included): replaces poly.py:443-503 called through
 * core/module.py:221-227.  X [C,n] -> F [C,m], J [C,m,n] (J may be NULL). */
int bfb_poly_eval_batch(bfb_handle h, const double *X, int64_t C, double *F, double *J, int loc);

/* Density.logp_and_grad(x, original_space=False, use_surrogate=True) for C points of the TRANSFORMED space:
 * replaces core/density.py:724-754 (+ Pipeline.fun_and_jac :487-566) for a surrogate-only density whose
 * logp is output 0 of the PolyModel.  X [C,n] -> logp [C], grad [C,n]. */
int bfb_logp_and_grad_batch(bfb_handle h, const double *X, int64_t C, double *logp, double *grad, int loc);
/* which evaluator served the last bfb_logp_and_grad_batch: 0 = generic warp-per-point (bfb_eval.cuh), 2 = FP64 tensor core
 * (bfb_eval_dmma.cu), 3 = tensor-core likelihood pipeline (bfb_lik_dmma.cu); -1 before the first call */
int bfb_eval_last_path(bfb_handle h);

/* Second module of a two-module pipeline (core/density.py:487-566; examples/2d-donut.ipynb f_1, the chi^2 module of
 * examples/des-y1-w-cosmosis.ipynb): kind 1 = Gaussian likelihood logp = c0 - 1/2 sum_o f_o^2 of the m outputs of the model
 * set with bfb_set_model, pre-whitened by the caller (bayesfast_b200/density.py: whiten_spec); kind 0 removes it.
 * Density-level calls (bfb_logp_and_grad_batch, the samplers) then evaluate the pipeline; bfb_poly_eval_batch still
 * returns the (whitened) outputs.  bfb_set_model / bfb_fit_solve reset it. */
int bfb_set_epilogue(bfb_handle h, int kind, double c0);
/* Third module of the DES-Y1 example's pipeline (examples/des-y1-w-cosmosis.ipynb cells 12-14, des_post_f / des_post_fj:
 * logp = like + prior(x), a user Module with inputs ['like', 'x'] in the reference): independent Gaussian prior on the
 * ORIGINAL-space inputs, logp += c0 - 1/2 sum_j w[j] (x_j - mu[j])^2, w [n] = 1 / sigma^2 (0: no prior on that input),
 * mu [n]; host pointers; w == NULL removes it.  After bfb_set_model, before bfb_set_epilogue. */
int bfb_set_prior(bfb_handle h, const double *w, const double *mu, double c0);

/* ------------------------------------------------------------------------------------------------
 * Fit: replaces PolyModel.fit (poly.py:505-589): the design-matrix builders _lsq_* (_poly.pyx:143-177),
 * scipy.linalg.lstsq (poly.py:570) and _set_bound (poly.py:262-292).  One design matrix per recipe row
 * is shared by all outputs that use the same configs.
 * Rows may be accumulated in several calls (and on several GPUs: bfb_fit_export/import carry the
 * packed partial sums through an all-reduce).  The model set by bfb_set_model supplies the configs
 * (coefficients there are ignored).  y [N,m]; w NULL or [N] (rows are scaled by w like poly.py:566-568).
 * Limits, checked by bfb_fit_begin (BFB_ERR_ARG): input_size <= 128, the evaluators' limit, and P <= 16384 parameters per
 * output (the configs serving one output together): full quadratic models up to n = 128 (P = 8385), cubic-2 up to n = 104
 * (P = 16381), cubic-3 up to n = 44 (P = 16215).  The bound and decay ellipsoids (bfb_fit_moments, bfb_fit_max_beta) take
 * input_size <= 128.
 * ---------------------------------------------------------------------------------------------- */
int bfb_fit_begin(bfb_handle h, const double *shift /* [n] or NULL: reference point of the shifted moments, identical on all ranks */);
int bfb_fit_accumulate(bfb_handle h, const double *x, const double *y, const double *w, int64_t N, int loc);
/* number of doubles in the partial-sum buffer (Gram blocks, X^T y, moments) */
int64_t bfb_fit_buffer_size(bfb_handle h);
/* device pointer of that buffer (for an in-place NCCL all-reduce by the host framework) */
int bfb_fit_buffer(bfb_handle h, double **dev_ptr);
/* The exchange step of a fit whose rows are sharded over GPUs (replaces nothing in the reference: its fit is single-process,
 * modules/poly.py:505-589): pack the partial sums -- the upper block triangle of every Gram, X^T y, the shifted moments, the
 * row count -- into ONE contiguous device buffer of *len doubles (10.6 MB at P = 1585), all-reduce it (sum) over the ranks
 * (NCCL on *dev_ptr; or staged through the host with bfb_fit_exchange_host, dir 0 device -> host, 1 host -> device), unpack. */
int bfb_fit_exchange_pack(bfb_handle h, double **dev_ptr, int64_t *len);
int bfb_fit_exchange_host(bfb_handle h, double *host, int dir);
int bfb_fit_exchange_unpack(bfb_handle h);
/* solve the normal equations (equilibrated Cholesky + refinement), write packed coefficients in the
 * layout of bfb_model_desc.cfg_coef; also installs them into the handle's model. */
int bfb_fit_solve(bfb_handle h, double *coef_out, double *rel_resid);
/* _set_bound pieces: mean and covariance^-1 of the accumulated x (unweighted), max Mahalanobis radius of
 * the rows given here (second pass), all reductions on device. */
int bfb_fit_moments(bfb_handle h, double *mu, double *cov);
int bfb_fit_max_beta(bfb_handle h, const double *x, int64_t N, const double *mu, const double *hess,
                     double *max_beta, double *beta_out /* NULL or [N] */, int loc);

/* ------------------------------------------------------------------------------------------------
 * Sampler: replaces bayesfast.core.sample.sample()'s worker pool (core/sample.py:165-214,
 * utils/parallel.py:130-150) and NUTS/HMC.run (samplers/hmc_utils/base_hmc.py:62-172, samplers/nuts.py,
 * samplers/hmc.py, hmc_utils/integration.py, metrics.py, step_size.py) for C chains at once (eight chains per warp on the
 * FP64 tensor cores for input_size <= 32 without multi-output / n > 28 cubic-3 models; one warp per chain otherwise).
 * Random stream: include/bfb_rng.h, chain ids chain0 .. chain0+C-1.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_warmup, max_treedepth, n_int_step;
    double max_change;
    int32_t adapt_step_size;
    double target_accept, gamma, k, t0;
    int32_t adapt_metric;
    double initial_weight;
    int32_t adapt_window, update_window, doubling;
    uint64_t seed;
    int64_t chain0;
} bfb_sampler_cfg;

/* Outputs of one bfb_sampler_run call, chain-major [C, n_iter(, n)]; any pointer may be NULL. */
typedef struct {
    double *samples;
    double *logp, *energy, *mean_tree_accept, *step_size, *step_size_bar, *energy_change, *max_energy_change;
    int32_t *tree_depth, *tree_size, *diverging;  /* HMC: tree_depth = accepted, tree_size = n_int_step */
} bfb_run_out;

/* x0 [C,n] (transformed space), step0 [C] (DualAverageAdaptation initial_step, i.e. already / n^0.25,
 * sample_trace.py:365-373), var0 [C,n], mean0 [C,n] (initial_mean, sample_trace.py:437-444). Host pointers. */
int bfb_sampler_init(bfb_handle h, const bfb_sampler_cfg *cfg, int64_t C, const double *x0,
                     const double *step0, const double *var0, const double *mean0);
/* Dense mass matrix: replaces QuadMetricFull / QuadMetricFullAdapt (samplers/hmc_utils/metrics.py:94-132, 240-330,
 * 374-417; NTrace(metric='full') or a covariance, samplers/sample_trace.py:430-453).  cov0 [C,n,n] initial covariances
 * (positive definite, else BFB_ERR_ARG like metrics.py:105-106); everything else as bfb_sampler_init.  The chains then run
 * on the generic warp-per-chain kernel.  bfb_sampler_get_cov: final covariances [C,n,n] and per-chain flag "a Cholesky
 * factorisation failed during adaptation" (metrics.py:284-287); host pointers, either may be NULL. */
int bfb_sampler_init_dense(bfb_handle h, const bfb_sampler_cfg *cfg, int64_t C, const double *x0,
                           const double *step0, const double *cov0, const double *mean0);
int bfb_sampler_get_cov(bfb_handle h, double *cov, int32_t *chol_error);
/* restore every chain to its state right after bfb_sampler_init (device-to-device copies only) */
int bfb_sampler_reset(bfb_handle h);
/* advance every chain by n_iter iterations; out pointers in `loc`; total_tree_size (host, may be NULL) =
 * sum over chains and iterations of tree_size = leapfrog steps performed in trees. */
int bfb_sampler_run(bfb_handle h, int sampler, int32_t n_iter, const bfb_run_out *out, int loc,
                    int64_t *total_tree_size);
/* Reduced outputs: what SampleTrace.get hands to its callers (samplers/sample_trace.py:762-787: the samples after
 * warm-up, flattened) instead of every record of every iteration -- a 4096 x 1500 run at n = 26 is 1.7 GB per GPU otherwise.
 * skip: the records of the first `skip` iterations of this call are not written at all; thin >= 1: of the following
 * iterations every thin-th is kept, the out arrays are then [C, n_keep(, n)] with n_keep = ceil((n_iter - skip) / thin)
 * (host outputs only for thin > 1); mean [n] / cov [n,n] (host, may be NULL): mean and unbiased covariance (np.cov) of the
 * samples of ALL iterations after `skip` over all chains, accumulated on the device.  opts == NULL: bfb_sampler_run.
 * diag [n, (n_iter - diag_from) / 2 + 3] (host, may be NULL): the partials of bfb_chain_diagnostics over the samples of iterations
 * diag_from .. n_iter - 1 of this call, whatever skip, thin and out ask for; skip <= diag_from <= n_iter - 4.  They are computed on
 * the device from the buffer the samples are staged in, or from one [C, n_iter - diag_from, n] buffer that holds them otherwise
 * (BFB_ERR_CUDA naming the size when it cannot be allocated). */
typedef struct {
    int32_t skip, thin;
    double *mean, *cov;
    int32_t diag_from;
    double *diag;
} bfb_run_opts;
int bfb_sampler_run_ex(bfb_handle h, int sampler, int32_t n_iter, const bfb_run_out *out, int loc,
                       const bfb_run_opts *opts, int64_t *total_tree_size);
/* Tempered samplers: replace TNUTS / THMC (samplers/tnuts.py, thmc.py), BaseTHMC.astep (samplers/hmc_utils/base_hmc.py:220-262)
 * and TCpuLeapfrogIntegrator (samplers/hmc_utils/integration.py:98-222) for C chains at once.  The Hamiltonian lives on (u, q) with
 * potential beta(u) phi(q) + (1 - beta(u)) psi(q) + U(u), phi = -logp of h's model, psi = -(logp of h_base's model + logxi)
 * (TNTrace.density_base / logxi, samplers/sample_trace.py:540-567); h_base is a second handle on the same device that must outlive
 * the run.  u0 [C] (host): the tempering variable of the first iteration (the reference draws it from numpy's global generator,
 * base_hmc.py:242).  Everything else as bfb_sampler_init (diagonal metric only); draw order per iteration: n normals (momentum),
 * 1 normal (momentum of u), then as NUTS / HMC.  bfb_tsampler_run: sampler = BFB_NUTS (TNUTS) or BFB_HMC (THMC); u / weight
 * [C, n_iter] = the stats 'u' and 'weight' (stats.py TNStepStats / THStepStats), the rest as bfb_sampler_run; pointers in `loc`,
 * any may be NULL.  Runs on a warp-per-chain kernel (bfb_sampler_tempered.cu); bfb_sampler_reset / bfb_sampler_get_state apply. */
int bfb_tsampler_init(bfb_handle h, bfb_handle h_base, double logxi, const bfb_sampler_cfg *cfg, int64_t C, const double *x0,
                      const double *u0, const double *step0, const double *var0, const double *mean0);
int bfb_tsampler_run(bfb_handle h, int sampler, int32_t n_iter, const bfb_run_out *out, double *u, double *weight, int loc,
                     int64_t *total_tree_size);
/* which kernel family ran the last bfb_sampler_run / bfb_tsampler_run of this handle: 0 = warp-per-chain (bfb_sampler.cu,
 * bfb_sampler_tempered.cu), 2 = FP64 tensor core, one warp per 8 chains (bfb_sampler_dmma.cu), 3 = tensor core, four-warp team per
 * 8 chains (bfb_sampler_team.cu; NUTS for 32 < n <= 64 only), 4 = tensor core, integrator warp + tree warp (bfb_sampler_pair.cu,
 * NUTS only); -1 before the first run.  The environment variable BFB200_SAMPLER = dmma | team | pair | generic pins one (tests,
 * profiles); bfb_sampler_run fails with BFB_ERR_ARG when the pinned family cannot run the model. */
int bfb_sampler_last_path(bfb_handle h);
/* page-locked host memory for the outputs of bfb_sampler_run: with it the device-to-host copies of one chunk of
 * iterations overlap the kernel of the next chunk */
int bfb_host_alloc(size_t bytes, void **ptr);
int bfb_host_free(void *ptr);
/* final adaptation state for the host-side trace objects: final_step [C,4] = log_step, log_bar, hbar, count;
 * final_var [C,n]; n_draws [C]; status [C] (0 ok, 1 non-finite logp/grad at x0, 2 non-finite start energy,
 * 3 nan in logbern); q [C,n] current position.  Host pointers, any may be NULL. */
int bfb_sampler_get_state(bfb_handle h, double *final_step, double *final_var, int64_t *n_draws,
                          int32_t *status, double *q);
/* The steps on either side of the sampler inside Recipe._sam_step / _pos_step on device-resident (loc == BFB_DEVICE) or host
 * arrays (SURVEY.md 8f rank 2):
 * bfb_importance_weights -- PostStep, core/recipe.py:1286-1297: weights [N] = exp(logp - logq), weights_trunc [N] =
 *   clip(weights, 0, mean(weights) * N^k_trunc) (k_trunc < 0: no truncation); either output may be NULL; stats [5] (host, may be
 *   NULL) = sum weights | cap | sum weights_trunc | sum weights_trunc^2 | max weights_trunc.
 * bfb_argsort_gather -- SystematicResampler.run, utils/misc.py:62-108: out[i] = argsort(a)[pos[i]] for the n systematic positions
 *   pos (which the host mirror computes exactly like the reference's np.linspace(...).astype(int)); ties are ordered by index,
 *   NaN sorts last; N < 2^31. */
int bfb_importance_weights(bfb_handle h, const double *logp, const double *logq, int64_t N, double k_trunc,
                           double *weights, double *weights_trunc, double *stats, int loc);
int bfb_argsort_gather(bfb_handle h, const double *a, int64_t N, const int64_t *pos, int64_t n, int64_t *out, int loc);
/* Convergence diagnostics of sampled chains (replaces nothing in the reference, which leaves them to the caller; the definitions are
 * those of Stan's and ArviZ's non-rank-normalised split-R-hat and ESS, bayesfast_b200/diag.py): x [C, T_total, n] in `loc`, draws
 * t0 .. t0 + N - 1 of every chain (N >= 4), split into M' = 2 C half-chains of L = N / 2 draws.  partials [n, L + 3] (host) per
 * coordinate: M' | mean of the half-chain means | sum of their squared deviations from it | the lag sums S(k) = sum over half-chains
 * of sum_t y[t] y[t + k], k = 0 .. L - 1, of the centred half-chains y.  All are sums over chains: shards of chains combine with a
 * pairwise (Chan) update of the first three and a sum of the rest.  The lag sums run on the FP64 tensor cores; repeated calls are
 * bit-identical. */
int bfb_chain_diagnostics(bfb_handle h, const double *x, int64_t C, int64_t T_total, int64_t t0, int64_t N, int n, int loc,
                          double *partials);
/* device time of the last bfb_sampler_run / bfb_fit_accumulate / bfb_poly_eval_batch / bfb_chain_diagnostics kernel(s), CUDA events
 * on the handle's stream, milliseconds */
int bfb_last_kernel_ms(bfb_handle h, float *ms);
/* number of kernels launched by this handle since creation */
int64_t bfb_launch_count(bfb_handle h);

/* draws t0..t0+count-1 of the stream (seed, chain) computed ON THE DEVICE: u (uniform view) and z (normal
 * view).  Host pointers.  Used by the parity tests to teacher-force the oracle. */
int bfb_rng_fill(bfb_handle h, uint64_t seed, uint64_t chain, uint64_t t0, int64_t count, double *u, double *z);
/* Phi^-1 of count probabilities p in (0, 1) computed ON THE DEVICE, twice: z by the restatement the tensor-core samplers
 * draw their momenta with, z_ref by bfb_norminv of bfb_rng.h.  Host pointers.  The two must agree bit for bit. */
int bfb_norminv_fill(bfb_handle h, const double *p, int64_t count, double *z, double *z_ref);

/* FP64 peak microbenchmarks for the roofline denominator (MEASURED_PEAKS.json has no FP64 entry):
 * kind 0 = DFMA, 1 = DMMA m8n8k4, 2 = both interleaved.  Returns TFLOP/s. */
int bfb_fp64_peak(bfb_handle h, int kind, double *tflops);
/* cycles one warp needs per dependent-free m8n8k4 DMMA with `nacc` (1, 2, 4, 8 or 15) independent accumulators, B operand
 * from registers (src 0) or one shared-memory load per DMMA (src 1), `warps_per_sm` (4 or 8) resident warps: the issue
 * model behind the tensor-core sampler (DESIGN.md 4.1). */
int bfb_dmma_issue_test(bfb_handle h, int nacc, int src, int warps_per_sm, double *cycles_per_dmma);

#ifdef __cplusplus
}
#endif
#endif
