// bfb_common.cuh -- shared declarations of libbfb200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/bfb200.h"
#include "../../include/bfb_rng.h"

#define BFB_NSTAGE 3    // device staging buffers of the host-output pipeline of bfb_sampler_run
#define BFB_WARP 32
#define BFB_FULL 0xffffffffu
// ChainState::tree_total: [0] leapfrogs in trees, [1..19] round / section counters and cycle sums of the timing builds
#define BFB_TREE_TOTAL_LEN 20

void bfb_set_error(const char *fmt, ...);

#define BFB_CUDA(call)                                                                           \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            bfb_set_error("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__));   \
            return BFB_ERR_CUDA;                                                                 \
        }                                                                                        \
    } while (0)

#define BFB_REQUIRE(cond, code, ...)                                                             \
    do {                                                                                         \
        if (!(cond)) { bfb_set_error(__VA_ARGS__); return (code); }                              \
    } while (0)

// ----------------------------------------------------------------------------------------------
// Device-side model tables.  Every output o of the PolyModel is flattened on the host into a full-n
// polynomial (masked configs scattered into full tensors, zeros elsewhere), so one evaluator serves
// masks, multiple configs and multiple outputs.  Matrices are stored "k-major": T[k][j] with the lane
// index j contiguous and padded to np = 32*ceil(n/32) columns (zeros), so lane j reads T[k*np + j].
// ----------------------------------------------------------------------------------------------
struct DevModel {
    int n, np, m;
    int has_quad, has_c2, has_c3;
    const double *c0;    // [m]
    const double *lin;   // [m][np]
    const double *S;     // [m][n][np]   symmetrised quadratic: S[k][j] = a_kj (k<j), 2 a_jj, a_jk (k>j)
    const double *A1T;   // [m][n][np]   A1T[k][j] = A[j][k]     (t_j = sum_k A[j][k] x_k)
    const double *A2;    // [m][n][np]   A2[k][j]  = A[k][j]     (u_j = sum_k A[k][j] x_k^2)
    const double *c3;    // [m][C(n,3)]  packed j<k<l
    int64_t n_c3;
    const int *c3_row;   // [n][n]  offset of the packed row (j, k), j < k < n - 1, i.e. of a_(j,k,k+1); -1 elsewhere
    int use_bound;
    const double *mu;    // [np]
    const double *HT;    // [n][np]  HT[k][j] = H[j][k]
    double alpha;
    const double *f_mu;  // [m]
    int use_scales;
    const double *s0, *sdiff;   // [np] (sdiff padded with 1)
    int use_decay;
    const double *d_mu;  // [np]
    const double *d_H;   // [n][np]  d_H[k][j] = Hd[k][j]
    double d_alpha2, d_gamma;
    int use_transform;
    const double *r_lo, *r_w;   // [np] ranges[:,0], ranges[:,1]-ranges[:,0]
    const int *hb;       // [np] bit0 = lower bound hard, bit1 = upper bound hard
    // DMMA operand table of output 0 (bfb_dmma.cuh): bfrag[kt][tile][lane]; frag_nr = 0 when the model does not qualify
    const double *bfrag;
    int frag_nr, frag_nt, frag_ext;
    // operand table of the four-warp team evaluator (bfb_team.cuh): tfrag[w][kt][tile][lane]; null when the model does not qualify
    const double *tfrag;
    int team_nr;         // dimensions per lane-quad of the team tables: frag_nr for n <= 32, 16 for 32 < n <= 64 (team kernels only)
    // cubic-3 block of the team evaluator: tfrag3[kt][warp][tile][lane] (streamed from L2), pair table tpair[4 kt] = k | l << 8,
    // t3_kt k-tiles (padded to a multiple of 8)
    const double *tfrag3;
    const int *tpair;
    int t3_kt;
    // cubic-3 block of the tensor-core evaluator: operand table bfrag3[kt][tile][lane], pair table c3pair[4 kt] = k | l << 8
    const double *bfrag3;
    const int *c3pair;
    int c3_kt, c3_n3t;
    // second module of the pipeline (bfb_set_epilogue): 1 = Gaussian likelihood of the m (pre-whitened) outputs,
    // logp = e_c0 - 1/2 sum_o f_o^2
    int epilogue;
    double e_c0;
    // operand table of the tensor-core likelihood pipeline (bfb_lik_dmma.cu: one record per output), or null
    const double *lik_tab;
    int lik_nr;
    // feature form of the likelihood pipeline (model variant bit 4, bfb_dmma.cuh): outputs = Phi(x) C^T over the features
    // 1 | x_j | x_a x_b (a <= b in the UNION of the quadratic configs' masks); records of 8 outputs, feature / gradient tables
    const double *lik_ftab;
    const int *lik_fpt;  // [4 KT1][2] feature -> (a, b): -1,-1 constant; a,-1 linear; a,b product; -2,-2 padding
    const int *lik_fgt;  // [32][1 + 3 QMAX] per dimension: count, then (feature index, partner dimension, factor) triples
    int lik_kt1, lik_nt2, lik_nt1, lik_frec;
    int lik_ext;         // the pipeline has a radial bound / module rescale / variable transform / prior: model variant bits 3 | 1
    // third module of the pipeline (bfb_set_prior): independent Gaussian prior on the original-space inputs,
    // logp += p_c0 - 1/2 sum_j p_w[j] (x_j - p_mu[j])^2
    int use_prior;
    const double *p_w, *p_mu;   // [np]
    double p_c0;
};

struct HostConfig {
    int order, n_in, n_out;
    std::vector<int64_t> in_mask, out_mask;
    int64_t coef_off;   // offset of this config's packed coefficients in the concatenated buffer
    int64_t n_packed;   // packed coefficients per output
};

// Chain state kept on the device between bfb_sampler_run calls (SoA, chain-major).
struct ChainState {
    int64_t C;
    int n, np;
    double *q;        // [C][np]
    double *logp;     // [C]  cached logp at q
    double *g;        // [C][np] cached grad at q
    double *var;      // [C][np]
    double *fg_mean, *fg_raw, *bg_mean, *bg_raw;   // [C][np]
    double *fg_n, *bg_n;                             // [C]
    double *log_step, *log_bar, *hbar, *mu_da;       // [C]
    int64_t *count;                                  // [C]
    int64_t *n_samples, *previous_update;            // [C]
    int32_t *adapt_window;                           // [C]
    int64_t *t_draw;                                 // [C]
    int64_t *iter;                                   // [C] iterations done
    int32_t *status;                                 // [C]
    unsigned long long *tree_total;                  // [BFB_TREE_TOTAL_LEN]: leapfrogs in trees; debug counters of the multi-chain kernels
    // dense mass matrix (bfb_sampler_init_dense; generic kernel only): [C][n][np], transposed XT[k][j] = X[j][k]
    double *covT, *cholT, *cholW, *fgcT, *bgcT;      // covariance, its Cholesky factor (+ work copy), Welford fore/background
    int32_t *chol_error;                             // [C]
};

struct FitState;

struct bfb_context {
    int device;
    cudaStream_t stream;
    bool own_stream;
    cudaEvent_t ev0, ev1;
    float last_ms;
    int64_t launches;
    int sm_count;
    // model
    bool has_model;
    int n, m, np;
    std::vector<HostConfig> configs;
    std::vector<double> packed;          // host copy of packed coefficients
    bfb_model_desc desc_flags;           // scalar flags only (pointers invalid)
    std::vector<double> h_mu, h_hess, h_fmu, h_s0, h_sdiff, h_dmu, h_dhess, h_ranges, h_pw, h_pmu;
    double h_pc0;
    std::vector<uint8_t> h_hb;
    std::vector<void *> model_allocs;
    DevModel dm;
    // sampler
    bool has_chains;
    bool dense_metric;         // chains were set up by bfb_sampler_init_dense
    std::vector<void *> dense_allocs;
    bfb_sampler_cfg scfg;
    ChainState cs;
    std::vector<void *> chain_allocs;
    std::vector<void *> chain_snapshot;
    int64_t alloc_C;           // shape the chain arrays were allocated for (reused by bfb_sampler_init)
    int alloc_np;
    cudaStream_t copy_stream;  // device-to-host output pipeline of bfb_sampler_run
    cudaEvent_t ev_k[BFB_NSTAGE], ev_c[BFB_NSTAGE];
    void *stage[BFB_NSTAGE];
    size_t stage_len[BFB_NSTAGE];
    int *queue;                // work queue of the multi-chain kernel
    size_t queue_len;
    int last_path;             // kernel family of the last sampler launch: 0 generic, 2 dmma, 3 team, 4 pair (bfb_sampler.cu: FAM_*)
    int64_t iters_done;        // iterations completed by every chain since bfb_sampler_init / reset
    double *lik_tab;           // operand table of the tensor-core likelihood evaluator (bfb_lik_dmma.cu), or null
    int lik_nr;
    int last_eval_path;        // evaluator of the last bfb_logp_and_grad_batch: 0 generic, 2 tensor core, 3 tensor-core likelihood pipeline
    double *gstack;            // deep NUTS stack levels of the multi-chain kernel (L2 resident)
    size_t gstack_len;
    // progress reporting of a single-launch run (bfb_sampler_run_ex, host outputs): the kernel counts the groups that finished
    // iteration chunk k in a block behind its work queue; the last one writes k + 1 to *progress_host (mapped pinned memory), and
    // the host thread starts the device-to-host copy of that chunk while the kernel goes on
    int *progress_host;        // host address of the flag; progress_host_dev = the same word as seen from the device
    int *progress_host_dev;
    int progress_arm;          // > 0: the next NUTS launch should report progress in about this many chunks
    int progress_chunk_iters;  // set by the launcher that honoured the request (0: not honoured)
    int progress_n_chunks;
    // tempered samplers (bfb_sampler_tempered.cu): handle of the base density, log xi, tempering variable [C] current | [C] initial
    const bfb_context *t_base;
    double t_logxi;
    double *t_u;
    // fit
    FitState *fit;
    // chain diagnostics (bfb_diag.cu): device workspace, grown on demand
    double *diag_ws;
    size_t diag_ws_len;
};

int bfb_upload_model(bfb_context *h);          // (re)build the device tables from configs/packed
void bfb_free_list(std::vector<void *> &v);
// queue the split-R-hat / ESS partials of device draws x [C, T, n], kept range t0 .. t0 + N, on h->stream (bfb_diag.cu)
int bfb_diag_enqueue(bfb_context *h, const double *x, int64_t C, int64_t T, int64_t t0, int64_t N, int n, const double **dev_partials);

// ----------------------------------------------------------------------------------------------
// warp helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(BFB_FULL, v, o);
    return v;   // butterfly: bitwise identical on every lane
}

__device__ __forceinline__ double np_logaddexp(double a, double b)
{
    // numpy's logaddexp (the reference: nuts.py:85,163)
    if (a == b) return a + 0.6931471805599453;
    double tmp = a - b;
    if (tmp > 0) return a + log1p(exp(-tmp));
    else if (tmp <= 0) return b + log1p(exp(tmp));
    return tmp;
}
