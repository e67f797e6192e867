// bfb_model.cu -- handle life cycle, model upload (host-side flattening into device tables),
// batched evaluation entry points, RNG exposure.
#include "bfb_common.cuh"
#include "bfb_eval.cuh"
#include "bfb_team.cuh"
int bfb_launch_eval_dmma(bfb_context *h, const double *X, int64_t C, double *LP, double *G);
int bfb_launch_eval_team(bfb_context *h, const double *X, int64_t C, double *LP, double *G);    // bfb_eval_team.cu: 32 < n <= 64
int bfb_launch_lik_dmma(bfb_context *h, const double *X, int64_t C, double *LP, double *G);   // bfb_lik_dmma.cu
int bfb_build_lik_table(bfb_context *h);
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>

static thread_local char g_err[1024] = "";

void bfb_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *bfb_last_error(void) { return g_err; }
extern "C" int bfb_version(void) { return 100; }

extern "C" int bfb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void bfb_free_list(std::vector<void *> &v)
{
    for (void *p : v) cudaFree(p);
    v.clear();
}

void bfb_fit_free(bfb_context *h);

extern "C" int bfb_create(int device, bfb_handle *out)
{
    BFB_REQUIRE(out != nullptr, BFB_ERR_ARG, "bfb_create: out is NULL");
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) {
        bfb_set_error("bfb_create: no CUDA device available (%s); libbfb200 has no CPU fallback",
                      e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        cudaGetLastError();
        return BFB_ERR_CUDA;
    }
    BFB_REQUIRE(device >= 0 && device < cnt, BFB_ERR_ARG, "bfb_create: device %d out of range [0,%d)", device, cnt);
    BFB_CUDA(cudaSetDevice(device));
    bfb_context *h = new bfb_context();
    h->device = device;
    h->own_stream = true;
    h->last_ms = 0.f;
    h->launches = 0;
    h->has_model = false;
    h->has_chains = false;
    h->dense_metric = false;
    h->lik_tab = nullptr; h->lik_nr = 0; h->last_eval_path = -1;
    h->fit = nullptr;
    h->diag_ws = nullptr; h->diag_ws_len = 0;
    h->t_base = nullptr; h->t_logxi = 0.; h->t_u = nullptr;
    h->gstack = nullptr;
    h->gstack_len = 0;
    h->progress_host = nullptr; h->progress_host_dev = nullptr;
    h->progress_arm = 0; h->progress_chunk_iters = 0; h->progress_n_chunks = 0;
    h->copy_stream = nullptr;
    h->queue = nullptr;
    h->queue_len = 0;
    h->iters_done = 0;
    h->last_path = -1;
    h->alloc_C = 0; h->alloc_np = 0;
    for (int i = 0; i < BFB_NSTAGE; ++i) { h->stage[i] = nullptr; h->stage_len[i] = 0; }
    memset(&h->dm, 0, sizeof(h->dm));
    memset(&h->cs, 0, sizeof(h->cs));
    BFB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    BFB_CUDA(cudaEventCreate(&h->ev0));
    BFB_CUDA(cudaEventCreate(&h->ev1));
    cudaDeviceProp prop;
    BFB_CUDA(cudaGetDeviceProperties(&prop, device));
    h->sm_count = prop.multiProcessorCount;
    *out = h;
    return BFB_OK;
}

extern "C" int bfb_destroy(bfb_handle h)
{
    if (!h) return BFB_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    bfb_free_list(h->model_allocs);
    bfb_free_list(h->chain_allocs);
    bfb_free_list(h->dense_allocs);
    bfb_fit_free(h);
    if (h->gstack) cudaFree(h->gstack);
    if (h->diag_ws) cudaFree(h->diag_ws);
    if (h->t_u) cudaFree(h->t_u);
    if (h->queue) cudaFree(h->queue);
    if (h->progress_host) cudaFreeHost(h->progress_host);
    for (int i = 0; i < BFB_NSTAGE; ++i) if (h->stage[i]) cudaFree(h->stage[i]);
    if (h->copy_stream) {
        for (int i = 0; i < BFB_NSTAGE; ++i) { cudaEventDestroy(h->ev_k[i]); cudaEventDestroy(h->ev_c[i]); }
        cudaStreamDestroy(h->copy_stream);
    }
    cudaEventDestroy(h->ev0);
    cudaEventDestroy(h->ev1);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
    return BFB_OK;
}

extern "C" int bfb_set_stream(bfb_handle h, void *cuda_stream)
{
    BFB_REQUIRE(h, BFB_ERR_ARG, "null handle");
    BFB_CUDA(cudaSetDevice(h->device));
    if (h->own_stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); h->own_stream = false; }
    h->stream = (cudaStream_t)cuda_stream;
    return BFB_OK;
}

extern "C" int bfb_synchronize(bfb_handle h)
{
    BFB_REQUIRE(h, BFB_ERR_ARG, "null handle");
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    return BFB_OK;
}

extern "C" int bfb_last_kernel_ms(bfb_handle h, float *ms)
{
    BFB_REQUIRE(h && ms, BFB_ERR_ARG, "null argument");
    *ms = h->last_ms;
    return BFB_OK;
}

extern "C" int64_t bfb_launch_count(bfb_handle h) { return h ? h->launches : 0; }

// ----------------------------------------------------------------------------------------------
// model
// ----------------------------------------------------------------------------------------------
static int64_t packed_size(int order, int64_t ni)
{
    switch (order) {
    case BFB_LINEAR: return ni + 1;
    case BFB_QUADRATIC: return ni * (ni + 1) / 2;
    case BFB_CUBIC_2: return ni * ni;
    case BFB_CUBIC_3: return ni * (ni - 1) * (ni - 2) / 6;
    }
    return -1;
}

static int64_t c3_index_host(int a, int b, int c, int n)
{
    int64_t na = n - a;
    int64_t before_a = ((int64_t)n * (n - 1) * (n - 2) - na * (na - 1) * (na - 2)) / 6;
    int64_t nb = n - b;
    int64_t before_b = ((na - 1) * (na - 2) - nb * (nb - 1)) / 2;
    return before_a + before_b + (c - b - 1);
}

template <class T>
static int upload(bfb_context *h, const std::vector<T> &v, const T **dst)
{
    void *p = nullptr;
    size_t bytes = sizeof(T) * (v.empty() ? 1 : v.size());
    BFB_CUDA(cudaMalloc(&p, bytes));
    h->model_allocs.push_back(p);
    if (!v.empty()) BFB_CUDA(cudaMemcpyAsync(p, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice, h->stream));
    *dst = (const T *)p;
    return BFB_OK;
}

int bfb_upload_model(bfb_context *h)
{
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    bfb_free_list(h->model_allocs);
    h->lik_tab = nullptr; h->lik_nr = 0;
    const int n = h->n, m = h->m, np = h->np;
    DevModel &D = h->dm;
    memset(&D, 0, sizeof(D));
    D.n = n; D.np = np; D.m = m;
    bool hq = false, h2 = false, h3 = false;
    for (auto &c : h->configs) {
        hq |= c.order == BFB_QUADRATIC; h2 |= c.order == BFB_CUBIC_2; h3 |= c.order == BFB_CUBIC_3;
    }
    D.has_quad = hq; D.has_c2 = h2; D.has_c3 = h3;
    int64_t nc3 = (int64_t)n * (n - 1) * (n - 2) / 6;
    D.n_c3 = nc3;
    std::vector<double> c0(m, 0.), lin((size_t)m * np, 0.), S, A1T, A2, c3;
    if (hq) S.assign((size_t)m * n * np, 0.);
    if (h2) { A1T.assign((size_t)m * n * np, 0.); A2.assign((size_t)m * n * np, 0.); }
    if (h3) c3.assign((size_t)m * (nc3 > 0 ? nc3 : 1), 0.);
    for (auto &c : h->configs) {
        const int ni = c.n_in;
        for (int q = 0; q < c.n_out; ++q) {
            const int o = (int)c.out_mask[q];
            const double *a = h->packed.data() + c.coef_off + (int64_t)q * c.n_packed;
            if (c.order == BFB_LINEAR) {
                c0[o] += a[0];
                for (int k = 0; k < ni; ++k) lin[(size_t)o * np + c.in_mask[k]] += a[1 + k];
            } else if (c.order == BFB_QUADRATIC) {
                int64_t idx = 0;
                double *So = S.data() + (size_t)o * n * np;
                for (int k = 0; k < ni; ++k)
                    for (int l = k; l < ni; ++l) {
                        double v = a[idx++];
                        int64_t K = c.in_mask[k], L = c.in_mask[l];
                        if (k == l) So[K * np + K] += 2. * v;
                        else { So[K * np + L] += v; So[L * np + K] += v; }
                    }
            } else if (c.order == BFB_CUBIC_2) {
                double *T1 = A1T.data() + (size_t)o * n * np, *T2 = A2.data() + (size_t)o * n * np;
                for (int k = 0; k < ni; ++k)
                    for (int l = 0; l < ni; ++l) {
                        double v = a[(int64_t)k * ni + l];
                        int64_t K = c.in_mask[k], L = c.in_mask[l];
                        T1[L * np + K] += v;   // A1T[k'][j] = A[j][k']
                        T2[K * np + L] += v;   // A2[k'][j]  = A[k'][j]
                    }
            } else {
                int64_t idx = 0;
                double *Co = c3.data() + (size_t)o * nc3;
                for (int k = 0; k < ni; ++k)
                    for (int l = k + 1; l < ni; ++l)
                        for (int p = l + 1; p < ni; ++p)
                            Co[c3_index_host((int)c.in_mask[k], (int)c.in_mask[l], (int)c.in_mask[p], n)] += a[idx++];
            }
        }
    }
    int rc;
    if ((rc = upload(h, c0, &D.c0))) return rc;
    if ((rc = upload(h, lin, &D.lin))) return rc;
    if ((rc = upload(h, S, &D.S))) return rc;
    if ((rc = upload(h, A1T, &D.A1T))) return rc;
    if ((rc = upload(h, A2, &D.A2))) return rc;
    if ((rc = upload(h, c3, &D.c3))) return rc;
    {
        std::vector<int> c3row(h3 ? (size_t)n * n : 1, -1);
        if (h3)
            for (int j = 0; j < n - 2; ++j)
                for (int k = j + 1; k < n - 1; ++k) c3row[(size_t)j * n + k] = (int)c3_index_host(j, k, k + 1, n);
        if ((rc = upload(h, c3row, &D.c3_row))) return rc;
    }

    const bfb_model_desc &F = h->desc_flags;
    auto pad = [&](const std::vector<double> &v, double fill) {
        std::vector<double> o(np, fill);
        for (int j = 0; j < n && j < (int)v.size(); ++j) o[j] = v[j];
        return o;
    };
    D.use_bound = F.use_bound; D.alpha = F.alpha;
    std::vector<double> DH((size_t)n * np, 0.);          // decay ellipsoid, d_H[k][j] = Hd[k][j]
    if (F.use_decay)
        for (int k = 0; k < n; ++k)
            for (int j = 0; j < n; ++j) DH[(size_t)k * np + j] = h->h_dhess[(size_t)k * n + j];
    {
        std::vector<double> HT((size_t)n * np, 0.);
        if (F.use_bound)
            for (int j = 0; j < n; ++j)
                for (int k = 0; k < n; ++k) HT[(size_t)k * np + j] = h->h_hess[(size_t)j * n + k];
        if ((rc = upload(h, pad(h->h_mu, 0.), &D.mu))) return rc;
        if ((rc = upload(h, HT, &D.HT))) return rc;
        // operand table of the team evaluator (bfb_team.cuh) for `nr` dimensions per lane-quad: warp w owns the rows r = NRW w + v
        auto build_team_table = [&](int nr) -> int {
            const bool c2 = h2;
            const int nrw = (nr + 3) / 4, ntw = bfb_team_tiles(nr, c2);
            const int TDw = (nrw + 1) / 2, TXw = c2 ? nrw : (nrw + 1) / 2;
            std::vector<double> tf((size_t)4 * nr * ntw * 32, 0.);
            for (int w = 0; w < 4; ++w)
                for (int kt = 0; kt < nr; ++kt)
                    for (int t = 0; t < ntw; ++t)
                        for (int lane = 0; lane < 32; ++lane) {
                            const int k = 4 * kt + (lane & 3), gid = lane >> 2, own = gid >> 1, e = gid & 1;
                            const std::vector<double> *T = nullptr;
                            int v;
                            if (t < TDw) { v = 2 * t + e; if (v < nrw) T = &HT; }
                            else if (t < TDw + TXw) { v = 2 * (t - TDw) + e; if (v < nrw) T = &S; else if (c2 && v < 2 * nrw) { T = &A1T; v -= nrw; } }
                            else { v = 2 * (t - TDw - TXw) + e; if (v < nrw) T = &A2; }
                            const int j = 4 * (nrw * w + v) + own;
                            if (T && !T->empty() && k < n && j < n) tf[(((size_t)w * nr + kt) * ntw + t) * 32 + lane] = (*T)[(size_t)k * np + j];
                        }
            const int rc_ = upload(h, tf, &D.tfrag);
            if (!rc_) D.team_nr = nr;
            return rc_;
        };
        // operand table of the tensor-core evaluator (bfb_dmma.cuh), output 0
        const int nr = bfb_frag_nr(n);
        if (nr > 0 && np == 32) {
            const bool c2 = h2;
            const bool ext = F.use_decay || F.use_transform || F.use_scales;     // MV bit 1 (bfb_dmma.cuh)
            const int TX = c2 ? nr : (nr + 1) / 2, NT = bfb_frag_tiles(nr, c2, ext);
            const int NTP = (NT + 1) / 2;
            std::vector<double> fr((size_t)nr * NTP * 64, 0.);
            for (int kt = 0; kt < nr; ++kt)
                for (int t = 0; t < NT; ++t)
                    for (int lane = 0; lane < 32; ++lane) {
                        const int k = 4 * kt + (lane & 3), gid = lane >> 2, own = gid >> 1, e = gid & 1;
                        const std::vector<double> *T = nullptr;
                        int v;
                        const int TD = (nr + 1) / 2, TD2 = ext ? TD : 0;   // tile order: D | D2 (decay) | x block | x^2 block
                        if (t < TD) { v = 2 * t + e; if (v < nr) T = &HT; }
                        else if (t < TD + TD2) { v = 2 * (t - TD) + e; if (v < nr) T = &DH; }
                        else if (t < TD + TD2 + TX) { v = 2 * (t - TD - TD2) + e; if (v < nr) T = &S; else if (c2 && v < 2 * nr) { T = &A1T; v -= nr; } }
                        else { v = 2 * (t - TD - TD2 - TX) + e; if (v < nr) T = &A2; }
                        const int j = 4 * v + own;
                        if (T && !T->empty() && k < n && j < n) fr[(((size_t)kt * NTP + t / 2) * 32 + lane) * 2 + (t & 1)] = (*T)[(size_t)k * np + j];
                    }
            if ((rc = upload(h, fr, &D.bfrag))) return rc;
            D.frag_nr = nr; D.frag_nt = NT; D.frag_ext = ext ? 1 : 0;
            if (!ext) {
                if ((rc = build_team_table(nr))) return rc;
            }
        }
        // 32 < n <= 64: only the team kernels (four warps per 8-chain group, 16 dimensions per warp) reach the tensor cores; with
        // cubic-3 configs their pair-product operand (1 MB at n = 64) is streamed from L2 (bfb_team.cuh)
        if (n > 32 && n <= 64 && !(F.use_decay || F.use_transform || F.use_scales) && (!h3 || h2)) {
            if ((rc = build_team_table(16))) return rc;
            if (h3) {
                const int nrw = 4, tn3 = 2, n_pairs = n * (n - 1) / 2, kt3 = ((n_pairs + 3) / 4 + 7) / 8 * 8;
                std::vector<int> pairs((size_t)kt3 * 4, 0);
                {
                    int p = 0;
                    for (int k = 0; k < n; ++k)
                        for (int l = k + 1; l < n; ++l) pairs[p++] = k | (l << 8);
                }
                std::vector<double> f3((size_t)kt3 * 4 * tn3 * 32, 0.);
                for (int kt = 0; kt < kt3; ++kt)
                    for (int w = 0; w < 4; ++w)
                        for (int t = 0; t < tn3; ++t)
                            for (int lane = 0; lane < 32; ++lane) {
                                const int p = 4 * kt + (lane & 3), gid = lane >> 2, own = gid >> 1, e = gid & 1;
                                const int v = 2 * t + e, j = 4 * (nrw * w + v) + own;
                                if (p >= n_pairs || v >= nrw || j >= n) continue;
                                const int k = pairs[p] & 0xff, l = pairs[p] >> 8;
                                if (j == k || j == l) continue;
                                int a = j, b = k, c = l;
                                if (a > b) std::swap(a, b);
                                if (b > c) std::swap(b, c);
                                if (a > b) std::swap(a, b);
                                f3[(((size_t)kt * 4 + w) * tn3 + t) * 32 + lane] = c3[c3_index_host(a, b, c, n)];     // output 0
                            }
                if ((rc = upload(h, f3, &D.tfrag3))) return rc;
                // the device reads a pair as the offsets of its two factors inside a chain's quad of the exchange buffer
                for (int &pe : pairs) { const int k = pe & 0xff, l = pe >> 8; pe = ((k >> 2) * 32 + (k & 3)) | (((l >> 2) * 32 + (l & 3)) << 16); }
                if ((rc = upload(h, pairs, &D.tpair))) return rc;
                D.t3_kt = kt3;
            }
        }
        // cubic-3 block (bfb_dmma.cuh, MV bit 2): pairs (k < l) in lexicographic order, 4 per k-tile; column (tile t, lane
        // quad-owner `own`, e) holds dimension j = 4 (2 t + e) + own like the other blocks
        if (nr > 0 && h3 && np == 32 && nr <= 7) {
            const int n3t = (nr + 1) / 2, n_pairs = n * (n - 1) / 2, kt3 = (n_pairs + 3) / 4;
            std::vector<int> pairs((size_t)kt3 * 4, 0);
            {
                int p = 0;
                for (int k = 0; k < n; ++k)
                    for (int l = k + 1; l < n; ++l) pairs[p++] = k | (l << 8);
            }
            std::vector<double> f3((size_t)kt3 * n3t * 32, 0.);
            for (int kt = 0; kt < kt3; ++kt)
                for (int t = 0; t < n3t; ++t)
                    for (int lane = 0; lane < 32; ++lane) {
                        const int p = 4 * kt + (lane & 3), gid = lane >> 2, own = gid >> 1, e = gid & 1;
                        const int v = 2 * t + e, j = 4 * v + own;
                        if (p >= n_pairs || v >= nr || j >= n) continue;
                        const int k = pairs[p] & 0xff, l = pairs[p] >> 8;
                        if (j == k || j == l) continue;
                        int a = j, b = k, c = l;
                        if (a > b) std::swap(a, b);
                        if (b > c) std::swap(b, c);
                        if (a > b) std::swap(a, b);
                        f3[((size_t)kt * n3t + t) * 32 + lane] = c3[c3_index_host(a, b, c, n)];     // output 0
                    }
            if ((rc = upload(h, f3, &D.bfrag3))) return rc;
            if ((rc = upload(h, pairs, &D.c3pair))) return rc;
            D.c3_kt = kt3; D.c3_n3t = n3t;
        }
        std::vector<double> fm(m, 0.);
        for (int o = 0; o < m && o < (int)h->h_fmu.size(); ++o) fm[o] = h->h_fmu[o];
        if ((rc = upload(h, fm, &D.f_mu))) return rc;
    }
    D.use_scales = F.use_scales;
    if ((rc = upload(h, pad(h->h_s0, 0.), &D.s0))) return rc;
    if ((rc = upload(h, pad(h->h_sdiff, 1.), &D.sdiff))) return rc;
    D.use_decay = F.use_decay; D.d_alpha2 = F.d_alpha2; D.d_gamma = F.d_gamma;
    {
        if ((rc = upload(h, pad(h->h_dmu, 0.), &D.d_mu))) return rc;
        if ((rc = upload(h, DH, &D.d_H))) return rc;
    }
    D.use_transform = F.use_transform;
    {
        std::vector<double> lo(np, 0.), w(np, 1.);
        std::vector<int> hb(np, 0);
        if (F.use_transform)
            for (int j = 0; j < n; ++j) {
                lo[j] = h->h_ranges[2 * j];
                w[j] = h->h_ranges[2 * j + 1] - h->h_ranges[2 * j];
                hb[j] = (h->h_hb[2 * j] ? 1 : 0) | (h->h_hb[2 * j + 1] ? 2 : 0);
            }
        if ((rc = upload(h, lo, &D.r_lo))) return rc;
        if ((rc = upload(h, w, &D.r_w))) return rc;
        if ((rc = upload(h, hb, &D.hb))) return rc;
    }
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    return BFB_OK;
}

extern "C" int bfb_set_model(bfb_handle h, const bfb_model_desc *d)
{
    BFB_REQUIRE(h && d, BFB_ERR_ARG, "bfb_set_model: null argument");
    BFB_REQUIRE(d->n > 0 && d->m > 0 && d->n_config > 0, BFB_ERR_ARG, "bfb_set_model: n, m, n_config must be positive");
    BFB_REQUIRE(d->n <= 128, BFB_ERR_ARG, "bfb_set_model: input_size %d > 128 is not supported", d->n);
    h->n = d->n; h->m = d->m; h->np = 32 * ((d->n + 31) / 32);
    h->configs.clear();
    int64_t ioff = 0, ooff = 0, coff = 0;
    for (int c = 0; c < d->n_config; ++c) {
        HostConfig hc;
        hc.order = d->cfg_order[c]; hc.n_in = d->cfg_n_in[c]; hc.n_out = d->cfg_n_out[c];
        BFB_REQUIRE(hc.order >= BFB_LINEAR && hc.order <= BFB_CUBIC_3, BFB_ERR_ARG, "config %d: bad order %d", c, hc.order);
        BFB_REQUIRE(hc.n_in > 0 && hc.n_in <= d->n && hc.n_out > 0 && hc.n_out <= d->m, BFB_ERR_ARG,
                    "config %d: bad mask sizes", c);
        hc.in_mask.assign(d->cfg_in_mask + ioff, d->cfg_in_mask + ioff + hc.n_in);
        hc.out_mask.assign(d->cfg_out_mask + ooff, d->cfg_out_mask + ooff + hc.n_out);
        for (int k = 0; k < hc.n_in; ++k)
            BFB_REQUIRE(hc.in_mask[k] >= 0 && hc.in_mask[k] < d->n && (k == 0 || hc.in_mask[k] > hc.in_mask[k - 1]),
                        BFB_ERR_ARG, "config %d: input_mask must be sorted unique indices in [0,n)", c);
        for (int k = 0; k < hc.n_out; ++k)
            BFB_REQUIRE(hc.out_mask[k] >= 0 && hc.out_mask[k] < d->m && (k == 0 || hc.out_mask[k] > hc.out_mask[k - 1]),
                        BFB_ERR_ARG, "config %d: output_mask must be sorted unique indices in [0,m)", c);
        hc.n_packed = packed_size(hc.order, hc.n_in);
        hc.coef_off = coff;
        ioff += hc.n_in; ooff += hc.n_out; coff += hc.n_packed * hc.n_out;
        h->configs.push_back(hc);
    }
    h->packed.assign((size_t)coff, 0.);
    if (d->cfg_coef) memcpy(h->packed.data(), d->cfg_coef, sizeof(double) * (size_t)coff);
    h->desc_flags = *d;
    const int n = d->n, m = d->m;
    auto cp = [](std::vector<double> &dst, const double *src, size_t cnt) {
        dst.clear();
        if (src) dst.assign(src, src + cnt);
    };
    if (d->use_bound) {
        BFB_REQUIRE(d->mu && d->hess && d->f_mu, BFB_ERR_ARG, "use_bound set but mu/hess/f_mu missing");
        cp(h->h_mu, d->mu, n); cp(h->h_hess, d->hess, (size_t)n * n); cp(h->h_fmu, d->f_mu, m);
    } else { h->h_mu.clear(); h->h_hess.clear(); h->h_fmu.clear(); }
    if (d->use_scales) {
        BFB_REQUIRE(d->s0 && d->sdiff, BFB_ERR_ARG, "use_scales set but s0/sdiff missing");
        cp(h->h_s0, d->s0, n); cp(h->h_sdiff, d->sdiff, n);
    } else { h->h_s0.clear(); h->h_sdiff.clear(); }
    if (d->use_decay) {
        BFB_REQUIRE(d->d_mu && d->d_hess, BFB_ERR_ARG, "use_decay set but d_mu/d_hess missing");
        cp(h->h_dmu, d->d_mu, n); cp(h->h_dhess, d->d_hess, (size_t)n * n);
    } else { h->h_dmu.clear(); h->h_dhess.clear(); }
    if (d->use_transform) {
        BFB_REQUIRE(d->ranges && d->hard_bounds, BFB_ERR_ARG, "use_transform set but ranges/hard_bounds missing");
        cp(h->h_ranges, d->ranges, (size_t)2 * n);
        h->h_hb.assign(d->hard_bounds, d->hard_bounds + 2 * n);
    } else { h->h_ranges.clear(); h->h_hb.clear(); }
    int rc = bfb_upload_model(h);
    if (rc) return rc;
    h->has_model = true;
    return BFB_OK;
}

// Third module of the DES-Y1 example's pipeline (examples/des-y1-w-cosmosis.ipynb cells 12-14: des_post_f(like, x) = like +
// prior(x)): independent Gaussian prior on original-space inputs, logp += c0 - 1/2 sum_j w[j] (x_j - mu[j])^2 with w = 1 /
// sigma^2 (0 where an input has no prior).  w == NULL removes it.  Call after bfb_set_model and before bfb_set_epilogue.
extern "C" int bfb_set_prior(bfb_handle h, const double *w, const double *mu, double c0)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_set_prior: no model set");
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    DevModel &D = h->dm;
    if (!w) { D.use_prior = 0; h->h_pw.clear(); h->h_pmu.clear(); return BFB_OK; }
    BFB_REQUIRE(mu, BFB_ERR_ARG, "bfb_set_prior: mu missing");
    const int n = h->n, np = h->np;
    for (int j = 0; j < n; ++j) BFB_REQUIRE(w[j] >= 0. && std::isfinite(w[j]) && std::isfinite(mu[j]), BFB_ERR_ARG, "bfb_set_prior: bad weight / mean at input %d", j);
    h->h_pw.assign(w, w + n); h->h_pmu.assign(mu, mu + n); h->h_pc0 = c0;
    std::vector<double> pw(np, 0.), pm(np, 0.);
    for (int j = 0; j < n; ++j) { pw[j] = w[j]; pm[j] = mu[j]; }
    int rc;
    if ((rc = upload(h, pw, &D.p_w))) return rc;
    if ((rc = upload(h, pm, &D.p_mu))) return rc;
    D.use_prior = 1; D.p_c0 = c0;
    D.frag_nr = 0;                       // logp is no longer output 0 alone: the single-output tensor-core evaluators are off
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    return BFB_OK;
}

// Second module of a two-module pipeline (core/density.py:487-566: surrogate x -> m outputs, then a user Module m -> logp):
// kind 1 = Gaussian likelihood logp = c0 - 1/2 |f|^2 of the m outputs of the model set before, which the caller has
// pre-whitened (f' = Lt (f - d) with Cinv = Lt^T Lt folds into the polynomial coefficients, the constants and f_mu because
// all of them are linear in the outputs: bayesfast_b200/density.py whiten_spec).  kind 0 removes it.  Evaluated by the
// generic kernels (density_eval, bfb_eval.cuh); the tensor-core evaluators take logp = output 0 and are switched off.
extern "C" int bfb_set_epilogue(bfb_handle h, int kind, double c0)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_set_epilogue: no model set");
    BFB_REQUIRE(kind == 0 || kind == 1, BFB_ERR_ARG, "bfb_set_epilogue: unknown kind %d", kind);
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    if (kind == 0 && h->dm.epilogue) return bfb_upload_model(h);      // rebuilds the tensor-core tables
    h->dm.epilogue = kind;
    h->dm.e_c0 = kind ? c0 : 0.;
    if (kind) h->dm.frag_nr = 0;
    if (kind && !h->lik_tab) return bfb_build_lik_table(h);      // tensor-core evaluator of the pipeline, if it applies
    return BFB_OK;
}

// ----------------------------------------------------------------------------------------------
// batched evaluation kernels: one warp per (point, output)
// ----------------------------------------------------------------------------------------------
template <int NPL>
__global__ void __launch_bounds__(128) poly_eval_kernel(DevModel M, const double *__restrict__ X, int64_t C,
                                                        double *__restrict__ F, double *__restrict__ J)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double *xsm = smem + (size_t)wib * 2 * M.np, *dsm = xsm + M.np;
    const int64_t total = C * M.m;
    for (int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib; w < total; w += (int64_t)gridDim.x * (blockDim.x >> 5)) {
        const int64_t c = w / M.m;
        const int o = (int)(w % M.m);
        double x[NPL], Jr[NPL], f;
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            int j = lane + 32 * r;
            x[r] = (j < M.n) ? X[c * M.n + j] : 0.;
        }
        module_fg<NPL>(M, o, x, lane, xsm, dsm, f, Jr);
        if (lane == 0) F[c * M.m + o] = f;
        if (J) {
#pragma unroll
            for (int r = 0; r < NPL; ++r) {
                int j = lane + 32 * r;
                if (j < M.n) J[(c * M.m + o) * M.n + j] = Jr[r];
            }
        }
        __syncwarp();
    }
}

template <int NPL>
__global__ void __launch_bounds__(128) density_eval_kernel(DevModel M, const double *__restrict__ X, int64_t C,
                                                           double *__restrict__ LP, double *__restrict__ G)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    double *xsm = smem + (size_t)wib * 2 * M.np, *dsm = xsm + M.np;
    for (int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib; c < C; c += (int64_t)gridDim.x * (blockDim.x >> 5)) {
        double x[NPL], g[NPL], lp;
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            int j = lane + 32 * r;
            x[r] = (j < M.n) ? X[c * M.n + j] : 0.;
        }
        density_eval<NPL>(M, x, lane, xsm, dsm, lp, g);
        if (lane == 0) LP[c] = lp;
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            int j = lane + 32 * r;
            if (j < M.n) G[c * M.n + j] = g[r];
        }
        __syncwarp();
    }
}

struct DevBuf {
    // stages a caller buffer on the device when it lives on the host
    void *dev = nullptr; const void *host_src = nullptr; void *host_dst = nullptr; size_t bytes = 0; bool owned = false;
    ~DevBuf() { if (owned && dev) cudaFree(dev); }        // every early return of the callers frees the staged copies
};

static int stage_in(bfb_context *h, const void *p, size_t bytes, int loc, DevBuf &b)
{
    b.bytes = bytes;
    if (loc == BFB_DEVICE) { b.dev = (void *)p; return BFB_OK; }
    BFB_CUDA(cudaMalloc(&b.dev, bytes ? bytes : 8));
    b.owned = true;
    BFB_CUDA(cudaMemcpyAsync(b.dev, p, bytes, cudaMemcpyHostToDevice, h->stream));
    return BFB_OK;
}
static int stage_out(bfb_context *h, void *p, size_t bytes, int loc, DevBuf &b)
{
    b.bytes = bytes;
    if (!p) { b.dev = nullptr; return BFB_OK; }
    if (loc == BFB_DEVICE) { b.dev = p; return BFB_OK; }
    BFB_CUDA(cudaMalloc(&b.dev, bytes ? bytes : 8));
    b.owned = true; b.host_dst = p;
    return BFB_OK;
}
static int finish(bfb_context *h, DevBuf &b)
{
    if (b.owned && b.host_dst) BFB_CUDA(cudaMemcpyAsync(b.host_dst, b.dev, b.bytes, cudaMemcpyDeviceToHost, h->stream));
    return BFB_OK;
}
static void release(DevBuf &b) { if (b.owned && b.dev) cudaFree(b.dev); b.dev = nullptr; }

extern "C" int bfb_poly_eval_batch(bfb_handle h, const double *X, int64_t C, double *F, double *J, int loc)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_poly_eval_batch: no model set");
    BFB_REQUIRE(X && F && C >= 0, BFB_ERR_ARG, "bfb_poly_eval_batch: bad arguments");
    if (C == 0) return BFB_OK;
    BFB_CUDA(cudaSetDevice(h->device));
    const int n = h->n, m = h->m, npl = h->np / 32;
    DevBuf bx, bf, bj;
    int rc;
    if ((rc = stage_in(h, X, sizeof(double) * C * n, loc, bx))) return rc;
    if ((rc = stage_out(h, F, sizeof(double) * C * m, loc, bf))) return rc;
    if ((rc = stage_out(h, J, sizeof(double) * C * m * n, loc, bj))) return rc;
    const int wpb = 4;
    int64_t blocks64 = (C * m + wpb - 1) / wpb;
    int blocks = (int)(blocks64 < (int64_t)h->sm_count * 16 ? blocks64 : (int64_t)h->sm_count * 16);
    size_t smem = sizeof(double) * wpb * 2 * h->np;
    BFB_CUDA(cudaEventRecord(h->ev0, h->stream));
    // single-output PolyModel (value + Jacobian row): the tensor-core evaluator computes exactly module_fg
    int fast = 1;
    if (m == 1 && bj.dev && !h->dm.use_decay && !h->dm.use_transform)
        fast = bfb_launch_eval_dmma(h, (const double *)bx.dev, C, (double *)bf.dev, (double *)bj.dev);
    if (fast == 1 && m == 1 && bj.dev && !h->dm.use_decay && !h->dm.use_transform)
        fast = bfb_launch_eval_team(h, (const double *)bx.dev, C, (double *)bf.dev, (double *)bj.dev);
    if (fast < 0) return fast;
    if (fast == 1) {
    switch (npl) {
    case 1: poly_eval_kernel<1><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bf.dev, (double *)bj.dev); break;
    case 2: poly_eval_kernel<2><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bf.dev, (double *)bj.dev); break;
    case 3: poly_eval_kernel<3><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bf.dev, (double *)bj.dev); break;
    default: poly_eval_kernel<4><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bf.dev, (double *)bj.dev); break;
    }
    h->launches++;
    }
    BFB_CUDA(cudaGetLastError());
    BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
    if ((rc = finish(h, bf))) return rc;
    if ((rc = finish(h, bj))) return rc;
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    BFB_CUDA(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    release(bx); release(bf); release(bj);
    return BFB_OK;
}

extern "C" int bfb_logp_and_grad_batch(bfb_handle h, const double *X, int64_t C, double *logp, double *grad, int loc)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_logp_and_grad_batch: no model set");
    BFB_REQUIRE(X && logp && grad && C >= 0, BFB_ERR_ARG, "bfb_logp_and_grad_batch: bad arguments");
    if (C == 0) return BFB_OK;
    BFB_CUDA(cudaSetDevice(h->device));
    const int n = h->n, npl = h->np / 32;
    DevBuf bx, bl, bg;
    int rc;
    if ((rc = stage_in(h, X, sizeof(double) * C * n, loc, bx))) return rc;
    if ((rc = stage_out(h, logp, sizeof(double) * C, loc, bl))) return rc;
    if ((rc = stage_out(h, grad, sizeof(double) * C * n, loc, bg))) return rc;
    const int wpb = 4;
    int64_t blocks64 = (C + wpb - 1) / wpb;
    int blocks = (int)(blocks64 < (int64_t)h->sm_count * 16 ? blocks64 : (int64_t)h->sm_count * 16);
    size_t smem = sizeof(double) * wpb * 2 * h->np;
    BFB_CUDA(cudaEventRecord(h->ev0, h->stream));
    rc = bfb_launch_lik_dmma(h, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev);
    h->last_eval_path = (h->dm.lik_ftab && !getenv("BFB200_LIK_DENSE")) ? 4 : 3;
    if (rc == 1) { rc = bfb_launch_eval_dmma(h, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev); h->last_eval_path = 2; }
    if (rc == 1) { rc = bfb_launch_eval_team(h, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev); h->last_eval_path = 5; }
    if (rc < 0) return rc;
    if (rc == 1) h->last_eval_path = 0;
    if (rc == 1) {
    switch (npl) {
    case 1: density_eval_kernel<1><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev); break;
    case 2: density_eval_kernel<2><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev); break;
    case 3: density_eval_kernel<3><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev); break;
    default: density_eval_kernel<4><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, (const double *)bx.dev, C, (double *)bl.dev, (double *)bg.dev); break;
    }
    h->launches++;
    }
    BFB_CUDA(cudaGetLastError());
    BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
    if ((rc = finish(h, bl))) return rc;
    if ((rc = finish(h, bg))) return rc;
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    BFB_CUDA(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    release(bx); release(bl); release(bg);
    return BFB_OK;
}

extern "C" int bfb_eval_last_path(bfb_handle h)
{
    return h ? h->last_eval_path : -1;
}

// ----------------------------------------------------------------------------------------------
// RNG exposure
// ----------------------------------------------------------------------------------------------
__global__ void rng_fill_kernel(uint64_t seed, uint64_t chain, uint64_t t0, int64_t count, double *u, double *z)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double uu = bfb_draw_uniform(seed, chain, t0 + (uint64_t)i);
    u[i] = uu;
    z[i] = bfb_norminv(uu);
}

extern "C" int bfb_rng_fill(bfb_handle h, uint64_t seed, uint64_t chain, uint64_t t0, int64_t count, double *u, double *z)
{
    BFB_REQUIRE(h && u && z && count >= 0, BFB_ERR_ARG, "bfb_rng_fill: bad arguments");
    if (count == 0) return BFB_OK;
    BFB_CUDA(cudaSetDevice(h->device));
    double *du, *dz;
    BFB_CUDA(cudaMalloc(&du, sizeof(double) * count));
    BFB_CUDA(cudaMalloc(&dz, sizeof(double) * count));
    rng_fill_kernel<<<(unsigned)((count + 255) / 256), 256, 0, h->stream>>>(seed, chain, t0, count, du, dz);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    BFB_CUDA(cudaMemcpyAsync(u, du, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaMemcpyAsync(z, dz, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(du); cudaFree(dz);
    return BFB_OK;
}
