// bfb_fit.cu -- PolyModel.fit on the device (reference: bayesfast/modules/poly.py:505-589).
//
//   accumulate : fused feature expansion (the _lsq_* builders of _poly.pyx:143-177, never materialised in HBM)
//                + Gram  G = [Phi_w | w y]^T [Phi_w | w y]  on FP64 tensor cores (DMMA m8n8k4), upper block
//                triangle only, split over row chunks with a deterministic two-stage reduction;
//                + shifted first/second moments of x for _set_bound (poly.py:262-276).
//   all-reduce : the partial sums live in ONE contiguous device buffer (bfb_fit_buffer) that the host framework
//                all-reduces over NCCL when the rows are sharded over GPUs.
//   solve      : symmetric diagonal equilibration, blocked right-looking Cholesky, triangular solves for all
//                outputs at once, one step of iterative refinement; replaces scipy.linalg.lstsq (poly.py:570).
//
// Outputs that are served by the same set of configs (same recipe row, poly.py:298-337) share one Gram.
#include "bfb_common.cuh"
#include "bfb_gram.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>

// temporary device allocations of one call: freed on every return path (the error paths used to leak them)
struct TmpList : std::vector<void *> {
    ~TmpList() { for (void *p : *this) cudaFree(p); }
};

struct FitGroup {
    std::vector<int> cfg_ids, outputs;
    int P, Pt, Ptp, nt;
    short4 *d_feat;     // [Ptp]  (i0,i1,i2,kind): kind 0 monomial x[i0]*x[i1]*x[i2] (-1 -> 1), 1 y column i0, 2 padding
    size_t g_off;       // offset of the Ptp x Ptp Gram inside FitState::buf
};

struct FitState {
    std::vector<FitGroup> groups;
    double *buf = nullptr;
    int64_t buf_len = 0;
    double *xbuf = nullptr;      // packed exchange buffer (bfb_fit_exchange_pack)
    size_t off_s1 = 0, off_s2 = 0, off_cnt = 0;
    double *d_shift = nullptr;
    std::vector<double> shift;
    double *ws = nullptr;
    size_t ws_len = 0;
    std::vector<void *> allocs;
};

void bfb_fit_free(bfb_context *h)
{
    if (!h->fit) return;
    for (void *p : h->fit->allocs) cudaFree(p);
    if (h->fit->ws) cudaFree(h->fit->ws);
    delete h->fit;
    h->fit = nullptr;
}

// ----------------------------------------------------------------------------------------------
// Gram kernel
// ----------------------------------------------------------------------------------------------
// One CTA = one 64 x 64 tile (ti <= tj) of the Gram over one chunk of rows.  Per stage of KC rows:
//   1. the x rows are staged in shared memory with a constant-1 column appended at index n, so that a monomial with
//      fewer than three factors needs no branch (missing factors index the 1);
//   2. every thread owns ONE feature column of each of the two tiles (its three factor indices sit in registers for
//      the whole kernel) and expands it for its 16 rows: (x[i0] * x[i1]) * x[i2] * w -- the multiplication order of
//      _lsq_quadratic / _lsq_cubic_2 / _lsq_cubic_3; y columns are read from global memory;
//   3. 4 warps (2 x 2) multiply the two 64-feature panels with DMMA m8n8k4, 32 x 32 per warp.
__global__ void __launch_bounds__(128) gram_kernel(const double *__restrict__ x, const double *__restrict__ y,
                                                   const double *__restrict__ w, int64_t N, int n, int m,
                                                   const short4 *__restrict__ feat, int nt, int64_t rows_per_chunk,
                                                   double *__restrict__ ws)
{
    extern __shared__ double sm[];
    int t = blockIdx.x, ti = 0;
    while (t >= nt - ti) { t -= nt - ti; ++ti; }
    const int tj = ti + t;
    const bool diag = (ti == tj);
    const int ldx = n + 2;                   // n values + the constant 1 (+1 pad)
    double *xs = sm;                         // [KC][ldx]
    double *wk = xs + KC * ldx;              // [KC]
    double *phiI = wk + KC;                  // [KC][LDP]
    double *phiJ = diag ? phiI : phiI + KC * LDP;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // this thread's feature column in each tile
    const int fcol = tid & (TS - 1), khalf = tid >> 6;          // rows khalf, khalf + 2, ...
    const short4 fi = feat[ti * TS + fcol], fj = feat[tj * TS + fcol];
    const int i0 = fi.x >= 0 ? fi.x : n, i1 = fi.y >= 0 ? fi.y : n, i2 = fi.z >= 0 ? fi.z : n;
    const int j0 = fj.x >= 0 ? fj.x : n, j1 = fj.y >= 0 ? fj.y : n, j2 = fj.z >= 0 ? fj.z : n;
    const int wm = warp >> 1, wn = warp & 1;
    double acc[4][4][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.;
    const int64_t r_begin = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r_end = min(N, r_begin + rows_per_chunk);
    // flat, division-free walk over the KC x n block of x (contiguous in global memory): element e = tid + 128 s
    const int k_init = tid / n, j_init = tid - k_init * n, dk = 128 / n, dj = 128 - dk * n;
    const int n_el = KC * n;
    for (int64_t r0 = r_begin; r0 < r_end; r0 += KC) {
        __syncthreads();
        {
            const int64_t last = (r_end - 1 - r0) * n;          // rows past the end re-read the last row (their w is 0)
            const double *xb = x + r0 * n;
            int k = k_init, j = j_init;
            for (int e = tid; e < n_el; e += 128) {
                const int64_t src = (int64_t)k * n + j;
                xs[k * ldx + j] = xb[src <= last + n - 1 ? src : last + j];
                j += dj; k += dk;
                if (j >= n) { j -= n; k += 1; }
            }
            if (tid < KC) {
                xs[tid * ldx + n] = 1.;
                wk[tid] = (r0 + tid < r_end) ? (w ? w[r0 + tid] : 1.) : 0.;
            }
        }
        __syncthreads();
        if (fi.w == 0) {
#pragma unroll 8
            for (int k = khalf; k < KC; k += 2) {
                const double *xr = xs + k * ldx;
                phiI[k * LDP + fcol] = ((xr[i0] * xr[i1]) * xr[i2]) * wk[k];
            }
        } else {
            for (int k = khalf; k < KC; k += 2) {
                const int64_t row = min(r0 + k, r_end - 1);
                phiI[k * LDP + fcol] = (fi.w == 1 ? y[row * m + fi.x] : 0.) * wk[k];
            }
        }
        if (!diag) {
            if (fj.w == 0) {
#pragma unroll 8
                for (int k = khalf; k < KC; k += 2) {
                    const double *xr = xs + k * ldx;
                    phiJ[k * LDP + fcol] = ((xr[j0] * xr[j1]) * xr[j2]) * wk[k];
                }
            } else {
                for (int k = khalf; k < KC; k += 2) {
                    const int64_t row = min(r0 + k, r_end - 1);
                    phiJ[k * LDP + fcol] = (fj.w == 1 ? y[row * m + fj.x] : 0.) * wk[k];
                }
            }
        }
        __syncthreads();
        gram_tile_mma(phiI, phiJ, lane, wm, wn, acc);
    }
    double *out = ws + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (TS * TS);
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int r = 32 * wm + 8 * a + (lane >> 2), c = 32 * wn + 8 * b + 2 * (lane & 3);
            out[r * TS + c] = acc[a][b][0];
            out[r * TS + c + 1] = acc[a][b][1];
        }
}

// G[tile] += sum over chunks (fixed order: deterministic)
__global__ void gram_reduce_kernel(const double *__restrict__ ws, int n_tiles, int n_chunks, int nt, int Ptp,
                                   double *__restrict__ G)
{
    int t = blockIdx.x, ti = 0;
    const int tile = t;
    while (t >= nt - ti) { t -= nt - ti; ++ti; }
    const int tj = ti + t;
    for (int e = threadIdx.x; e < TS * TS; e += blockDim.x) {
        double s = 0.;
        for (int c = 0; c < n_chunks; ++c) s += ws[((size_t)c * n_tiles + tile) * (TS * TS) + e];
        int r = e / TS, cidx = e - r * TS;
        G[(size_t)(ti * TS + r) * Ptp + tj * TS + cidx] += s;
    }
}

// shifted moments: S1 = sum (x - s), S2 = sum (x - s)(x - s)^T, count.  One block per row range; fixed-order reduce.
__global__ void __launch_bounds__(256) moments_kernel(const double *__restrict__ x, int64_t N, int n,
                                                      const double *__restrict__ shift, int64_t rows_per_block,
                                                      double *__restrict__ ws)
{
    extern __shared__ double sm[];
    double *xs = sm;   // [64][n+1]
    const int ldx = n + 1, tid = threadIdx.x;
    const int npair = n * n;
    const int PER = 16;                      // n <= 64 -> n^2 <= 4096 = 256 * 16
    double acc[PER];
#pragma unroll
    for (int i = 0; i < PER; ++i) acc[i] = 0.;
    double acc1 = 0.;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_block, r_end = min(N, r_begin + rows_per_block);
    for (int64_t r0 = r_begin; r0 < r_end; r0 += 64) {
        __syncthreads();
        for (int e = tid; e < 64 * n; e += 256) {
            int k = e / n, j = e - k * n;
            int64_t row = r0 + k;
            xs[k * ldx + j] = (row < r_end) ? x[row * n + j] - shift[j] : 0.;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            int pidx = tid + 256 * i;
            if (pidx < npair) {
                int a = pidx / n, b = pidx - a * n;
                double s = acc[i];
                for (int k = 0; k < 64; ++k) s = fma(xs[k * ldx + a], xs[k * ldx + b], s);
                acc[i] = s;
            }
        }
        if (tid < n) {
            double s = acc1;
            for (int k = 0; k < 64; ++k) s += xs[k * ldx + tid];
            acc1 = s;
        }
    }
    double *out = ws + (size_t)blockIdx.x * (npair + n);
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        int pidx = tid + 256 * i;
        if (pidx < npair) out[n + pidx] = acc[i];
    }
    if (tid < n) out[tid] = acc1;
}

__global__ void moments_reduce_kernel(const double *__restrict__ ws, int n_blocks, int len, double *__restrict__ dst)
{
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= len) return;
    double s = 0.;
    for (int b = 0; b < n_blocks; ++b) s += ws[(size_t)b * len + e];
    dst[e] += s;
}

// ----------------------------------------------------------------------------------------------
// host: groups / begin / accumulate
// ----------------------------------------------------------------------------------------------
static void push_feat(std::vector<short4> &v, int a, int b, int c, int kind)
{
    short4 s; s.x = (short)a; s.y = (short)b; s.z = (short)c; s.w = (short)kind;
    v.push_back(s);
}

extern "C" int bfb_fit_begin(bfb_handle h, const double *shift)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_fit_begin: set the model (configs) first");
    BFB_REQUIRE(h->n <= 64, BFB_ERR_ARG, "fit supports input_size <= 64 (got %d)", h->n);
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    bfb_fit_free(h);
    FitState *fs = new FitState();
    h->fit = fs;
    const int n = h->n, m = h->m;
    // recipe rows (poly.py:298-337): per output, the config serving each order
    std::map<std::vector<int>, int> key2group;
    for (int o = 0; o < m; ++o) {
        std::vector<int> key(4, -1);
        for (size_t c = 0; c < h->configs.size(); ++c) {
            const HostConfig &hc = h->configs[c];
            if (std::find(hc.out_mask.begin(), hc.out_mask.end(), (int64_t)o) != hc.out_mask.end()) {
                BFB_REQUIRE(key[hc.order - 1] < 0, BFB_ERR_ARG,
                            "multiple PolyConfigs of the same order share output %d", o);
                key[hc.order - 1] = (int)c;
            }
        }
        BFB_REQUIRE(key[0] >= 0 || key[1] >= 0 || key[2] >= 0 || key[3] >= 0, BFB_ERR_ARG,
                    "no PolyConfig has output for variable %d", o);
        auto it = key2group.find(key);
        if (it == key2group.end()) {
            FitGroup g;
            for (int k = 0; k < 4; ++k) if (key[k] >= 0) g.cfg_ids.push_back(key[k]);
            g.outputs.push_back(o);
            key2group[key] = (int)fs->groups.size();
            fs->groups.push_back(g);
        } else fs->groups[it->second].outputs.push_back(o);
    }
    size_t off = 0;
    for (FitGroup &g : fs->groups) {
        std::vector<short4> feat;
        for (int cid : g.cfg_ids) {
            const HostConfig &hc = h->configs[cid];
            const std::vector<int64_t> &im = hc.in_mask;
            const int ni = hc.n_in;
            if (hc.order == BFB_LINEAR) {
                push_feat(feat, -1, -1, -1, 0);
                for (int k = 0; k < ni; ++k) push_feat(feat, (int)im[k], -1, -1, 0);
            } else if (hc.order == BFB_QUADRATIC) {
                for (int k = 0; k < ni; ++k) for (int l = k; l < ni; ++l) push_feat(feat, (int)im[k], (int)im[l], -1, 0);
            } else if (hc.order == BFB_CUBIC_2) {
                for (int k = 0; k < ni; ++k) for (int l = 0; l < ni; ++l) push_feat(feat, (int)im[k], (int)im[k], (int)im[l], 0);
            } else {
                for (int k = 0; k < ni; ++k) for (int l = k + 1; l < ni; ++l) for (int p = l + 1; p < ni; ++p)
                    push_feat(feat, (int)im[k], (int)im[l], (int)im[p], 0);
            }
        }
        g.P = (int)feat.size();
        for (int o : g.outputs) push_feat(feat, o, -1, -1, 1);
        g.Pt = (int)feat.size();
        g.nt = (g.Pt + TS - 1) / TS;
        g.Ptp = g.nt * TS;
        while ((int)feat.size() < g.Ptp) push_feat(feat, -1, -1, -1, 2);
        BFB_REQUIRE(g.P <= 16384, BFB_ERR_ARG, "fit: %d parameters per output exceed the single-GPU limit 16384", g.P);
        void *p = nullptr;
        BFB_CUDA(cudaMalloc(&p, sizeof(short4) * feat.size()));
        fs->allocs.push_back(p);
        BFB_CUDA(cudaMemcpy(p, feat.data(), sizeof(short4) * feat.size(), cudaMemcpyHostToDevice));
        g.d_feat = (short4 *)p;
        g.g_off = off;
        off += (size_t)g.Ptp * g.Ptp;
    }
    fs->off_s1 = off; off += n;
    fs->off_s2 = off; off += (size_t)n * n;
    fs->off_cnt = off; off += 1;
    fs->buf_len = (int64_t)off;
    void *p = nullptr;
    BFB_CUDA(cudaMalloc(&p, sizeof(double) * off));
    fs->allocs.push_back(p);
    fs->buf = (double *)p;
    BFB_CUDA(cudaMemset(fs->buf, 0, sizeof(double) * off));
    fs->shift.assign(n, 0.);
    if (shift) for (int j = 0; j < n; ++j) fs->shift[j] = shift[j];
    BFB_CUDA(cudaMalloc(&p, sizeof(double) * n));
    fs->allocs.push_back(p);
    fs->d_shift = (double *)p;
    BFB_CUDA(cudaMemcpy(fs->d_shift, fs->shift.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
    return BFB_OK;
}

extern "C" int64_t bfb_fit_buffer_size(bfb_handle h) { return (h && h->fit) ? h->fit->buf_len : -1; }

// ---- exchange buffer of the sharded fit: only the upper block triangle of every Gram (the kernel writes no other tile)
// plus the moments, contiguous: P = 1585 (+ 1 y column) is 325 tiles = 10.6 MB instead of the 25 x 25 tiles = 20.5 MB of
// the working buffer ----
// dir 0: tiles (ti <= tj) of the Ptp x Ptp matrix -> packed, dir 1: packed -> matrix
static __global__ void fit_pack_tiles_kernel(double *__restrict__ gram, double *__restrict__ packed, int nt, int Ptp, int dir)
{
    int t = blockIdx.x, ti = 0;
    while (t >= nt - ti) { t -= nt - ti; ++ti; }              // tile index -> (ti, tj = ti + t)
    const int tj = ti + t;
    double *dst = packed + (size_t)blockIdx.x * TS * TS;
    for (int e = threadIdx.x; e < TS * TS; e += blockDim.x) {
        const size_t g = (size_t)(ti * TS + e / TS) * Ptp + (size_t)tj * TS + e % TS;
        if (dir == 0) dst[e] = gram[g]; else gram[g] = dst[e];
    }
}

static int fit_exchange_len(const FitState *fs, int n, int64_t *len)
{
    int64_t l = 0;
    for (const FitGroup &g : fs->groups) l += (int64_t)g.nt * (g.nt + 1) / 2 * TS * TS;
    *len = l + n + (int64_t)n * n + 1;
    return BFB_OK;
}

static int fit_exchange_copy(bfb_context *h, int dir)
{
    FitState *fs = h->fit;
    const int n = h->n;
    int64_t len;
    fit_exchange_len(fs, n, &len);
    if (!fs->xbuf) {
        void *p = nullptr;
        BFB_CUDA(cudaMalloc(&p, sizeof(double) * len));
        fs->allocs.push_back(p);
        fs->xbuf = (double *)p;
    }
    size_t off = 0;
    for (FitGroup &g : fs->groups) {
        const int ntile = g.nt * (g.nt + 1) / 2;
        fit_pack_tiles_kernel<<<ntile, 256, 0, h->stream>>>(fs->buf + g.g_off, fs->xbuf + off, g.nt, g.Ptp, dir);
        h->launches++;
        off += (size_t)ntile * TS * TS;
    }
    const size_t tail = (size_t)n + (size_t)n * n + 1;       // s1 | s2 | count are contiguous in the working buffer
    if (dir == 0) BFB_CUDA(cudaMemcpyAsync(fs->xbuf + off, fs->buf + fs->off_s1, sizeof(double) * tail, cudaMemcpyDeviceToDevice, h->stream));
    else BFB_CUDA(cudaMemcpyAsync(fs->buf + fs->off_s1, fs->xbuf + off, sizeof(double) * tail, cudaMemcpyDeviceToDevice, h->stream));
    BFB_CUDA(cudaGetLastError());
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    return BFB_OK;
}

extern "C" int bfb_fit_exchange_pack(bfb_handle h, double **dev_ptr, int64_t *len)
{
    BFB_REQUIRE(h && h->fit && dev_ptr && len, BFB_ERR_STATE, "bfb_fit_exchange_pack: call bfb_fit_begin first");
    BFB_CUDA(cudaSetDevice(h->device));
    int rc = fit_exchange_copy(h, 0);
    if (rc) return rc;
    *dev_ptr = h->fit->xbuf;
    return fit_exchange_len(h->fit, h->n, len);
}

extern "C" int bfb_fit_exchange_unpack(bfb_handle h)
{
    BFB_REQUIRE(h && h->fit && h->fit->xbuf, BFB_ERR_STATE, "bfb_fit_exchange_unpack: call bfb_fit_exchange_pack first");
    BFB_CUDA(cudaSetDevice(h->device));
    return fit_exchange_copy(h, 1);
}

// host staging of the packed exchange buffer (a backend without device collectives: gloo); dir 0: device -> host, 1: host -> device
extern "C" int bfb_fit_exchange_host(bfb_handle h, double *host, int dir)
{
    BFB_REQUIRE(h && h->fit && h->fit->xbuf && host, BFB_ERR_STATE, "bfb_fit_exchange_host: call bfb_fit_exchange_pack first");
    BFB_CUDA(cudaSetDevice(h->device));
    int64_t len;
    fit_exchange_len(h->fit, h->n, &len);
    if (dir == 0) BFB_CUDA(cudaMemcpy(host, h->fit->xbuf, sizeof(double) * len, cudaMemcpyDeviceToHost));
    else BFB_CUDA(cudaMemcpy(h->fit->xbuf, host, sizeof(double) * len, cudaMemcpyHostToDevice));
    return BFB_OK;
}

extern "C" int bfb_fit_buffer(bfb_handle h, double **dev_ptr)
{
    BFB_REQUIRE(h && h->fit && dev_ptr, BFB_ERR_STATE, "bfb_fit_buffer: call bfb_fit_begin first");
    *dev_ptr = h->fit->buf;
    return BFB_OK;
}

static int ensure_ws(FitState *fs, size_t len)
{
    if (fs->ws_len >= len) return BFB_OK;
    if (fs->ws) cudaFree(fs->ws);
    fs->ws = nullptr; fs->ws_len = 0;
    BFB_CUDA(cudaMalloc((void **)&fs->ws, sizeof(double) * len));
    fs->ws_len = len;
    return BFB_OK;
}

__global__ void add_count_kernel(double *cnt, double v) { *cnt += v; }

extern "C" int bfb_fit_accumulate(bfb_handle h, const double *x, const double *y, const double *w, int64_t N, int loc)
{
    BFB_REQUIRE(h && h->fit, BFB_ERR_STATE, "bfb_fit_accumulate: call bfb_fit_begin first");
    BFB_REQUIRE(x && y && N >= 0, BFB_ERR_ARG, "bfb_fit_accumulate: bad arguments");
    if (N == 0) return BFB_OK;
    BFB_CUDA(cudaSetDevice(h->device));
    FitState *fs = h->fit;
    const int n = h->n, m = h->m;
    const double *dx = x, *dy = y, *dw = w;
    TmpList tmp;
    if (loc == BFB_HOST) {
        void *p;
        BFB_CUDA(cudaMalloc(&p, sizeof(double) * N * n)); tmp.push_back(p);
        BFB_CUDA(cudaMemcpyAsync(p, x, sizeof(double) * N * n, cudaMemcpyHostToDevice, h->stream)); dx = (double *)p;
        BFB_CUDA(cudaMalloc(&p, sizeof(double) * N * m)); tmp.push_back(p);
        BFB_CUDA(cudaMemcpyAsync(p, y, sizeof(double) * N * m, cudaMemcpyHostToDevice, h->stream)); dy = (double *)p;
        if (w) {
            BFB_CUDA(cudaMalloc(&p, sizeof(double) * N)); tmp.push_back(p);
            BFB_CUDA(cudaMemcpyAsync(p, w, sizeof(double) * N, cudaMemcpyHostToDevice, h->stream)); dw = (double *)p;
        }
    }
    BFB_CUDA(cudaEventRecord(h->ev0, h->stream));
    for (FitGroup &g : fs->groups) {
        const int n_tiles = g.nt * (g.nt + 1) / 2;
        // enough (tile, chunk) CTAs for ~4 waves, but at least 8 stages of rows per chunk
        int64_t want = ((int64_t)h->sm_count * 4 * 4 + n_tiles - 1) / n_tiles;
        int64_t max_chunks = (N + 8 * KC - 1) / (8 * KC);
        int n_chunks = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(want, max_chunks), 65535));
        int64_t rows_per_chunk = ((N + n_chunks - 1) / n_chunks + KC - 1) / KC * KC;
        n_chunks = (int)((N + rows_per_chunk - 1) / rows_per_chunk);
        int rc = ensure_ws(fs, (size_t)n_tiles * n_chunks * TS * TS);
        if (rc) return rc;
        size_t smem = sizeof(double) * (KC * (n + 2) + KC + 2 * KC * LDP);
        dim3 grid(n_tiles, n_chunks);
        gram_kernel<<<grid, 128, smem, h->stream>>>(dx, dy, dw, N, n, m, g.d_feat, g.nt, rows_per_chunk, fs->ws);
        h->launches++;
        BFB_CUDA(cudaGetLastError());
        gram_reduce_kernel<<<n_tiles, 256, 0, h->stream>>>(fs->ws, n_tiles, n_chunks, g.nt, g.Ptp, fs->buf + g.g_off);
        h->launches++;
        BFB_CUDA(cudaGetLastError());
    }
    BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
    {
        int nb = (int)std::max<int64_t>(1, std::min<int64_t>((N + 1023) / 1024, (int64_t)h->sm_count * 2));
        int64_t rpb = ((N + nb - 1) / nb + 63) / 64 * 64;
        nb = (int)((N + rpb - 1) / rpb);
        const int len = n * n + n;
        int rc = ensure_ws(fs, (size_t)nb * len);
        if (rc) return rc;
        moments_kernel<<<nb, 256, sizeof(double) * 64 * (n + 1), h->stream>>>(dx, N, n, fs->d_shift, rpb, fs->ws);
        h->launches++;
        BFB_CUDA(cudaGetLastError());
        moments_reduce_kernel<<<(len + 255) / 256, 256, 0, h->stream>>>(fs->ws, nb, len, fs->buf + fs->off_s1);
        h->launches++;
        add_count_kernel<<<1, 1, 0, h->stream>>>(fs->buf + fs->off_cnt, (double)N);
        h->launches++;
        BFB_CUDA(cudaGetLastError());
    }
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    BFB_CUDA(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    for (void *p : tmp) cudaFree(p);
    tmp.clear();
    return BFB_OK;
}

// mean and covariance (unbiased, like np.cov) of the accumulated rows, from the shifted moments
extern "C" int bfb_fit_moments(bfb_handle h, double *mu, double *cov)
{
    BFB_REQUIRE(h && h->fit && mu && cov, BFB_ERR_STATE, "bfb_fit_moments: call bfb_fit_begin / accumulate first");
    BFB_CUDA(cudaSetDevice(h->device));
    FitState *fs = h->fit;
    const int n = h->n;
    std::vector<double> s1(n), s2((size_t)n * n);
    double cnt = 0.;
    BFB_CUDA(cudaMemcpy(s1.data(), fs->buf + fs->off_s1, sizeof(double) * n, cudaMemcpyDeviceToHost));
    BFB_CUDA(cudaMemcpy(s2.data(), fs->buf + fs->off_s2, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    BFB_CUDA(cudaMemcpy(&cnt, fs->buf + fs->off_cnt, sizeof(double), cudaMemcpyDeviceToHost));
    BFB_REQUIRE(cnt >= 2., BFB_ERR_NUMERIC, "bfb_fit_moments: need at least 2 rows");
    for (int i = 0; i < n; ++i) mu[i] = fs->shift[i] + s1[i] / cnt;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            double a = 0.5 * (s2[(size_t)i * n + j] + s2[(size_t)j * n + i]);
            cov[(size_t)i * n + j] = (a - s1[i] * s1[j] / cnt) / (cnt - 1.);
        }
    return BFB_OK;
}

// ----------------------------------------------------------------------------------------------
// Mahalanobis radii of rows (poly.py:270-276): one warp per row
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) beta_kernel(const double *__restrict__ x, int64_t N, int n,
                                                   const double *__restrict__ mu, const double *__restrict__ hess,
                                                   double *__restrict__ beta_out, unsigned long long *__restrict__ maxbits)
{
    extern __shared__ double sm[];
    double *Hs = sm;                 // [n][n]
    double *ds = sm + n * n;         // [4][n]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) Hs[e] = hess[e];
    __syncthreads();
    double *d = ds + wib * n;
    double best = 0.;
    for (int64_t row = (int64_t)blockIdx.x * 4 + wib; row < N; row += (int64_t)gridDim.x * 4) {
        for (int j = lane; j < n; j += 32) d[j] = x[row * n + j] - mu[j];
        __syncwarp();
        double part = 0.;
        for (int k = lane; k < n; k += 32) {
            double t = 0.;
            for (int i = 0; i < n; ++i) t = fma(d[i], Hs[i * n + k], t);    // (d^T H)_k
            part = fma(t, d[k], part);
        }
        double b = sqrt(warp_sum(part));
        if (beta_out && lane == 0) beta_out[row] = b;
        best = fmax(best, b);
        __syncwarp();
    }
    if (lane == 0 && best > 0.) atomicMax(maxbits, (unsigned long long)__double_as_longlong(best));
}

extern "C" int bfb_fit_max_beta(bfb_handle h, const double *x, int64_t N, const double *mu, const double *hess,
                                double *max_beta, double *beta_out, int loc)
{
    BFB_REQUIRE(h && h->has_model && x && mu && hess && max_beta && N > 0, BFB_ERR_ARG, "bfb_fit_max_beta: bad arguments");
    BFB_CUDA(cudaSetDevice(h->device));
    const int n = h->n;
    TmpList tmp;
    auto dmal = [&](size_t bytes, void **p) -> int { BFB_CUDA(cudaMalloc(p, bytes)); tmp.push_back(*p); return BFB_OK; };
    int rc;
    void *dmu, *dh, *dmax, *dxv = (void *)x, *dbeta = (void *)beta_out;
    if ((rc = dmal(sizeof(double) * n, &dmu)) || (rc = dmal(sizeof(double) * n * n, &dh)) || (rc = dmal(8, &dmax))) return rc;
    BFB_CUDA(cudaMemcpyAsync(dmu, mu, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    BFB_CUDA(cudaMemcpyAsync(dh, hess, sizeof(double) * n * n, cudaMemcpyHostToDevice, h->stream));
    BFB_CUDA(cudaMemsetAsync(dmax, 0, 8, h->stream));
    if (loc == BFB_HOST) {
        if ((rc = dmal(sizeof(double) * N * n, &dxv))) return rc;
        BFB_CUDA(cudaMemcpyAsync(dxv, x, sizeof(double) * N * n, cudaMemcpyHostToDevice, h->stream));
        if (beta_out && (rc = dmal(sizeof(double) * N, &dbeta))) return rc;
    }
    int blocks = (int)std::min<int64_t>((N + 3) / 4, (int64_t)h->sm_count * 16);
    beta_kernel<<<blocks, 128, sizeof(double) * (n * n + 4 * n), h->stream>>>((const double *)dxv, N, n, (const double *)dmu,
                                                                              (const double *)dh, (double *)dbeta,
                                                                              (unsigned long long *)dmax);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    unsigned long long bits = 0;
    BFB_CUDA(cudaMemcpyAsync(&bits, dmax, 8, cudaMemcpyDeviceToHost, h->stream));
    if (loc == BFB_HOST && beta_out)
        BFB_CUDA(cudaMemcpyAsync(beta_out, dbeta, sizeof(double) * N, cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(max_beta, &bits, 8);
    for (void *p : tmp) cudaFree(p);
    tmp.clear();
    return BFB_OK;
}

// ----------------------------------------------------------------------------------------------
// solve: equilibrate, blocked Cholesky, triangular solves, refinement
// ----------------------------------------------------------------------------------------------
#define NB 32

// A (P x P, both triangles) = D G D, Bs (P x nr) = D G[:, P:P+nr], D = diag(G)^-1/2
__global__ void assemble_kernel(const double *__restrict__ G, int Ptp, int P, int nr, double *__restrict__ A,
                                double *__restrict__ Bs, double *__restrict__ dscale)
{
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t total = (int64_t)P * (P + nr);
    if (e >= total) return;
    int i = (int)(e / (P + nr)), j = (int)(e - (int64_t)i * (P + nr));
    double di = rsqrt(G[(size_t)i * Ptp + i]);
    if (j < P) {
        double dj = rsqrt(G[(size_t)j * Ptp + j]);
        // only block-upper tiles hold data
        double g = (i / TS <= j / TS) ? G[(size_t)i * Ptp + j] : G[(size_t)j * Ptp + i];
        A[(size_t)i * P + j] = (i == j) ? 1. : g * di * dj;
        if (j == 0) dscale[i] = di;
    } else {
        Bs[(size_t)i * nr + (j - P)] = G[(size_t)i * Ptp + j] * di;     // y columns sit right of the features
    }
}

__global__ void __launch_bounds__(1024) chol_diag_kernel(double *A, int lda, int P, int kb, int *info)
{
    __shared__ double s[NB][NB + 1];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int nb = min(NB, P - kb);
    s[ty][tx] = (ty < nb && tx < nb) ? A[(size_t)(kb + ty) * lda + kb + tx] : (ty == tx ? 1. : 0.);
    for (int j = 0; j < nb; ++j) {
        __syncthreads();
        if (tx == j && ty == j) {
            double v = s[j][j];
            if (!(v > 0.)) { atomicMax(info, kb + j + 1); v = 1.; }
            s[j][j] = sqrt(v);
        }
        __syncthreads();
        if (tx == j && ty > j) s[ty][j] /= s[j][j];
        __syncthreads();
        if (ty > j && tx > j && tx <= ty) s[ty][tx] -= s[ty][j] * s[tx][j];
    }
    __syncthreads();
    if (ty < nb && tx < nb) A[(size_t)(kb + ty) * lda + kb + tx] = (tx <= ty) ? s[ty][tx] : 0.;
}

__global__ void __launch_bounds__(128) chol_trsm_kernel(double *A, int lda, int P, int kb)
{
    __shared__ double L[NB][NB + 1];
    const int nb = min(NB, P - kb);
    for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) {
        int r = e / NB, c = e - r * NB;
        L[r][c] = (r < nb && c < nb) ? A[(size_t)(kb + r) * lda + kb + c] : (r == c ? 1. : 0.);
    }
    __syncthreads();
    const int i = kb + nb + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    double r[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) r[j] = (j < nb) ? A[(size_t)i * lda + kb + j] : 0.;
#pragma unroll
    for (int j = 0; j < NB; ++j) {
        double s = r[j];
#pragma unroll
        for (int k = 0; k < j; ++k) s = fma(-r[k], L[j][k], s);
        r[j] = s / L[j][j];
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) if (j < nb) A[(size_t)i * lda + kb + j] = r[j];
}

__global__ void __launch_bounds__(256) chol_syrk_kernel(double *A, int lda, int P, int kb)
{
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    const int nb = min(NB, P - kb);
    const int base = kb + nb;
    const int i0 = base + bi * 64, j0 = base + bj * 64;
    __shared__ double Pi[64][NB + 1], Pj[64][NB + 1];
    for (int e = threadIdx.x; e < 64 * NB; e += 256) {
        int r = e / NB, c = e - r * NB;
        Pi[r][c] = (i0 + r < P && c < nb) ? A[(size_t)(i0 + r) * lda + kb + c] : 0.;
        Pj[r][c] = (j0 + r < P && c < nb) ? A[(size_t)(j0 + r) * lda + kb + c] : 0.;
    }
    __syncthreads();
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.;
#pragma unroll 8
    for (int k = 0; k < NB; ++k) {
        double pa[4], pb[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) { pa[a] = Pi[ty * 4 + a][k]; pb[a] = Pj[tx * 4 + a][k]; }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = fma(pa[a], pb[b], acc[a][b]);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int i = i0 + ty * 4 + a, j = j0 + tx * 4 + b;
            if (i < P && j < P && j <= i) A[(size_t)i * lda + j] -= acc[a][b];
        }
}

__global__ void transpose_lower_kernel(const double *__restrict__ L, int P, double *__restrict__ U)
{
    __shared__ double t[32][33];
    int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    int i = by + threadIdx.y, j = bx + threadIdx.x;
    t[threadIdx.y][threadIdx.x] = (i < P && j < P) ? L[(size_t)i * P + j] : 0.;
    __syncthreads();
    int ii = bx + threadIdx.y, jj = by + threadIdx.x;
    if (ii < P && jj < P) U[(size_t)ii * P + jj] = t[threadIdx.x][threadIdx.y];
}

// one CTA per right-hand side: L z = b (using U = L^T for coalesced rows), then L^T c = z.  Column-oriented substitution: step j
// fixes one unknown and updates the rest with one AXPY over a row of U (of L on the way back), one barrier per step.  The row of
// step j + 1 is loaded into registers while step j runs (the steps are latency bound: 2 P dependent steps, each a barrier, a shared-
// memory read, a division and the row load -- unpipelined the L2 latency of that load was most of the 1.7 ms at P = 1054).
__global__ void __launch_bounds__(1024) chol_solve_kernel(const double *__restrict__ L, const double *__restrict__ U, int P,
                                                          const double *__restrict__ B, int nr, double *__restrict__ X)
{
    extern __shared__ double sm[];
    double *z = sm, *o = sm + P;
    const int col = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    constexpr int PF = 4;                                   // row elements per thread held in registers: P <= PF * blockDim.x
    for (int i = tid; i < P; i += nt) z[i] = B[(size_t)i * nr + col];
    if (P > PF * nt) {                                      // (not reached: the fit caps P far below) unpipelined fall-back
        for (int j = 0; j < P; ++j) {
            __syncthreads();
            const double zj = z[j] / U[(size_t)j * P + j];
            if (tid == 0) o[j] = zj;
            const double *Uj = U + (size_t)j * P;
            for (int i = j + 1 + tid; i < P; i += nt) z[i] = fma(-Uj[i], zj, z[i]);
        }
        __syncthreads();
        for (int j = P - 1; j >= 0; --j) {
            __syncthreads();
            const double cj = o[j] / L[(size_t)j * P + j];
            if (tid == 0) z[j] = cj;
            const double *Lj = L + (size_t)j * P;
            for (int k = tid; k < j; k += nt) o[k] = fma(-Lj[k], cj, o[k]);
        }
    } else {
        double u[PF], d;
        auto load_u = [&](int j) {                          // row j of U right of the diagonal, and the diagonal
            const double *Uj = U + (size_t)j * P;
            d = Uj[j];
#pragma unroll
            for (int e = 0; e < PF; ++e) { const int i = j + 1 + tid + e * nt; u[e] = (i < P) ? Uj[i] : 0.; }
        };
        load_u(0);
        for (int j = 0; j < P; ++j) {
            __syncthreads();
            const double zj = z[j] / d;
            if (tid == 0) o[j] = zj;
            double un[PF];
#pragma unroll
            for (int e = 0; e < PF; ++e) un[e] = u[e];
            const int jn = (j + 1 < P) ? j + 1 : j;
            load_u(jn);                                     // in flight across the barrier of the next step
#pragma unroll
            for (int e = 0; e < PF; ++e) { const int i = j + 1 + tid + e * nt; if (i < P) z[i] = fma(-un[e], zj, z[i]); }
        }
        __syncthreads();
        auto load_l = [&](int j) {                          // row j of L left of the diagonal, and the diagonal
            const double *Lj = L + (size_t)j * P;
            d = Lj[j];
#pragma unroll
            for (int e = 0; e < PF; ++e) { const int k = tid + e * nt; u[e] = (k < j) ? Lj[k] : 0.; }
        };
        load_l(P - 1);
        for (int j = P - 1; j >= 0; --j) {
            __syncthreads();
            const double cj = o[j] / d;
            if (tid == 0) z[j] = cj;                        // z now collects the solution
            double un[PF];
#pragma unroll
            for (int e = 0; e < PF; ++e) un[e] = u[e];
            const int jn = (j > 0) ? j - 1 : 0;
            load_l(jn);
#pragma unroll
            for (int e = 0; e < PF; ++e) { const int k = tid + e * nt; if (k < j) o[k] = fma(-un[e], cj, o[k]); }
        }
    }
    __syncthreads();
    for (int i = tid; i < P; i += nt) X[(size_t)i * nr + col] = z[i];
}

// R = Bs - As * X   (As symmetric P x P, X and Bs are P x nr); one warp per (row, rhs)
__global__ void __launch_bounds__(128) residual_kernel(const double *__restrict__ As, int P, const double *__restrict__ X,
                                                       const double *__restrict__ Bs, int nr, double *__restrict__ R)
{
    const int lane = threadIdx.x & 31;
    int64_t wid = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (wid >= (int64_t)P * nr) return;
    int i = (int)(wid / nr), c = (int)(wid - (int64_t)i * nr);
    double s = 0.;
    for (int k = lane; k < P; k += 32) s = fma(As[(size_t)i * P + k], X[(size_t)k * nr + c], s);
    s = warp_sum(s);
    if (lane == 0) R[(size_t)i * nr + c] = Bs[(size_t)i * nr + c] - s;
}

__global__ void axpy_kernel(double *x, const double *d, int64_t len)
{
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < len) x[e] += d[e];
}

static int cholesky_device(bfb_context *h, double *A, int P, int *d_info)
{
    for (int kb = 0; kb < P; kb += NB) {
        chol_diag_kernel<<<1, dim3(NB, NB), 0, h->stream>>>(A, P, P, kb, d_info);
        h->launches++;
        const int rest = P - kb - NB;
        if (rest > 0) {
            chol_trsm_kernel<<<(rest + 127) / 128, 128, 0, h->stream>>>(A, P, P, kb);
            const int nblk = (rest + 63) / 64;
            chol_syrk_kernel<<<dim3(nblk, nblk), 256, 0, h->stream>>>(A, P, P, kb);
            h->launches += 2;
        }
    }
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

extern "C" int bfb_fit_solve(bfb_handle h, double *coef_out, double *rel_resid)
{
    BFB_REQUIRE(h && h->fit, BFB_ERR_STATE, "bfb_fit_solve: call bfb_fit_begin / accumulate first");
    BFB_CUDA(cudaSetDevice(h->device));
    FitState *fs = h->fit;
    double worst = 0.;
    for (FitGroup &g : fs->groups) {
        const int P = g.P, nr = (int)g.outputs.size();
        double *A, *As, *U, *Bs, *X, *R, *D, *dsc;
        int *d_info;
        TmpList tmp;
        auto dmal = [&](size_t bytes, void **p) -> int { BFB_CUDA(cudaMalloc(p, bytes)); tmp.push_back(*p); return BFB_OK; };
        int rc;
        if ((rc = dmal(sizeof(double) * P * P, (void **)&A)) || (rc = dmal(sizeof(double) * P * P, (void **)&As)) ||
            (rc = dmal(sizeof(double) * P * P, (void **)&U)) || (rc = dmal(sizeof(double) * P * nr, (void **)&Bs)) ||
            (rc = dmal(sizeof(double) * P * nr, (void **)&X)) || (rc = dmal(sizeof(double) * P * nr, (void **)&R)) ||
            (rc = dmal(sizeof(double) * P * nr, (void **)&D)) || (rc = dmal(sizeof(double) * P, (void **)&dsc)) ||
            (rc = dmal(sizeof(int), (void **)&d_info)))
            return rc;
        BFB_CUDA(cudaMemsetAsync(d_info, 0, sizeof(int), h->stream));
        const int64_t tot = (int64_t)P * (P + nr);
        assemble_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(fs->buf + g.g_off, g.Ptp, P, nr, A, Bs, dsc);
        h->launches++;
        BFB_CUDA(cudaMemcpyAsync(As, A, sizeof(double) * P * P, cudaMemcpyDeviceToDevice, h->stream));
        if ((rc = cholesky_device(h, A, P, d_info))) return rc;
        transpose_lower_kernel<<<dim3((P + 31) / 32, (P + 31) / 32), dim3(32, 32), 0, h->stream>>>(A, P, U);
        h->launches++;
        const size_t smem = sizeof(double) * 2 * P;
        BFB_CUDA(cudaFuncSetAttribute(chol_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        chol_solve_kernel<<<nr, 1024, smem, h->stream>>>(A, U, P, Bs, nr, X);
        h->launches++;
        const int64_t nw = (int64_t)P * nr;
        for (int it = 0; it < 2; ++it) {      // iterative refinement on the equilibrated system
            residual_kernel<<<(unsigned)((nw + 3) / 4), 128, 0, h->stream>>>(As, P, X, Bs, nr, R);
            chol_solve_kernel<<<nr, 1024, smem, h->stream>>>(A, U, P, R, nr, D);
            axpy_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, h->stream>>>(X, D, nw);
            h->launches += 3;
        }
        residual_kernel<<<(unsigned)((nw + 3) / 4), 128, 0, h->stream>>>(As, P, X, Bs, nr, R);
        h->launches++;
        BFB_CUDA(cudaGetLastError());
        std::vector<double> hx((size_t)P * nr), hr((size_t)P * nr), hb((size_t)P * nr), hd(P);
        int info = 0;
        BFB_CUDA(cudaMemcpyAsync(hx.data(), X, sizeof(double) * P * nr, cudaMemcpyDeviceToHost, h->stream));
        BFB_CUDA(cudaMemcpyAsync(hr.data(), R, sizeof(double) * P * nr, cudaMemcpyDeviceToHost, h->stream));
        BFB_CUDA(cudaMemcpyAsync(hb.data(), Bs, sizeof(double) * P * nr, cudaMemcpyDeviceToHost, h->stream));
        BFB_CUDA(cudaMemcpyAsync(hd.data(), dsc, sizeof(double) * P, cudaMemcpyDeviceToHost, h->stream));
        BFB_CUDA(cudaMemcpyAsync(&info, d_info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        BFB_CUDA(cudaStreamSynchronize(h->stream));
        for (void *p : tmp) cudaFree(p);
    tmp.clear();
        BFB_REQUIRE(info == 0, BFB_ERR_NUMERIC,
                    "fit: the normal equations are not positive definite (pivot %d of %d): the design matrix is rank "
                    "deficient (duplicated / too few points?)", info, P);
        double rn = 0., bn = 0.;
        for (size_t e = 0; e < hr.size(); ++e) { rn += hr[e] * hr[e]; bn += hb[e] * hb[e]; }
        worst = std::max(worst, bn > 0. ? std::sqrt(rn / bn) : 0.);
        // un-scale and scatter into the packed per-config layout
        for (int c = 0; c < nr; ++c) {
            const int o = g.outputs[c];
            int row = 0;
            for (int cid : g.cfg_ids) {
                const HostConfig &hc = h->configs[cid];
                int q = (int)(std::find(hc.out_mask.begin(), hc.out_mask.end(), (int64_t)o) - hc.out_mask.begin());
                double *dst = h->packed.data() + hc.coef_off + (int64_t)q * hc.n_packed;
                for (int64_t k = 0; k < hc.n_packed; ++k, ++row) dst[k] = hx[(size_t)row * nr + c] * hd[row];
            }
        }
    }
    if (coef_out) memcpy(coef_out, h->packed.data(), sizeof(double) * h->packed.size());
    if (rel_resid) *rel_resid = worst;
    return bfb_upload_model(h);
}
