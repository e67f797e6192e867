// bfb_diag.cu -- split-R-hat and effective sample size of sampled chains on the device: the per-coordinate partial sums that
// bayesfast_b200/diag.py finishes on the host (and all-reduces first when the chains are sharded over GPUs).
//
// The draws x[c, t, j] of the kept iterations t0 .. t0 + N are split into M' = 2 C half-chains of L = N / 2 draws (the middle draw
// of an odd N is dropped).  Per coordinate j the partials are, in this order (bfb200.h: bfb_chain_diagnostics):
//   M' | mean of the half-chain means m_c | sum_c (m_c - mean)^2 | S(k) = sum_c sum_t y_c[t] y_c[t + k], k = 0 .. L - 1,
// y_c = x_c - m_c.  S(k) is the sum of the k-th superdiagonal of the Gram G_j = Y_j^T Y_j of the M' x L matrix of centred half-chains:
//   means     : one pass over the rows (n contiguous), half-chain means in a fixed summation order;
//   meanstat  : mean and M2 of the M' means per coordinate, two passes with a fixed tree reduction;
//   center    : the centred draws transposed to Y [n][M'][Lp] (time contiguous, zero padded to Lp = 64 ceil(L / 64)): a staged block
//               of rows serves every coordinate of a slab, and the Gram kernel then reads one coordinate's panels contiguously;
//   lagsum    : the upper block triangle of every G_j on FP64 tensor cores (the 64 x 64 tiles of bfb_gram.cuh, half-chains are the K
//               dimension), split over chunks of half-chains; a tile's epilogue folds its 127 diagonals into S partials, G is never
//               stored; a second kernel adds tiles and chunks in a fixed order.  No atomics: repeated calls are bit-identical.
#include "bfb_common.cuh"
#include "bfb_gram.cuh"
#include <algorithm>

namespace {

constexpr int DIAG_TW = 32;      // time steps per block of the transposing kernel
constexpr int DIAG_SLAB = 64;    // coordinates per block of the transposing kernel
constexpr int NDIAG = 2 * TS - 1;

// hm[hc][j] = mean of half-chain hc = 2 c + h of coordinate j; one block per chain, thread (h, j) walks its L draws in order
__global__ void __launch_bounds__(256) diag_means_kernel(const double *__restrict__ x, int64_t T, int64_t t0, int64_t N, int n,
                                                         double *__restrict__ hm)
{
    const int64_t c = blockIdx.x;
    const int64_t L = N / 2;
    for (int e = threadIdx.x; e < 2 * n; e += blockDim.x) {
        const int h = e / n, j = e - h * n;
        const double *p = x + (c * T + t0 + h * (N - L)) * n + j;
        double s0 = 0., s1 = 0., s2 = 0., s3 = 0.;
        int64_t t = 0;
        for (; t + 4 <= L; t += 4) {
            s0 += p[t * n]; s1 += p[(t + 1) * n]; s2 += p[(t + 2) * n]; s3 += p[(t + 3) * n];
        }
        for (; t < L; ++t) s0 += p[t * n];
        hm[(2 * c + h) * n + j] = ((s0 + s1) + (s2 + s3)) / (double)L;
    }
}

// fixed-order tree sum of the 256 values of a block
__device__ double block_sum256(double v, double *red)
{
    red[threadIdx.x] = v;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

// P[j][0..2] = M', mean of the half-chain means, sum of squared deviations from it; one block per coordinate
__global__ void __launch_bounds__(256) diag_meanstat_kernel(const double *__restrict__ hm, int64_t Mp, int n, int64_t ldp,
                                                            double *__restrict__ P)
{
    __shared__ double red[256];
    const int j = blockIdx.x;
    double s = 0.;
    for (int64_t c = threadIdx.x; c < Mp; c += 256) s += hm[c * n + j];
    const double mean = block_sum256(s, red) / (double)Mp;
    double q = 0.;
    for (int64_t c = threadIdx.x; c < Mp; c += 256) { const double d = hm[c * n + j] - mean; q += d * d; }
    const double m2 = block_sum256(q, red);
    if (threadIdx.x == 0) { P[j * ldp] = (double)Mp; P[j * ldp + 1] = mean; P[j * ldp + 2] = m2; }
}

// Y[j][hc][t] = x[c, t0 + h (N - L) + t, j] - hm[hc][j] for t < L, 0 for L <= t < Lp.  Block = (half-chain, window of DIAG_TW steps)
// x (slab of DIAG_SLAB coordinates): reads whole row segments, writes DIAG_TW contiguous steps per coordinate.
__global__ void __launch_bounds__(256) diag_center_kernel(const double *__restrict__ x, int64_t T, int64_t t0, int64_t N, int n,
                                                          int64_t Mp, int Lp, const double *__restrict__ hm, double *__restrict__ Y)
{
    __shared__ double tile[DIAG_TW][DIAG_SLAB + 1];
    const int nw = Lp / DIAG_TW;
    const int64_t hc = blockIdx.x / nw;
    const int w = (int)(blockIdx.x - hc * nw);
    const int j0 = blockIdx.y * DIAG_SLAB, nj = min(DIAG_SLAB, n - j0);
    const int64_t L = N / 2, c = hc >> 1;
    const int64_t row0 = c * T + t0 + (hc & 1) * (N - L) + (int64_t)w * DIAG_TW;
    for (int e = threadIdx.x; e < DIAG_TW * DIAG_SLAB; e += 256) {
        const int u = e / DIAG_SLAB, jj = e - u * DIAG_SLAB;
        if (jj < nj)
            tile[u][jj] = ((int64_t)w * DIAG_TW + u < L) ? x[(row0 + u) * n + j0 + jj] - hm[hc * n + j0 + jj] : 0.;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < DIAG_TW * DIAG_SLAB; e += 256) {
        const int jj = e / DIAG_TW, u = e - jj * DIAG_TW;
        if (jj < nj) Y[((size_t)(j0 + jj) * Mp + hc) * Lp + (size_t)w * DIAG_TW + u] = tile[u][jj];
    }
}

// One CTA = tile (ti <= tj) of G_j over one chunk of half-chains: stages the two KC x 64 panels of Y_j (rows past M' are zero),
// multiplies them on the tensor cores, and folds the tile's diagonals d = c - r into ws[chunk][j][tile][d + 63]
// (lag 64 (tj - ti) + d; the lower half of a diagonal tile repeats its upper half and is left out).
__global__ void __launch_bounds__(128) lagsum_kernel(const double *__restrict__ Y, int64_t Mp, int Lp, int nt, int n_tiles,
                                                     int64_t rows_per_chunk, double *__restrict__ ws)
{
    extern __shared__ double sm[];
    const int j = blockIdx.x / n_tiles, tile = blockIdx.x - j * n_tiles;
    int t = tile, ti = 0;
    while (t >= nt - ti) { t -= nt - ti; ++ti; }
    const int tj = ti + t;
    const bool diag = (ti == tj);
    double *phiI = sm, *phiJ = diag ? sm : sm + KC * LDP;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
    const int u = tid & (TS - 1), khalf = tid >> 6;
    double acc[4][4][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.;
    const double *Yj = Y + (size_t)j * Mp * Lp;
    const int64_t r_begin = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r_end = min(Mp, r_begin + rows_per_chunk);
    for (int64_t r0 = r_begin; r0 < r_end; r0 += KC) {
        __syncthreads();
#pragma unroll 4
        for (int k = khalf; k < KC; k += 2) {
            const bool in = r0 + k < r_end;
            const double *yr = Yj + (size_t)(r0 + k) * Lp;
            phiI[k * LDP + u] = in ? yr[ti * TS + u] : 0.;
            if (!diag) phiJ[k * LDP + u] = in ? yr[tj * TS + u] : 0.;
        }
        __syncthreads();
        gram_tile_mma(phiI, phiJ, lane, wm, wn, acc);
    }
    __syncthreads();
    double *E = sm;                                   // [TS][TS + 1]: the tile, rows r, columns c
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int r = 32 * wm + 8 * a + (lane >> 2), c = 32 * wn + 8 * b + 2 * (lane & 3);
            E[r * (TS + 1) + c] = acc[a][b][0];
            E[r * (TS + 1) + c + 1] = acc[a][b][1];
        }
    __syncthreads();
    if (tid < NDIAG) {
        const int d = tid - (TS - 1);
        double s = 0.;
        if (!(diag && d < 0))
            for (int r = max(0, -d); r < min(TS, TS - d); ++r) s += E[r * (TS + 1) + r + d];
        ws[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * NDIAG + tid] = s;    // blockIdx.x = j n_tiles + tile
    }
}

// P[j][3 + k] = S(k): over chunks, then the (at most two) tile diagonals holding lag k, then their tiles, in a fixed order
__global__ void lagsum_reduce_kernel(const double *__restrict__ ws, int n, int nt, int n_tiles, int n_chunks, int64_t L,
                                     int64_t ldp, double *__restrict__ P)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * L) return;
    const int j = (int)(i / L);
    const int k = (int)(i - (int64_t)j * L);
    double s = 0.;
    for (int ch = 0; ch < n_chunks; ++ch) {
        const double *w = ws + ((size_t)ch * n + j) * n_tiles * NDIAG;
        for (int dt = k / TS; dt <= k / TS + 1 && dt < nt; ++dt) {
            const int d = k - TS * dt;
            if (d < -(TS - 1)) continue;
            for (int ti = 0; ti + dt < nt; ++ti) {
                const int tile = ti * nt - ti * (ti - 1) / 2 + dt;
                s += w[(size_t)tile * NDIAG + d + TS - 1];
            }
        }
    }
    P[j * ldp + 3 + k] = s;
}

int ensure_diag_ws(bfb_context *h, size_t len)
{
    if (h->diag_ws_len >= len) return BFB_OK;
    if (h->diag_ws) cudaFree(h->diag_ws);
    h->diag_ws = nullptr; h->diag_ws_len = 0;
    const cudaError_t e = cudaMalloc((void **)&h->diag_ws, sizeof(double) * len);
    if (e != cudaSuccess) {
        cudaGetLastError();
        bfb_set_error("chain diagnostics: cannot allocate the %.2f GB device workspace (%s)", 8e-9 * (double)len, cudaGetErrorString(e));
        return BFB_ERR_CUDA;
    }
    h->diag_ws_len = len;
    return BFB_OK;
}

} // namespace

// Queue the diagnostics of the device draws x [C, T, n] (kept range t0 .. t0 + N) on h->stream; *dev_partials receives the device
// address of the n x (L + 3) partials, valid until the next call on this handle.
int bfb_diag_enqueue(bfb_context *h, const double *x, int64_t C, int64_t T, int64_t t0, int64_t N, int n, const double **dev_partials)
{
    const int64_t L = N / 2, Mp = 2 * C, ldp = L + 3;
    const int nt = (int)((L + TS - 1) / TS), Lp = nt * TS, n_tiles = nt * (nt + 1) / 2;
    // enough (tile, coordinate, chunk) CTAs for ~4 waves, but at least 8 stages of half-chains per chunk
    const int64_t ctas = (int64_t)n_tiles * n;
    const int64_t want = ((int64_t)h->sm_count * 16 + ctas - 1) / ctas, max_chunks = (Mp + 8 * KC - 1) / (8 * KC);
    int n_chunks = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(want, max_chunks), 65535));
    const int64_t rows_per_chunk = ((Mp + n_chunks - 1) / n_chunks + KC - 1) / KC * KC;
    n_chunks = (int)((Mp + rows_per_chunk - 1) / rows_per_chunk);
    BFB_REQUIRE(ctas < (1ll << 31), BFB_ERR_ARG, "chain diagnostics: too many coordinates x lag tiles");
    const size_t lenY = (size_t)n * Mp * Lp, lenM = (size_t)Mp * n, lenW = (size_t)n_chunks * ctas * NDIAG, lenP = (size_t)n * ldp;
    int rc = ensure_diag_ws(h, lenY + lenM + lenW + lenP);
    if (rc) return rc;
    double *Y = h->diag_ws, *hm = Y + lenY, *ws = hm + lenM, *P = ws + lenW;
    const int thr = (int)std::min<int64_t>(256, (2 * n + 31) / 32 * 32);
    diag_means_kernel<<<(unsigned)C, thr, 0, h->stream>>>(x, T, t0, N, n, hm);
    diag_meanstat_kernel<<<n, 256, 0, h->stream>>>(hm, Mp, n, ldp, P);
    diag_center_kernel<<<dim3((unsigned)(Mp * (Lp / DIAG_TW)), (n + DIAG_SLAB - 1) / DIAG_SLAB), 256, 0, h->stream>>>(
        x, T, t0, N, n, Mp, Lp, hm, Y);
    const size_t smem = sizeof(double) * 2 * KC * LDP;
    static_assert(2 * KC * LDP >= TS * (TS + 1), "the epilogue tile reuses the panels' shared memory");
    lagsum_kernel<<<dim3((unsigned)ctas, n_chunks), 128, smem, h->stream>>>(Y, Mp, Lp, nt, n_tiles, rows_per_chunk, ws);
    const int64_t nk = (int64_t)n * L;
    lagsum_reduce_kernel<<<(unsigned)((nk + 127) / 128), 128, 0, h->stream>>>(ws, n, nt, n_tiles, n_chunks, L, ldp, P);
    h->launches += 5;
    BFB_CUDA(cudaGetLastError());
    *dev_partials = P;
    return BFB_OK;
}

extern "C" int bfb_chain_diagnostics(bfb_handle h, const double *x, int64_t C, int64_t T_total, int64_t t0, int64_t N, int n,
                                     int loc, double *partials)
{
    BFB_REQUIRE(h && x && partials, BFB_ERR_ARG, "bfb_chain_diagnostics: null argument");
    BFB_REQUIRE(loc == BFB_HOST || loc == BFB_DEVICE, BFB_ERR_ARG, "bfb_chain_diagnostics: bad location");
    BFB_REQUIRE(C >= 1 && n >= 1 && N >= 4 && t0 >= 0 && t0 + N <= T_total && N / 2 < (1ll << 30), BFB_ERR_ARG,
                "bfb_chain_diagnostics: need C >= 1, n >= 1, N >= 4 and 0 <= t0, t0 + N <= T_total (C=%lld T_total=%lld t0=%lld N=%lld n=%d)",
                (long long)C, (long long)T_total, (long long)t0, (long long)N, n);
    BFB_CUDA(cudaSetDevice(h->device));
    const double *dx = x;
    void *tmp = nullptr;
    struct Guard { void *&p; ~Guard() { if (p) cudaFree(p); } } guard{tmp};
    if (loc == BFB_HOST) {
        const size_t bytes = sizeof(double) * (size_t)C * (size_t)T_total * (size_t)n;
        BFB_CUDA(cudaMalloc(&tmp, bytes));
        BFB_CUDA(cudaMemcpyAsync(tmp, x, bytes, cudaMemcpyHostToDevice, h->stream));
        dx = (const double *)tmp;
    }
    const double *P = nullptr;
    BFB_CUDA(cudaEventRecord(h->ev0, h->stream));
    int rc = bfb_diag_enqueue(h, dx, C, T_total, t0, N, n, &P);
    if (rc) return rc;
    BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
    BFB_CUDA(cudaMemcpyAsync(partials, P, sizeof(double) * (size_t)n * (size_t)(N / 2 + 3), cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    BFB_CUDA(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    return BFB_OK;
}
