// bfb_nuts_common.cuh -- pieces shared by the multi-chain-per-warp NUTS kernels (bfb_sampler_dmma.cu, bfb_sampler_team.cu,
// bfb_sampler_pair.cu): linear-domain multinomial weights, the run-output descriptor, the work queue and the deep tree stack.
#pragma once
#include "bfb_common.cuh"
#include <cstdlib>

struct RunOutDevF {
    bfb_run_out o;
    int32_t n_iter;
};

struct WT { double m; int k; };   // weight = m * 2^k, m in [1, 2) (or m == 0)

__device__ __forceinline__ double pow2i(int d)   // 2^d for d in [-1022, 1023], 0 below, +inf above
{
    if (d < -1022) return 0.;
    if (d > 1023) return INFINITY;
    return __longlong_as_double((long long)(d + 1023) << 52);
}
__device__ __forceinline__ WT wt_from_dE(double dE)
{
    // exp(-dE) = 2^y, y = -dE * log2(e)
    const double y = -dE * 1.4426950408889634;
    const double kf = floor(y);
    WT w;
    w.m = exp2(y - kf);
    w.k = (int)kf;
    return w;
}
__device__ __forceinline__ WT wt_add(WT a, WT b)
{
    WT r;
    if (a.k >= b.k) { r.m = fma(b.m, pow2i(b.k - a.k), a.m); r.k = a.k; }
    else { r.m = fma(a.m, pow2i(a.k - b.k), b.m); r.k = b.k; }
    if (r.m >= 2.) { r.m *= 0.5; r.k += 1; }
    return r;
}
// u * a < b
__device__ __forceinline__ bool wt_select(double u, WT a, WT b)
{
    return u * a.m < b.m * pow2i(b.k - a.k);
}
__device__ __forceinline__ double wt_min1(WT w) { return (w.k >= 0) ? 1. : w.m * pow2i(w.k); }

#define BFB_NSLOT 12   // proposal slots per chain: tree proposal + one per pending subtree (<= L - 1) + the current one

// queue[0] = head, queue[1] = tail, queue[2 .. 2 + n_groups) = chunks finished per group, then ring[n_units]: ids of the
// groups whose next chunk can start (initially every group once; a group is appended again when one of its chunks completes)
// head0 > 0: the first head0 units are pre-assigned (warp slot s = blockIdx.x + gridDim.x * warp takes unit s without an atomic),
// which deals the groups evenly over ALL blocks when there are fewer groups than warp slots
static __global__ void queue_init_kernel(int *queue, int n_groups, int n_units, int head0 = 0)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { queue[0] = head0; queue[1] = n_groups; }
    if (i < n_groups) queue[2 + i] = 0;
    if (i < n_units) queue[2 + n_groups + i] = (i < n_groups) ? i : -1;
}

// Work queue of a persistent sampler kernel for n_iter iterations of n_groups groups: units of chunk_iters iterations
// (default_chunks per group, at least 16 iterations each, BFB200_CHUNK_ITERS overrides), h->queue grown to hold the queue and
// `extra` ints behind it, and the initialiser launched on h->stream.
static inline int queue_setup(bfb_context *h, int n_groups, int n_iter, int default_chunks, int head0, size_t extra,
                              int &chunk_iters, int &n_units)
{
    chunk_iters = (n_iter + default_chunks - 1) / default_chunks;
    if (chunk_iters < 16) chunk_iters = n_iter < 16 ? n_iter : 16;
    if (const char *e = getenv("BFB200_CHUNK_ITERS")) { int v = atoi(e); if (v >= 1) chunk_iters = v; }
    const int n_chunks = (n_iter + chunk_iters - 1) / chunk_iters;
    const int64_t n_units64 = (int64_t)n_groups * n_chunks;
    BFB_REQUIRE(n_units64 < (1ll << 31), BFB_ERR_ARG, "too many work units");
    n_units = (int)n_units64;
    const size_t qlen = 2 + (size_t)n_groups + (size_t)n_units64 + extra;
    if (qlen > h->queue_len) {
        if (h->queue) cudaFree(h->queue);
        h->queue = nullptr; h->queue_len = 0;
        BFB_CUDA(cudaMalloc((void **)&h->queue, sizeof(int) * qlen));
        h->queue_len = qlen;
    }
    queue_init_kernel<<<(unsigned)((n_units64 + 255) / 256), 256, 0, h->stream>>>(h->queue, n_groups, n_units, head0);
    h->launches++;
    return BFB_OK;
}

// h->gstack of a tree-building kernel, grown on demand: per group the stack levels LS + 1 .. L - 1 that do not fit in shared
// memory (3 vectors of `slot` doubles each) at h->gstack, then per group the proposal pool (n_prop x 2 vectors) at *gprop
static inline int gstack_reserve(bfb_context *h, int n_groups, int L, int LS, int slot, int n_prop, double **gprop)
{
    const size_t deep = (size_t)(L - 1 > LS ? L - 1 - LS : 0) * 3 * slot, prop = (size_t)n_prop * 2 * slot;
    if ((deep + prop) * (size_t)n_groups > h->gstack_len) {
        if (h->gstack) cudaFree(h->gstack);
        h->gstack = nullptr; h->gstack_len = 0;
        BFB_CUDA(cudaMalloc((void **)&h->gstack, sizeof(double) * (deep + prop) * (size_t)n_groups));
        h->gstack_len = (deep + prop) * (size_t)n_groups;
    }
    *gprop = h->gstack + deep * (size_t)n_groups;
    return BFB_OK;
}
