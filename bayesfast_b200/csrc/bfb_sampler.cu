// bfb_sampler.cu -- lock-step NUTS / HMC: one warp per chain, the whole transition (tree building,
// U-turn tests, multinomial selection, dual averaging, windowed Welford metric) on the device.
//
// Mapping.  Lane j of a warp owns dimension j (+32r) of every state vector of its chain; the binary tree
// of nuts.py:134-178 is built iteratively: leaf i of a depth-D subtree is followed by ctz(~i) merges
// against a per-level stack of completed left siblings kept in shared memory (lane-private columns, so
// no synchronisation is needed for it).  Chains in different warps never wait for each other, so chains
// with different tree depths do not mask one another; within a warp every decision is warp-uniform
// (butterfly reductions give bitwise identical sums on all lanes).
//
// Reference restated here: samplers/hmc_utils/base_hmc.py:62-85 (astep), samplers/nuts.py:27-217,
// samplers/hmc.py:16-49, hmc_utils/integration.py:28-95, hmc_utils/metrics.py:73-91,186-211,333-371,
// hmc_utils/step_size.py:10-51.  Draw order: SURVEY.md 8(a) row N-RNG; stream: include/bfb_rng.h.
#include "bfb_common.cuh"
#include "bfb_eval.cuh"
#include <algorithm>
#include <cstring>
#include <cstdio>
#include <cstdlib>

// the kernel of the family select_family chose for the model: 0 on launch, 1 when its shared memory does not fit, < 0 on error
int bfb_launch_nuts_dmma(bfb_context *h, const bfb_run_out &o, int n_iter);   // bfb_sampler_dmma.cu
int bfb_launch_hmc_dmma(bfb_context *h, const bfb_run_out &o, int n_iter);    // bfb_sampler_dmma.cu
int bfb_launch_nuts_team(bfb_context *h, const bfb_run_out &o, int n_iter);   // bfb_sampler_team.cu
int bfb_launch_hmc_team(bfb_context *h, const bfb_run_out &o, int n_iter);    // bfb_sampler_team.cu
int bfb_launch_nuts_pair(bfb_context *h, const bfb_run_out &o, int n_iter);   // bfb_sampler_pair.cu

struct RunOutDev {
    bfb_run_out o;
    int32_t n_iter;
};

// dense metric (QuadMetricFull, metrics.py:94-132): every stored momentum that can become a tree end also carries its
// velocity cov . p (3 more fixed vectors, 2 more per stack level)
__host__ __device__ inline size_t warp_smem_doubles(int np, int L, bool dense = false)
{
    size_t s = (size_t)((dense ? 15 : 12) + (dense ? 7 : 5) * L) * np + 3 * (size_t)L;
    return (s + 1) & ~(size_t)1;
}

// v = cov . p with the covariance stored transposed and padded, covT[k * np + j] = cov[j][k] (lane j reads row k coalesced;
// the Welford covariance of metrics.py:374-417 is not bitwise symmetric, so the reference's element order is kept).
// scr: np doubles of per-warp scratch.
template <int NPL>
__device__ __forceinline__ void dense_velocity(const double *__restrict__ covT, int n, int np, const double (&p)[NPL],
                                               double (&v)[NPL], int lane, double *scr)
{
    __syncwarp();
#pragma unroll
    for (int r = 0; r < NPL; ++r) { scr[lane + 32 * r] = p[r]; v[r] = 0.; }
    __syncwarp();
#pragma unroll 4
    for (int k = 0; k < n; ++k) {
        const double pk = scr[k];
#pragma unroll
        for (int r = 0; r < NPL; ++r) v[r] = fma(covT[(size_t)k * np + lane + 32 * r], pk, v[r]);
    }
    __syncwarp();
}

template <int NPL>
__device__ __forceinline__ double pdot(const double (&a)[NPL], const double (&b)[NPL])
{
    double part = 0.;
#pragma unroll
    for (int r = 0; r < NPL; ++r) part = fma(a[r], b[r], part);
    return warp_sum(part);
}

// scipy.linalg.cholesky(cov, lower=True) (metrics.py:108, 282-287) of the lower triangle of cov, left-looking by columns with
// the lanes over the rows: out[k * np + j] = L[j][k].  Returns false on a non-positive pivot (the reference then keeps its
// old factor).  diag: 1 double of per-warp scratch.
template <int NPL>
__device__ __forceinline__ bool dense_cholesky(const double *__restrict__ covT, double *__restrict__ out, int n, int np, int lane,
                                               double *diag)
{
    bool ok = true;
    for (int k = 0; k < n; ++k) {
        double s_[NPL];
#pragma unroll
        for (int r = 0; r < NPL; ++r) s_[r] = covT[(size_t)k * np + lane + 32 * r];
#pragma unroll 4
        for (int m = 0; m < k; ++m) {
            const double lkm = out[(size_t)m * np + k];
#pragma unroll
            for (int r = 0; r < NPL; ++r) s_[r] = fma(-out[(size_t)m * np + lane + 32 * r], lkm, s_[r]);
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < NPL; ++r) if (lane + 32 * r == k) diag[0] = s_[r];
        __syncwarp();
        const double d2 = diag[0];
        if (!(d2 > 0.)) { ok = false; break; }
        const double d = sqrt(d2);
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            const int j = lane + 32 * r;
            out[(size_t)k * np + j] = (j == k) ? d : (j > k && j < n) ? s_[r] / d : 0.;
        }
        __syncwarp();
    }
    return ok;
}

// QuadMetricFull.random (metrics.py:123-127): solve_triangular(chol.T, z), back substitution; cholT[k * np + j] = L[j][k],
// so row i of L^T is one coalesced load.  z / the result are lane-owned (dimension j = lane + 32 r).
template <int NPL>
__device__ __forceinline__ void dense_momentum(const double *__restrict__ cholT, int n, int np, const double (&z)[NPL],
                                               double (&x)[NPL], int lane)
{
#pragma unroll
    for (int r = 0; r < NPL; ++r) x[r] = 0.;
    double row[NPL];
#pragma unroll
    for (int r = 0; r < NPL; ++r) row[r] = cholT[(size_t)(n - 1) * np + lane + 32 * r];
    for (int i = n - 1; i >= 0; --i) {
        double nxt[NPL];
#pragma unroll
        for (int r = 0; r < NPL; ++r) nxt[r] = (i > 0) ? cholT[(size_t)(i - 1) * np + lane + 32 * r] : 0.;
        double part = 0., zi = 0., lii = 0.;
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            const int j = lane + 32 * r;
            if (j > i) part = fma(row[r], x[r], part);      // x_j of the rows already solved; zeros elsewhere
            if (j == i) { zi = z[r]; lii = row[r]; }
        }
        const double sum = warp_sum(part);
        const int src = i & 31;
        zi = __shfl_sync(BFB_FULL, zi, src); lii = __shfl_sync(BFB_FULL, lii, src);
        const double xi = (zi - sum) / lii;
#pragma unroll
        for (int r = 0; r < NPL; ++r) { if (lane + 32 * r == i) x[r] = xi; row[r] = nxt[r]; }
    }
}

template <int NPL, bool DENSE>
__device__ __forceinline__ void leapfrog(const DevModel &M, double eps, const double (&var)[NPL], const double *covT,
                                         double (&q)[NPL], double (&p)[NPL], double (&g)[NPL], double (&v)[NPL], int lane,
                                         double *xsm, double *dsm, double &logp, double &energy)
{
    // integration.py:68-95 (kick - drift - kick), metrics.py:88-91 / 129-132 (velocity_energy); v = velocity of the new state
    // (dense metric only)
    const double dt = 0.5 * eps;
#pragma unroll
    for (int r = 0; r < NPL; ++r) p[r] = fma(dt, g[r], p[r]);
    if (DENSE) {
        dense_velocity<NPL>(covT, M.n, M.np, p, v, lane, dsm);
#pragma unroll
        for (int r = 0; r < NPL; ++r) q[r] = fma(eps, v[r], q[r]);
    } else {
#pragma unroll
        for (int r = 0; r < NPL; ++r) q[r] = fma(eps, var[r] * p[r], q[r]);
    }
    density_eval<NPL>(M, q, lane, xsm, dsm, logp, g);
    double part = 0.;
#pragma unroll
    for (int r = 0; r < NPL; ++r) p[r] = fma(dt, g[r], p[r]);
    if (DENSE) {
        dense_velocity<NPL>(covT, M.n, M.np, p, v, lane, dsm);
#pragma unroll
        for (int r = 0; r < NPL; ++r) part = fma(p[r], v[r], part);
    } else {
#pragma unroll
        for (int r = 0; r < NPL; ++r) part = fma(p[r], var[r] * p[r], part);
    }
    energy = 0.5 * warp_sum(part) - logp;
}

template <int NPL>
__device__ __forceinline__ double vdot(const double (&a)[NPL], const double (&var)[NPL], const double (&b)[NPL])
{
    double part = 0.;
#pragma unroll
    for (int r = 0; r < NPL; ++r) part = fma(a[r], var[r] * b[r], part);
    return warp_sum(part);
}

#define VLD(dst, off)                                                     \
    _Pragma("unroll") for (int r_ = 0; r_ < NPL; ++r_) dst[r_] = wsm[(off) + lane + 32 * r_]
#define VST(off, src)                                                     \
    _Pragma("unroll") for (int r_ = 0; r_ < NPL; ++r_) wsm[(off) + lane + 32 * r_] = src[r_]

// U-turn products p_sum . velocity(end): the velocity is var * p (diagonal metric, recomputed) or the stored cov . p
#define UDOT(a, bp, bv) (DENSE ? pdot<NPL>(a, bv) : vdot<NPL>(a, var, bp))

template <int NPL, int SAMPLER, bool DENSE>
__global__ void __launch_bounds__(256) sampler_kernel(DevModel M, bfb_sampler_cfg cfg, ChainState st, RunOutDev out, int L)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    if (c >= st.C) return;
    const int n = M.n, np = M.np;
    double *wsm = smem + (size_t)wib * warp_smem_doubles(np, L, DENSE);
    double *xsm = wsm, *dsm = wsm + np;
    const int oTL = 2 * np, oTR = 5 * np, oPS = 8 * np, oPQ = 9 * np, oPG = 10 * np, oPB = 11 * np;
    const int oTLv = 12 * np, oTRv = 13 * np, oPBv = 14 * np;            // dense metric: velocities of the tree ends
    const int oST = (DENSE ? 15 : 12) * np, SV = DENSE ? 7 : 5;          // stack entry: pl, pr, ps, q', g' (, vl, vr)
    double *ssc = wsm + (size_t)((DENSE ? 15 : 12) + SV * L) * np;   // [3][L] scalars of the stack: log_size, energy, logp
    if (st.status[c] != 0) return;
    // dense metric state of this chain (transposed, padded: XT[k * np + j] = X[j][k]); the Welford covariances and the
    // Cholesky factor stay in global memory (L2): they are touched once per warm-up iteration / momentum draw
    const size_t mb = (size_t)c * n * np;
    double *covT = DENSE ? st.covT + mb : nullptr, *cholT = DENSE ? st.cholT + mb : nullptr, *cholW = DENSE ? st.cholW + mb : nullptr;
    double *fgcT = DENSE ? st.fgcT + mb : nullptr, *bgcT = DENSE ? st.bgcT + mb : nullptr;

    const uint64_t seed = cfg.seed, chain = (uint64_t)(cfg.chain0 + c);
    int64_t t = st.t_draw[c];
    int64_t it0 = st.iter[c];
    const size_t vb = (size_t)c * np;

    double q[NPL], g[NPL], p[NPL], v[NPL], var[NPL], inv_std[NPL];
    double fgm[NPL], fgr[NPL], bgm[NPL], bgr[NPL];
#pragma unroll
    for (int r = 0; r < NPL; ++r) {
        const int j = lane + 32 * r;
        q[r] = st.q[vb + j]; g[r] = st.g[vb + j]; var[r] = st.var[vb + j];
        inv_std[r] = 1. / sqrt(var[r]);
        fgm[r] = st.fg_mean[vb + j]; fgr[r] = st.fg_raw[vb + j];
        bgm[r] = st.bg_mean[vb + j]; bgr[r] = st.bg_raw[vb + j];
        p[r] = 0.; v[r] = 0.;
    }
    double logp_q = st.logp[c];
    double fg_n = st.fg_n[c], bg_n = st.bg_n[c];
    double log_step = st.log_step[c], log_bar = st.log_bar[c], hbar = st.hbar[c];
    const double mu_da = st.mu_da[c];
    int64_t count = st.count[c], n_samples = st.n_samples[c], previous_update = st.previous_update[c];
    int adapt_window = st.adapt_window[c];
    int status = 0;
    unsigned long long tree_total = 0;

    for (int it = 0; it < out.n_iter; ++it) {
        const bool warmup = (it0 + it) < cfg.n_warmup;
        // momentum: metrics.py:83-86
        double p0[NPL], v0[NPL];
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            const int j = lane + 32 * r;
            p0[r] = (j < n) ? (DENSE ? 1. : inv_std[r]) * bfb_draw_normal(seed, chain, (uint64_t)(t + j)) : 0.;
            v0[r] = 0.;
        }
        t += n;
        if (DENSE) {                                                  // metrics.py:123-127, 113-121
            double z[NPL];
#pragma unroll
            for (int r = 0; r < NPL; ++r) z[r] = p0[r];
            dense_momentum<NPL>(cholT, n, np, z, p0, lane);
            dense_velocity<NPL>(covT, n, np, p0, v0, lane, dsm);
        }
        const double E0 = 0.5 * UDOT(p0, p0, v0) - logp_q;           // integration.py:28-34
        if (!isfinite(E0)) { status = 2; break; }                     // base_hmc.py:72-76
        const double eps = warmup ? exp(log_step) : exp(log_bar);     // step_size.py:25-29

        double accept_stat, s_logp, s_energy, s_dE, s_maxdE = 0.;
        int s_depth, s_size, diverging = 0;

        if (SAMPLER == BFB_NUTS) {
            // Tree.__init__, nuts.py:27-43
            VST(oTL, q); VST(oTL + np, p0); VST(oTL + 2 * np, g);
            VST(oTR, q); VST(oTR + np, p0); VST(oTR + 2 * np, g);
            VST(oPS, p0); VST(oPQ, q); VST(oPG, g);
            if (DENSE) { VST(oTLv, v0); VST(oTRv, v0); }
            double prop_E = E0, prop_lp = logp_q, tree_ls = 0., acc_sum = 0., maxdE = 0.;
            int depth = 0, n_prop = 0;
            bool turn = false, nan_flag = false;
            for (int d = 0; d < cfg.max_treedepth; ++d) {
                // nuts.py:210 direction = logbern(log 0.5) * 2 - 1
                const double ud = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                const int dir = (log(ud) < -0.6931471805599453) ? 1 : -1;
                const int oEnd = dir > 0 ? oTR : oTL;
                const int oEndv = dir > 0 ? oTRv : oTLv;
                VLD(q, oEnd); VLD(p, oEnd + np); VLD(g, oEnd + 2 * np);
                VST(oPB, p);
                if (DENSE) { VLD(v, oEndv); VST(oPBv, v); }
                const double step = dir > 0 ? eps : -eps;
                const int nleaf = 1 << depth;
                double Rpl[NPL], Rps[NPL], Rqp[NPL], Rgp[NPL], Rvl[NPL];
#pragma unroll
                for (int r = 0; r < NPL; ++r) Rvl[r] = 0.;
                double Rls = 0., REp = 0., Rlpp = 0.;
                // ---- _build_subtree(depth), nuts.py:134-178, iteratively ----
                for (int i = 0; i < nleaf; ++i) {
                    double lp, E;
                    leapfrog<NPL, DENSE>(M, step, var, covT, q, p, g, v, lane, xsm, dsm, lp, E);
                    // _single_step, nuts.py:105-132
                    double dE = E - E0;
                    if (isnan(dE)) dE = INFINITY;
                    if (fabs(dE) > fabs(maxdE)) maxdE = dE;
                    n_prop += 1;
                    if (!(fabs(dE) < cfg.max_change)) { diverging = 1; break; }
                    { const double e = exp(-dE); acc_sum += e < 1. ? e : 1.; }
#pragma unroll
                    for (int r = 0; r < NPL; ++r) { Rpl[r] = p[r]; Rps[r] = p[r]; Rqp[r] = q[r]; Rgp[r] = g[r]; if (DENSE) Rvl[r] = v[r]; }
                    Rls = -dE; REp = E; Rlpp = lp;
                    int lvl = 0;
                    while ((i >> lvl) & 1) {
                        const int oS = oST + lvl * SV * np;
                        double T1pl[NPL], T1pr[NPL], T1ps[NPL], ps[NPL], T1vl[NPL], T1vr[NPL];
                        VLD(T1pl, oS); VLD(T1pr, oS + np); VLD(T1ps, oS + 2 * np);
                        if (DENSE) { VLD(T1vl, oS + 5 * np); VLD(T1vr, oS + 6 * np); }
                        else {
#pragma unroll
                            for (int r = 0; r < NPL; ++r) T1vl[r] = T1vr[r] = 0.;
                        }
#pragma unroll
                        for (int r = 0; r < NPL; ++r) ps[r] = T1ps[r] + Rps[r];
                        bool turning = (UDOT(ps, T1pl, T1vl) <= 0.) | (UDOT(ps, p, v) <= 0.);
                        if (lvl >= 1) {
                            double ps1[NPL], ps2[NPL];
#pragma unroll
                            for (int r = 0; r < NPL; ++r) { ps1[r] = T1ps[r] + Rpl[r]; ps2[r] = T1pr[r] + Rps[r]; }
                            turning |= (UDOT(ps1, T1pl, T1vl) <= 0.) | (UDOT(ps1, Rpl, Rvl) <= 0.);
                            turning |= (UDOT(ps2, T1pr, T1vr) <= 0.) | (UDOT(ps2, p, v) <= 0.);
                        }
                        const double T1ls = ssc[lvl];
                        const double ls = np_logaddexp(T1ls, Rls);
                        const double um = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                        const double lb = Rls - ls;
                        if (isnan(lb)) nan_flag = true;
                        if (!(log(um) < lb)) {   // keep tree1's proposal
                            VLD(Rqp, oS + 3 * np); VLD(Rgp, oS + 4 * np);
                            REp = ssc[L + lvl]; Rlpp = ssc[2 * L + lvl];
                        }
#pragma unroll
                        for (int r = 0; r < NPL; ++r) { Rpl[r] = T1pl[r]; Rps[r] = ps[r]; if (DENSE) Rvl[r] = T1vl[r]; }
                        Rls = ls;
                        if (turning) { turn = true; break; }
                        lvl++;
                    }
                    if (turn) break;
                    if (i + 1 < nleaf) {
                        const int oS = oST + lvl * SV * np;
                        VST(oS, Rpl); VST(oS + np, p); VST(oS + 2 * np, Rps); VST(oS + 3 * np, Rqp); VST(oS + 4 * np, Rgp);
                        if (DENSE) { VST(oS + 5 * np, Rvl); VST(oS + 6 * np, v); }
                        // every lane writes the same scalars (each lane later reads back its own write: no sync needed)
                        ssc[lvl] = Rls; ssc[L + lvl] = REp; ssc[2 * L + lvl] = Rlpp;
                    }
                }
                // Tree.extend, nuts.py:45-103
                VST(oEnd, q); VST(oEnd + np, p); VST(oEnd + 2 * np, g);
                if (DENSE) VST(oEndv, v);
                depth += 1;
                if (diverging || turn) break;
                {
                    const double ue = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                    const double lb = Rls - tree_ls;
                    if (isnan(lb)) nan_flag = true;
                    if (log(ue) < lb) { VST(oPQ, Rqp); VST(oPG, Rgp); prop_E = REp; prop_lp = Rlpp; }
                }
                tree_ls = np_logaddexp(tree_ls, Rls);
                double PS[NPL], PB[NPL], TLp[NPL], TRp[NPL], ps1[NPL], ps2[NPL], PBv[NPL], TLv[NPL], TRv[NPL];
                VLD(PS, oPS); VLD(PB, oPB); VLD(TLp, oTL + np); VLD(TRp, oTR + np);
                if (DENSE) { VLD(PBv, oPBv); VLD(TLv, oTLv); VLD(TRv, oTRv); }
                else {
#pragma unroll
                    for (int r = 0; r < NPL; ++r) PBv[r] = TLv[r] = TRv[r] = 0.;
                }
#pragma unroll
                for (int r = 0; r < NPL; ++r) PS[r] += Rps[r];
                VST(oPS, PS);
                bool turning = (UDOT(PS, TLp, TLv) <= 0.) | (UDOT(PS, TRp, TRv) <= 0.);
                // NB the reference updates self.p_sum in place before forming p_sum1 / p_sum2 (nuts.py:86-98),
                // so the "old tree" p_sum that enters them is already the total.
                if (dir > 0) {
#pragma unroll
                    for (int r = 0; r < NPL; ++r) { ps1[r] = PS[r] + Rpl[r]; ps2[r] = PB[r] + Rps[r]; }
                    turning |= (UDOT(ps1, TLp, TLv) <= 0.) | (UDOT(ps1, Rpl, Rvl) <= 0.);
                    turning |= (UDOT(ps2, PB, PBv) <= 0.) | (UDOT(ps2, p, v) <= 0.);
                } else {
#pragma unroll
                    for (int r = 0; r < NPL; ++r) { ps1[r] = Rps[r] + PB[r]; ps2[r] = Rpl[r] + PS[r]; }
                    turning |= (UDOT(ps1, p, v) <= 0.) | (UDOT(ps1, PB, PBv) <= 0.);
                    turning |= (UDOT(ps2, Rpl, Rvl) <= 0.) | (UDOT(ps2, TRp, TRv) <= 0.);
                }
                if (turning) { turn = true; break; }
            }
            if (nan_flag) { status = 3; break; }
            accept_stat = acc_sum / (double)n_prop;
            s_logp = prop_lp; s_energy = prop_E; s_depth = depth; s_size = n_prop;
            s_dE = prop_E - E0; s_maxdE = maxdE;
            VLD(q, oPQ); VLD(g, oPG);
            logp_q = prop_lp;
            tree_total += (unsigned long long)n_prop;
        } else {
            // HMC._hamiltonian_step, hmc.py:16-49
            double qs[NPL], gs[NPL];
#pragma unroll
            for (int r = 0; r < NPL; ++r) { qs[r] = q[r]; gs[r] = g[r]; p[r] = p0[r]; }
            double lp = logp_q, E = E0;
            for (int s = 0; s < cfg.n_int_step; ++s) leapfrog<NPL, DENSE>(M, eps, var, covT, q, p, g, v, lane, xsm, dsm, lp, E);
            double dE;
            if (isfinite(E)) { dE = E0 - E; diverging = fabs(dE) > cfg.max_change; }
            else { dE = -INFINITY; diverging = 1; }
            { const double e = exp(dE); accept_stat = e < 1. ? e : 1.; }
            bool accepted = false;
            if (!diverging) {
                const double ua = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                accepted = !(ua >= accept_stat);
            }
            s_logp = lp; s_energy = E; s_depth = accepted ? 1 : 0; s_size = cfg.n_int_step; s_dE = dE;
            if (accepted) logp_q = lp;
            else {
#pragma unroll
                for (int r = 0; r < NPL; ++r) { q[r] = qs[r]; g[r] = gs[r]; }
            }
            tree_total += (unsigned long long)cfg.n_int_step;
        }

        // DualAverageAdaptation.update, step_size.py:31-45
        if (warmup && cfg.adapt_step_size) {
            const double cnt = (double)count;
            const double w = 1. / (cnt + cfg.t0);
            hbar = ((1. - w) * hbar + w * (cfg.target_accept - accept_stat));
            log_step = mu_da - hbar * sqrt(cnt) / cfg.gamma;
            const double mk = pow(cnt, -cfg.k);
            log_bar = mk * log_step + (1. - mk) * log_bar;
            count += 1;
        }
        // QuadMetricDiagAdapt.update, metrics.py:186-211 with _WeightedVariance.add_sample :351-357
        if (DENSE && warmup && cfg.adapt_metric) {
            // QuadMetricFullAdapt.update, metrics.py:289-313 with _WeightedCovariance.add_sample :398-404
            // (raw_cov[i][j] += new_diff[i] * old_diff[j]; stored transposed, lane j owns new_diff[j])
            const int64_t delta = n_samples - previous_update;
            const bool upd = ((delta + 1) % cfg.update_window == 0), swap = delta >= adapt_window;
            fg_n += 1.; bg_n += 1.;
            double fn[NPL], bn[NPL];
            __syncwarp();
#pragma unroll
            for (int r = 0; r < NPL; ++r) {
                const double fo = q[r] - fgm[r], bo = q[r] - bgm[r];
                fgm[r] += fo / fg_n; bgm[r] += bo / bg_n;
                fn[r] = q[r] - fgm[r]; bn[r] = q[r] - bgm[r];
                xsm[lane + 32 * r] = fo; dsm[lane + 32 * r] = bo;
            }
            __syncwarp();
            for (int k = 0; k < n; ++k) {
                const double fok = xsm[k], bok = dsm[k];
#pragma unroll
                for (int r = 0; r < NPL; ++r) {
                    const size_t idx = (size_t)k * np + lane + 32 * r;
                    const double f = fgcT[idx] + 1. * fn[r] * fok, b = bgcT[idx] + 1. * bn[r] * bok;
                    if (upd) covT[idx] = f / fg_n;
                    // end of the adaptation window: foreground <- background, fresh background (identity x weight 10)
                    fgcT[idx] = swap ? b : f;
                    bgcT[idx] = swap ? ((lane + 32 * r == k) ? 10. : 0.) : b;
                }
            }
            __syncwarp();
            if (upd) {
                if (dense_cholesky<NPL>(covT, cholW, n, np, lane, ssc)) {
                    for (int i = lane; i < n * np; i += 32) cholT[i] = cholW[i];
                } else if (lane == 0) st.chol_error[c] = 1;      // metrics.py:284-287: the old factor stays in use
                __syncwarp();
            }
            if (swap) {
#pragma unroll
                for (int r = 0; r < NPL; ++r) { fgm[r] = bgm[r]; bgm[r] = 0.; }
                fg_n = bg_n; bg_n = 10.;
                previous_update = n_samples;
                if (cfg.doubling) adapt_window *= 2;
            }
            n_samples += 1;
        }
        if (!DENSE && warmup && cfg.adapt_metric) {
            const int64_t delta = n_samples - previous_update;
            fg_n += 1.; bg_n += 1.;
#pragma unroll
            for (int r = 0; r < NPL; ++r) {
                double od = q[r] - fgm[r];
                fgm[r] += od / fg_n;
                fgr[r] += 1. * od * (q[r] - fgm[r]);
                od = q[r] - bgm[r];
                bgm[r] += od / bg_n;
                bgr[r] += 1. * od * (q[r] - bgm[r]);
            }
            if ((delta + 1) % cfg.update_window == 0) {
#pragma unroll
                for (int r = 0; r < NPL; ++r) {
                    if (lane + 32 * r < n) { var[r] = fgr[r] / fg_n; inv_std[r] = 1. / sqrt(var[r]); }
                }
            }
            if (delta >= adapt_window) {
#pragma unroll
                for (int r = 0; r < NPL; ++r) { fgm[r] = bgm[r]; fgr[r] = bgr[r]; bgm[r] = 0.; bgr[r] = 0.; }
                fg_n = bg_n; bg_n = 10.;     // _WeightedVariance(self._n): default initial_weight 10, zero mean / variance
                previous_update = n_samples;
                if (cfg.doubling) adapt_window *= 2;
            }
            n_samples += 1;
        }

        // outputs: base_hmc.py:82-85, stats.py:12-14
        const size_t o = (size_t)c * out.n_iter + it;
        if (out.o.samples) {
#pragma unroll
            for (int r = 0; r < NPL; ++r) {
                const int j = lane + 32 * r;
                if (j < n) out.o.samples[o * n + j] = q[r];
            }
        }
        if (lane == 0) {
            if (out.o.logp) out.o.logp[o] = s_logp;
            if (out.o.energy) out.o.energy[o] = s_energy;
            if (out.o.tree_depth) out.o.tree_depth[o] = s_depth;
            if (out.o.tree_size) out.o.tree_size[o] = s_size;
            if (out.o.mean_tree_accept) out.o.mean_tree_accept[o] = accept_stat;
            if (out.o.step_size) out.o.step_size[o] = exp(log_step);
            if (out.o.step_size_bar) out.o.step_size_bar[o] = exp(log_bar);
            if (out.o.energy_change) out.o.energy_change[o] = s_dE;
            if (out.o.max_energy_change) out.o.max_energy_change[o] = s_maxdE;
            if (out.o.diverging) out.o.diverging[o] = diverging;
        }
        if (status) break;
    }

    // persist chain state
#pragma unroll
    for (int r = 0; r < NPL; ++r) {
        const int j = lane + 32 * r;
        st.q[vb + j] = q[r]; st.g[vb + j] = g[r]; st.var[vb + j] = var[r];
        st.fg_mean[vb + j] = fgm[r]; st.fg_raw[vb + j] = fgr[r];
        st.bg_mean[vb + j] = bgm[r]; st.bg_raw[vb + j] = bgr[r];
    }
    if (lane == 0) {
        st.logp[c] = logp_q; st.fg_n[c] = fg_n; st.bg_n[c] = bg_n;
        st.log_step[c] = log_step; st.log_bar[c] = log_bar; st.hbar[c] = hbar;
        st.count[c] = count; st.n_samples[c] = n_samples; st.previous_update[c] = previous_update;
        st.adapt_window[c] = adapt_window; st.t_draw[c] = t; st.iter[c] = it0 + out.n_iter;
        st.status[c] = status;
        if (tree_total) atomicAdd(st.tree_total, tree_total);
    }
}

// logp / grad at x0 and the finite check of base_hmc.py:42-46
template <int NPL>
__global__ void __launch_bounds__(128) chain_init_kernel(DevModel M, ChainState st)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    if (c >= st.C) return;
    double *xsm = smem + (size_t)wib * 2 * M.np, *dsm = xsm + M.np;
    double q[NPL], g[NPL], lp;
#pragma unroll
    for (int r = 0; r < NPL; ++r) q[r] = st.q[(size_t)c * M.np + lane + 32 * r];
    density_eval<NPL>(M, q, lane, xsm, dsm, lp, g);
    bool ok = isfinite(lp);
#pragma unroll
    for (int r = 0; r < NPL; ++r) {
        ok = ok && isfinite(g[r]);
        st.g[(size_t)c * M.np + lane + 32 * r] = g[r];
    }
    ok = __all_sync(BFB_FULL, ok);
    if (lane == 0) { st.logp[c] = lp; st.status[c] = ok ? 0 : 1; }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
template <class T>
static int dalloc(bfb_context *h, T **p, size_t count)
{
    void *v = nullptr;
    BFB_CUDA(cudaMalloc(&v, sizeof(T) * (count ? count : 1)));
    BFB_CUDA(cudaMemsetAsync(v, 0, sizeof(T) * (count ? count : 1), h->stream));
    h->chain_allocs.push_back(v);
    *p = (T *)v;
    return BFB_OK;
}

template <class T>
static int h2d(bfb_context *h, T *dst, const std::vector<T> &src)
{
    BFB_CUDA(cudaMemcpyAsync(dst, src.data(), sizeof(T) * src.size(), cudaMemcpyHostToDevice, h->stream));
    return BFB_OK;
}

// (pointer, bytes) list of every chain-state array, for snapshot / reset
static std::vector<std::pair<void *, size_t>> state_arrays(const ChainState &s)
{
    const size_t V = (size_t)s.C * s.np * sizeof(double), D = (size_t)s.C * sizeof(double), I = (size_t)s.C * sizeof(int64_t);
    return {{s.q, V}, {s.g, V}, {s.var, V}, {s.fg_mean, V}, {s.fg_raw, V}, {s.bg_mean, V}, {s.bg_raw, V},
            {s.logp, D}, {s.fg_n, D}, {s.bg_n, D}, {s.log_step, D}, {s.log_bar, D}, {s.hbar, D}, {s.mu_da, D},
            {s.count, I}, {s.n_samples, I}, {s.previous_update, I}, {s.adapt_window, (size_t)s.C * sizeof(int32_t)},
            {s.t_draw, I}, {s.iter, I}, {s.status, (size_t)s.C * sizeof(int32_t)}};
}

extern "C" int bfb_sampler_reset(bfb_handle h)
{
    BFB_REQUIRE(h && h->has_chains && !h->chain_snapshot.empty(), BFB_ERR_STATE, "bfb_sampler_reset: no chains");
    BFB_CUDA(cudaSetDevice(h->device));
    auto arrs = state_arrays(h->cs);
    for (size_t i = 0; i < arrs.size(); ++i)
        BFB_CUDA(cudaMemcpyAsync(arrs[i].first, h->chain_snapshot[i], arrs[i].second, cudaMemcpyDeviceToDevice, h->stream));
    if (h->dense_metric) {
        const ChainState &s = h->cs;
        const size_t MB = (size_t)s.C * s.n * s.np * sizeof(double);
        double *live[4] = {s.covT, s.cholT, s.fgcT, s.bgcT};
        for (int i = 0; i < 4; ++i)
            BFB_CUDA(cudaMemcpyAsync(live[i], h->dense_allocs[6 + i], MB, cudaMemcpyDeviceToDevice, h->stream));
        BFB_CUDA(cudaMemsetAsync(s.chol_error, 0, sizeof(int32_t) * s.C, h->stream));
    }
    if (h->t_u)      // tempered chains: u back to u_0
        BFB_CUDA(cudaMemcpyAsync(h->t_u, h->t_u + h->cs.C, sizeof(double) * h->cs.C, cudaMemcpyDeviceToDevice, h->stream));
    h->iters_done = 0;
    return BFB_OK;
}

static int sampler_init_common(bfb_handle h, const bfb_sampler_cfg *cfg, int64_t C, const double *x0,
                               const double *step0, const double *var0, const double *mean0)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_sampler_init: no model set");
    BFB_REQUIRE(cfg && x0 && step0 && var0 && mean0 && C > 0, BFB_ERR_ARG, "bfb_sampler_init: bad arguments");
    BFB_REQUIRE(cfg->max_treedepth > 0 && cfg->max_treedepth <= 20, BFB_ERR_ARG, "max_treedepth must be in [1,20]");
    BFB_REQUIRE(cfg->update_window > 0 && cfg->adapt_window > 0, BFB_ERR_ARG, "adapt/update window must be positive");
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    h->has_chains = false;
    h->scfg = *cfg;
    const int n = h->n, np = h->np;
    ChainState &s = h->cs;
    int rc;
    const size_t V = (size_t)C * np;
    // device arrays are kept between calls with the same shape: cudaMalloc / cudaFree are slow (and contended when every
    // GPU of a box has its own process), and sample() calls this once per run
    const bool reuse = !h->chain_allocs.empty() && h->alloc_C == C && h->alloc_np == np && !h->chain_snapshot.empty();
    if (reuse) {
        for (auto &a : state_arrays(s)) BFB_CUDA(cudaMemsetAsync(a.first, 0, a.second, h->stream));
        BFB_CUDA(cudaMemsetAsync(s.tree_total, 0, BFB_TREE_TOTAL_LEN * sizeof(unsigned long long), h->stream));
    } else {
        bfb_free_list(h->chain_allocs);
        h->chain_snapshot.clear();
        h->alloc_C = 0; h->alloc_np = 0;
        memset(&s, 0, sizeof(s));
        s.C = C; s.n = n; s.np = np;
        if ((rc = dalloc(h, &s.q, V)) || (rc = dalloc(h, &s.g, V)) || (rc = dalloc(h, &s.var, V)) ||
            (rc = dalloc(h, &s.fg_mean, V)) || (rc = dalloc(h, &s.fg_raw, V)) || (rc = dalloc(h, &s.bg_mean, V)) ||
            (rc = dalloc(h, &s.bg_raw, V)) || (rc = dalloc(h, &s.logp, C)) || (rc = dalloc(h, &s.fg_n, C)) ||
            (rc = dalloc(h, &s.bg_n, C)) || (rc = dalloc(h, &s.log_step, C)) || (rc = dalloc(h, &s.log_bar, C)) ||
            (rc = dalloc(h, &s.hbar, C)) || (rc = dalloc(h, &s.mu_da, C)) || (rc = dalloc(h, &s.count, C)) ||
            (rc = dalloc(h, &s.n_samples, C)) || (rc = dalloc(h, &s.previous_update, C)) ||
            (rc = dalloc(h, &s.adapt_window, C)) || (rc = dalloc(h, &s.t_draw, C)) || (rc = dalloc(h, &s.iter, C)) ||
            (rc = dalloc(h, &s.status, C)) || (rc = dalloc(h, &s.tree_total, BFB_TREE_TOTAL_LEN)))
            return rc;
        for (auto &a : state_arrays(s)) {
            void *p = nullptr;
            BFB_CUDA(cudaMalloc(&p, a.second));
            h->chain_allocs.push_back(p);
            h->chain_snapshot.push_back(p);
        }
        h->alloc_C = C; h->alloc_np = np;
    }
    s.C = C; s.n = n; s.np = np;
    std::vector<double> vq(V, 0.), vvar(V, 1.), vfm(V, 0.), vfr(V, 0.);
    std::vector<double> fgn(C), bgn(C, 10.), ls(C), mu(C);
    std::vector<int64_t> cnt(C, 1);
    std::vector<int32_t> aw(C, cfg->adapt_window);
    for (int64_t c = 0; c < C; ++c) {
        for (int j = 0; j < n; ++j) {
            vq[c * np + j] = x0[c * n + j];
            vvar[c * np + j] = var0[c * n + j];
            vfm[c * np + j] = mean0[c * n + j];
            vfr[c * np + j] = var0[c * n + j] * cfg->initial_weight;     // metrics.py:348
            BFB_REQUIRE(var0[c * n + j] > 0., BFB_ERR_ARG, "the input diagonal covariance is not positive definite.");
        }
        fgn[c] = cfg->initial_weight;
        BFB_REQUIRE(step0[c] > 0., BFB_ERR_ARG, "initial step size must be positive");
        ls[c] = log(step0[c]);                 // step_size.py:13
        mu[c] = log(10. * step0[c]);           // step_size.py:20
    }
    if ((rc = h2d(h, s.q, vq)) || (rc = h2d(h, s.var, vvar)) || (rc = h2d(h, s.fg_mean, vfm)) ||
        (rc = h2d(h, s.fg_raw, vfr)) || (rc = h2d(h, s.fg_n, fgn)) || (rc = h2d(h, s.bg_n, bgn)) ||
        (rc = h2d(h, s.log_step, ls)) || (rc = h2d(h, s.log_bar, ls)) || (rc = h2d(h, s.mu_da, mu)) ||
        (rc = h2d(h, s.count, cnt)) || (rc = h2d(h, s.adapt_window, aw)))
        return rc;
    const int wpb = 4;
    const int blocks = (int)((C + wpb - 1) / wpb);
    const size_t smem = sizeof(double) * wpb * 2 * np;
    switch (np / 32) {
    case 1: chain_init_kernel<1><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, s); break;
    case 2: chain_init_kernel<2><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, s); break;
    case 3: chain_init_kernel<3><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, s); break;
    default: chain_init_kernel<4><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, s); break;
    }
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    // device-resident snapshot of the initial state (bfb_sampler_reset restarts the same run without host traffic)
    {
        auto arrs = state_arrays(s);
        for (size_t i = 0; i < arrs.size(); ++i)
            BFB_CUDA(cudaMemcpyAsync(h->chain_snapshot[i], arrs[i].first, arrs[i].second, cudaMemcpyDeviceToDevice, h->stream));
    }
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    h->has_chains = true;
    h->iters_done = 0;
    return BFB_OK;
}

extern "C" int bfb_sampler_init(bfb_handle h, const bfb_sampler_cfg *cfg, int64_t C, const double *x0,
                                const double *step0, const double *var0, const double *mean0)
{
    BFB_REQUIRE(h, BFB_ERR_STATE, "bfb_sampler_init: null handle");
    bfb_free_list(h->dense_allocs);
    h->dense_metric = false;
    if (h->t_u) { cudaSetDevice(h->device); cudaStreamSynchronize(h->stream); cudaFree(h->t_u); h->t_u = nullptr; }
    h->t_base = nullptr;
    return sampler_init_common(h, cfg, C, x0, step0, var0, mean0);
}

// Dense mass matrix: QuadMetricFull / QuadMetricFullAdapt (hmc_utils/metrics.py:94-132, 240-330, 374-417).  cov0 [C,n,n].
// The chains then run on the generic warp-per-chain kernel (sampler_kernel<.., DENSE = true>).
extern "C" int bfb_sampler_init_dense(bfb_handle h, const bfb_sampler_cfg *cfg, int64_t C, const double *x0,
                                      const double *step0, const double *cov0, const double *mean0)
{
    BFB_REQUIRE(h && h->has_model, BFB_ERR_STATE, "bfb_sampler_init_dense: no model set");
    BFB_REQUIRE(cfg && x0 && step0 && cov0 && mean0 && C > 0, BFB_ERR_ARG, "bfb_sampler_init_dense: bad arguments");
    const int n = h->n, np = h->np;
    const size_t M1 = (size_t)n * np, MT = (size_t)C * M1;
    // host-side factorisation of the initial covariances (scipy.linalg.cholesky(cov, lower=True), metrics.py:108 / 271)
    std::vector<double> covT(MT, 0.), cholT(MT, 0.), fgT(MT, 0.), bgT(MT, 0.), L((size_t)n * n);
    for (int64_t c = 0; c < C; ++c) {
        const double *A = cov0 + (size_t)c * n * n;
        std::fill(L.begin(), L.end(), 0.);
        for (int j = 0; j < n; ++j)
            for (int i = j; i < n; ++i) {
                double s_ = A[(size_t)i * n + j];
                for (int k = 0; k < j; ++k) s_ -= L[(size_t)i * n + k] * L[(size_t)j * n + k];
                if (i == j) {
                    BFB_REQUIRE(s_ > 0., BFB_ERR_ARG, "the input covariance is not positive definite.");
                    L[(size_t)j * n + j] = sqrt(s_);
                } else L[(size_t)i * n + j] = s_ / L[(size_t)j * n + j];
            }
        for (int k = 0; k < n; ++k)
            for (int j = 0; j < n; ++j) {
                const size_t d = (size_t)c * M1 + (size_t)k * np + j;
                covT[d] = A[(size_t)j * n + k];
                cholT[d] = L[(size_t)j * n + k];
                fgT[d] = A[(size_t)j * n + k] * cfg->initial_weight;       // metrics.py:392
                bgT[d] = (j == k) ? 10. : 0.;                               // _WeightedCovariance(self._n): eye * 10
            }
    }
    bfb_free_list(h->dense_allocs);
    h->dense_metric = false;
    if (h->t_u) { cudaSetDevice(h->device); cudaStreamSynchronize(h->stream); cudaFree(h->t_u); h->t_u = nullptr; }
    h->t_base = nullptr;
    std::vector<double> ones((size_t)C * n, 1.);
    int rc = sampler_init_common(h, cfg, C, x0, step0, ones.data(), mean0);
    if (rc) return rc;
    h->has_chains = false;
    ChainState &s = h->cs;
    // [0..4] covT cholT cholW fgcT bgcT, [5] chol_error, [6..9] snapshots of covT cholT fgcT bgcT (bfb_sampler_reset)
    for (int i = 0; i < 10; ++i) {
        void *p = nullptr;
        const size_t bytes = (i == 5) ? sizeof(int32_t) * C : sizeof(double) * MT;
        BFB_CUDA(cudaMalloc(&p, bytes));
        h->dense_allocs.push_back(p);
        BFB_CUDA(cudaMemsetAsync(p, 0, bytes, h->stream));
    }
    s.covT = (double *)h->dense_allocs[0]; s.cholT = (double *)h->dense_allocs[1]; s.cholW = (double *)h->dense_allocs[2];
    s.fgcT = (double *)h->dense_allocs[3]; s.bgcT = (double *)h->dense_allocs[4]; s.chol_error = (int32_t *)h->dense_allocs[5];
    const std::vector<double> *src[4] = {&covT, &cholT, &fgT, &bgT};
    double *dst[4] = {s.covT, s.cholT, s.fgcT, s.bgcT};
    for (int i = 0; i < 4; ++i) {
        BFB_CUDA(cudaMemcpyAsync(dst[i], src[i]->data(), sizeof(double) * MT, cudaMemcpyHostToDevice, h->stream));
        BFB_CUDA(cudaMemcpyAsync(h->dense_allocs[6 + i], dst[i], sizeof(double) * MT, cudaMemcpyDeviceToDevice, h->stream));
    }
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    h->dense_metric = true;
    h->has_chains = true;
    return BFB_OK;
}

// final covariances [C,n,n] of a dense-metric run (QuadMetricFullAdapt._cov) and, per chain, whether a Cholesky
// factorisation failed during adaptation (metrics.py:284-287, 315-317)
extern "C" int bfb_sampler_get_cov(bfb_handle h, double *cov, int32_t *chol_error)
{
    BFB_REQUIRE(h && h->has_chains && h->dense_metric, BFB_ERR_STATE, "bfb_sampler_get_cov: no dense-metric chains");
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    const ChainState &s = h->cs;
    const int n = s.n, np = s.np;
    if (cov) {
        std::vector<double> t((size_t)s.C * n * np);
        BFB_CUDA(cudaMemcpy(t.data(), s.covT, sizeof(double) * t.size(), cudaMemcpyDeviceToHost));
        for (int64_t c = 0; c < s.C; ++c)
            for (int j = 0; j < n; ++j)
                for (int k = 0; k < n; ++k) cov[((size_t)c * n + j) * n + k] = t[((size_t)c * n + k) * np + j];
    }
    if (chol_error) BFB_CUDA(cudaMemcpy(chol_error, s.chol_error, sizeof(int32_t) * s.C, cudaMemcpyDeviceToHost));
    return BFB_OK;
}

template <int NPL, int SAMPLER, bool DENSE>
static int launch_sampler(bfb_context *h, const RunOutDev &out, int wpb)
{
    const int L = h->scfg.max_treedepth;
    const size_t smem = sizeof(double) * wpb * warp_smem_doubles(h->np, L, DENSE);
    BFB_REQUIRE(smem <= 227 * 1024, BFB_ERR_ARG, "sampler needs %zu bytes of shared memory per block (> 227 KB)", smem);
    BFB_CUDA(cudaFuncSetAttribute(sampler_kernel<NPL, SAMPLER, DENSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int blocks = (int)((h->cs.C + wpb - 1) / wpb);
    sampler_kernel<NPL, SAMPLER, DENSE><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, h->scfg, h->cs, out, L);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

template <int NPL, int SAMPLER>
static int launch_sampler(bfb_context *h, const RunOutDev &out, int wpb)
{
    return h->dense_metric ? launch_sampler<NPL, SAMPLER, true>(h, out, wpb) : launch_sampler<NPL, SAMPLER, false>(h, out, wpb);
}

// kernel families of the sampler, numbered as bfb_sampler_last_path reports them
enum { FAM_GENERIC = 0, FAM_DMMA = 2, FAM_TEAM = 3, FAM_PAIR = 4 };
static const char *const fam_name[] = {"generic", nullptr, "dmma", "team", "pair"};
// what the family's kernels take, for the error when a pinned family cannot run the model
static const char *const fam_needs[] = {nullptr, nullptr,
    "n <= 32 without a prior (with cubic-3 configs: n <= 28 and cubic-2 ones), or the likelihood pipeline's tensor-core table",
    "n <= 64 for HMC and 32 < n <= 64 for NUTS, without decay / transform / rescale / likelihood pipeline",
    "NUTS with n <= 32, without a prior / cubic-3 configs / likelihood pipeline"};

// The kernel family that runs `sampler` on the model and chains of h.  By default a dense mass matrix runs on the generic
// warp-per-chain kernel.  NUTS runs on the team kernel for 32 < n <= 64, else on the one-warp kernel (dmma) where that takes
// the model.  HMC runs on the team kernel for 32 < n <= 64 and up to four groups of 8 chains per SM (4736 chains on a B200:
// 4096 chains 2.20e9 leapfrogs/s against 2.06e9 with one warp per group), above that on the one-warp kernel, which then has
// enough warps and fewer instructions (16384 chains: 3.2e9 against 2.5e9).  Everything else runs on the generic kernel.
// BFB200_SAMPLER = generic | dmma | team | pair pins a family for tests and profiles (*pinned); a pinned family that cannot
// run the model is an error (< 0).
static int select_family(bfb_context *h, int sampler, bool *pinned)
{
    const DevModel &M = h->dm;
    const bool nuts = sampler == BFB_NUTS;
    const bool team = !M.epilogue && M.tfrag && M.team_nr != 0 && !M.frag_ext && (!nuts || M.team_nr == 16) &&
                      (!M.has_c3 || (M.team_nr == 16 && M.tfrag3 && M.has_c2));
    const bool dmma = M.epilogue ? M.lik_tab != nullptr : M.frag_nr != 0 && (!M.has_c3 || (M.c3_kt != 0 && M.has_c2));
    const bool pair = nuts && !M.epilogue && M.frag_nr != 0 && !M.has_c3;
    const bool depth_ok = !nuts || h->scfg.max_treedepth <= 10;        // the tensor-core NUTS kernels keep at most 10 tree levels
    const char *sel = getenv("BFB200_SAMPLER");
    *pinned = sel != nullptr;
    if (!sel) {
        if (h->dense_metric || !depth_ok) return FAM_GENERIC;
        if (team && (nuts || M.team_nr == 16 || (h->cs.C + 7) / 8 <= (int64_t)h->sm_count * 4)) return FAM_TEAM;
        return dmma ? FAM_DMMA : FAM_GENERIC;
    }
    int fam = -1;
    for (int f = 0; f <= FAM_PAIR; ++f)
        if (fam_name[f] && !strcmp(sel, fam_name[f])) fam = f;
    BFB_REQUIRE(fam >= 0, BFB_ERR_ARG, "BFB200_SAMPLER=%s: unknown kernel family (generic, dmma, team or pair)", sel);
    if (fam == FAM_GENERIC) return fam;
    BFB_REQUIRE(!h->dense_metric, BFB_ERR_ARG, "BFB200_SAMPLER=%s: a dense mass matrix runs on the generic kernel only", sel);
    BFB_REQUIRE(depth_ok, BFB_ERR_ARG, "BFB200_SAMPLER=%s: the tensor-core NUTS kernels take max_treedepth <= 10", sel);
    BFB_REQUIRE(fam == FAM_DMMA ? dmma : fam == FAM_TEAM ? team : pair, BFB_ERR_ARG,
                "BFB200_SAMPLER=%s: the %s kernels cannot run this model; they take %s", sel, sel, fam_needs[fam]);
    return fam;
}

// launch the kernel(s) that advance every chain by n_iter iterations, outputs (device pointers) laid out [C, n_iter(, n)]
static int launch_run(bfb_context *h, int sampler, int n_iter, const bfb_run_out &dev_out)
{
    RunOutDev od;
    od.n_iter = n_iter;
    od.o = dev_out;
    bool pinned;
    const int fam = select_family(h, sampler, &pinned);
    if (fam < 0) return fam;
    int rc = 1;
    if (fam == FAM_TEAM) rc = sampler == BFB_NUTS ? bfb_launch_nuts_team(h, od.o, n_iter) : bfb_launch_hmc_team(h, od.o, n_iter);
    else if (fam == FAM_DMMA) rc = sampler == BFB_NUTS ? bfb_launch_nuts_dmma(h, od.o, n_iter) : bfb_launch_hmc_dmma(h, od.o, n_iter);
    else if (fam == FAM_PAIR) rc = bfb_launch_nuts_pair(h, od.o, n_iter);
    if (rc == 0) h->last_path = fam;
    if (rc <= 0) return rc;
    // the family's shared memory does not fit the model: the generic kernel runs it, unless the family was pinned
    BFB_REQUIRE(!pinned || fam == FAM_GENERIC, BFB_ERR_ARG,
                "BFB200_SAMPLER=%s: the kernel needs more than 227 KB of shared memory per block for this model", fam_name[fam]);
    h->last_path = FAM_GENERIC;
    // warps per block: as many as the per-warp tree state leaves room for in shared memory (the evaluation is latency bound:
    // at n = 64 a warp needs 32 KB, and 7 resident warps per SM instead of 4 are 1.7x the throughput)
    const int npl = h->np / 32;
    int wpb = 1;
    {
        const size_t per_warp = sizeof(double) * warp_smem_doubles(h->np, h->scfg.max_treedepth, h->dense_metric), cap = 227 * 1024;
        size_t best = 0;
        for (int w = 1; w <= 8; ++w) {                       // resident warps per SM = blocks that fit x warps per block
            const size_t resident = (cap / (w * per_warp + 1024)) * w;
            if (resident > best) { best = resident; wpb = w; }
        }
    }
    if (sampler == BFB_NUTS) {
        switch (npl) {
        case 1: rc = launch_sampler<1, BFB_NUTS>(h, od, wpb); break;
        case 2: rc = launch_sampler<2, BFB_NUTS>(h, od, wpb); break;
        case 3: rc = launch_sampler<3, BFB_NUTS>(h, od, wpb); break;
        default: rc = launch_sampler<4, BFB_NUTS>(h, od, wpb); break;
        }
    } else {
        switch (npl) {
        case 1: rc = launch_sampler<1, BFB_HMC>(h, od, wpb); break;
        case 2: rc = launch_sampler<2, BFB_HMC>(h, od, wpb); break;
        case 3: rc = launch_sampler<3, BFB_HMC>(h, od, wpb); break;
        default: rc = launch_sampler<4, BFB_HMC>(h, od, wpb); break;
        }
    }
    return rc;
}

// byte size of one (chain, iteration) record of output field f (order of bfb_run_out)
static size_t field_bytes(int f, int n) { return f == 0 ? sizeof(double) * n : (f <= 7 ? sizeof(double) : sizeof(int32_t)); }

static int launch_run(bfb_context *h, int sampler, int n_iter, const bfb_run_out &dev_out);

// Host outputs from ONE launch (the tensor-core NUTS kernel reports progress; anything else returns 1 before launching and the
// caller falls back to the chunked launches): device buffer [C, R(, n)] per field, the host thread polls the progress word the
// kernel writes into mapped pinned memory and queues the strided copy of every finished chunk on the copy stream.
// diag_t0 >= 0: the diagnostics of iterations diag_t0 .. R - 1 are queued behind the kernel (they overlap the last copies), *diag_P
// receives their device partials.
// Returns BFB_OK when the run was done (ev1 recorded, copies complete), 1 when this path does not apply, < 0 on error.
static int single_launch_host_outputs(bfb_context *h, int sampler, int R, void *const user[11], int n_keep, int diag_t0,
                                      const double **diag_P)
{
    const DevModel &M = h->dm;
    // only nuts_dmma_kernel reports progress, and only when it runs by default with eight chains per group
    bool pinned;
    if (select_family(h, sampler, &pinned) != FAM_DMMA || pinned || M.epilogue || M.has_c3 || getenv("BFB200_CHAINS_PER_GROUP")) return 1;
    const int64_t C = h->cs.C;
    const int n = h->n;
    size_t rec = 0;
    for (int f = 0; f < 11; ++f) if (user[f]) rec += field_bytes(f, n);
    if (rec == 0) return 1;
    const size_t need = rec * (size_t)C * (size_t)R;
    if (!h->copy_stream) {
        BFB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < BFB_NSTAGE; ++i) { BFB_CUDA(cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
                                               BFB_CUDA(cudaEventCreateWithFlags(&h->ev_c[i], cudaEventDisableTiming)); }
    }
    if (h->stage_len[0] < need) {
        if (h->stage[0]) cudaFree(h->stage[0]);
        h->stage[0] = nullptr; h->stage_len[0] = 0;
        if (cudaMalloc(&h->stage[0], need) != cudaSuccess) { cudaGetLastError(); return 1; }     // does not fit: chunked launches
        h->stage_len[0] = need;
    }
    if (!h->progress_host) {
        BFB_CUDA(cudaHostAlloc((void **)&h->progress_host, 64, cudaHostAllocMapped));
        BFB_CUDA(cudaHostGetDevicePointer((void **)&h->progress_host_dev, h->progress_host, 0));
    }
    void *dptr[11];
    char *base = (char *)h->stage[0];
    for (int f = 0; f < 11; ++f) {
        dptr[f] = nullptr;
        if (user[f]) { dptr[f] = base; base += field_bytes(f, n) * (size_t)C * (size_t)R; }
    }
    bfb_run_out dev = {(double *)dptr[0], (double *)dptr[1], (double *)dptr[2], (double *)dptr[3], (double *)dptr[4],
                       (double *)dptr[5], (double *)dptr[6], (double *)dptr[7], (int32_t *)dptr[8],
                       (int32_t *)dptr[9], (int32_t *)dptr[10]};
    volatile int *flag = h->progress_host;
    *flag = 0;
    // report chunks: the kernel counts, per chain, the chains that finished each chunk of iterations (independent of its work units) and
    // the host copies a chunk out as soon as the last chain is through.  Finer chunks start the copies earlier and leave a smaller last
    // chunk behind the kernel; what bounds the drain with eight GPUs on one host is that host's aggregate ingest (94 GB/s whatever the
    // copy pattern, scripts/d2h_probe.py), see DESIGN.md 7
    int want = 64;
    if (const char *e = getenv("BFB200_E2E_CHUNKS")) { int v = atoi(e); if (v >= 1) want = v; }
    h->progress_arm = want; h->progress_chunk_iters = 0; h->progress_n_chunks = 0;
    // After the warm-up (or with a fixed step) a chain's step_size / step_size_bar records repeat one value (step_size.py:25-45: dual
    // averaging only moves in the warm-up): ONE column of each crosses PCIe and the host thread replicates it over the iterations while
    // it waits for the kernel -- 16 of the 276 bytes of a record at n = 26, which matters when eight GPUs drain into one host.
    const bool const_steps = h->iters_done >= (int64_t)h->scfg.n_warmup || !h->scfg.adapt_step_size;
    int rc = launch_run(h, sampler, R, dev);
    h->progress_arm = 0;
    if (rc) return rc;
    h->iters_done += R;
    BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
    if (diag_t0 >= 0 && (rc = bfb_diag_enqueue(h, (const double *)dptr[0], C, R, diag_t0, R - diag_t0, n, diag_P))) return rc;
    const bool rep[2] = {const_steps && user[4] != nullptr, const_steps && user[5] != nullptr};
    double *col = nullptr;                          // pinned [2][C]: the first record of the two fields
    struct ColGuard { double *&p; ~ColGuard() { if (p) cudaFreeHost(p); } } col_guard{col};
    if (rep[0] || rep[1]) BFB_CUDA(cudaHostAlloc((void **)&col, sizeof(double) * 2 * (size_t)C, cudaHostAllocDefault));
    bool col_queued = false, col_ready = false;
    int filled = 0;                                 // iterations of the replicated fields already written on the host
    auto fill_to = [&](int it_end) {
        for (int k = 0; k < 2; ++k) {
            if (!rep[k]) continue;
            double *dst = (double *)user[4 + k];
            const double *src = col + (size_t)k * C;
            for (int64_t c = 0; c < C; ++c) {
                double *row = dst + (size_t)c * n_keep;
                const double v = src[c];
                for (int i = filled; i < it_end; ++i) row[i] = v;
            }
        }
        filled = it_end;
    };
    auto copy_range = [&](int it_begin, int its) -> int {
        for (int f = 0; f < 11; ++f) {
            if (!user[f]) continue;
            if ((f == 4 && rep[0]) || (f == 5 && rep[1])) continue;
            const size_t fb = field_bytes(f, n);
            BFB_CUDA(cudaMemcpy2DAsync((char *)user[f] + fb * (size_t)it_begin, fb * (size_t)n_keep, (char *)dptr[f] + fb * (size_t)it_begin,
                                       fb * (size_t)R, fb * (size_t)its, (size_t)C, cudaMemcpyDeviceToHost, h->copy_stream));
        }
        if (!col_queued && (rep[0] || rep[1])) {     // first record of the replicated fields (the kernel has written it by now)
            for (int k = 0; k < 2; ++k)
                if (rep[k])
                    BFB_CUDA(cudaMemcpy2DAsync(col + (size_t)k * C, sizeof(double), dptr[4 + k], sizeof(double) * (size_t)R, sizeof(double),
                                               (size_t)C, cudaMemcpyDeviceToHost, h->copy_stream));
            BFB_CUDA(cudaEventRecord(h->ev_c[0], h->copy_stream));
            col_queued = true;
        }
        return BFB_OK;
    };
    // replicate up to the iterations whose copies are queued, as soon as the column has arrived (never blocks before the end)
    auto replicate = [&](int it_end, bool wait) -> int {
        if (!(rep[0] || rep[1]) || !col_queued) return BFB_OK;
        if (!col_ready) {
            if (wait) BFB_CUDA(cudaEventSynchronize(h->ev_c[0]));
            else if (cudaEventQuery(h->ev_c[0]) != cudaSuccess) { cudaGetLastError(); return BFB_OK; }
            col_ready = true;
        }
        fill_to(it_end);
        return BFB_OK;
    };
    if (h->last_path != FAM_DMMA || h->progress_chunk_iters == 0) {
        // another kernel family took the launch: no progress reports, one copy after the kernel
        BFB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev1, 0));
        if ((rc = copy_range(0, R))) return rc;
        if ((rc = replicate(R, true))) return rc;
        BFB_CUDA(cudaStreamSynchronize(h->copy_stream));
        return BFB_OK;
    }
    const int K = h->progress_chunk_iters, nch = h->progress_n_chunks;
    int copied = 0;                                  // chunks whose copies are queued
    unsigned spins = 0;
    while (copied < nch) {
        int seen = *flag;
        if (seen <= copied) {
            if ((++spins & 0x3ff) == 0) {
                const cudaError_t q = cudaStreamQuery(h->stream);     // the kernel ended (or failed) without the last report?
                if (q == cudaSuccess) seen = (*flag > copied) ? *flag : nch;
                else if (q != cudaErrorNotReady) { bfb_set_error("bfb_sampler_run_ex: %s", cudaGetErrorString(q)); return BFB_ERR_CUDA; }
            }
            if (seen <= copied) continue;
        }
        const int it_begin = copied * K, it_end = (seen * K < R) ? seen * K : R;
        if ((rc = copy_range(it_begin, it_end - it_begin))) return rc;
        copied = seen;
        if (copied < nch && (rc = replicate(it_end, false))) return rc;     // host work while the kernel goes on
    }
    if ((rc = replicate(R, true))) return rc;
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->copy_stream));
    return BFB_OK;
}

// ---- reduced outputs (bfb_sampler_run_ex): thinning and summaries on the device ----
// dst[c][i] = src[c][i * thin] for records of `rec` doubles (samples: n) or of one 4-byte / 8-byte word
template <class T>
__global__ void thin_kernel(const T *__restrict__ src, T *__restrict__ dst, int64_t C, int K, int kk, int thin, int rec)
{
    const int64_t total = C * (int64_t)kk * rec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(i % rec);
        const int64_t r = i / rec;
        const int it = (int)(r % kk);
        const int64_t c = r / kk;
        dst[i] = src[(c * K + (int64_t)it * thin) * rec + j];
    }
}
// shifted first and second moments of the rows x[r][0..n): per-block partials part[b][n + n*n] (sum (x - s), sum (x - s)(x - s)^T),
// rows dealt to the blocks in tiles of 32; a second kernel adds the partials in a fixed order (deterministic)
static __global__ void __launch_bounds__(256) trace_moments_partial_kernel(const double *__restrict__ x, int64_t rows, int n, const double *__restrict__ shift,
                                                             double *__restrict__ part)
{
    extern __shared__ double xs[];        // [32][n]
    const int ne = n + n * n;
    double acc[72];                       // entries tid, tid + 256, ...: n <= 128 -> at most 65 per thread
    const int nacc = (ne + 255) / 256;
    for (int a = 0; a < nacc; ++a) acc[a] = 0.;
    for (int64_t r0 = (int64_t)blockIdx.x * 32; r0 < rows; r0 += (int64_t)gridDim.x * 32) {
        const int nr = (int)((rows - r0 < 32) ? rows - r0 : 32);
        __syncthreads();
        for (int i = threadIdx.x; i < nr * n; i += 256) xs[i] = x[r0 * n + i] - shift[i % n];
        __syncthreads();
        for (int a = 0; a < nacc; ++a) {
            const int e = threadIdx.x + a * 256;
            if (e >= ne) break;
            double v = acc[a];
            if (e < n) { for (int r = 0; r < nr; ++r) v += xs[r * n + e]; }
            else { const int j = (e - n) / n, k = (e - n) % n; for (int r = 0; r < nr; ++r) v = fma(xs[r * n + j], xs[r * n + k], v); }
            acc[a] = v;
        }
    }
    for (int a = 0; a < nacc; ++a) { const int e = threadIdx.x + a * 256; if (e < ne) part[(size_t)blockIdx.x * ne + e] = acc[a]; }
}
static __global__ void trace_moments_reduce_kernel(const double *__restrict__ part, int nb, int ne, double *__restrict__ accum)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ne) return;
    double v = accum[e];
    for (int b = 0; b < nb; ++b) v += part[(size_t)b * ne + e];
    accum[e] = v;
}

extern "C" int bfb_sampler_run(bfb_handle h, int sampler, int32_t n_iter, const bfb_run_out *out, int loc,
                               int64_t *total_tree_size)
{
    return bfb_sampler_run_ex(h, sampler, n_iter, out, loc, nullptr, total_tree_size);
}

extern "C" int bfb_sampler_run_ex(bfb_handle h, int sampler, int32_t n_iter, const bfb_run_out *out, int loc,
                                  const bfb_run_opts *opts, int64_t *total_tree_size)
{
    BFB_REQUIRE(h && h->has_model && h->has_chains, BFB_ERR_STATE, "bfb_sampler_run: call bfb_sampler_init first");
    BFB_REQUIRE(sampler == BFB_NUTS || sampler == BFB_HMC, BFB_ERR_ARG, "unknown sampler %d", sampler);
    BFB_REQUIRE(n_iter > 0 && out, BFB_ERR_ARG, "bfb_sampler_run: bad arguments");
    BFB_REQUIRE(sampler != BFB_HMC || h->scfg.n_int_step > 0, BFB_ERR_ARG, "n_int_step must be positive");
    const int skip = opts ? opts->skip : 0, thin = opts ? opts->thin : 1;
    const bool want_mom = opts && (opts->mean || opts->cov);
    const bool want_diag = opts && opts->diag;
    const int dfrom = want_diag ? opts->diag_from : 0;
    BFB_REQUIRE(skip >= 0 && skip <= n_iter && thin >= 1, BFB_ERR_ARG, "bfb_sampler_run_ex: need 0 <= skip <= n_iter and thin >= 1");
    BFB_REQUIRE(!want_diag || (dfrom >= skip && n_iter - dfrom >= 4), BFB_ERR_ARG,
                "bfb_sampler_run_ex: the diagnostics need skip <= diag_from <= n_iter - 4 (skip %d, diag_from %d, n_iter %d)", skip, dfrom, n_iter);
    BFB_REQUIRE(loc == BFB_HOST || (thin == 1 && !want_mom), BFB_ERR_ARG, "bfb_sampler_run_ex: thinning and summaries need host outputs");
    BFB_CUDA(cudaSetDevice(h->device));
    const int64_t C = h->cs.C;
    const int n = h->n;
    void *const user[11] = {out->samples, out->logp, out->energy, out->mean_tree_accept, out->step_size, out->step_size_bar,
                            out->energy_change, out->max_energy_change, out->tree_depth, out->tree_size, out->diverging};
    BFB_CUDA(cudaMemsetAsync(h->cs.tree_total, 0, BFB_TREE_TOTAL_LEN * sizeof(unsigned long long), h->stream));
    unsigned long long tt = 0;
    const bfb_run_out none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    BFB_CUDA(cudaEventRecord(h->ev0, h->stream));
    if (skip > 0) {                         // warm-up iterations whose records nobody wants: no output traffic at all
        int rc = launch_run(h, sampler, skip, none);
        if (rc) return rc;
        h->iters_done += skip;
    }
    const int R = n_iter - skip;            // iterations with records
    const int n_keep = (R + thin - 1) / thin;
    // diagnostics: iterations dfrom .. n_iter - 1 are draws diag_t0 .. of diag_src [C, diag_T, n]; diag_buf holds them when no
    // buffer of the run does
    const int Rd = n_iter - dfrom;
    const double *diag_P = nullptr, *diag_src = nullptr;
    int64_t diag_T = 0, diag_t0 = 0;
    double *diag_buf = nullptr;
    struct DiagGuard { double *&p; ~DiagGuard() { if (p) cudaFree(p); } } diag_guard{diag_buf};
    auto alloc_diag_buf = [&](int iters) -> int {
        const size_t bytes = sizeof(double) * (size_t)C * (size_t)iters * (size_t)n;
        const cudaError_t e = cudaMalloc((void **)&diag_buf, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            diag_buf = nullptr;
            bfb_set_error("bfb_sampler_run_ex: the diagnostics need the samples of %d iterations x %lld chains resident on the device, "
                          "a %.2f GB buffer that cannot be allocated (%s)", iters, (long long)C, 1e-9 * (double)bytes, cudaGetErrorString(e));
            return BFB_ERR_CUDA;
        }
        return BFB_OK;
    };
    int single_rc = 1;
    if (R >= 64 && loc == BFB_HOST && sampler == BFB_NUTS && !h->dense_metric && thin == 1 && !want_mom && (!want_diag || user[0]) &&
        !getenv("BFB200_E2E_MULTI_LAUNCH")) {
        single_rc = single_launch_host_outputs(h, sampler, R, user, n_keep, want_diag ? dfrom - skip : -1, &diag_P);
        if (single_rc < 0) return single_rc;
    }
    if (R == 0) {
    } else if (loc == BFB_DEVICE) {
        bfb_run_out dev = *out;
        if (want_diag && !dev.samples) {
            int rc = alloc_diag_buf(R);
            if (rc) return rc;
            dev.samples = diag_buf;
        }
        int rc = launch_run(h, sampler, R, dev);
        if (rc) return rc;
        h->iters_done += R;
        diag_src = dev.samples; diag_T = R; diag_t0 = dfrom - skip;
    } else if (single_rc == BFB_OK) {
        // done: ONE launch for all R iterations into a device buffer laid out like the caller's arrays; the kernel reported every
        // finished chunk of iterations and the host copied it out while the kernel went on (no launch boundaries, no tails)
    } else {
        // Host outputs: the run is cut into chunks of iterations; chunk k's kernel writes a device staging buffer while
        // chunk k-1 is copied to the caller's arrays on a second stream (strided 2-D copies: the host layout is
        // chain-major).  With pinned host memory (bfb_host_alloc) the copies are hidden behind the kernels.  Thinned
        // records are compacted on the device first; the summaries are accumulated from the staging buffer.
        int n_chunks = R >= 512 ? 6 : (R >= 128 ? 3 : 1);
        if (const char *e = getenv("BFB200_E2E_CHUNKS")) { int v = atoi(e); if (v >= 1 && v <= R) n_chunks = v; }
        int K = (R + n_chunks - 1) / n_chunks;
        K = ((K + thin - 1) / thin) * thin;                 // chunk boundaries on kept iterations
        n_chunks = (R + K - 1) / K;
        size_t rec = 0;
        for (int f = 0; f < 11; ++f) if (user[f]) rec += field_bytes(f, n);
        const bool stage_samples = (want_mom || want_diag) && !user[0];    // the summaries need the samples even if the caller does not
        if (stage_samples) rec += field_bytes(0, n);
        const size_t full = rec * (size_t)C * K;
        const size_t need = full + (thin > 1 ? rec * (size_t)C * ((K + thin - 1) / thin) : 0);
        if (!h->copy_stream) {
            BFB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
            for (int i = 0; i < BFB_NSTAGE; ++i) { BFB_CUDA(cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
                                                   BFB_CUDA(cudaEventCreateWithFlags(&h->ev_c[i], cudaEventDisableTiming)); }
        }
        for (int i = 0; i < BFB_NSTAGE; ++i) {
            if (h->stage_len[i] < need) {
                if (h->stage[i]) cudaFree(h->stage[i]);
                h->stage[i] = nullptr; h->stage_len[i] = 0;
                BFB_CUDA(cudaMalloc(&h->stage[i], need ? need : 8));
                h->stage_len[i] = need;
            }
        }
        const int ne = n + n * n, nb = h->sm_count * 2;
        if (want_diag) {
            int rc = alloc_diag_buf(Rd);
            if (rc) return rc;
            diag_src = diag_buf; diag_T = Rd; diag_t0 = 0;
        }
        double *mom = nullptr;              // [n] shift | [ne] accumulators | [nb][ne] partials
        if (want_mom) {
            BFB_CUDA(cudaMalloc((void **)&mom, sizeof(double) * ((size_t)n + ne + (size_t)nb * ne)));
            BFB_CUDA(cudaMemsetAsync(mom, 0, sizeof(double) * ((size_t)n + ne), h->stream));
        }
        for (int k = 0; k < n_chunks; ++k) {
            const int it_begin = k * K, Kk = (it_begin + K <= R) ? K : R - it_begin;
            const int kk = (Kk + thin - 1) / thin, keep_begin = it_begin / thin;
            const int sb = k % BFB_NSTAGE;
            if (k >= BFB_NSTAGE) BFB_CUDA(cudaStreamWaitEvent(h->stream, h->ev_c[sb], 0));   // staging buffer free again
            void *dptr[11], *cptr[11];
            char *base = (char *)h->stage[sb], *cbase = (char *)h->stage[sb] + full;
            for (int f = 0; f < 11; ++f) {
                dptr[f] = cptr[f] = nullptr;
                if (user[f] || (f == 0 && stage_samples)) {
                    dptr[f] = base; base += field_bytes(f, n) * (size_t)C * Kk;
                    cptr[f] = cbase; cbase += field_bytes(f, n) * (size_t)C * kk;
                }
            }
            bfb_run_out dev = {(double *)dptr[0], (double *)dptr[1], (double *)dptr[2], (double *)dptr[3], (double *)dptr[4],
                               (double *)dptr[5], (double *)dptr[6], (double *)dptr[7], (int32_t *)dptr[8],
                               (int32_t *)dptr[9], (int32_t *)dptr[10]};
            int rc = launch_run(h, sampler, Kk, dev);
            if (rc) { if (mom) cudaFree(mom); return rc; }
            h->iters_done += Kk;
            if (want_mom) {
                if (k == 0) BFB_CUDA(cudaMemcpyAsync(mom, dptr[0], sizeof(double) * n, cudaMemcpyDeviceToDevice, h->stream));   // shift = first record
                trace_moments_partial_kernel<<<nb, 256, sizeof(double) * 32 * n, h->stream>>>((const double *)dptr[0], C * (int64_t)Kk, n, mom, mom + n + ne);
                trace_moments_reduce_kernel<<<(ne + 127) / 128, 128, 0, h->stream>>>(mom + n + ne, nb, ne, mom + n);
                h->launches += 2;
            }
            if (want_diag) {                // this chunk's iterations from dfrom on, into the resident buffer
                const int lo = std::max(it_begin, dfrom - skip), hi = it_begin + Kk;
                if (hi > lo)
                    BFB_CUDA(cudaMemcpy2DAsync(diag_buf + (size_t)(lo - (dfrom - skip)) * n, sizeof(double) * n * (size_t)Rd,
                                               (const double *)dptr[0] + (size_t)(lo - it_begin) * n, sizeof(double) * n * (size_t)Kk,
                                               sizeof(double) * n * (size_t)(hi - lo), (size_t)C, cudaMemcpyDeviceToDevice, h->stream));
            }
            if (thin > 1) {
                for (int f = 0; f < 11; ++f) {
                    if (!user[f]) continue;
                    const int64_t tot = C * (int64_t)kk * (f == 0 ? n : 1);
                    const unsigned gb = (unsigned)((tot + 255) / 256 < 4096 ? (tot + 255) / 256 : 4096);
                    if (f <= 7) thin_kernel<double><<<gb, 256, 0, h->stream>>>((const double *)dptr[f], (double *)cptr[f], C, Kk, kk, thin, f == 0 ? n : 1);
                    else thin_kernel<int32_t><<<gb, 256, 0, h->stream>>>((const int32_t *)dptr[f], (int32_t *)cptr[f], C, Kk, kk, thin, 1);
                    h->launches++;
                }
            }
            BFB_CUDA(cudaGetLastError());
            BFB_CUDA(cudaEventRecord(h->ev_k[sb], h->stream));
            BFB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_k[sb], 0));
            for (int f = 0; f < 11; ++f) {
                if (!user[f]) continue;
                const size_t fb = field_bytes(f, n);
                BFB_CUDA(cudaMemcpy2DAsync((char *)user[f] + fb * (size_t)keep_begin, fb * (size_t)n_keep, thin > 1 ? cptr[f] : dptr[f],
                                           fb * (size_t)kk, fb * (size_t)kk, (size_t)C, cudaMemcpyDeviceToHost, h->copy_stream));
            }
            BFB_CUDA(cudaEventRecord(h->ev_c[sb], h->copy_stream));
        }
        if (want_mom) {
            // mean = s + S1 / N, cov = (S2 - S1 S1^T / N) / (N - 1)   (np.cov: unbiased)
            std::vector<double> m((size_t)n + ne);
            BFB_CUDA(cudaMemcpyAsync(m.data(), mom, sizeof(double) * m.size(), cudaMemcpyDeviceToHost, h->stream));
            BFB_CUDA(cudaStreamSynchronize(h->stream));
            const double N = (double)C * (double)R;
            if (opts->mean) for (int j = 0; j < n; ++j) opts->mean[j] = m[j] + m[n + j] / N;
            if (opts->cov)
                for (int j = 0; j < n; ++j)
                    for (int k2 = 0; k2 < n; ++k2)
                        opts->cov[(size_t)j * n + k2] = (m[2 * n + (size_t)j * n + k2] - m[n + j] * m[n + k2] / N) / (N - 1.);
            cudaFree(mom);
        }
        BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
        BFB_CUDA(cudaStreamSynchronize(h->copy_stream));
    }
    if (R == 0 || loc == BFB_DEVICE) BFB_CUDA(cudaEventRecord(h->ev1, h->stream));
    if (diag_src) {
        int rc = bfb_diag_enqueue(h, diag_src, C, diag_T, diag_t0, Rd, n, &diag_P);
        if (rc) return rc;
    }
    if (want_diag) BFB_CUDA(cudaMemcpyAsync(opts->diag, diag_P, sizeof(double) * (size_t)n * (size_t)(Rd / 2 + 3), cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaMemcpyAsync(&tt, h->cs.tree_total, sizeof(tt), cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    BFB_CUDA(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    if (total_tree_size) *total_tree_size = (int64_t)tt;
    if (getenv("BFB200_DEBUG")) {
        unsigned long long dbg[BFB_TREE_TOTAL_LEN];
        BFB_CUDA(cudaMemcpy(dbg, h->cs.tree_total, sizeof(dbg), cudaMemcpyDeviceToHost));
        fprintf(stderr, "[bfb200] leaves %llu warp-rounds %llu merge-passes %llu iter-end-sections %llu  ms %.3f\n", dbg[0], dbg[1], dbg[2], dbg[3], h->last_ms);
        if (dbg[1] && h->last_path == FAM_TEAM)
            fprintf(stderr, "[bfb200] team kernel, leader-warp cycles per round: apply %.0f boundary %.0f leapfrog+eval %.0f owners %.0f tasks+leaf %.0f decisions %.0f command-barrier %.0f\n",
                    (double)dbg[4] / dbg[1], (double)dbg[5] / dbg[1], (double)dbg[6] / dbg[1], (double)dbg[7] / dbg[1],
                    (double)dbg[8] / dbg[1], (double)dbg[9] / dbg[1], (double)dbg[10] / dbg[1]);
        else if (dbg[1] && h->last_path == FAM_PAIR)
            fprintf(stderr, "[bfb200] pair kernel, tree warp cycles per round: boundary %.0f rng+dbl %.0f wait-for-leaves %.0f leaf-pair %.0f merges %.0f push %.0f extend %.0f hand-over %.0f | integrator (%llu rounds): wait-unit %.0f wait-tree %.0f compute %.0f\n",
                    (double)dbg[4] / dbg[1], (double)dbg[5] / dbg[1], (double)dbg[6] / dbg[1], (double)dbg[7] / dbg[1],
                    (double)dbg[8] / dbg[1], (double)dbg[9] / dbg[1], (double)dbg[10] / dbg[1], (double)dbg[11] / dbg[1], dbg[12],
                    (double)dbg[13] / (dbg[12] ? dbg[12] : 1), (double)dbg[14] / (dbg[12] ? dbg[12] : 1), (double)dbg[15] / (dbg[12] ? dbg[12] : 1));
        else if (dbg[1]) {
            const double bnd = (double)(dbg[4] + dbg[16] + dbg[17] + dbg[18] + dbg[19]);
            fprintf(stderr, "[bfb200] cycles per warp-round: boundary %.0f rng+dbl %.0f (unused) %.0f leaves %.0f merge-loop %.0f push %.0f extend %.0f | unit setup+teardown per round %.0f\n",
                    bnd / dbg[1], (double)dbg[5] / dbg[1], (double)dbg[6] / dbg[1], (double)dbg[7] / dbg[1],
                    (double)dbg[8] / dbg[1], (double)dbg[9] / dbg[1], (double)dbg[10] / dbg[1], (double)dbg[11] / dbg[1]);
            fprintf(stderr, "[bfb200] boundary cycles per warp-round: statistics %.0f lane-per-dimension %.0f progress-report %.0f new-state %.0f rest %.0f | rounds with a boundary %.3f\n",
                    (double)dbg[16] / dbg[1], (double)dbg[17] / dbg[1], (double)dbg[18] / dbg[1], (double)dbg[19] / dbg[1],
                    (double)dbg[4] / dbg[1], (double)dbg[3] / dbg[1]);
        }
    }
    return BFB_OK;
}

extern "C" int bfb_sampler_last_path(bfb_handle h)
{
    return h ? h->last_path : -1;
}

// pinned host memory for the outputs of bfb_sampler_run (asynchronous, full-speed device-to-host copies)
extern "C" int bfb_host_alloc(size_t bytes, void **ptr)
{
    BFB_REQUIRE(ptr, BFB_ERR_ARG, "bfb_host_alloc: null pointer");
    BFB_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 8, cudaHostAllocDefault));
    return BFB_OK;
}
extern "C" int bfb_host_free(void *ptr)
{
    if (ptr) BFB_CUDA(cudaFreeHost(ptr));
    return BFB_OK;
}

extern "C" int bfb_sampler_get_state(bfb_handle h, double *final_step, double *final_var, int64_t *n_draws,
                                     int32_t *status, double *q)
{
    BFB_REQUIRE(h && h->has_chains, BFB_ERR_STATE, "bfb_sampler_get_state: no chains");
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    const ChainState &s = h->cs;
    const int64_t C = s.C;
    const int n = s.n, np = s.np;
    if (final_step) {
        std::vector<double> a(C), b(C), c(C);
        std::vector<int64_t> k(C);
        BFB_CUDA(cudaMemcpy(a.data(), s.log_step, sizeof(double) * C, cudaMemcpyDeviceToHost));
        BFB_CUDA(cudaMemcpy(b.data(), s.log_bar, sizeof(double) * C, cudaMemcpyDeviceToHost));
        BFB_CUDA(cudaMemcpy(c.data(), s.hbar, sizeof(double) * C, cudaMemcpyDeviceToHost));
        BFB_CUDA(cudaMemcpy(k.data(), s.count, sizeof(int64_t) * C, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < C; ++i) {
            final_step[4 * i] = a[i]; final_step[4 * i + 1] = b[i]; final_step[4 * i + 2] = c[i];
            final_step[4 * i + 3] = (double)k[i];
        }
    }
    auto getvec = [&](const double *dev, double *host) -> int {
        std::vector<double> tmp((size_t)C * np);
        BFB_CUDA(cudaMemcpy(tmp.data(), dev, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < C; ++i)
            for (int j = 0; j < n; ++j) host[i * n + j] = tmp[i * np + j];
        return BFB_OK;
    };
    int rc;
    if (final_var && (rc = getvec(s.var, final_var))) return rc;
    if (q && (rc = getvec(s.q, q))) return rc;
    if (n_draws) BFB_CUDA(cudaMemcpy(n_draws, s.t_draw, sizeof(int64_t) * C, cudaMemcpyDeviceToHost));
    if (status) BFB_CUDA(cudaMemcpy(status, s.status, sizeof(int32_t) * C, cudaMemcpyDeviceToHost));
    return BFB_OK;
}
