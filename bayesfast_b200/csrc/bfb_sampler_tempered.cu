// bfb_sampler_tempered.cu -- the tempered samplers TNUTS / THMC (SURVEY.md 8f rank 4) on the device, sm_100a.
//
// Replaces bayesfast/samplers/tnuts.py, thmc.py, hmc_utils/base_hmc.py:220-262 (BaseTHMC.astep) and
// hmc_utils/integration.py:98-222 (TCpuLeapfrogIntegrator) for C chains at once: one warp per chain (lane j owns the
// dimensions j, j + 32, ...), the organisation of the generic kernel of bfb_sampler.cu.  The Hamiltonian lives on (u, q):
// potential = beta(u) phi(q) + (1 - beta(u)) psi(q) + U(u) with phi = -logp of the handle's model, psi = -(logp of the BASE
// handle's model + log xi), beta the logistic function; the integrator is drift(1/2) - kick - drift(1/2) with the gradients
// of BOTH densities taken at the midpoint and both values taken again at the end point (4 evaluations per leapfrog).  The tree
// (nuts.py:27-178) runs on the n momenta / velocities only -- the tempering momentum never enters a U-turn test -- and a
// proposal carries (q, u, weight, energy, logp) (tnuts.py:12-19).  Diagonal metric.
#include "bfb_common.cuh"
#include "bfb_eval.cuh"
#include <cmath>
#include <cstring>

namespace {

struct TRunOutDev {
    bfb_run_out o;
    double *u, *weight;
    int32_t n_iter;
};

// per-warp shared memory: evaluation scratch (2 np) | tree ends L, R: q, p (4 np) | p_sum | proposal q | momentum at the begin of
// the doubling | stack levels: p_left, p_right, p_sum, proposal q (4 np each) | stack scalars [5][L]
__host__ __device__ inline size_t t_warp_smem_doubles(int np, int L)
{
    size_t s = (size_t)(9 + 4 * L) * np + 5 * (size_t)L;
    return (s + 1) & ~(size_t)1;
}

// shared memory in front of the per-warp areas: the two DevModels
constexpr size_t T_MODEL_DOUBLES = (2 * sizeof(DevModel) + 15) / 16 * 2;

// integration.py:104-128
__device__ __forceinline__ double t_beta(double u) { return 1. / (1. + exp(-u)); }
__device__ __forceinline__ double t_d_beta(double u) { const double e = exp(-u); return e / ((1. + e) * (1. + e)); }
__device__ __forceinline__ double t_temp_potential(double u) { return u + 2. * log(1. + exp(-u)); }
__device__ __forceinline__ double t_d_temp_potential(double u) { const double e = exp(u); return (e - 1.) / (e + 1.); }

// ONE out-of-line copy of the evaluator for both densities and all six call sites of an iteration (start state: 2, leapfrog: 4).
// Inlined six times the kernel was bound by instruction fetch (ncu, profiles/r02_i_tsampler_tnuts_ncu_summary.md:
// sm__icc_request_hit_rate 43 %, 17.9 no_instruction stall cycles per issued instruction with 14 warps per SM at different places of
// ~6 x the evaluator's code); the two models sit in shared memory so that the callee reads their fields through one pointer.
template <int NPL> struct TVec { double v[NPL]; };
template <int NPL> struct TEval { double lp; double g[NPL]; };

template <int NPL>
__device__ __noinline__ TEval<NPL> t_eval_ool(const DevModel *M, TVec<NPL> q, int lane, double *xsm, double *dsm)
{
    TEval<NPL> r;
    density_eval<NPL>(*M, q.v, lane, xsm, dsm, r.lp, r.g);
    return r;
}

template <int NPL>
__device__ __forceinline__ void t_eval(const DevModel *M, const double (&q)[NPL], int lane, double *xsm, double *dsm, double &lp,
                                       double (&g)[NPL])
{
    TVec<NPL> a;
#pragma unroll
    for (int r = 0; r < NPL; ++r) a.v[r] = q[r];
    const TEval<NPL> e = t_eval_ool<NPL>(M, a, lane, xsm, dsm);
    lp = e.lp;
#pragma unroll
    for (int r = 0; r < NPL; ++r) g[r] = e.g[r];
}

// the tail compute_state (integration.py:139-150) and _step (:205-222) share: energy, logp, weight of a state
template <int NPL>
__device__ __forceinline__ void t_finish(const double (&var)[NPL], const double (&p)[NPL], double u, double vt, double lp, double lpb,
                                         double logxi, double &energy, double &weight)
{
    double part = 0.;
#pragma unroll
    for (int r = 0; r < NPL; ++r) part = fma(p[r], var[r] * p[r], part);
    const double kin = 0.5 * warp_sum(part) + vt * vt / 2.;
    const double phi = -lp, psi = -(lpb + logxi);
    const double beta = t_beta(u), U = t_temp_potential(u);
    const double potential = beta * phi + (1. - beta) * psi + U;
    energy = kin + potential;
    const double delta = phi - psi;
    weight = delta == 0. ? 1. : delta / expm1(delta);
}

// integration.py:152-222 TCpuLeapfrogIntegrator._step
template <int NPL>
__device__ __forceinline__ void t_leapfrog(const DevModel *M, const DevModel *MB, double logxi, double eps, const double (&var)[NPL],
                                           double (&q)[NPL], double (&p)[NPL], double &u, double &vt, int lane, double *xsm,
                                           double *dsm, double &logp, double &energy, double &weight)
{
    const double dt = 0.5 * eps;
    double g1[NPL], g2[NPL], lp, lpb;
    u += vt * dt;
#pragma unroll
    for (int r = 0; r < NPL; ++r) q[r] = fma(dt, var[r] * p[r], q[r]);
    t_eval<NPL>(M, q, lane, xsm, dsm, lp, g1);
    t_eval<NPL>(MB, q, lane, xsm, dsm, lpb, g2);
    {
        const double phi = -lp, psi = -(lpb + logxi);
        const double beta = t_beta(u), d_beta = t_d_beta(u), dU = t_d_temp_potential(u);
        const double d_pot_du = d_beta * (phi - psi) + dU;
        vt += -d_pot_du * eps;
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            const double d_pot_dq = beta * (-g1[r]) + (1. - beta) * (-g2[r]);
            p[r] = fma(eps, -d_pot_dq, p[r]);
        }
    }
    u += vt * dt;
#pragma unroll
    for (int r = 0; r < NPL; ++r) q[r] = fma(dt, var[r] * p[r], q[r]);
    t_eval<NPL>(M, q, lane, xsm, dsm, lp, g1);
    t_eval<NPL>(MB, q, lane, xsm, dsm, lpb, g2);
    logp = lp;
    t_finish<NPL>(var, p, u, vt, lp, lpb, logxi, energy, weight);
}

template <int NPL>
__device__ __forceinline__ double t_vdot(const double (&a)[NPL], const double (&var)[NPL], const double (&b)[NPL])
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
#define UDOT(a, b) t_vdot<NPL>(a, var, b)

template <int NPL, int SAMPLER>
__global__ void __launch_bounds__(256) tsampler_kernel(DevModel Mpar, DevModel MBpar, double logxi, bfb_sampler_cfg cfg, ChainState st,
                                                       double *__restrict__ tu, TRunOutDev out, int L)
{
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    // both models at the head of the block's shared memory (read by the out-of-line evaluator through a pointer)
    DevModel *M = reinterpret_cast<DevModel *>(smem), *MB = M + 1;
    if (threadIdx.x == 0) { *M = Mpar; *MB = MBpar; }
    __syncthreads();
    const int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    if (c >= st.C) return;
    const int n = Mpar.n, np = Mpar.np;
    double *wsm = smem + T_MODEL_DOUBLES + (size_t)wib * t_warp_smem_doubles(np, L);
    double *xsm = wsm, *dsm = wsm + np;
    const int oTL = 2 * np, oTR = 4 * np, oPS = 6 * np, oPQ = 7 * np, oPB = 8 * np, oST = 9 * np, SV = 4;
    double *ssc = wsm + (size_t)(9 + SV * L) * np;      // [5][L]: log_size, energy, logp, u, weight of the stacked proposals
    if (st.status[c] != 0) return;

    const uint64_t seed = cfg.seed, chain = (uint64_t)(cfg.chain0 + c);
    int64_t t = st.t_draw[c];
    const int64_t it0 = st.iter[c];
    const size_t vb = (size_t)c * np;

    double q[NPL], p[NPL], var[NPL], inv_std[NPL];
    double fgm[NPL], fgr[NPL], bgm[NPL], bgr[NPL];
#pragma unroll
    for (int r = 0; r < NPL; ++r) {
        const int j = lane + 32 * r;
        q[r] = st.q[vb + j]; var[r] = st.var[vb + j];
        inv_std[r] = 1. / sqrt(var[r]);
        fgm[r] = st.fg_mean[vb + j]; fgr[r] = st.fg_raw[vb + j];
        bgm[r] = st.bg_mean[vb + j]; bgr[r] = st.bg_raw[vb + j];
        p[r] = 0.;
    }
    double u_cur = tu[c];
    double fg_n = st.fg_n[c], bg_n = st.bg_n[c];
    double log_step = st.log_step[c], log_bar = st.log_bar[c], hbar = st.hbar[c];
    const double mu_da = st.mu_da[c];
    int64_t count = st.count[c], n_samples = st.n_samples[c], previous_update = st.previous_update[c];
    int adapt_window = st.adapt_window[c];
    int status = 0;
    unsigned long long tree_total = 0;

    for (int it = 0; it < out.n_iter; ++it) {
        const bool warmup = (it0 + it) < cfg.n_warmup;
        // base_hmc.py:244-247: P0 = (v0, p0), p0 = metric.random (n normals), then v0 (one normal)
        double p0[NPL];
#pragma unroll
        for (int r = 0; r < NPL; ++r) {
            const int j = lane + 32 * r;
            p0[r] = (j < n) ? inv_std[r] * bfb_draw_normal(seed, chain, (uint64_t)(t + j)) : 0.;
        }
        t += n;
        const double vt0 = bfb_draw_normal(seed, chain, (uint64_t)t); t++;
        // compute_state, integration.py:130-150 (values of both densities at the current point)
        double E0, w0, lp0;
        {
            double gt[NPL], lpb;
            t_eval<NPL>(M, q, lane, xsm, dsm, lp0, gt);
            t_eval<NPL>(MB, q, lane, xsm, dsm, lpb, gt);
            t_finish<NPL>(var, p0, u_cur, vt0, lp0, lpb, logxi, E0, w0);
        }
        if (!isfinite(E0)) { status = 2; break; }                     // base_hmc.py:249-253
        const double eps = warmup ? exp(log_step) : exp(log_bar);     // step_size.py:25-29

        double accept_stat, s_logp, s_energy, s_dE, s_maxdE = 0., s_u, s_w;
        int s_depth, s_size, diverging = 0;

        if (SAMPLER == BFB_NUTS) {
            // Tree.__init__, nuts.py:27-43 (TTree: the proposal also carries u and weight, tnuts.py:16-19)
            VST(oTL, q); VST(oTL + np, p0);
            VST(oTR, q); VST(oTR + np, p0);
            VST(oPS, p0); VST(oPQ, q);
            double uL = u_cur, vL = vt0, uR = u_cur, vR = vt0;
            double prop_E = E0, prop_lp = lp0, prop_u = u_cur, prop_w = w0, tree_ls = 0., acc_sum = 0., maxdE = 0.;
            int depth = 0, n_prop = 0;
            bool turn = false, nan_flag = false;
            for (int d = 0; d < cfg.max_treedepth; ++d) {
                // nuts.py:210 direction = logbern(log 0.5) * 2 - 1
                const double ud = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                const int dir = (log(ud) < -0.6931471805599453) ? 1 : -1;
                const int oEnd = dir > 0 ? oTR : oTL;
                VLD(q, oEnd); VLD(p, oEnd + np);
                VST(oPB, p);
                double u = dir > 0 ? uR : uL, vt = dir > 0 ? vR : vL;
                const double step = dir > 0 ? eps : -eps;
                const int nleaf = 1 << depth;
                double Rpl[NPL], Rps[NPL], Rqp[NPL];
                double Rls = 0., REp = 0., Rlpp = 0., Rup = 0., Rwp = 1.;
                // ---- _build_subtree(depth), nuts.py:134-178, iteratively ----
                for (int i = 0; i < nleaf; ++i) {
                    double lp, E, w;
                    t_leapfrog<NPL>(M, MB, logxi, step, var, q, p, u, vt, lane, xsm, dsm, lp, E, w);
                    // _single_step, nuts.py:105-132
                    double dE = E - E0;
                    if (isnan(dE)) dE = INFINITY;
                    if (fabs(dE) > fabs(maxdE)) maxdE = dE;
                    n_prop += 1;
                    if (!(fabs(dE) < cfg.max_change)) { diverging = 1; break; }
                    { const double e = exp(-dE); acc_sum += e < 1. ? e : 1.; }
#pragma unroll
                    for (int r = 0; r < NPL; ++r) { Rpl[r] = p[r]; Rps[r] = p[r]; Rqp[r] = q[r]; }
                    Rls = -dE; REp = E; Rlpp = lp; Rup = u; Rwp = w;
                    int lvl = 0;
                    while ((i >> lvl) & 1) {
                        const int oS = oST + lvl * SV * np;
                        double T1pl[NPL], T1pr[NPL], T1ps[NPL], ps[NPL];
                        VLD(T1pl, oS); VLD(T1pr, oS + np); VLD(T1ps, oS + 2 * np);
#pragma unroll
                        for (int r = 0; r < NPL; ++r) ps[r] = T1ps[r] + Rps[r];
                        bool turning = (UDOT(ps, T1pl) <= 0.) | (UDOT(ps, p) <= 0.);
                        if (lvl >= 1) {
                            double ps1[NPL], ps2[NPL];
#pragma unroll
                            for (int r = 0; r < NPL; ++r) { ps1[r] = T1ps[r] + Rpl[r]; ps2[r] = T1pr[r] + Rps[r]; }
                            turning |= (UDOT(ps1, T1pl) <= 0.) | (UDOT(ps1, Rpl) <= 0.);
                            turning |= (UDOT(ps2, T1pr) <= 0.) | (UDOT(ps2, p) <= 0.);
                        }
                        const double T1ls = ssc[lvl];
                        const double ls = np_logaddexp(T1ls, Rls);
                        const double um = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                        const double lb = Rls - ls;
                        if (isnan(lb)) nan_flag = true;
                        if (!(log(um) < lb)) {   // keep tree1's proposal
                            VLD(Rqp, oS + 3 * np);
                            REp = ssc[L + lvl]; Rlpp = ssc[2 * L + lvl]; Rup = ssc[3 * L + lvl]; Rwp = ssc[4 * L + lvl];
                        }
#pragma unroll
                        for (int r = 0; r < NPL; ++r) { Rpl[r] = T1pl[r]; Rps[r] = ps[r]; }
                        Rls = ls;
                        if (turning) { turn = true; break; }
                        lvl++;
                    }
                    if (turn) break;
                    if (i + 1 < nleaf) {
                        const int oS = oST + lvl * SV * np;
                        VST(oS, Rpl); VST(oS + np, p); VST(oS + 2 * np, Rps); VST(oS + 3 * np, Rqp);
                        // every lane writes the same scalars (each lane later reads back its own write: no sync needed)
                        ssc[lvl] = Rls; ssc[L + lvl] = REp; ssc[2 * L + lvl] = Rlpp; ssc[3 * L + lvl] = Rup; ssc[4 * L + lvl] = Rwp;
                    }
                }
                // Tree.extend, nuts.py:45-103
                VST(oEnd, q); VST(oEnd + np, p);
                if (dir > 0) { uR = u; vR = vt; } else { uL = u; vL = vt; }
                depth += 1;
                if (diverging || turn) break;
                {
                    const double ue = bfb_draw_uniform(seed, chain, (uint64_t)t); t++;
                    const double lb = Rls - tree_ls;
                    if (isnan(lb)) nan_flag = true;
                    if (log(ue) < lb) { VST(oPQ, Rqp); prop_E = REp; prop_lp = Rlpp; prop_u = Rup; prop_w = Rwp; }
                }
                tree_ls = np_logaddexp(tree_ls, Rls);
                double PS[NPL], PB[NPL], TLp[NPL], TRp[NPL], ps1[NPL], ps2[NPL];
                VLD(PS, oPS); VLD(PB, oPB); VLD(TLp, oTL + np); VLD(TRp, oTR + np);
#pragma unroll
                for (int r = 0; r < NPL; ++r) PS[r] += Rps[r];
                VST(oPS, PS);
                bool turning = (UDOT(PS, TLp) <= 0.) | (UDOT(PS, TRp) <= 0.);
                // the reference updates self.p_sum in place before forming p_sum1 / p_sum2 (nuts.py:86-98): the "old tree"
                // p_sum that enters them is already the total
                if (dir > 0) {
#pragma unroll
                    for (int r = 0; r < NPL; ++r) { ps1[r] = PS[r] + Rpl[r]; ps2[r] = PB[r] + Rps[r]; }
                    turning |= (UDOT(ps1, TLp) <= 0.) | (UDOT(ps1, Rpl) <= 0.);
                    turning |= (UDOT(ps2, PB) <= 0.) | (UDOT(ps2, p) <= 0.);
                } else {
#pragma unroll
                    for (int r = 0; r < NPL; ++r) { ps1[r] = Rps[r] + PB[r]; ps2[r] = Rpl[r] + PS[r]; }
                    turning |= (UDOT(ps1, p) <= 0.) | (UDOT(ps1, PB) <= 0.);
                    turning |= (UDOT(ps2, Rpl) <= 0.) | (UDOT(ps2, TRp) <= 0.);
                }
                if (turning) { turn = true; break; }
            }
            if (nan_flag) { status = 3; break; }
            accept_stat = acc_sum / (double)n_prop;
            s_logp = prop_lp; s_energy = prop_E; s_depth = depth; s_size = n_prop;
            s_dE = prop_E - E0; s_maxdE = maxdE; s_u = prop_u; s_w = prop_w;      // tnuts.py:21-33
            VLD(q, oPQ);
            tree_total += (unsigned long long)n_prop;
        } else {
            // HMC._hamiltonian_step, hmc.py:16-49, on the tempered integrator; stats of thmc.py:16-27
            double qs[NPL];
#pragma unroll
            for (int r = 0; r < NPL; ++r) { qs[r] = q[r]; p[r] = p0[r]; }
            double lp = lp0, E = E0, w = w0, u = u_cur, vt = vt0;
            for (int s = 0; s < cfg.n_int_step; ++s) t_leapfrog<NPL>(M, MB, logxi, eps, var, q, p, u, vt, lane, xsm, dsm, lp, E, w);
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
            s_u = u; s_w = w;       // of the integrated state, accepted or not (thmc.py:18-19); the next iteration starts from this u
            if (!accepted) {
#pragma unroll
                for (int r = 0; r < NPL; ++r) q[r] = qs[r];
            }
            tree_total += (unsigned long long)cfg.n_int_step;
        }
        u_cur = s_u;                // base_hmc.py:237 u0 = stats._u[-1]

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
        if (warmup && cfg.adapt_metric) {
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
                fg_n = bg_n; bg_n = 10.;
                previous_update = n_samples;
                if (cfg.doubling) adapt_window *= 2;
            }
            n_samples += 1;
        }

        // outputs: base_hmc.py:259-262, stats.py (TNStepStats / THStepStats)
        const size_t o = (size_t)c * out.n_iter + it;
        if (out.o.samples) {
#pragma unroll
            for (int r = 0; r < NPL; ++r) {
                const int j = lane + 32 * r;
                if (j < n) out.o.samples[o * n + j] = q[r];
            }
        }
        if (lane == 0) {
            if (out.u) out.u[o] = s_u;
            if (out.weight) out.weight[o] = s_w;
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
    }

    // persist chain state
#pragma unroll
    for (int r = 0; r < NPL; ++r) {
        const int j = lane + 32 * r;
        st.q[vb + j] = q[r]; st.var[vb + j] = var[r];
        st.fg_mean[vb + j] = fgm[r]; st.fg_raw[vb + j] = fgr[r];
        st.bg_mean[vb + j] = bgm[r]; st.bg_raw[vb + j] = bgr[r];
    }
    if (lane == 0) {
        tu[c] = u_cur;
        st.fg_n[c] = fg_n; st.bg_n[c] = bg_n;
        st.log_step[c] = log_step; st.log_bar[c] = log_bar; st.hbar[c] = hbar;
        st.count[c] = count; st.n_samples[c] = n_samples; st.previous_update[c] = previous_update;
        st.adapt_window[c] = adapt_window; st.t_draw[c] = t; st.iter[c] = it0 + out.n_iter;
        st.status[c] = status;
        if (tree_total) atomicAdd(st.tree_total, tree_total);
    }
}

template <int NPL, int SAMPLER>
int launch_t(bfb_context *h, const bfb_context *hb, const TRunOutDev &out)
{
    const int L = h->scfg.max_treedepth;
    const size_t per_warp = sizeof(double) * t_warp_smem_doubles(h->np, L), cap = 227 * 1024;
    int wpb = 1;
    size_t best = 0;
    for (int w = 1; w <= 8; ++w) {                       // resident warps per SM = blocks that fit x warps per block
        const size_t resident = (cap / (w * per_warp + sizeof(double) * T_MODEL_DOUBLES + 1024)) * w;
        if (resident > best) { best = resident; wpb = w; }
    }
    const size_t smem = per_warp * wpb + sizeof(double) * T_MODEL_DOUBLES;
    BFB_REQUIRE(smem <= cap, BFB_ERR_ARG, "tempered sampler needs %zu bytes of shared memory per block (> 227 KB)", smem);
    BFB_CUDA(cudaFuncSetAttribute(tsampler_kernel<NPL, SAMPLER>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int blocks = (int)((h->cs.C + wpb - 1) / wpb);
    tsampler_kernel<NPL, SAMPLER><<<blocks, 32 * wpb, smem, h->stream>>>(h->dm, hb->dm, h->t_logxi, h->scfg, h->cs, h->t_u, out, L);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

}  // namespace

extern "C" int bfb_tsampler_init(bfb_handle h, bfb_handle h_base, double logxi, const bfb_sampler_cfg *cfg, int64_t C,
                                 const double *x0, const double *u0, const double *step0, const double *var0, const double *mean0)
{
    BFB_REQUIRE(h && h_base && h->has_model && h_base->has_model, BFB_ERR_STATE, "bfb_tsampler_init: both handles need a model");
    BFB_REQUIRE(h != h_base && h->device == h_base->device, BFB_ERR_ARG, "bfb_tsampler_init: the base density needs a handle of its own on the same device");
    BFB_REQUIRE(h->n == h_base->n, BFB_ERR_ARG, "bfb_tsampler_init: density (%d inputs) and base density (%d) differ in input size", h->n, h_base->n);
    BFB_REQUIRE(u0 && std::isfinite(logxi), BFB_ERR_ARG, "bfb_tsampler_init: bad arguments");
    int rc = bfb_sampler_init(h, cfg, C, x0, step0, var0, mean0);     // diagonal metric; clears any tempered state
    if (rc) return rc;
    BFB_CUDA(cudaSetDevice(h->device));
    BFB_CUDA(cudaMalloc((void **)&h->t_u, sizeof(double) * 2 * (size_t)C));       // [C] current u | [C] u_0 (for bfb_sampler_reset)
    BFB_CUDA(cudaMemcpyAsync(h->t_u, u0, sizeof(double) * C, cudaMemcpyHostToDevice, h->stream));
    BFB_CUDA(cudaMemcpyAsync(h->t_u + C, u0, sizeof(double) * C, cudaMemcpyHostToDevice, h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    h->t_base = h_base;
    h->t_logxi = logxi;
    return BFB_OK;
}

extern "C" int bfb_tsampler_run(bfb_handle h, int sampler, int32_t n_iter, const bfb_run_out *out, double *u, double *weight,
                                int loc, int64_t *total_tree_size)
{
    BFB_REQUIRE(h && h->has_chains && h->t_base && h->t_u, BFB_ERR_STATE, "bfb_tsampler_run: call bfb_tsampler_init first");
    BFB_REQUIRE(h->t_base->has_model && h->t_base->n == h->n, BFB_ERR_STATE, "bfb_tsampler_run: the base handle's model changed");
    BFB_REQUIRE(out && n_iter > 0, BFB_ERR_ARG, "bfb_tsampler_run: bad arguments");
    BFB_REQUIRE(sampler == BFB_NUTS || sampler == BFB_HMC, BFB_ERR_ARG, "bfb_tsampler_run: sampler must be BFB_NUTS (TNUTS) or BFB_HMC (THMC)");
    BFB_REQUIRE(loc == BFB_HOST || loc == BFB_DEVICE, BFB_ERR_ARG, "bfb_tsampler_run: bad location");
    BFB_CUDA(cudaSetDevice(h->device));
    // the base handle's tables must be complete before this stream reads them
    BFB_CUDA(cudaStreamSynchronize(h->t_base->stream));
    const int64_t C = h->cs.C;
    const int n = h->n;
    const size_t R = (size_t)C * n_iter;
    // the 13 output fields: samples | 7 doubles of bfb_run_out | 3 int32 of bfb_run_out | u | weight
    void *user[13] = {out->samples, out->logp, out->energy, out->mean_tree_accept, out->step_size, out->step_size_bar,
                      out->energy_change, out->max_energy_change, out->tree_depth, out->tree_size, out->diverging, u, weight};
    size_t bytes[13];
    for (int f = 0; f < 13; ++f) bytes[f] = R * (f == 0 ? sizeof(double) * n : (f >= 8 && f <= 10 ? sizeof(int32_t) : sizeof(double)));
    void *dev[13];
    char *pool = nullptr;
    if (loc == BFB_HOST) {
        size_t total = 0;
        for (int f = 0; f < 13; ++f) if (user[f]) total += (bytes[f] + 255) & ~(size_t)255;
        if (total) BFB_CUDA(cudaMalloc((void **)&pool, total));
        size_t off = 0;
        for (int f = 0; f < 13; ++f) {
            dev[f] = user[f] ? pool + off : nullptr;
            if (user[f]) off += (bytes[f] + 255) & ~(size_t)255;
        }
    } else {
        for (int f = 0; f < 13; ++f) dev[f] = user[f];
    }
    TRunOutDev od;
    od.n_iter = n_iter;
    od.o.samples = (double *)dev[0];
    od.o.logp = (double *)dev[1]; od.o.energy = (double *)dev[2]; od.o.mean_tree_accept = (double *)dev[3];
    od.o.step_size = (double *)dev[4]; od.o.step_size_bar = (double *)dev[5]; od.o.energy_change = (double *)dev[6];
    od.o.max_energy_change = (double *)dev[7];
    od.o.tree_depth = (int32_t *)dev[8]; od.o.tree_size = (int32_t *)dev[9]; od.o.diverging = (int32_t *)dev[10];
    od.u = (double *)dev[11]; od.weight = (double *)dev[12];
    cudaError_t e = cudaMemsetAsync(h->cs.tree_total, 0, BFB_TREE_TOTAL_LEN * sizeof(unsigned long long), h->stream);
    int rc = BFB_OK;
    if (e == cudaSuccess) {
        cudaEventRecord(h->ev0, h->stream);
        const int npl = h->np / 32;
        if (sampler == BFB_NUTS) {
            switch (npl) {
            case 1: rc = launch_t<1, BFB_NUTS>(h, h->t_base, od); break;
            case 2: rc = launch_t<2, BFB_NUTS>(h, h->t_base, od); break;
            case 3: rc = launch_t<3, BFB_NUTS>(h, h->t_base, od); break;
            default: rc = launch_t<4, BFB_NUTS>(h, h->t_base, od); break;
            }
        } else {
            switch (npl) {
            case 1: rc = launch_t<1, BFB_HMC>(h, h->t_base, od); break;
            case 2: rc = launch_t<2, BFB_HMC>(h, h->t_base, od); break;
            case 3: rc = launch_t<3, BFB_HMC>(h, h->t_base, od); break;
            default: rc = launch_t<4, BFB_HMC>(h, h->t_base, od); break;
            }
        }
        cudaEventRecord(h->ev1, h->stream);
    }
    if (rc == BFB_OK && e == cudaSuccess && loc == BFB_HOST) {
        for (int f = 0; f < 13 && e == cudaSuccess; ++f)
            if (user[f]) e = cudaMemcpyAsync(user[f], dev[f], bytes[f], cudaMemcpyDeviceToHost, h->stream);
    }
    unsigned long long tt = 0;
    if (rc == BFB_OK && e == cudaSuccess) e = cudaMemcpyAsync(&tt, h->cs.tree_total, sizeof(tt), cudaMemcpyDeviceToHost, h->stream);
    if (rc == BFB_OK && e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (pool) cudaFree(pool);
    if (rc) return rc;
    if (e != cudaSuccess) { bfb_set_error("bfb_tsampler_run: %s", cudaGetErrorString(e)); return BFB_ERR_CUDA; }
    cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1);
    if (total_tree_size) *total_tree_size = (int64_t)tt;
    h->last_path = 0;
    h->iters_done += n_iter;
    return BFB_OK;
}
