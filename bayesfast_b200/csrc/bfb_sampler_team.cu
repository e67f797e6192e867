// bfb_sampler_team.cu -- NUTS / HMC with EIGHT chains per TEAM of four warps (bfb_team.cuh): the tensor-core sampler for
// linear + quadratic (+ cubic-2, + cubic-3 above 32 dimensions) surrogates with or without radial bound, HMC for input_size
// <= 64, NUTS for 32 < input_size <= 64.
//
// Reference restated here: samplers/hmc_utils/base_hmc.py:62-85, samplers/nuts.py:27-217, samplers/hmc.py:16-49,
// hmc_utils/integration.py:28-95, hmc_utils/metrics.py:73-91,186-211,333-371, hmc_utils/step_size.py:10-51.
#include "bfb_team.cuh"
#include "bfb_nuts_common.cuh"
#include <cstring>
#include <cstdlib>

static __device__ __noinline__ double team_draw_normal(uint64_t seed, uint64_t chain, uint64_t t) { return bfb_draw_normal(seed, chain, t); }
static __device__ __noinline__ double team_draw_uniform(uint64_t seed, uint64_t chain, uint64_t t) { return bfb_draw_uniform(seed, chain, t); }

// Nesterov dual averaging of the step size, step_size.py:31-45 (one instance in the kernel image: pow and exp are large)
static __device__ __noinline__ void team_dual_average(double cnt, double hbar0, double mu_da, double accept_stat, double log_bar,
                                                      double t0, double target, double gamma, double kk,
                                                      double &hbar, double &log_step, double &log_bar_new, double &e_step, double &e_bar)
{
    const double ww = 1. / (cnt + t0);
    hbar = ((1. - ww) * hbar0 + ww * (target - accept_stat));
    log_step = mu_da - hbar * sqrt(cnt) / gamma;
    const double mk = pow(cnt, -kk);
    log_bar_new = mk * log_step + (1. - mk) * log_bar;
    e_step = exp(log_step); e_bar = exp(log_bar_new);
}

// shared memory of a team of the HMC kernel: exchange buffers (x | x - mu | x^2) | reduction buffers | control words
template <int NR, int MV>
__host__ __device__ constexpr int team_base_doubles() { return 3 * TeamShape<NR, MV>::SLOT + TeamShape<NR, MV>::RED_DOUBLES + 24; }

// next work unit of the team (leader pops, everybody reads after the barrier); false when the queue is exhausted
__device__ __forceinline__ bool team_next_unit(int *queue, volatile int *ring, int n_units, bool &first, int slot, volatile int *tctl,
                                               int bar_id, bool leader, int &group)
{
    if (leader) {
        int idx = first ? slot : atomicAdd(queue, 1);
        int grp = -1;
        if (idx < n_units) { while ((grp = ring[idx]) < 0) __nanosleep(2000); }
        tctl[0] = grp;
    }
    first = false;
    team_bar(bar_id);
    group = tctl[0];
    team_bar(bar_id);              // everybody has read the word before the leader may write the next one
    __threadfence();
    return group >= 0;
}

// ----------------------------------------------------------------------------------------------------------------------
// HMC (samplers/hmc.py:16-49): n_int_step leapfrogs per iteration for every chain, no tree.
// ----------------------------------------------------------------------------------------------------------------------
template <int NR, int MV, int G>
__global__ void __launch_bounds__(128 * G, 1) hmc_team_kernel(DevModel M, bfb_sampler_cfg cfg, ChainState st, RunOutDevF out,
                                                              int base_iter, int chunk_iters, int n_groups, int n_units,
                                                              int *__restrict__ queue)
{
    using TS = TeamShape<NR, MV>;
    constexpr int NRW = TS::NRW;
    extern __shared__ double smem[];
    double *tab = smem, *msm = smem + TS::TAB_DOUBLES;
    for (int i = threadIdx.x; i < TS::TAB_DOUBLES; i += blockDim.x) tab[i] = M.tfrag[i];
    for (int i = threadIdx.x; i < TS::MSM_HALF && i < M.np; i += blockDim.x) { msm[i] = M.use_bound ? M.mu[i] : 0.; msm[TS::MSM_HALF + i] = M.lin[i]; }
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, team = wib >> 2, w = wib & 3, gi = lane >> 2, lg = lane & 3;
    double *tsm = smem + TS::TAB_DOUBLES + TS::MSM + (size_t)team * team_base_doubles<NR, MV>();
    double *xbuf = tsm, *red = tsm + 3 * TS::SLOT;
    const double *mu_t = msm;
    volatile int *tctl = reinterpret_cast<volatile int *>(red + TS::RED_DOUBLES);
    double *bcast = red + TS::RED_DOUBLES + 8;         // [2][8 chains]: value and energy of the end point, from the leader warp
    const int bar_id = 1 + team;
    const double *tab_w = tab + (size_t)w * NR * TS::NTW * 32;
    const bool leader = (w == 0 && lane == 0), scribe = (w == 0 && lg == 0);
    const int n = M.n;
    const DmmaConsts K = dmma_consts(M);
    volatile int *qv = queue;
    volatile int *ring = queue + 2 + n_groups;
    int rbuf = 0;
    bool first = true;
    const int slot = blockIdx.x + gridDim.x * team;
#pragma unroll 1
    for (;;) {
    int group;
    if (!team_next_unit(queue, ring, n_units, first, slot, tctl, bar_id, leader, group)) break;
    const int chunk = qv[2 + group];
    const int it_lo = chunk * chunk_iters;
    const int it_hi = min(out.n_iter, it_lo + chunk_iters);
    const int64_t c_raw = (int64_t)group * 8 + gi;
    const bool exists = c_raw < st.C;
    const int64_t c = exists ? c_raw : st.C - 1;
    const size_t vb = (size_t)c * M.np;
    double q[NRW], p[NRW], g[NRW], var[NRW];
#pragma unroll
    for (int i = 0; i < NRW; ++i) {
        const int j = 4 * (NRW * w + i) + lg;
        q[i] = st.q[vb + j]; g[i] = st.g[vb + j]; var[i] = st.var[vb + j]; p[i] = 0.;
    }
    const uint64_t seed = cfg.seed, chain_id = (uint64_t)(cfg.chain0 + c);
    int64_t t = st.t_draw[c];
    const int it0 = base_iter;
    double logp_q = st.logp[c];
    double log_step = st.log_step[c], log_bar = st.log_bar[c], hbar = st.hbar[c];
    const double mu_da = st.mu_da[c];
    int64_t count = st.count[c], n_samples = st.n_samples[c], previous_update = st.previous_update[c];
    int adapt_window = st.adapt_window[c];
    double fg_n = st.fg_n[c], bg_n = st.bg_n[c];
    int status = exists ? st.status[c] : 9;
    unsigned long long tree_total = 0;

#pragma unroll 1
    for (int it = it_lo; it < it_hi; ++it) {
        const bool warm = (it0 + it) < cfg.n_warmup;
        // momentum: metrics.py:83-86 (every lane draws the normals of its own dimensions)
        double qs[NRW], gs[NRW], part = 0.;
#pragma unroll
        for (int i = 0; i < NRW; ++i) {
            const int j = 4 * (NRW * w + i) + lg;
            const double z = (j < n) ? team_draw_normal(seed, chain_id, (uint64_t)(t + j)) : 0.;
            p[i] = (j < n) ? z / sqrt(var[i]) : 0.;
            part = fma(p[i], var[i] * p[i], part);
            qs[i] = q[i]; gs[i] = g[i];
        }
        double z0 = 0., z1 = 0., z2 = 0.;
        team_sum4(part, z0, z1, z2, red, rbuf, bar_id, lane, w);
        const double ke0 = part;
        bool live = status == 0;
        double E0 = 0.5 * ke0 - logp_q;
        if (live) {
            t += n;
            if (!isfinite(E0)) { status = 2; live = false; }                 // base_hmc.py:72-76
        }
        const double eps = warm ? exp(log_step) : exp(log_bar);               // step_size.py:25-29
        const double dt = 0.5 * eps;
        double lp = logp_q, E = E0;
#pragma unroll 1
        for (int s_ = 0; s_ < cfg.n_int_step; ++s_) {
            // integration.py:68-95
#pragma unroll
            for (int i = 0; i < NRW; ++i) {
                p[i] = fma(dt, g[i], p[i]);
                q[i] = fma(eps, var[i] * p[i], q[i]);
                const int e = (NRW * w + i) * 32 + lane;
                xbuf[e] = q[i]; xbuf[TS::SLOT + e] = q[i] - mu_t[4 * (NRW * w + i) + lg]; xbuf[2 * TS::SLOT + e] = q[i] * q[i];
            }
            team_bar(bar_id);
            double gn[NRW], ke2;
            team_logp_grad<NR, MV>(tab_w, msm, xbuf, red, rbuf, bar_id, lane, w, K, live, q, p, var, dt, lp, gn, ke2);
#pragma unroll
            for (int i = 0; i < NRW; ++i) { g[i] = gn[i]; p[i] = fma(dt, gn[i], p[i]); }
            E = 0.5 * ke2 - lp;
        }
        // the value and the kinetic energy are complete in the leader warp only (team_logp_grad)
        if (cfg.n_int_step > 0) {
            if (scribe) { bcast[gi] = lp; bcast[8 + gi] = E; }
            team_bar(bar_id);
            lp = bcast[gi]; E = bcast[8 + gi];
        }
        // HMC._hamiltonian_step, hmc.py:31-49
        double dE;
        int diverging = 0;
        if (isfinite(E)) { dE = E0 - E; diverging = fabs(dE) > cfg.max_change; }
        else { dE = -INFINITY; diverging = 1; }
        double accept_stat;
        { const double e_ = exp(dE); accept_stat = e_ < 1. ? e_ : 1.; }
        const double ua = team_draw_uniform(seed, chain_id, (uint64_t)t);
        bool accepted = false;
        if (live && !diverging) { t += 1; accepted = !(ua >= accept_stat); }
        const double s_logp = lp, s_energy = E;
        if (accepted) logp_q = lp;
        else {
#pragma unroll
            for (int i = 0; i < NRW; ++i) { q[i] = qs[i]; g[i] = gs[i]; }
        }
        if (live) {
            tree_total += (unsigned long long)cfg.n_int_step;
            if (warm && cfg.adapt_step_size) {          // step_size.py:31-45
                const double cnt = (double)count;
                const double ww = 1. / (cnt + cfg.t0);
                hbar = ((1. - ww) * hbar + ww * (cfg.target_accept - accept_stat));
                log_step = mu_da - hbar * sqrt(cnt) / cfg.gamma;
                const double mk = pow(cnt, -cfg.k);
                log_bar = mk * log_step + (1. - mk) * log_bar;
                count += 1;
            }
            if (warm && cfg.adapt_metric) {             // metrics.py:186-211, 351-357; Welford state in global memory
                const int64_t delta = n_samples - previous_update;
                const bool upd = ((delta + 1) % cfg.update_window == 0);
                const bool swap = delta >= adapt_window;
                fg_n += 1.; bg_n += 1.;
#pragma unroll
                for (int i = 0; i < NRW; ++i) {
                    const int j = 4 * (NRW * w + i) + lg;
                    if (j < n) {
                        double fgm = st.fg_mean[vb + j], fgr = st.fg_raw[vb + j], bgm = st.bg_mean[vb + j], bgr = st.bg_raw[vb + j];
                        double od = q[i] - fgm;
                        fgm += od / fg_n;
                        fgr += 1. * od * (q[i] - fgm);
                        od = q[i] - bgm;
                        bgm += od / bg_n;
                        bgr += 1. * od * (q[i] - bgm);
                        if (upd) var[i] = fgr / fg_n;
                        if (swap) { fgm = bgm; fgr = bgr; bgm = 0.; bgr = 0.; }
                        st.fg_mean[vb + j] = fgm; st.fg_raw[vb + j] = fgr; st.bg_mean[vb + j] = bgm; st.bg_raw[vb + j] = bgr;
                    }
                }
                if (swap) { fg_n = bg_n; bg_n = 10.; previous_update = n_samples; if (cfg.doubling) adapt_window *= 2; }
                n_samples += 1;
            }
            const size_t o = (size_t)c * out.n_iter + it;
            if (out.o.samples) {
#pragma unroll
                for (int i = 0; i < NRW; ++i) { const int j = 4 * (NRW * w + i) + lg; if (j < n) out.o.samples[o * n + j] = q[i]; }
            }
            if (scribe) {
                if (out.o.logp) out.o.logp[o] = s_logp;
                if (out.o.energy) out.o.energy[o] = s_energy;
                if (out.o.tree_depth) out.o.tree_depth[o] = accepted ? 1 : 0;
                if (out.o.tree_size) out.o.tree_size[o] = cfg.n_int_step;
                if (out.o.mean_tree_accept) out.o.mean_tree_accept[o] = accept_stat;
                if (out.o.step_size) out.o.step_size[o] = exp(log_step);
                if (out.o.step_size_bar) out.o.step_size_bar[o] = exp(log_bar);
                if (out.o.energy_change) out.o.energy_change[o] = dE;
                if (out.o.max_energy_change) out.o.max_energy_change[o] = 0.;
                if (out.o.diverging) out.o.diverging[o] = diverging;
            }
        }
    }
    // ---- persist chain state ----
    if (exists && st.status[c] == 0) {
#pragma unroll
        for (int i = 0; i < NRW; ++i) {
            const int j = 4 * (NRW * w + i) + lg;
            st.q[vb + j] = q[i]; st.g[vb + j] = g[i]; st.var[vb + j] = var[i];
        }
    }
    team_bar(bar_id);                // every warp has read st.status before the scribe overwrites it
    if (exists && scribe && st.status[c] == 0) {
        st.logp[c] = logp_q; st.fg_n[c] = fg_n; st.bg_n[c] = bg_n;
        st.log_step[c] = log_step; st.log_bar[c] = log_bar; st.hbar[c] = hbar;
        st.count[c] = count; st.n_samples[c] = n_samples; st.previous_update[c] = previous_update;
        st.adapt_window[c] = adapt_window; st.t_draw[c] = t; st.iter[c] = it0 + it_hi;
        st.status[c] = status;
        if (tree_total) atomicAdd(st.tree_total, tree_total);
    }
    __threadfence();
    team_bar(bar_id);
    if (leader) {
        qv[2 + group] = chunk + 1;
        if ((chunk + 1) * chunk_iters < out.n_iter) {
            const int ti = atomicAdd(queue + 1, 1);
            __threadfence();
            ring[ti] = group;
        }
    }
    }   // unit loop
}

template <int NR, int MV, int G>
static int launch_hmc_team(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    using TS = TeamShape<NR, MV>;
    const int64_t C = h->cs.C;
    const int n_groups = (int)((C + 7) / 8);
    const size_t smem = sizeof(double) * (TS::TAB_DOUBLES + TS::MSM + (size_t)G * team_base_doubles<NR, MV>());
    if (smem > (size_t)(227 * 1024)) return 1;
    BFB_CUDA(cudaFuncSetAttribute(hmc_team_kernel<NR, MV, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    RunOutDevF od;
    od.o = o; od.n_iter = n_iter;
    int blocks = h->sm_count;
    if ((int64_t)blocks > n_groups) blocks = n_groups;
    int chunk_iters, n_units, rc;
    if ((rc = queue_setup(h, n_groups, n_iter, 6, blocks * G, 0, chunk_iters, n_units))) return rc;
    hmc_team_kernel<NR, MV, G><<<blocks, 128 * G, smem, h->stream>>>(h->dm, h->scfg, h->cs, od, (int)h->iters_done, chunk_iters,
                                                                    n_groups, n_units, h->queue);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

template <int NR, int MV>
static int launch_hmc_team_g(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    int G = 4;
    if (const char *e = getenv("BFB200_TEAMS_PER_SM")) { int v = atoi(e); if (v >= 1 && v <= 5) G = v; }
    switch (G) {
    case 1: return launch_hmc_team<NR, MV, 1>(h, o, n_iter);
    case 3: return launch_hmc_team<NR, MV, 3>(h, o, n_iter);
    case 5: return launch_hmc_team<NR, MV, 5>(h, o, n_iter);
    }
    return launch_hmc_team<NR, MV, 4>(h, o, n_iter);
}

// launches the HMC kernel of the model (select_family, bfb_sampler.cu, chose this family): 0 on launch, 1 when its shared memory
// does not fit, < 0 on error
int bfb_launch_hmc_team(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    const DevModel &M = h->dm;
    if (M.team_nr == 16) {            // 32 < n <= 64: one team per SM (the operand table alone is 128 KB), more groups than SMs queue
        if (M.has_c3) return launch_hmc_team<16, 5, 1>(h, o, n_iter);
        return M.has_c2 ? launch_hmc_team<16, 1, 1>(h, o, n_iter) : launch_hmc_team<16, 0, 1>(h, o, n_iter);
    }
    const int mv = M.has_c2 ? 1 : 0;
#define BFB_CASE(NR_, MV_) if (M.team_nr == NR_ && mv == MV_) return launch_hmc_team_g<NR_, MV_>(h, o, n_iter);
    BFB_CASE(4, 0) BFB_CASE(4, 1) BFB_CASE(7, 0) BFB_CASE(7, 1) BFB_CASE(8, 0) BFB_CASE(8, 1)
#undef BFB_CASE
    bfb_set_error("bfb_launch_hmc_team: no kernel instantiation for this model");
    return BFB_ERR_ARG;
}

// ----------------------------------------------------------------------------------------------------------------------
// NUTS.  One round = one leapfrog of every live chain of the team, then whatever each chain needs (the 8 chains are NOT in
// lock step: own iteration / depth / leaf counters).  Work is split three ways:
//   * owners (all four warps, own dimensions): leapfrog, evaluation, every elementwise vector update -- proposal store,
//     sub-tree momentum sums, stack push, tree ends -- done SPECULATIVELY before the decisions (a pushed entry or a stored
//     proposal of a doubling that turns out to end here is dead data);
//   * tasks (one warp per tree level, whole vectors, reduction inside the quad only): the U-turn dot products of the merge
//     at level l for every chain whose leaf index has bit l set, and of Tree.extend for chains at the last leaf of a
//     doubling -- all levels of a leaf at once, in parallel on different warps (the merge order only matters for the
//     scalars);
//   * control (warp w owns the scalars of the chains 2 w and 2 w + 1, 16 lanes each): energies, multinomial weights, uniforms,
//     proposal slots, dual averaging, statistics, published as one command word per chain.  With two chains per warp most
//     rounds take the short path of every section (an iteration ends in 14 % of a warp's rounds instead of 44 % of a
//     single leader's), and the four warps decide in parallel.
// A lane therefore wears two hats: as owner / task lane it belongs to the row chain gi = lane >> 2, as control lane to the
// chain cc = 2 w + (lane >> 4); what crosses between the two goes through shared memory (command words, leaf energies).
// Barriers per round: 3-4 in the evaluation, pbuf, flags, command (+2 when a chain of the team crosses an iteration boundary).
// ----------------------------------------------------------------------------------------------------------------------
#define TC_FIN 1
#define TC_OK 2
#define TC_IEND 4
#define TC_RIGHT 8
#define TC_START (1 << 12)
#define TC_ENDP (1 << 13)
#define TC_STOP (1 << 14)
#define TC_FRESH (1 << 15)
#define TC_PNEW (1 << 16)

// doubles of shared memory per team: 14 fixed vector slots + 3 per stack level 1..LS | reduction | per-level scalars | flags
__host__ __device__ inline int team_nuts_doubles(int slot, int LS) { return (14 + 3 * LS) * slot + 256 + 400 + 96; }

template <int NR, int MV>
__global__ void __launch_bounds__(128, 1) nuts_team_kernel(DevModel M, bfb_sampler_cfg cfg, ChainState st, RunOutDevF out,
                                                           int L, int LS, double *__restrict__ gstack, double *__restrict__ gprop,
                                                           int base_iter, int chunk_iters, int n_groups, int n_units,
                                                           int *__restrict__ queue)
{
    using TS = TeamShape<NR, MV>;
    constexpr int NRW = TS::NRW, SLOT = TS::SLOT;
    extern __shared__ double smem[];
    double *tab = smem, *msm = smem + TS::TAB_DOUBLES;
    for (int i = threadIdx.x; i < TS::TAB_DOUBLES; i += blockDim.x) tab[i] = M.tfrag[i];
    for (int i = threadIdx.x; i < TS::MSM_HALF && i < M.np; i += blockDim.x) { msm[i] = M.use_bound ? M.mu[i] : 0.; msm[TS::MSM_HALF + i] = M.lin[i]; }
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, gi = lane >> 2, lg = lane & 3;
    const int cc = 2 * w + (lane >> 4), cl = lane & 15;         // control chain of this lane, lane index within its half warp
    double *tsm = smem + TS::TAB_DOUBLES + TS::MSM;
    double *xb = tsm, *sRL = tsm + SLOT, *sRS = tsm + 2 * SLOT, *sPBUF = tsm + 3 * SLOT;
    double *sTLQ = tsm + 4 * SLOT, *sTLP = tsm + 5 * SLOT, *sTLG = tsm + 6 * SLOT;
    double *sTRQ = tsm + 7 * SLOT, *sTRP = tsm + 8 * SLOT, *sTRG = tsm + 9 * SLOT;
    double *sPS = tsm + 10 * SLOT, *sPB = tsm + 11 * SLOT, *sVAR = tsm + 12 * SLOT, *sS0 = tsm + 13 * SLOT;
    double *red = tsm + 14 * SLOT;
    double *sSTK = red + 256 + 400 + 96;               // stack levels 1..LS last: everything else at a constant offset
    double *ssc = red + 256 + cc;                      // scalar (field f, level l) of the control chain at ssc[(f * 10 + l) * 8]
    double *flg = red + 256 + 400;
    volatile int *ci = reinterpret_cast<volatile int *>(flg);     // [0, 8) command words | [8, 20) level flags | 20 extend flags | 24 unit
    // [0,8) step | [8,16) logp | [16,24) draw counter | [24,32) kinetic energy | [32,40) first direction draw | [40,48) leaf logp | [48,56) leaf energy
    volatile double *cdv = flg + 16;
    const int bar_id = 1;
    const double *tab_w = tab + (size_t)w * NR * TS::NTW * 32;
    const double *mu_t = msm;
    const bool leader = (w == 0 && lane == 0), chief = (cl == 0);
    const int n = M.n;
    const DmmaConsts K = dmma_consts(M);
    volatile int *qv = queue;
    volatile int *ring = queue + 2 + n_groups;
    int rbuf = 0;
    bool first = true;
    const int slot_id = blockIdx.x;
#ifdef BFB_TEAM_TIMING     // per-phase cycle counters of warp 0 (printed with BFB200_DEBUG=1)
#define TTICK(k_) { const long long now_ = clock64(); tacc[k_] += now_ - tlast; tlast = now_; }
#else
#define TTICK(k_)
#endif
#define OWN(i_) ((NRW * w + (i_)) * 32 + lane)
#define OLD(dst, base) _Pragma("unroll") for (int i_ = 0; i_ < NRW; ++i_) dst[i_] = (base)[OWN(i_)];
#define OST(base, src) _Pragma("unroll") for (int i_ = 0; i_ < NRW; ++i_) (base)[OWN(i_)] = src[i_];

#pragma unroll 1
    for (;;) {
    int group;
    if (!team_next_unit(queue, ring, n_units, first, slot_id, ci + 24, bar_id, leader, group)) break;
    const int chunk = qv[2 + group];
    const int it_lo = chunk * chunk_iters;
    const int it_hi = min(out.n_iter, it_lo + chunk_iters);
    const int64_t c_raw = (int64_t)group * 8 + gi;
    const bool exists = c_raw < st.C;
    const int64_t c = exists ? c_raw : st.C - 1;
    const size_t vb = (size_t)c * M.np;
    const int64_t k_raw = (int64_t)group * 8 + cc;                 // control chain
    const bool k_exists = k_raw < st.C;
    const int64_t kc = k_exists ? k_raw : st.C - 1;
    double *gst = gstack + (size_t)group * (size_t)(L - 1 > LS ? L - 1 - LS : 0) * 3 * SLOT;      // deep stack levels (L2 resident)
    double *gpr = gprop + (size_t)group * BFB_NSLOT * 2 * SLOT;                                   // proposal pool (q, grad) per slot
    auto stk = [&](int lvl) -> double * { return (lvl <= LS) ? (sSTK + (lvl - 1) * 3 * SLOT) : (gst + (size_t)(lvl - 1 - LS) * 3 * SLOT); };

    // ---- row chain: vectors (own dimensions) and the counters every warp keeps in step ----
    double q[NRW], p[NRW], g[NRW], var[NRW], rpsf[NRW], pq[NRW], pg[NRW];
#pragma unroll
    for (int i = 0; i < NRW; ++i) {
        const int j = 4 * (NRW * w + i) + lg;
        q[i] = st.q[vb + j]; g[i] = st.g[vb + j]; var[i] = st.var[vb + j]; p[i] = 0.; rpsf[i] = 0.; pq[i] = q[i]; pg[i] = g[i];
    }
    const uint64_t seed = cfg.seed;
    const int it0 = base_iter;
    const int status0 = exists ? st.status[c] : 9;
    int status = status0;
    int it = it_lo, depth = 0, ileaf = 0, nslot = 1;
    bool done = (status != 0) || it_lo >= it_hi;
    double step = 0.;
    int n_samples = (int)st.n_samples[c], previous_update = (int)st.previous_update[c];      // < 2^31 iterations
    int adapt_window = st.adapt_window[c];
    double fg_n = st.fg_n[c], bg_n = st.bg_n[c];
    // ---- control chain: the scalars of the transition ----
    const uint64_t k_chain_id = (uint64_t)(cfg.chain0 + kc);
    int64_t t = st.t_draw[kc];
    double logp_q = st.logp[kc], log_step = st.log_step[kc], log_bar = st.log_bar[kc];
    double e_step = exp(log_step), e_bar = exp(log_bar);
    double E0 = 0., prop_E = 0., prop_lp = 0., acc_sum = 0., maxdE = 0.;
    WT Wtree; Wtree.m = 1.; Wtree.k = 0;
    int n_prop = 0, diverging = 0, prop_slot = 0, k_status = k_exists ? st.status[kc] : 9;
    unsigned freemask = 0, tree_total = 0;
    double ub0 = 0., ub1 = 0.;            // prefetched uniforms: lane cl holds draws tb2 + 2 cl + {0, 1} of the control chain
    int64_t tb2 = -(1ll << 40);

    // ---- the first command: start the first iteration of the unit ----
    {
        int cm = 0;
        if (k_status == 0 && it_lo < it_hi) {
            const bool warm_new = (it0 + it) < cfg.n_warmup;
            if (chief) { cdv[cc] = warm_new ? e_step : e_bar; cdv[8 + cc] = logp_q; cdv[16 + cc] = __longlong_as_double(t); }
            t += n + 1;                                   // the momentum normals and the direction of the first doubling
            prop_slot = 0;
            freemask = ((1u << BFB_NSLOT) - 1u) & ~1u;
            cm = TC_START | TC_FRESH | (1 << 4);
        }
        if (chief) ci[cc] = cm;
    }
    team_bar(bar_id);
    bool first_round = true;
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64(); (void)tacc; (void)tlast;
    unsigned dbg_rounds = 0; (void)dbg_rounds;

#pragma unroll 1
    for (;;) {
        // ================= apply the command: Tree.extend bookkeeping, next doubling, iteration boundary =================
        TTICK(6)
        const int cm = ci[gi];
        {
            const bool live = !done;
            const bool fin = live && (cm & TC_FIN);
            if (fin) {
                const bool right_cur = step > 0.;
                OST(right_cur ? sTRQ : sTLQ, q) OST(right_cur ? sTRP : sTLP, p) OST(right_cur ? sTRG : sTLG, g)
                depth += 1;
                if (cm & TC_OK) {
#pragma unroll
                    for (int i = 0; i < NRW; ++i) sPS[OWN(i)] += rpsf[i];
                }
                if (cm & TC_PNEW) {                             // the tree's proposal changed: fetch it now, it is needed at the boundary
                    const double *src = gpr + (size_t)((cm >> 8) & 15) * 2 * SLOT;
                    OLD(pq, src) OLD(pg, src + SLOT)
                }
                if (!(cm & TC_IEND)) {                          // next doubling: nuts.py:210 + the first lines of Tree.extend
                    const bool right = cm & TC_RIGHT;
                    OLD(q, right ? sTRQ : sTLQ) OLD(p, right ? sTRP : sTLP) OLD(g, right ? sTRG : sTLG)
                    OST(sPB, p)
                    step = right ? fabs(step) : -fabs(step);
                    ileaf = 0;
                }
            } else if (live && !first_round) ileaf += 1;
            if (live) nslot = (cm >> 4) & 15;
            const bool endp = live && (cm & TC_ENDP), startp = live && (cm & TC_START);
            TTICK(0)
            if (__any_sync(BFB_FULL, endp || startp)) {
                // ---- iteration boundary: base_hmc.py:62-85, Tree.__init__ nuts.py:27-43 ----
                const bool warm_old = (it0 + it) < cfg.n_warmup;            // of the iteration that ends
                if (endp) {
#pragma unroll
                    for (int i = 0; i < NRW; ++i) { q[i] = pq[i]; g[i] = pg[i]; }
                    if (out.o.samples) {
#pragma unroll
                        for (int i = 0; i < NRW; ++i) {
                            const int j = 4 * (NRW * w + i) + lg;
                            if (j < n) out.o.samples[((size_t)c * out.n_iter + it) * n + j] = q[i];
                        }
                    }
                    if (warm_old && cfg.adapt_metric) {       // windowed Welford metric: metrics.py:186-211, 333-371
                        const int delta = n_samples - previous_update;
                        const bool upd = ((delta + 1) % (int)cfg.update_window == 0);
                        const bool swap = delta >= adapt_window;
                        fg_n += 1.; bg_n += 1.;
#pragma unroll
                        for (int i = 0; i < NRW; ++i) {
                            const int j = 4 * (NRW * w + i) + lg;
                            if (j < n) {
                                double fgm = st.fg_mean[vb + j], fgr = st.fg_raw[vb + j], bgm = st.bg_mean[vb + j], bgr = st.bg_raw[vb + j];
                                double od = q[i] - fgm;
                                fgm += od / fg_n;
                                fgr += 1. * od * (q[i] - fgm);
                                od = q[i] - bgm;
                                bgm += od / bg_n;
                                bgr += 1. * od * (q[i] - bgm);
                                if (upd) var[i] = fgr / fg_n;
                                if (swap) { fgm = bgm; fgr = bgr; bgm = 0.; bgr = 0.; }
                                st.fg_mean[vb + j] = fgm; st.fg_raw[vb + j] = fgr; st.bg_mean[vb + j] = bgm; st.bg_raw[vb + j] = bgr;
                            }
                        }
                        if (swap) { fg_n = bg_n; bg_n = 10.; previous_update = n_samples; if (cfg.doubling) adapt_window *= 2; }
                        n_samples += 1;
                    }
                    it += 1;
                    if (cm & TC_STOP) done = true;
                }
                if (endp || startp) { OST(sVAR, var) }
                team_bar(bar_id);
                // momentum draw (metrics.py:83-86), lane = dimension, one chain at a time, the chains dealt to the four warps;
                // lane n draws the uniform that follows the normals: the direction of the first doubling (nuts.py:210)
                {
                    unsigned mask = __ballot_sync(BFB_FULL, startp && !done) & 0x11111111u;
                    int idx = 0;
#pragma unroll 1
                    while (mask) {
                        const int src = __ffs(mask) - 1;
                        mask &= mask - 1;
                        if ((idx & 3) == w) {
                            const int ch = src >> 2;
                            const int64_t t_s = __double_as_longlong(cdv[16 + ch]);
                            const uint64_t cid = (uint64_t)(cfg.chain0 + (int64_t)group * 8 + ch);
                            double kpart = 0.;
                            const int npass = n / 32 + 1;            // lane-indexed dimensions j = 32 pass + lane <= n (dimension n = the uniform)
#pragma unroll 1
                            for (int pass = 0; pass < npass; ++pass) {
                                const int j = 32 * pass + lane, e = (j >> 2) * 32 + src + (j & 3);
                                double p0j = 0., vj = 0.;
                                if (j < n) { vj = sVAR[e]; p0j = team_draw_normal(seed, cid, (uint64_t)(t_s + j)) / sqrt(vj); }
                                else if (j == n) cdv[32 + ch] = team_draw_uniform(seed, cid, (uint64_t)(t_s + n));
                                if (j < 4 * TS::NRP) sPBUF[e] = p0j;
                                kpart = fma(p0j, vj * p0j, kpart);
                            }
                            const double ke = warp_sum(kpart);
                            if (lane == 0) cdv[24 + ch] = ke;
                        }
                        ++idx;
                    }
                }
                team_bar(bar_id);
                if (startp && !done) {
                    OLD(p, sPBUF)
                    const double e0 = 0.5 * cdv[24 + gi] - cdv[8 + gi];
                    if (!isfinite(e0)) { status = 2; done = true; }        // base_hmc.py:72-76
                    else {
                        const bool right = cdv[32 + gi] < 0.5;
                        step = right ? cdv[gi] : -cdv[gi];
                        OST(sTLQ, q) OST(sTLP, p) OST(sTLG, g) OST(sTRQ, q) OST(sTRP, p) OST(sTRG, g) OST(sPS, p) OST(sPB, p)
                        if (cm & TC_FRESH) { OST(gpr, q) OST(gpr + SLOT, g) }       // starting point = slot 0 = the accepted proposal
#pragma unroll
                        for (int i = 0; i < NRW; ++i) { pq[i] = q[i]; pg[i] = g[i]; }
                        depth = 0; ileaf = 0;
                    }
                }
                // control chain: the new transition
                {
                    const int kcm = ci[cc];
                    if ((kcm & TC_START) && k_status == 0) {
                        const double lq = cdv[8 + cc];
                        const double e0 = 0.5 * cdv[24 + cc] - lq;
                        if (!isfinite(e0)) { k_status = 2; t -= 1; }               // the direction draw is not consumed
                        else { E0 = e0; prop_E = e0; prop_lp = lq; Wtree.m = 1.; Wtree.k = 0; acc_sum = 0.; maxdE = 0.; n_prop = 0; diverging = 0; }
                    }
                }
            }
        }
        first_round = false;
        TTICK(1)
        if (!__any_sync(BFB_FULL, !done)) break;
#ifdef BFB_TEAM_TIMING
        ++dbg_rounds;
#endif
        const bool live = !done;
        // control-chain view of the counters (every warp holds all 8 row chains)
        const int k_ileaf = __shfl_sync(BFB_FULL, ileaf, 4 * cc), k_depth = __shfl_sync(BFB_FULL, depth, 4 * cc);
        const int k_it = __shfl_sync(BFB_FULL, it, 4 * cc), k_nslot = __shfl_sync(BFB_FULL, nslot, 4 * cc);
        const bool k_live = __shfl_sync(BFB_FULL, (int)live, 4 * cc) != 0;
        // uniforms of the control chain: refilled when the window of 32 draws could run out within this round
        if (__any_sync(BFB_FULL, k_live && (t < tb2 || t - tb2 > 18))) {
            const bool rf = k_live && (t < tb2 || t - tb2 > 18);
            const uint64_t blk = (uint64_t)(t >> 1) + (uint64_t)cl;
            const bfb_philox_block b = bfb_philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)k_chain_id, (uint32_t)(k_chain_id >> 32),
                                                         (uint32_t)seed, (uint32_t)(seed >> 32));
            if (rf) {
                ub0 = bfb_u64_to_uniform((uint64_t)b.v[0] | ((uint64_t)b.v[1] << 32));
                ub1 = bfb_u64_to_uniform((uint64_t)b.v[2] | ((uint64_t)b.v[3] << 32));
                tb2 = (t >> 1) << 1;
            }
        }
        // ================= leapfrog (integration.py:68-95) and evaluation =================
        const double dt = 0.5 * step;
#pragma unroll
        for (int i = 0; i < NRW; ++i) {
            if (live) {
                p[i] = fma(dt, g[i], p[i]);
                q[i] = fma(step, var[i] * p[i], q[i]);
            }
            const int e = OWN(i);
            xb[e] = q[i]; xb[SLOT + e] = q[i] - mu_t[4 * (NRW * w + i) + lg]; xb[2 * SLOT + e] = q[i] * q[i];
        }
        team_bar(bar_id);
        {
            double gn[NRW], lp, ke2;
            team_logp_grad<NR, MV>(tab_w, msm, xb, red, rbuf, bar_id, lane, w, K, live, q, p, var, dt, lp, gn, ke2);
            if (live) {
#pragma unroll
                for (int i = 0; i < NRW; ++i) { g[i] = gn[i]; p[i] = fma(dt, gn[i], p[i]); }
            }
            if (w == 0 && lg == 0) { cdv[40 + gi] = lp; cdv[48 + gi] = 0.5 * ke2 - lp; }     // value and energy are complete in warp 0
        }
        TTICK(2)
        // ================= owners: proposal store, sub-tree sums, push (all speculative) =================
        const int k = live ? (__ffs(~ileaf) - 1) : 0;                       // merges this leaf completes (Tree._build_subtree)
        const bool last = live && (ileaf + 1 == (1 << depth));
        const int kmax = __reduce_max_sync(BFB_FULL, k);
        {
            OST(sPBUF, p)
            if (live) { double *slot = gpr + (size_t)nslot * 2 * SLOT; OST(slot, q) OST(slot + SLOT, g) }
            double rpl[NRW], rps[NRW];
#pragma unroll
            for (int i = 0; i < NRW; ++i) { rpl[i] = p[i]; rps[i] = p[i]; }
            if (kmax >= 1) {
                double s0[NRW];
                OLD(s0, sS0)
                if (k >= 1) {
#pragma unroll
                    for (int i = 0; i < NRW; ++i) { rpl[i] = s0[i]; rps[i] += s0[i]; }
                }
#pragma unroll 1
                for (int l = 1; l < kmax; ++l) {
                    double a[NRW], b[NRW];
                    if (l <= LS) { const double *sp = sSTK + (l - 1) * 3 * SLOT; OLD(a, sp) OLD(b, sp + 2 * SLOT) }
                    else { const double *sp = gst + (size_t)(l - 1 - LS) * 3 * SLOT; OLD(a, sp) OLD(b, sp + 2 * SLOT) }
                    if (k > l) {
#pragma unroll
                        for (int i = 0; i < NRW; ++i) { rpl[i] = a[i]; rps[i] += b[i]; }
                    }
                }
            }
            if (last) {
                OST(sRL, rpl) OST(sRS, rps)
#pragma unroll
                for (int i = 0; i < NRW; ++i) rpsf[i] = rps[i];
            } else if (live) {
                if (k == 0) { OST(sS0, p) }
                else if (k <= LS) { double *sp = sSTK + (k - 1) * 3 * SLOT; OST(sp, rpl) OST(sp + SLOT, p) OST(sp + 2 * SLOT, rps) }
                else { double *sp = gst + (size_t)(k - 1 - LS) * 3 * SLOT; OST(sp, rpl) OST(sp + SLOT, p) OST(sp + 2 * SLOT, rps) }
            }
        }
        team_bar(bar_id);
        TTICK(3)
        // ================= tasks: U-turn dot products of all merges of this leaf and of Tree.extend =================
#pragma unroll 1
        for (int l = 0; l < kmax; ++l) {
            if ((l & 3) != w) continue;
            double v0 = 0., v1 = 0., v2 = 1., v3 = 1., v4 = 1., v5 = 1.;
            if (l == 0) {
#pragma unroll
                for (int r = 0; r < NR; ++r) {
                    const int e = r * 32 + lane;
                    const double pr = sPBUF[e], vr = sVAR[e], t1 = sS0[e];
                    const double ps = t1 + pr;
                    v0 = fma(ps, vr * t1, v0); v1 = fma(ps, vr * pr, v1);
                }
            } else {
                v2 = v3 = v4 = v5 = 0.;
                double Rps[NR];
#pragma unroll
                for (int r = 0; r < NR; ++r) Rps[r] = sPBUF[r * 32 + lane] + sS0[r * 32 + lane];
                auto dots = [&](const double *sp, const double *spm) {
#pragma unroll
                    for (int r = 0; r < NR; ++r) {
                        const int e = r * 32 + lane;
                        const double pr = sPBUF[e], vr = sVAR[e];
                        const double T1pl = sp[e], T1pr = sp[SLOT + e], T1ps = sp[2 * SLOT + e], Rpl = spm[e];
                        const double ps = T1ps + Rps[r], ps1 = T1ps + Rpl, ps2 = T1pr + Rps[r];
                        const double vT1pl = vr * T1pl, vp = vr * pr;
                        v0 = fma(ps, vT1pl, v0); v1 = fma(ps, vp, v1);
                        v2 = fma(ps1, vT1pl, v2); v3 = fma(ps1, vr * Rpl, v3);
                        v4 = fma(ps2, vr * T1pr, v4); v5 = fma(ps2, vp, v5);
                    }
                };
                if (l <= LS) {                                    // everything in shared memory (the common case)
#pragma unroll 1
                    for (int m = 1; m < l; ++m) {
                        const double *sq = sSTK + (m - 1) * 3 * SLOT + 2 * SLOT + lane;
#pragma unroll
                        for (int r = 0; r < NR; ++r) Rps[r] += sq[r * 32];
                    }
                    dots(sSTK + (l - 1) * 3 * SLOT, (l == 1) ? sS0 : sSTK + (l - 2) * 3 * SLOT);
                } else {
#pragma unroll 1
                    for (int m = 1; m < l; ++m) {
                        const double *sq = stk(m) + 2 * SLOT + lane;
#pragma unroll
                        for (int r = 0; r < NR; ++r) Rps[r] += sq[r * 32];
                    }
                    dots(stk(l), (l == 1) ? sS0 : stk(l - 1));
                }
            }
            const bool turning = team_any_nonpos6(v0, v1, v2, v3, v4, v5, lane);
            const unsigned bal = __ballot_sync(BFB_FULL, turning);
            if (lane == 0) ci[8 + l] = (int)bal;
        }
        if (w == 3 && __any_sync(BFB_FULL, last)) {
            // Tree.extend, nuts.py:86-101 (self.p_sum is updated in place BEFORE p_sum1 / p_sum2 are formed)
            const bool right = step > 0.;
            double v0 = 0., v1 = 0., v2 = 0., v3 = 0., v4 = 0., v5 = 0.;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const int e = r * 32 + lane;
                const double pr = sPBUF[e], vr = sVAR[e], Rpl = sRL[e], Rps = sRS[e], PBr = sPB[e];
                const double PSn = sPS[e] + Rps;
                const double TLp = right ? sTLP[e] : pr, TRp = right ? pr : sTRP[e];
                const double vp = vr * pr, vRpl = vr * Rpl, vPB = vr * PBr, vTL = vr * TLp, vTR = vr * TRp;
                v0 = fma(PSn, vTL, v0); v1 = fma(PSn, vTR, v1);
                const double ps1 = right ? PSn + Rpl : Rps + PBr, ps2 = right ? PBr + Rps : Rpl + PSn;
                v2 = fma(ps1, right ? vTL : vp, v2); v3 = fma(ps1, right ? vRpl : vPB, v3);
                v4 = fma(ps2, right ? vPB : vRpl, v4); v5 = fma(ps2, right ? vp : vTR, v5);
            }
            const bool turning = team_any_nonpos6(v0, v1, v2, v3, v4, v5, lane);
            const unsigned bal = __ballot_sync(BFB_FULL, turning);
            if (lane == 0) ci[20] = (int)bal;
        }
        // ================= control: the leaf (Tree._single_step, nuts.py:105-132) =================
        const double lp = cdv[40 + cc], E = cdv[48 + cc];
        bool div_leaf = false;
        double dE = E - E0;
        if (isnan(dE)) dE = INFINITY;
        if (k_live) {
            if (fabs(dE) > fabs(maxdE)) maxdE = dE;
            n_prop += 1;
            div_leaf = !(fabs(dE) < cfg.max_change);
        }
        const WT wl = wt_from_dE(div_leaf ? 0. : dE);
        const bool okl = k_live && !div_leaf;
        if (okl) { acc_sum += wt_min1(wl); freemask &= ~(1u << k_nslot); }
        if (div_leaf) diverging = 1;
        const bool k_last = k_live && (k_ileaf + 1 == (1 << k_depth));
        team_bar(bar_id);
        TTICK(4)
        // ================= control: merges (Tree._build_subtree, nuts.py:134-178), Tree.extend, iteration end =================
        {
            auto uni = [&](int64_t tt) -> double {
                const int kk = (int)(tt - tb2) & 31;
                const int sl = (lane & 16) | (kk >> 1);
                const double a0 = __shfl_sync(BFB_FULL, ub0, sl), a1 = __shfl_sync(BFB_FULL, ub1, sl);
                return (kk & 1) ? a1 : a0;
            };
            WT RW = wl;
            double REp = E, Rlpp = lp;
            int Rslot = k_nslot;
            bool turn = false;
            int lvl = 0;
            bool need = okl && (k_ileaf & 1);
#pragma unroll 1
            while (__any_sync(BFB_FULL, need)) {
                const int lv = need ? lvl : 0;
                const bool turning = (ci[8 + lv] >> (cc * 4)) & 1;
                const double um = uni(t);
                if (need) {
                    t += 1;
                    WT T1W; T1W.m = ssc[lv * 8]; T1W.k = (int)ssc[(10 + lv) * 8];
                    const int T1slot = (int)ssc[(40 + lv) * 8];
                    const WT tot = wt_add(T1W, RW);
                    if (!wt_select(um, tot, RW)) {               // keep tree1's proposal (nuts.py:164-167)
                        freemask |= 1u << Rslot;
                        Rslot = T1slot; REp = ssc[(20 + lv) * 8]; Rlpp = ssc[(30 + lv) * 8];
                    } else {
                        freemask |= 1u << T1slot;
                    }
                    RW = tot;
                    if (turning) turn = true;
                    lvl++;
                }
                need = need && !turn && ((k_ileaf >> lvl) & 1);
            }
            const bool fin = k_live && (div_leaf || turn || k_last);
            if (k_live && !fin && chief) {
                ssc[lvl * 8] = RW.m; ssc[(10 + lvl) * 8] = (double)RW.k; ssc[(20 + lvl) * 8] = REp; ssc[(30 + lvl) * 8] = Rlpp;
                ssc[(40 + lvl) * 8] = (double)Rslot;
            }
            int cmn = 0;
            if (__any_sync(BFB_FULL, fin)) {
                // ---- end of a doubling: Tree.extend, nuts.py:45-103 ----
                const double ue = uni(t);
                const bool ok = fin && !div_leaf && !turn;
                if (ok) {
                    const bool eturn = (ci[20] >> (cc * 4)) & 1;
                    t += 1;
                    const WT tot = wt_add(Wtree, RW);
                    if (wt_select(ue, Wtree, RW)) {               // nuts.py:81-83 biased progressive: log(u) < size2 - size1
                        freemask |= 1u << prop_slot;
                        prop_slot = Rslot; prop_E = REp; prop_lp = Rlpp;
                        cmn |= TC_PNEW;
                    } else {
                        freemask |= 1u << Rslot;
                    }
                    Wtree = tot;
                    if (eturn) turn = true;
                }
                const bool iter_end = fin && (div_leaf || turn || (k_depth + 1 >= cfg.max_treedepth));
                if (fin) cmn |= TC_FIN | (ok ? TC_OK : 0) | (iter_end ? TC_IEND : 0) | (prop_slot << 8);
                if (__any_sync(BFB_FULL, iter_end)) {
                    // ---- end of the iteration: base_hmc.py:77-85 ----
                    const bool warm_old = (it0 + k_it) < cfg.n_warmup;
                    const double accept_stat = acc_sum / (double)(n_prop > 0 ? n_prop : 1);
                    if (__any_sync(BFB_FULL, iter_end && warm_old && cfg.adapt_step_size)) {      // step_size.py:31-45
                        const bool da = iter_end && warm_old && cfg.adapt_step_size;
                        const double hbar0 = st.hbar[kc], mu_da = st.mu_da[kc];
                        const int64_t count = st.count[kc];
                        __syncwarp();
                        double hbar, ls_, lb_, es_, eb_;
                        team_dual_average((double)count, hbar0, mu_da, accept_stat, log_bar, cfg.t0, cfg.target_accept, cfg.gamma, cfg.k,
                                          hbar, ls_, lb_, es_, eb_);
                        if (da) {
                            log_step = ls_; log_bar = lb_; e_step = es_; e_bar = eb_;
                            if (chief) { st.hbar[kc] = hbar; st.log_step[kc] = log_step; st.log_bar[kc] = log_bar; st.count[kc] = count + 1; }
                        }
                    }
                    if (iter_end) {
                        if (chief) {
                            const size_t orow = (size_t)kc * out.n_iter + k_it;
                            if (out.o.logp) out.o.logp[orow] = prop_lp;
                            if (out.o.energy) out.o.energy[orow] = prop_E;
                            if (out.o.tree_depth) out.o.tree_depth[orow] = k_depth + 1;
                            if (out.o.tree_size) out.o.tree_size[orow] = n_prop;
                            if (out.o.mean_tree_accept) out.o.mean_tree_accept[orow] = accept_stat;
                            if (out.o.step_size) out.o.step_size[orow] = e_step;
                            if (out.o.step_size_bar) out.o.step_size_bar[orow] = e_bar;
                            if (out.o.energy_change) out.o.energy_change[orow] = prop_E - E0;
                            if (out.o.max_energy_change) out.o.max_energy_change[orow] = maxdE;
                            if (out.o.diverging) out.o.diverging[orow] = diverging;
                        }
                        logp_q = prop_lp;
                        tree_total += (unsigned)n_prop;
                        const bool stop = (k_it + 1 >= it_hi);
                        cmn |= TC_ENDP | (stop ? TC_STOP : TC_START);
                        freemask = ((1u << BFB_NSLOT) - 1u) & ~(1u << prop_slot);
                        if (!stop) {
                            const bool warm_new = (it0 + k_it + 1) < cfg.n_warmup;
                            if (chief) { cdv[cc] = warm_new ? e_step : e_bar; cdv[8 + cc] = logp_q; cdv[16 + cc] = __longlong_as_double(t); }
                            t += n + 1;                   // the momentum normals and the direction of the first doubling (drawn at the boundary)
                        }
                    }
                }
                // ---- direction of the next doubling of this iteration (nuts.py:210) ----
                const bool nd = fin && !iter_end;
                const double ud = uni(t);
                if (nd) { t += 1; if (ud < 0.5) cmn |= TC_RIGHT; }
            }
            if (k_live) cmn |= (__ffs(freemask) - 1) << 4;
            if (chief) ci[cc] = cmn;
        }
        TTICK(5)
        team_bar(bar_id);
    }

    // ---- persist chain state ----
    if (exists && status0 == 0) {
#pragma unroll
        for (int i = 0; i < NRW; ++i) {
            const int j = 4 * (NRW * w + i) + lg;
            st.q[vb + j] = q[i]; st.g[vb + j] = g[i]; st.var[vb + j] = var[i];
        }
        if (w == 0 && lg == 0) {
            st.iter[c] = it0 + it;
            st.fg_n[c] = fg_n; st.bg_n[c] = bg_n; st.n_samples[c] = n_samples; st.previous_update[c] = previous_update;
            st.adapt_window[c] = adapt_window;
        }
    }
    if (k_exists && chief && st.status[kc] == 0) {
        st.logp[kc] = logp_q; st.t_draw[kc] = t;
        if (tree_total) atomicAdd(st.tree_total, (unsigned long long)tree_total);
    }
    __threadfence();
    team_bar(bar_id);
    if (k_exists && chief && k_status != 0 && k_status != 9) st.status[kc] = k_status;
    __threadfence();
    team_bar(bar_id);
    if (leader) {
#ifdef BFB_TEAM_TIMING
        atomicAdd(st.tree_total + 1, (unsigned long long)dbg_rounds);
        for (int k_ = 0; k_ < 7; ++k_) atomicAdd(st.tree_total + 4 + k_, (unsigned long long)tacc[k_]);
#endif
        qv[2 + group] = chunk + 1;
        if ((chunk + 1) * chunk_iters < out.n_iter) {
            const int ti = atomicAdd(queue + 1, 1);
            __threadfence();
            ring[ti] = group;
        }
    }
    }   // unit loop
#undef OWN
#undef OLD
#undef OST
}

template <int NR, int MV>
static int launch_nuts_team(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    using TS = TeamShape<NR, MV>;
    constexpr int SLOT = TS::SLOT;
    const int L = h->scfg.max_treedepth;
    const int64_t C = h->cs.C;
    const int n_groups = (int)((C + 7) / 8);
    // one team per SM (the operand table alone is 128 KB), more groups than SMs queue; stack levels 1..LS in shared memory,
    // deeper (rarely touched) levels in an L2-resident buffer
    const size_t fixed = sizeof(double) * (TS::TAB_DOUBLES + TS::MSM);
    int LS = L - 1;
    while (LS > 0 && fixed + sizeof(double) * team_nuts_doubles(SLOT, LS) > (size_t)(227 * 1024)) --LS;
    if (const char *e = getenv("BFB200_STACK_LEVELS_SMEM")) { int v = atoi(e); if (v >= 0 && v < LS) LS = v; }
    const size_t smem = fixed + sizeof(double) * team_nuts_doubles(SLOT, LS);
    if (smem > (size_t)(227 * 1024)) return 1;
    BFB_CUDA(cudaFuncSetAttribute(nuts_team_kernel<NR, MV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    double *gprop;
    int rc;
    if ((rc = gstack_reserve(h, n_groups, L, LS, SLOT, BFB_NSLOT, &gprop))) return rc;
    RunOutDevF od;
    od.o = o; od.n_iter = n_iter;
    int blocks = h->sm_count;
    if ((int64_t)blocks > n_groups) blocks = n_groups;
    int chunk_iters, n_units;
    if ((rc = queue_setup(h, n_groups, n_iter, 6, blocks, 0, chunk_iters, n_units))) return rc;
    nuts_team_kernel<NR, MV><<<blocks, 128, smem, h->stream>>>(h->dm, h->scfg, h->cs, od, L, LS, h->gstack, gprop, (int)h->iters_done,
                                                               chunk_iters, n_groups, n_units, h->queue);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

// launches the NUTS kernel of the model (select_family, bfb_sampler.cu, chose this family: 32 < n <= 64): 0 on launch, 1 when
// its shared memory does not fit, < 0 on error
int bfb_launch_nuts_team(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    const DevModel &M = h->dm;
    if (M.has_c3) return launch_nuts_team<16, 5>(h, o, n_iter);
    return M.has_c2 ? launch_nuts_team<16, 1>(h, o, n_iter) : launch_nuts_team<16, 0>(h, o, n_iter);
}
