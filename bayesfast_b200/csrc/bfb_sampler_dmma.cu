// bfb_sampler_dmma.cu -- NUTS with the surrogate evaluated on the FP64 tensor cores: EIGHT chains per warp.
//
// Applies to input_size <= 32 (<= 28 with cubic-3 configs), logp = output 0 of a linear + quadratic (+ cubic-2 (+ cubic-3))
// PolyModel with or without radial bound, decay, variable transform and module rescale (model variants of bfb_dmma.cuh; the
// BASELINE.json headline configuration is NR = 7, MV = 1); anything else runs the generic kernel of
// bfb_sampler.cu.  Same algorithm, same draw order (SURVEY.md 8a N-RNG).
//
// Mapping (bfb_dmma.cuh): a chain is owned by the 4 lanes of a quad, lane lg owning the dimensions j = 4 r + lg; the
// 8 chains of a warp are the 8 rows of an m8n8k4 DMMA whose B operand is the (chain-independent) coefficient table, so one
// leapfrog of 8 chains is 105 DMMAs (n = 26, cubic-2) instead of ~1500 warp-wide DFMAs + their operand loads.
// Everything else is an asynchronous state machine: the chains of a warp are NOT in lock
// step (own iteration / depth / leaf counters); the warp loops over rounds -- "two leapfrogs for every live chain (one if
// its doubling has a single leaf), then whatever each chain needs" -- with every section entered on __any_sync and
// committed per chain by predication; the per-dimension work of an iteration boundary (sample output, Welford metric,
// momentum normals) is done cooperatively, lane per dimension, one chain at a time.  Multinomial weights in
// the linear domain (mantissa, exponent), U-turn dot products reduced packed over the quad, proposals referred to by slot
// index into an L2-resident pool, deep tree-stack levels in an L2-resident buffer, persistent warps fed by the ready ring
// of (chain group, iteration chunk) units.
//
// Reference restated here: samplers/hmc_utils/base_hmc.py:62-85, samplers/nuts.py:27-217, hmc_utils/integration.py:28-95,
// hmc_utils/metrics.py:73-91,186-211,333-371, hmc_utils/step_size.py:10-51.
#include "bfb_dmma.cuh"
#include "bfb_nuts_common.cuh"
#include "bfb_nuts_dmma_common.cuh"
#include <cstring>
#include <cstdlib>

#if defined(BFB_DMMA_PART_HEADLINE) && defined(BFB_CODE_PAD)
// Code-placement padding (BFB_CODE_PAD = number of 16-byte instructions): shifts the kernels of this module relative to the
// instruction-cache sets (a scan over 0..28 KB moved the run time by +-2 %).  Never launched.
template <int N>
__global__ void bfb_pad_kernel(double *p)
{
    double a = p[0];
#pragma unroll
    for (int i = 0; i < N; ++i) a = fma(a, 1.0000001, 0.5);
    p[0] = a;
}
void *bfb_pad_kernel_ref() { return (void *)bfb_pad_kernel<BFB_CODE_PAD>; }
#endif


// shared memory per warp, in doubles: TL q,p,g | TR q,p,g | PS | PB | stack levels 0..LS (pl, pr, psum) | per-level
// scalars [5][10][8 chains]: weight mantissa, weight exponent, proposal energy, proposal logp, proposal slot.  Level 0 holds
// the current subtree R; its scalars live in registers, and scalar level 0 holds the first leaf of a pair until it is merged.
// A vector slot holds element (r, lane) at r * 32 + lane: every access is one conflict-free 256-byte row.
__host__ __device__ inline int warp_smem_doubles(int NR, int LS) { return (11 + 3 * LS) * NR * 32 + 400; }

template <int NR, int MV, int W>
__global__ void __launch_bounds__(32 * W, 1) nuts_dmma_kernel(DevModel M, bfb_sampler_cfg cfg, ChainState st, RunOutDevF out,
                                                              int L, int LS, double *__restrict__ gstack,
                                                              double *__restrict__ gprop, int base_iter, int chunk_iters,
                                                              int n_groups, int n_units, int *__restrict__ queue, int cpg)
{
    // section: setup
    using SH = DmmaShape<NR, MV>;
    constexpr int SLOT = NR * 32;
    extern __shared__ double smem[];
    double *bsm = smem;                       // coefficient operand table
    double *msm = smem + SH::frag_doubles(W);    // per-dimension tables (dmma_stage_tables)
    if (!SH::LIK) { for (int i = threadIdx.x; i < SH::FRAG_DOUBLES; i += blockDim.x) bsm[i] = M.bfrag[i]; }
    dmma_stage_tables<MV>(M, msm);
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, gi = lane >> 2, lg = lane & 3;
    const int c3x = SH::C3 ? dmma_c3_doubles(NR, M.c3_kt, W) : 0;          // cubic-3 operand table, pair table, x scratch
    double *wsm = smem + SH::frag_doubles(W) + SH::MSM_DOUBLES + c3x + (size_t)wib * warp_smem_doubles(NR, LS);
    double *sTL = wsm, *sTR = wsm + 3 * SLOT, *sPS = wsm + 6 * SLOT, *sPB = wsm + 7 * SLOT, *sST = wsm + 8 * SLOT;
    double *ssc = wsm + (11 + 3 * LS) * SLOT + gi;       // scalar (field f, level l) of this chain at ssc[(f * 10 + l) * 8]
    const int n = M.n;
    const DmmaConsts K = dmma_consts(M);

#ifdef BFB_DMMA_TIMING     // per-section cycle counters and round / section counts (printed with BFB200_DEBUG=1); costs ~1 %
#define TICK(k) { const long long now_ = clock64(); tacc[k] += now_ - tlast; tlast = now_; }
#define DBG_COUNT(v) ++v;
#else
#define TICK(k)
#define DBG_COUNT(v)
#endif
#define VLD(dst, base)  _Pragma("unroll") for (int r_ = 0; r_ < NR; ++r_) dst[r_] = (base)[r_ * 32 + lane];
#define VST(base, src)  _Pragma("unroll") for (int r_ = 0; r_ < NR; ++r_) (base)[r_ * 32 + lane] = src[r_];

    volatile int *qv = queue;
    volatile int *ring = queue + 2 + n_groups;
    bool first_unit = true;                       // the first unit of a warp is pre-assigned: 512 groups spread over all 148 SMs
#pragma unroll 1
    for (;;) {
    int idx = 0, group = 0;
    if (lane == 0) {
        idx = first_unit ? (int)(blockIdx.x + gridDim.x * wib) : atomicAdd(queue, 1);
        if (idx < n_units) { while ((group = ring[idx]) < 0) __nanosleep(1000); }
    }
    first_unit = false;
    idx = __shfl_sync(BFB_FULL, idx, 0);
    if (idx >= n_units) break;
    group = __shfl_sync(BFB_FULL, group, 0);
    __threadfence();
    const int chunk = qv[2 + group];
    const int it_lo = chunk * chunk_iters;
    const int it_hi = min(out.n_iter, it_lo + chunk_iters);
    const long long t_unit0 = clock64(); (void)t_unit0;
    const int64_t c_raw = (int64_t)group * cpg + gi;          // cpg <= 8 chains per group (rows of the MMA); the other quads idle
    const bool exists = gi < cpg && c_raw < st.C;
    const int64_t c = exists ? c_raw : st.C - 1;
    double *gst = gstack + (size_t)group * (size_t)(L - 1 > LS ? L - 1 - LS : 0) * 3 * SLOT;   // deep stack levels (L2 resident)
    // proposals (q, grad) are written once, at the leaf, into a slot of an L2-resident pool and are afterwards only
    // referred to by their slot index: merges move no vectors.  Same thread writes and reads a given element.
    double *gpr = gprop + (size_t)group * BFB_NSLOT * 2 * SLOT;

    // ---- chain state (adaptation scalars stay in global memory: they are touched once per iteration) ----
    const size_t vb = (size_t)c * M.np;
    double q[NR], p[NR], g[NR], var[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int j = 4 * r + lg;
        q[r] = st.q[vb + j]; g[r] = st.g[vb + j]; var[r] = st.var[vb + j]; p[r] = 0.;
    }
    const uint64_t seed = cfg.seed, chain_id = (uint64_t)(cfg.chain0 + c);
    int64_t t = st.t_draw[c];
    const int it0 = base_iter;                 // iterations done before this launch (same for every chain)
    double logp_q = st.logp[c];
    double log_step = st.log_step[c], log_bar = st.log_bar[c];
    double e_step = exp(log_step), e_bar = exp(log_bar);    // refreshed only when dual averaging moves them
    int status = exists ? st.status[c] : 9;
    unsigned tree_total = 0, dbg_rounds = 0, dbg_merges = 0, dbg_iend = 0; (void)dbg_rounds; (void)dbg_merges; (void)dbg_iend;
    // tacc: 0..6 the sections of a round (0: the boundary outside its parts), 7 the loop head, 8..11 the boundary's parts
    long long tacc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64(); (void)tacc; (void)tlast;
    bool done = (status != 0) || it_lo >= it_hi;
    int it = it_lo;
    // progress reports (host outputs of a single launch, bfb_sampler_run_ex): every chain counts itself in when it has finished a
    // report chunk of rep_it iterations -- independent of the work units, whose ends synchronise the 8 chains of a group
    const int *pgb = queue + 2 + n_groups + n_units;            // [0] armed, [1..2] host flag address, [3] rep_it, [4 + k] counts
    const int rep_it = pgb[0] ? pgb[3] : 0;
    int next_rep = rep_it > 0 ? min((it_lo / rep_it + 1) * rep_it, out.n_iter) : -1;

    // transition state
    double E0 = 0., step = 0., prop_E = 0., prop_lp = 0., acc_sum = 0., maxdE = 0.;
    WT Wtree; Wtree.m = 1.; Wtree.k = 0;
    int depth = 0, ileaf = 0, n_prop = 0, diverging = 0, prop_slot = 0, Rslot = 0;
    unsigned freemask = 0;
    double REp = 0., Rlpp = 0.;
    WT RW; RW.m = 0.; RW.k = 0;
    // per-chain control flags: bnd = an iteration boundary is pending (end the previous iteration unless `fresh`,
    // start the next unless done), ns_dbl = a doubling must be started
    bool bnd = !done, fresh = true, ns_dbl = false;
    // the current subtree R (left-end p, right-end p, p_sum) is the level-0 stack entry
    double *sR = sST;
    // scratch vectors of the boundary section alias the (then empty) level-0 stack entry: the next state's position,
    // gradient and metric, staged by the chain's quad for the lane-per-dimension pass
    double *sGX = sST, *sVAR = sST + SLOT, *sQN = sST + 2 * SLOT;

    // stack entry of level lvl: levels 0..LS in shared memory, deeper ones in the L2-resident buffer
    auto stack_ptr = [&](int lvl) -> double * {
        return (lvl <= LS) ? (sST + lvl * 3 * SLOT) : (gst + (size_t)(lvl - 1 - LS) * 3 * SLOT);
    };

#pragma unroll 1
    while (__any_sync(BFB_FULL, !done)) {
        TICK(7)
        // section: boundary
        // ================= iteration boundary: base_hmc.py:62-85, Tree.__init__ nuts.py:27-43 =================
        if (__any_sync(BFB_FULL, bnd)) {
            DBG_COUNT(dbg_iend)
            const bool endp = bnd && !fresh;
            const bool warm_old = (it0 + it) < cfg.n_warmup;            // of the iteration that ends
            const size_t orow = (size_t)c * out.n_iter + it;
            // the accepted proposal (position, gradient) comes from the L2-resident pool: issue the loads first.  A fresh
            // chain's starting point becomes the accepted proposal in slot 0 of the pool, so every chain's next state is read
            // from there
            if (fresh && bnd) { VST(gpr, q) VST(gpr + SLOT, g) }
            double qn[NR], gx[NR];
            {
                const double *slot = gpr + (size_t)(endp ? prop_slot : 0) * 2 * SLOT;
                VLD(qn, slot) VLD(gx, slot + SLOT)
            }
            TICK(0)
            // section: boundary statistics
            // ---- (1) per chain (its quad), predicated: accept statistic, dual averaging, statistics ----
            const double accept_stat = acc_sum / (double)(n_prop > 0 ? n_prop : 1);
            if (__any_sync(BFB_FULL, endp && warm_old && cfg.adapt_step_size)) {      // step_size.py:31-45
                const double hbar0 = st.hbar[c], mu_da = st.mu_da[c];
                const int64_t count = st.count[c];
                __syncwarp();
                double hbar_, ls_, lb_, es_, eb_;
                dual_average_ni((double)count, hbar0, mu_da, accept_stat, log_bar, cfg.t0, cfg.target_accept, cfg.gamma, cfg.k, hbar_, ls_, lb_, es_, eb_);
                if (endp && warm_old && cfg.adapt_step_size) {
                    log_step = ls_; log_bar = lb_; e_step = es_; e_bar = eb_;
                    if (lg == 0) { st.hbar[c] = hbar_; st.log_step[c] = log_step; st.log_bar[c] = log_bar; st.count[c] = count + 1; }
                }
            }
            if (endp) {
                if (lg == 0) {
                    if (out.o.logp) out.o.logp[orow] = prop_lp;
                    if (out.o.energy) out.o.energy[orow] = prop_E;
                    if (out.o.tree_depth) out.o.tree_depth[orow] = depth;
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
                it += 1;
                if (it >= it_hi) done = true;
            }
            if (bnd) { VST(sQN, qn) VST(sGX, gx) VST(sVAR, var) }
            __syncwarp();
            TICK(8)
            // section: boundary lane per dimension
            // ---- (2) cooperative, lane j = dimension j, one chain at a time: new sample out, windowed Welford
            //      metric (metrics.py:186-211, 333-371), momentum draw (metrics.py:83-86), and the two ends and p_sum
            //      of the new tree (Tree.__init__): position, momentum and gradient of the new state ----
            unsigned mask = __ballot_sync(BFB_FULL, bnd);
#pragma unroll 1
            while (mask) {
                const int src = (__ffs(mask) - 1) & ~3;
                mask &= ~(0xfu << src);
                const int64_t c_s = shfl64(c, src), t_s = shfl64(t, src);
                const int it_s = __shfl_sync(BFB_FULL, it, src), slot_s = __shfl_sync(BFB_FULL, prop_slot, src);
                const int fl = __shfl_sync(BFB_FULL, (endp ? 1 : 0) | (done ? 2 : 0) | (warm_old ? 4 : 0), src);
                const int j = lane, e = (j >> 2) * 32 + src + (j & 3);     // element of a vector slot holding dim j of that chain
                if (fl & 1) {
                    const double qj = (j < 4 * NR) ? sQN[e] : 0.;
                    if (out.o.samples && j < n) out.o.samples[((size_t)c_s * out.n_iter + (it_s - 1)) * n + j] = qj;
                    if ((fl & 4) && cfg.adapt_metric) {
                        const int64_t n_samples = st.n_samples[c_s], previous_update = st.previous_update[c_s];
                        const int adapt_window = st.adapt_window[c_s];
                        const double fg_n = st.fg_n[c_s] + 1., bg_n = st.bg_n[c_s] + 1.;
                        __syncwarp();
                        const int64_t delta = n_samples - previous_update;
                        const bool upd = ((delta + 1) % cfg.update_window == 0);
                        const bool swap = delta >= adapt_window;
                        const size_t vi = (size_t)c_s * M.np + (j < n ? j : 0);
                        if (j < n) {
                        double fgm = st.fg_mean[vi], fgr = st.fg_raw[vi], bgm = st.bg_mean[vi], bgr = st.bg_raw[vi];
                        double od = qj - fgm;
                        fgm += od / fg_n;
                        fgr += 1. * od * (qj - fgm);
                        od = qj - bgm;
                        bgm += od / bg_n;
                        bgr += 1. * od * (qj - bgm);
                        if (upd) sVAR[e] = fgr / fg_n;
                        if (swap) { fgm = bgm; fgr = bgr; bgm = 0.; bgr = 0.; }
                        st.fg_mean[vi] = fgm; st.fg_raw[vi] = fgr; st.bg_mean[vi] = bgm; st.bg_raw[vi] = bgr;
                        }
                        if (lane == 0) {
                            st.fg_n[c_s] = swap ? bg_n : fg_n;
                            st.bg_n[c_s] = swap ? 10. : bg_n;
                            if (swap) { st.previous_update[c_s] = n_samples; if (cfg.doubling) st.adapt_window[c_s] = adapt_window * 2; }
                            st.n_samples[c_s] = n_samples + 1;
                        }
                    }
                }
                if (!(fl & 2)) {
                    double p0j = 0.;
                    if (j < n) p0j = draw_normal_ni(seed, (uint64_t)(cfg.chain0 + c_s), (uint64_t)(t_s + j)) / sqrt(sVAR[e]);
                    if (j < 4 * NR) {
                        const double qj = sQN[e], gj = sGX[e];
                        sTL[e] = qj; sTL[SLOT + e] = p0j; sTL[2 * SLOT + e] = gj;
                        sTR[e] = qj; sTR[SLOT + e] = p0j; sTR[2 * SLOT + e] = gj;
                        sPS[e] = p0j;
                    }
                }
            }
            __syncwarp();
            TICK(9)
            // section: boundary progress report
            {
                const bool hit = endp && it == next_rep;          // this chain's records of report chunk (it - 1) / rep_it are written
                if (__any_sync(BFB_FULL, hit)) {
                    __threadfence();                              // ... by several lanes (statistics: its quad, sample: lane per dimension)
                    __syncwarp();
                    if (hit) {
                        if (lg == 0) {
                            int *pg = queue + 2 + n_groups + n_units;
                            const int k = (it - 1) / rep_it;
                            if (atomicAdd(pg + 4 + k, 1) == (int)st.C - 1) {      // the last chain: tell the host (mapped pinned memory)
                                int *flag = reinterpret_cast<int *>(((unsigned long long)(unsigned)pg[2] << 32) | (unsigned long long)(unsigned)pg[1]);
                                *(volatile int *)flag = k + 1;
                                __threadfence_system();
                            }
                        }
                        next_rep = min(next_rep + rep_it, out.n_iter);
                    }
                }
            }
            TICK(10)
            // section: boundary new state
            // ---- (3) per chain, predicated: the new state and the empty tree ----
            double p0[NR], part = 0.;
            VLD(p0, sTL + SLOT)
            if (bnd) { VLD(q, sQN) VLD(g, sGX) VLD(var, sVAR) }
#pragma unroll
            for (int r = 0; r < NR; ++r) part = fma(p0[r], var[r] * p0[r], part);
            const double ke = qsum(part);
            const bool warm_new = (it0 + it) < cfg.n_warmup;
            const bool startp = bnd && !done;
            if (startp) {
                t += n;
                E0 = 0.5 * ke - logp_q;
                if (!isfinite(E0)) { status = 2; done = true; }
                step = warm_new ? e_step : e_bar;
                if (fresh) prop_slot = 0;
                freemask = ((1u << BFB_NSLOT) - 1u) & ~(1u << prop_slot);
                prop_E = E0; prop_lp = logp_q; Wtree.m = 1.; Wtree.k = 0; acc_sum = 0.; maxdE = 0.;
                depth = 0; n_prop = 0; diverging = 0;
                ns_dbl = !done;
            }
            bnd = false; fresh = false;
            TICK(11)
            if (!__any_sync(BFB_FULL, !done)) break;
        }
        const bool live = !done;
        DBG_COUNT(dbg_rounds)
        TICK(0)
        // section: round start
        // ---- uniforms of this round: lane lg of a quad holds draws 2 (t/2 + lg) + {0, 1} of its chain ----
        const int64_t tb2 = (t >> 1) << 1;
        const double2 ub = philox_pair_ni(seed, chain_id, (uint64_t)(t >> 1) + (uint64_t)lg);
        const double ub0 = ub.x, ub1 = ub.y;
        auto uni = [&](int64_t tt) -> double {
            const int k = (int)(tt - tb2);
            const int sl = (lane & ~3) | ((k >> 1) & 3);
            const double a0 = __shfl_sync(BFB_FULL, ub0, sl), a1 = __shfl_sync(BFB_FULL, ub1, sl);
            double u = (k & 1) ? a1 : a0;
            if (__any_sync(BFB_FULL, k >= 8)) { if (k >= 8) u = draw_uniform_ni(seed, chain_id, (uint64_t)tt); }
            return u;
        };
        // ================= start of a doubling: nuts.py:210 + the first lines of Tree.extend =================
        if (__any_sync(BFB_FULL, ns_dbl)) {
            const double ud = uni(t);
            if (ns_dbl) {
                t += 1;
                const bool right = ud < 0.5;                     // log(u) < log(0.5) on the draw grid of bfb_rng.h
                const double *src = right ? sTR : sTL;
                VLD(q, src) VLD(p, src + SLOT) VLD(g, src + 2 * SLOT)
                VST(sPB, p)
                step = right ? fabs(step) : -fabs(step);
                ileaf = 0;
                ns_dbl = false;
            }
        }
        TICK(1)
        // section: evaluation
        // ================= two leaves per round =================
        // A leaf with an even index is never followed by a decision (it is the left child of a level-0 merge), so a
        // round integrates a PAIR of leaves whenever the doubling has at least two: the fixed cost of a round (every
        // section below is paid per warp, not per chain) is spread over two leapfrogs.  Doublings of one leaf and
        // divergent first leaves skip the second half.
        const double dt = 0.5 * step;
        bool div_now = false, turn = false, did2 = false;
#ifdef BFB_UNROLL_HALVES
#pragma unroll
#else
#pragma unroll 1
#endif
        for (int half = 0; half < 2; ++half) {
            const bool go = live && (half == 0 || (!div_now && depth >= 1));
            if (half == 1 && !__any_sync(BFB_FULL, go)) break;
            // ---- leapfrog: integration.py:68-95.  In place (register diet: the state of a chain that sits this half out is
            // left untouched, its MMA row computes garbage that is ignored): p <- p + dt g, q <- q + step var p
            if (go) {
#pragma unroll
                for (int r = 0; r < NR; ++r) {
                    p[r] = fma(dt, g[r], p[r]);
                    q[r] = fma(step, var[r] * p[r], q[r]);
                }
            }
            double lp, ke2;
            {
                double gn[NR];
                dmma_logp_grad<NR, MV>(bsm, lane, K, q, msm, go, lp, gn,
                                       [&](const double (&gg)[NR]) {
                                           double s_ = 0.;
#pragma unroll
                                           for (int r = 0; r < NR; ++r) { const double pn = fma(dt, gg[r], p[r]); s_ = fma(pn, var[r] * pn, s_); }
                                           return s_;
                                       }, ke2);
                if (go) {
#pragma unroll
                    for (int r = 0; r < NR; ++r) {
                        g[r] = gn[r];
                        p[r] = fma(dt, gn[r], p[r]);
                    }
                }
            }
            // section: leaf
            const double E = 0.5 * ke2 - lp;
            // ---- leaf: Tree._single_step, nuts.py:105-132 ----
            double dE = E - E0;
            if (isnan(dE)) dE = INFINITY;
            bool div_leaf = false;
            if (go) {
                if (fabs(dE) > fabs(maxdE)) maxdE = dE;
                n_prop += 1;
                div_leaf = !(fabs(dE) < cfg.max_change);
                if (half == 1) ileaf += 1;
            }
            const WT wl = wt_from_dE(div_leaf ? 0. : dE);
            const bool okl = go && !div_leaf;
            if (okl) {
                acc_sum += wt_min1(wl);
                const int nslot = __ffs(freemask) - 1;
                freemask &= ~(1u << nslot);
                double *slot = gpr + (size_t)nslot * 2 * SLOT;
                VST(slot, q) VST(slot + SLOT, g)
                // the leaf becomes R; the first leaf of a pair waits at scalar level 0 for the level-0 merge, and its p
                // (left end and p_sum of R) is the left tree of that merge
                if (half == 1) {
                    ssc[0] = RW.m; ssc[10 * 8] = (double)RW.k; ssc[20 * 8] = REp; ssc[30 * 8] = Rlpp; ssc[40 * 8] = (double)Rslot;
                    did2 = true;
                } else {
                    VST(sR, p) VST(sR + 2 * SLOT, p)
                }
                VST(sR + SLOT, p)
                RW = wl; REp = E; Rlpp = lp; Rslot = nslot;
            }
            if (div_leaf) { diverging = 1; div_now = true; }
        }
        TICK(3)
        // section: merge
        // ================= merges: Tree._build_subtree nuts.py:134-178 and Tree.extend nuts.py:45-103 =================
        // Every live chain works through a queue, one merge per pass: the level-0 merge of a leaf pair, then the merges at
        // levels 1, 2, ... while (ileaf >> lvl) & 1 and no U-turn, then Tree.extend if the doubling ended.  A merge combines a
        // pending tree T with the current subtree R: T is a stack level (multinomial choice of the proposal, nuts.py:164-167)
        // or, for the extend, the whole tree (biased progressive choice, nuts.py:81-83).  The U-turn test runs on the two
        // trees in their order along the trajectory, X then Y, each given by the addresses of its left-end p, right-end p and
        // p_sum; a single leaf has all three at one address.
        int lvl = 0;
        int mq = live ? (did2 ? 0 : 1) : 3;      // next: 0 subtree merge at lvl, 1 decide on the extend, 2 extend, 3 none
        bool fin = false;
        const bool right = step > 0.;
#pragma unroll 1
        for (;;) {
            if (mq == 1) {
                fin = div_now || turn || (ileaf + 1 == (1 << depth));
                mq = (fin && !div_now && !turn) ? 2 : 3;
            }
            const bool go = mq == 0 || mq == 2, ext = mq == 2;
            if (!__any_sync(BFB_FULL, go)) break;
            DBG_COUNT(dbg_merges)
            // X, Y = stack level and R (level 0: the two leaves); extend: the whole tree and R, or R reversed and the whole tree
            const bool leaf0 = !ext && lvl == 0, extl = ext && !right;
            const double *tp = stack_ptr(go && !ext ? lvl : 0);
            const double *xl = ext ? (right ? sTL + SLOT : sR + SLOT) : tp;
            const double *xr = ext ? (right ? sPB : sR) : leaf0 ? tp : tp + SLOT;
            const double *xs = ext ? (right ? sPS : sR + 2 * SLOT) : leaf0 ? tp : tp + 2 * SLOT;
            const double *yl = extl ? sPB : leaf0 ? sR + SLOT : sR;
            const double *yr = extl ? sTR + SLOT : sR + SLOT;
            const double *ys = extl ? sPS : leaf0 ? sR + SLOT : sR + 2 * SLOT;
            double v0 = 0., v1 = 0., v2 = 0., v3 = 0., v4 = 0., v5 = 0.;
            double ps[NR], pl[NR];
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const int o = r * 32 + lane;
                const double xpl = xl[o], xpr = xr[o], xps = xs[o], ypl = yl[o], ypr = yr[o], yps = ys[o];
                ps[r] = xps + yps;
                pl[r] = xpl;
                // nuts.py:86-98: Tree.extend updates self.p_sum in place BEFORE p_sum1 / p_sum2 are formed, so the whole
                // tree's p_sum entering them is already the total (see the oracle, bf_oracle.c tree_extend)
                const double xq = (ext && right) ? ps[r] : xps, yq = (ext && !right) ? ps[r] : yps;
                const double vxl = var[r] * xpl, vyr = var[r] * ypr;
                const double ps1 = xq + ypl, ps2 = xpr + yq;
                v0 = fma(ps[r], vxl, v0); v1 = fma(ps[r], vyr, v1);
                v2 = fma(ps1, vxl, v2); v3 = fma(ps1, var[r] * ypl, v3);
                v4 = fma(ps2, var[r] * xpr, v4); v5 = fma(ps2, vyr, v5);
            }
            const bool turning = quad_any_nonpos6(v0, v1, v2, v3, v4, v5, lane);
            const double um = uni(t);
            if (go) {
                t += 1;
                WT TW; double TE, Tlp; int Tslot;
                if (ext) { TW = Wtree; TE = prop_E; Tlp = prop_lp; Tslot = prop_slot; }
                else {
                    TW.m = ssc[lvl * 8]; TW.k = (int)ssc[(10 + lvl) * 8];
                    TE = ssc[(20 + lvl) * 8]; Tlp = ssc[(30 + lvl) * 8]; Tslot = (int)ssc[(40 + lvl) * 8];
                }
                const WT tot = wt_add(TW, RW);
                const bool rwin = wt_select(um, ext ? TW : tot, RW);          // R's proposal wins
                freemask |= 1u << (rwin ? Tslot : Rslot);
                const int wslot = rwin ? Rslot : Tslot;
                const double wE = rwin ? REp : TE, wlp = rwin ? Rlpp : Tlp;
                if (ext) { Wtree = tot; prop_slot = wslot; prop_E = wE; prop_lp = wlp; }
                else { RW = tot; Rslot = wslot; REp = wE; Rlpp = wlp; }
                double *dps = ext ? sPS : sR + 2 * SLOT;
                VST(dps, ps)
                VST(sR, pl)                               // R's new left end (after the extend R is dead)
                if (turning) turn = true;
                if (ext) mq = 3;
                else { lvl++; mq = (!turn && ((ileaf >> lvl) & 1)) ? 0 : 1; }
            }
        }
        TICK(4)
        // section: push
        // ---- push R onto the stack at level lvl ----
        const bool push = live && !fin;
        if (__any_sync(BFB_FULL, push)) {
            double *sp = stack_ptr(push ? lvl : 1);
            if (push) {
                double a[NR], b[NR];
                VLD(a, sR) VLD(b, sR + 2 * SLOT)
                VST(sp, a) VST(sp + SLOT, p) VST(sp + 2 * SLOT, b)
                ssc[lvl * 8] = RW.m; ssc[(10 + lvl) * 8] = (double)RW.k; ssc[(20 + lvl) * 8] = REp; ssc[(30 + lvl) * 8] = Rlpp;
                ssc[(40 + lvl) * 8] = (double)Rslot;
                ileaf += 1;
            }
        }
        TICK(5)
        // section: extend
        // ================= end of a doubling: the rest of Tree.extend, nuts.py:45-103 =================
        if (fin) {
            double *dst = right ? sTR : sTL;
            VST(dst, q) VST(dst + SLOT, p) VST(dst + 2 * SLOT, g)
            depth += 1;
            const bool iter_end = div_now || turn || (depth >= cfg.max_treedepth);
            bnd = iter_end;
            ns_dbl = !iter_end;
        }
        TICK(6)
    }

    // section: persist
    // ---- persist chain state ----
    // the unit's group and chunk are recomputed rather than kept live across the loop (the register file is full)
    const int group_e = (int)((gpr - gprop) / (BFB_NSLOT * 2 * SLOT)), chunk_e = (it_hi - 1) / chunk_iters;
    if (gi < cpg && (int64_t)group_e * cpg + gi < st.C && st.status[c] == 0) {
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int j = 4 * r + lg;
            st.q[vb + j] = q[r]; st.g[vb + j] = g[r]; st.var[vb + j] = var[r];
        }
        if (lg == 0) {
            st.logp[c] = logp_q; st.t_draw[c] = t; st.iter[c] = it0 + it;
            st.status[c] = status;
            if (tree_total) atomicAdd(st.tree_total, (unsigned long long)tree_total);
        }
    }
    __threadfence();
    __syncwarp();
    if (lane == 0) {
#ifdef BFB_DMMA_TIMING
        atomicAdd(st.tree_total + 1, (unsigned long long)dbg_rounds);
        atomicAdd(st.tree_total + 2, (unsigned long long)dbg_merges);
        atomicAdd(st.tree_total + 3, (unsigned long long)dbg_iend);
        long long tsum = 0;
        for (int k_ = 0; k_ < 7; ++k_) { atomicAdd(st.tree_total + 4 + k_, (unsigned long long)tacc[k_]); tsum += tacc[k_]; }
        for (int k_ = 8; k_ < 12; ++k_) { atomicAdd(st.tree_total + 8 + k_, (unsigned long long)tacc[k_]); tsum += tacc[k_]; }
        atomicAdd(st.tree_total + 11, (unsigned long long)(clock64() - t_unit0 - tsum));
#endif
        qv[2 + group_e] = chunk_e + 1;
        if ((chunk_e + 1) * chunk_iters < out.n_iter) {
            const int ti = atomicAdd(queue + 1, 1);
            __threadfence();
            ring[ti] = group_e;
        }
    }
    }   // unit loop
#undef VLD
#undef VST
}

// ----------------------------------------------------------------------------------------------------------------------
// HMC (samplers/hmc.py:16-49): every chain makes n_int_step leapfrogs per iteration, so the 8 chains of a warp ARE in lock
// step and nothing of the tree machinery is needed: an iteration is momentum draw, n_int_step x (kick, drift, tensor-core
// evaluation, kick), Metropolis test, adaptation, outputs.  Same work units and queue as the NUTS kernel.
// ----------------------------------------------------------------------------------------------------------------------
template <int NR, int MV, int W>
__global__ void __launch_bounds__(32 * W, 1) hmc_dmma_kernel(DevModel M, bfb_sampler_cfg cfg, ChainState st, RunOutDevF out,
                                                             int base_iter, int chunk_iters, int n_groups, int n_units,
                                                             int *__restrict__ queue)
{
    using SH = DmmaShape<NR, MV>;
    extern __shared__ double smem[];
    double *bsm = smem;
    double *msm = smem + SH::frag_doubles(W);    // per-dimension tables (dmma_stage_tables)
    if (!SH::LIK) { for (int i = threadIdx.x; i < SH::FRAG_DOUBLES; i += blockDim.x) bsm[i] = M.bfrag[i]; }
    dmma_stage_tables<MV>(M, msm);
    __syncthreads();
    const int lane = threadIdx.x & 31, gi = lane >> 2, lg = lane & 3;
    const int n = M.n;
    const DmmaConsts K = dmma_consts(M);
    volatile int *qv = queue;
    volatile int *ring = queue + 2 + n_groups;
#pragma unroll 1
    for (;;) {
    int idx = 0, group = 0;
    if (lane == 0) {
        idx = atomicAdd(queue, 1);
        if (idx < n_units) { while ((group = ring[idx]) < 0) __nanosleep(100); }
    }
    idx = __shfl_sync(BFB_FULL, idx, 0);
    if (idx >= n_units) break;
    group = __shfl_sync(BFB_FULL, group, 0);
    __threadfence();
    const int chunk = qv[2 + group];
    const int it_lo = chunk * chunk_iters;
    const int it_hi = min(out.n_iter, it_lo + chunk_iters);
    const int64_t c_raw = (int64_t)group * 8 + gi;
    const bool exists = c_raw < st.C;
    const int64_t c = exists ? c_raw : st.C - 1;
    const size_t vb = (size_t)c * M.np;
    double q[NR], p[NR], g[NR], var[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int j = 4 * r + lg;
        q[r] = st.q[vb + j]; g[r] = st.g[vb + j]; var[r] = st.var[vb + j]; p[r] = 0.;
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
        if (!__any_sync(BFB_FULL, status == 0)) break;
        const bool warm = (it0 + it) < cfg.n_warmup;
        // momentum: metrics.py:83-86 (each quad draws the n normals of its chain, lane lg the dimensions 4 r + lg)
        double qs[NR], gs[NR], part = 0.;
#pragma unroll 1
        for (int r = 0; r < NR; ++r) {
            // rolled: one call site; the register arrays are indexed through the unrolled select below
            const int j = 4 * r + lg;
            const double z = (j < n) ? draw_normal_ni(seed, chain_id, (uint64_t)(t + j)) : 0.;
#pragma unroll
            for (int rr = 0; rr < NR; ++rr) if (rr == r) p[rr] = z;
        }
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            p[r] = (4 * r + lg < n) ? p[r] / sqrt(var[r]) : 0.;
            part = fma(p[r], var[r] * p[r], part);
            qs[r] = q[r]; gs[r] = g[r];
        }
        const double ke0 = qsum(part);
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
            for (int r = 0; r < NR; ++r) {
                p[r] = fma(dt, g[r], p[r]);
                q[r] = fma(eps, var[r] * p[r], q[r]);
            }
            double gn[NR], ke2;
            dmma_logp_grad<NR, MV>(bsm, lane, K, q, msm, live, lp, gn,
                                   [&](const double (&gg)[NR]) {
                                       double a_ = 0.;
#pragma unroll
                                       for (int r = 0; r < NR; ++r) { const double pn = fma(dt, gg[r], p[r]); a_ = fma(pn, var[r] * pn, a_); }
                                       return a_;
                                   }, ke2);
#pragma unroll
            for (int r = 0; r < NR; ++r) { g[r] = gn[r]; p[r] = fma(dt, gn[r], p[r]); }
            E = 0.5 * ke2 - lp;
        }
        // HMC._hamiltonian_step, hmc.py:31-49
        double dE;
        int diverging = 0;
        if (isfinite(E)) { dE = E0 - E; diverging = fabs(dE) > cfg.max_change; }
        else { dE = -INFINITY; diverging = 1; }
        double accept_stat;
        { const double e_ = exp(dE); accept_stat = e_ < 1. ? e_ : 1.; }
        const double ua = draw_uniform_ni(seed, chain_id, (uint64_t)t);
        bool accepted = false;
        if (live && !diverging) { t += 1; accepted = !(ua >= accept_stat); }
        const double s_logp = lp, s_energy = E;
        if (accepted) logp_q = lp;
        else {
#pragma unroll
            for (int r = 0; r < NR; ++r) { q[r] = qs[r]; g[r] = gs[r]; }
        }
        if (live) {
            tree_total += (unsigned long long)cfg.n_int_step;
            if (warm && cfg.adapt_step_size) {          // step_size.py:31-45
                const double cnt = (double)count;
                const double w = 1. / (cnt + cfg.t0);
                hbar = ((1. - w) * hbar + w * (cfg.target_accept - accept_stat));
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
                for (int r = 0; r < NR; ++r) {
                    const int j = 4 * r + lg;
                    if (j < n) {
                        double fgm = st.fg_mean[vb + j], fgr = st.fg_raw[vb + j], bgm = st.bg_mean[vb + j], bgr = st.bg_raw[vb + j];
                        double od = q[r] - fgm;
                        fgm += od / fg_n;
                        fgr += 1. * od * (q[r] - fgm);
                        od = q[r] - bgm;
                        bgm += od / bg_n;
                        bgr += 1. * od * (q[r] - bgm);
                        if (upd) var[r] = fgr / fg_n;
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
                for (int r = 0; r < NR; ++r) if (4 * r + lg < n) out.o.samples[o * n + 4 * r + lg] = q[r];
            }
            if (lg == 0) {
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
        for (int r = 0; r < NR; ++r) {
            const int j = 4 * r + lg;
            st.q[vb + j] = q[r]; st.g[vb + j] = g[r]; st.var[vb + j] = var[r];
        }
        if (lg == 0) {
            st.logp[c] = logp_q; st.fg_n[c] = fg_n; st.bg_n[c] = bg_n;
            st.log_step[c] = log_step; st.log_bar[c] = log_bar; st.hbar[c] = hbar;
            st.count[c] = count; st.n_samples[c] = n_samples; st.previous_update[c] = previous_update;
            st.adapt_window[c] = adapt_window; st.t_draw[c] = t; st.iter[c] = it0 + it_hi;
            st.status[c] = status;
            if (tree_total) atomicAdd(st.tree_total, tree_total);
        }
    }
    __threadfence();
    __syncwarp();
    if (lane == 0) {
        qv[2 + group] = chunk + 1;
        if ((chunk + 1) * chunk_iters < out.n_iter) {
            const int ti = atomicAdd(queue + 1, 1);
            __threadfence();
            ring[ti] = group;
        }
    }
    }   // unit loop
}

template <int NR, int MV, int W>
static int launch_hmc_dmma(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    using SH = DmmaShape<NR, MV>;
    const int64_t C = h->cs.C;
    const int n_groups = (int)((C + 7) / 8);
    const size_t smem = sizeof(double) * (SH::frag_doubles(W) + SH::MSM_DOUBLES + (SH::C3 ? dmma_c3_doubles(NR, h->dm.c3_kt, W) : 0));
    if (smem > (size_t)(227 * 1024)) return 1;
    BFB_CUDA(cudaFuncSetAttribute(hmc_dmma_kernel<NR, MV, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    RunOutDevF od;
    od.o = o; od.n_iter = n_iter;
    int chunk_iters, n_units, rc;
    if ((rc = queue_setup(h, n_groups, n_iter, 6, 0, 0, chunk_iters, n_units))) return rc;
    int blocks = h->sm_count;
    const int64_t want = (n_groups + W - 1) / W;
    if ((int64_t)blocks > want) blocks = (int)want;
    hmc_dmma_kernel<NR, MV, W><<<blocks, 32 * W, smem, h->stream>>>(h->dm, h->scfg, h->cs, od, (int)h->iters_done, chunk_iters,
                                                                   n_groups, n_units, h->queue);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

template <int NR, int MV>
static int launch_hmc_dmma_w(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    // warps per SM: the kernel needs no per-warp shared memory, so the register file is the only limit (255 registers up
    // to 8 warps, 168 at 12, 128 at 16: ptxas spills a few hundred bytes per thread, which the extra warps more than hide)
    const int64_t groups = (h->cs.C + 7) / 8, sms = h->sm_count;
    // measured (d=26 cubic-2, n_int_step=32): 16384 chains 52.5 % of the FP64 peak with 8 warps, 51.6 % with 12; 32768 chains
    // 56.0 / 57.9 / 57.9 % with 8 / 12 / 16
    int W = groups > sms * 16 ? 12 : groups > sms * 4 ? 8 : 4;
    if (const char *e = getenv("BFB200_HMC_WARPS_PER_SM")) { int v = atoi(e); if (v == 4 || v == 8 || v == 12 || v == 16) W = v; }
    if (DmmaShape<NR, MV>::LIK && W > 12) W = 12;        // 2 staged operand records per warp (15 KB): at most 12 warps per block
    if (DmmaShape<NR, MV>::FEAT) W = 4;                  // feature form: 28 KB of staged records, point and second-GEMM scratch per warp
    else if (const char *e2 = getenv("BFB200_WARPS_PER_SM")) { int v = atoi(e2); if (v == 4 || v == 8) W = v; }
    switch (W) {
    case 16: return launch_hmc_dmma<NR, MV, 16>(h, o, n_iter);
    case 12: return launch_hmc_dmma<NR, MV, 12>(h, o, n_iter);
    case 8: return launch_hmc_dmma<NR, MV, 8>(h, o, n_iter);
    }
    return launch_hmc_dmma<NR, MV, 4>(h, o, n_iter);
}

// The headline instantiation (d = 26 cubic-2: NR = 7, MV = 1) is compiled into a translation unit of its own
// (-DBFB_DMMA_PART_HEADLINE, see the Makefile): a small CUDA module loads in a few ms, whereas the first launch out of the
// ~60-kernel module of all instantiations paid 25-60 ms of lazy module loading (measured: 161-197 ms for the first
// 4096-chain run of a process against 137 ms for the following ones; scripts/variance.py).
int bfb_launch_hmc_dmma_headline(bfb_context *h, const bfb_run_out &o, int n_iter);
int bfb_launch_nuts_dmma_headline(bfb_context *h, const bfb_run_out &o, int n_iter);
#ifdef BFB_DMMA_PART_HEADLINE
int bfb_launch_hmc_dmma_headline(bfb_context *h, const bfb_run_out &o, int n_iter) { return launch_hmc_dmma_w<7, 1>(h, o, n_iter); }
#else
// launches the HMC kernel of the model (select_family, bfb_sampler.cu, chose this family): 0 on launch, 1 when its shared memory
// does not fit, < 0 on error
int bfb_launch_hmc_dmma(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    const DevModel &M = h->dm;
    if (M.epilogue && M.lik_ftab) {         // likelihood pipeline (model variant bit 3), feature form: two chained GEMMs per 8 outputs (bit 4)
        switch (M.lik_nr * 2 + (M.lik_ext ? 1 : 0)) {
        case 8: return launch_hmc_dmma_w<4, 24>(h, o, n_iter);
        case 14: return launch_hmc_dmma_w<7, 24>(h, o, n_iter);
        case 16: return launch_hmc_dmma_w<8, 24>(h, o, n_iter);
        case 9: return launch_hmc_dmma_w<4, 26>(h, o, n_iter);
        case 15: return launch_hmc_dmma_w<7, 26>(h, o, n_iter);
        case 17: return launch_hmc_dmma_w<8, 26>(h, o, n_iter);
        }
    } else if (M.epilogue) {                // likelihood pipeline: operand streamed from L2
        switch (M.lik_nr * 2 + (M.lik_ext ? 1 : 0)) {
        case 8: return launch_hmc_dmma_w<4, 8>(h, o, n_iter);
        case 14: return launch_hmc_dmma_w<7, 8>(h, o, n_iter);
        case 16: return launch_hmc_dmma_w<8, 8>(h, o, n_iter);
        case 9: return launch_hmc_dmma_w<4, 10>(h, o, n_iter);       // bound / rescale / transform / prior around the outputs
        case 15: return launch_hmc_dmma_w<7, 10>(h, o, n_iter);
        case 17: return launch_hmc_dmma_w<8, 10>(h, o, n_iter);
        }
    } else {
        const int mv = (M.has_c2 ? 1 : 0) | (M.frag_ext ? 2 : 0) | (M.has_c3 ? 4 : 0);
#ifdef BFB_NO_HEADLINE_SPLIT     // experiment: the headline instantiation inside the big module
        if (M.frag_nr == 7 && mv == 1) return launch_hmc_dmma_w<7, 1>(h, o, n_iter);
#else
        if (M.frag_nr == 7 && mv == 1) return bfb_launch_hmc_dmma_headline(h, o, n_iter);
#endif
#define BFB_CASE(NR_, MV_) if (M.frag_nr == NR_ && mv == MV_) return launch_hmc_dmma_w<NR_, MV_>(h, o, n_iter);
        BFB_CASE(4, 0) BFB_CASE(4, 1) BFB_CASE(4, 2) BFB_CASE(4, 3) BFB_CASE(7, 0) BFB_CASE(7, 2) BFB_CASE(7, 3)
        BFB_CASE(8, 0) BFB_CASE(8, 1) BFB_CASE(8, 2) BFB_CASE(8, 3)
        BFB_CASE(4, 5) BFB_CASE(4, 7) BFB_CASE(7, 5) BFB_CASE(7, 7)          // with cubic-3 configs (n <= 28)
#undef BFB_CASE
    }
    bfb_set_error("bfb_launch_hmc_dmma: no kernel instantiation for this model");
    return BFB_ERR_ARG;
}
#endif

template <int NR, int MV, int W>
static int launch_dmma(bfb_context *h, const bfb_run_out &o, int n_iter, int cpg)
{
    using SH = DmmaShape<NR, MV>;
    constexpr int SLOT = NR * 32;
    const int L = h->scfg.max_treedepth;
    const int64_t C = h->cs.C;
    const int n_groups = (int)((C + cpg - 1) / cpg);
    // one persistent block of W warps per SM (W = 4: one warp per scheduler, 4096 chains = 512 warps on 592 schedulers;
    // W = 8 when there are more groups than that); level 0 of the tree stack (the current subtree) and the next LS levels
    // live in shared memory, deeper (rarely touched) levels in an L2-resident buffer.  LS = 0 needs as much shared memory
    // as one stack level did when level 0 stayed in registers, so the same models fit.
    const size_t fixed = sizeof(double) * (SH::frag_doubles(W) + SH::MSM_DOUBLES + (SH::C3 ? dmma_c3_doubles(NR, h->dm.c3_kt, W) : 0));
    if (fixed + sizeof(double) * W * warp_smem_doubles(NR, 0) > (size_t)(227 * 1024)) return 1;      // does not fit: generic kernel
    const size_t budget = (size_t)(227 * 1024) - 1024 - fixed;
    int LS = L;
    while (LS > 0 && sizeof(double) * W * warp_smem_doubles(NR, LS) > budget) --LS;
    if (const char *e = getenv("BFB200_STACK_LEVELS_SMEM")) { int v = atoi(e); if (v >= 0 && v <= L) LS = v; }
    const size_t smem = fixed + sizeof(double) * W * warp_smem_doubles(NR, LS);
    BFB_REQUIRE(smem <= 227 * 1024, BFB_ERR_ARG, "sampler needs %zu bytes of shared memory per block (> 227 KB)", smem);
    BFB_CUDA(cudaFuncSetAttribute(nuts_dmma_kernel<NR, MV, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    double *gprop;
    int rc;
    if ((rc = gstack_reserve(h, n_groups, L, LS, SLOT, BFB_NSLOT, &gprop))) return rc;
    RunOutDevF od;
    od.o = o; od.n_iter = n_iter;
    // progress reports for host outputs: chunks of rep_iters iterations counted per CHAIN at its iteration boundary (the work units keep
    // their length: a unit end synchronises the 8 chains of a group, which costs ~3 % of the kernel at 48 units per group)
    const bool report = h->progress_arm > 0;
    int rep_iters = 0, n_rep = 0;
    if (report) {
        rep_iters = (n_iter + h->progress_arm - 1) / h->progress_arm;
        if (rep_iters < 4) rep_iters = n_iter < 4 ? n_iter : 4;
        n_rep = (n_iter + rep_iters - 1) / rep_iters;
    }
    // one block per SM whenever there are at least as many groups as SMs: with 512 groups (4096 chains) every SM then runs 3 or
    // 4 warps instead of 128 SMs running 4 and 20 none
    int blocks = h->sm_count;
    if ((int64_t)blocks > n_groups) blocks = n_groups;
    // iteration chunks = work units per group.  A group is bound to ONE warp at a time, but after every chunk it goes back to the queue
    // and the next free warp takes it: groups migrate between SMs that host 4 busy warps and SMs that host 3 (512 groups on 592 warp
    // slots), which evens out the finish times.  Measured at 4096 chains x 1500 iterations: 1 / 2 / 6 / 12 / 24 / 48 chunks =
    // 161 / 154 / 141 / 134.7 / 135.2 / 138.5 ms
    // work queue, then the progress block (see the iteration boundary of the kernel): 4 + n_rep ints
    int chunk_iters, n_units;
    if ((rc = queue_setup(h, n_groups, n_iter, 12, blocks * W, 4 + (size_t)n_rep, chunk_iters, n_units))) return rc;
    {
        int *pg = h->queue + 2 + (size_t)n_groups + (size_t)n_units;
        BFB_CUDA(cudaMemsetAsync(pg, 0, sizeof(int) * (4 + (size_t)n_rep), h->stream));
        if (report) {
            const unsigned long long fa = (unsigned long long)h->progress_host_dev;
            const int hdr[4] = {1, (int)(unsigned)(fa & 0xffffffffull), (int)(unsigned)(fa >> 32), rep_iters};
            BFB_CUDA(cudaMemcpyAsync(pg, hdr, sizeof(hdr), cudaMemcpyHostToDevice, h->stream));
            h->progress_chunk_iters = rep_iters; h->progress_n_chunks = n_rep;
        }
    }
    nuts_dmma_kernel<NR, MV, W><<<blocks, 32 * W, smem, h->stream>>>(h->dm, h->scfg, h->cs, od, L, LS, h->gstack, gprop,
                                                                    (int)h->iters_done, chunk_iters, n_groups, n_units, h->queue, cpg);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

template <int NR, int MV>
static int launch_dmma_w(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    // chains per group (MMA rows in use) and warps per SM.  Measured at 4096 chains (scripts/imbalance.py, full run): 8 per
    // group 184 ms, 7 (586 warps on the 592 schedulers) 187 ms, 6 212 ms, 4 with two warps per scheduler 214 ms -- the cost of
    // a round is per warp, not per live chain, so full MMAs win; BFB200_CHAINS_PER_GROUP overrides for experiments.
    const int64_t C = h->cs.C, slots4 = (int64_t)h->sm_count * 4;
    int cpg = 8;
    if (const char *e = getenv("BFB200_CHAINS_PER_GROUP")) { int v = atoi(e); if (v >= 1 && v <= 8) cpg = v; }
    int W = ((C + cpg - 1) / cpg > slots4) ? 8 : 4;
    if (const char *e = getenv("BFB200_WARPS_PER_SM")) { int v = atoi(e); if (v == 4 || v == 8) W = v; }
    if (DmmaShape<NR, MV>::LIK) W = 4;        // staged operand records + tree state of 8 warps do not fit; the persistent warps queue up
    return W == 8 ? launch_dmma<NR, MV, 8>(h, o, n_iter, cpg) : launch_dmma<NR, MV, 4>(h, o, n_iter, cpg);
}

#ifdef BFB_DMMA_PART_HEADLINE
int bfb_launch_nuts_dmma_headline(bfb_context *h, const bfb_run_out &o, int n_iter) { return launch_dmma_w<7, 1>(h, o, n_iter); }
#else
// launches the NUTS kernel of the model (select_family, bfb_sampler.cu, chose this family): 0 on launch, 1 when its shared memory
// does not fit, < 0 on error
int bfb_launch_nuts_dmma(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    const DevModel &M = h->dm;
    if (M.epilogue && M.lik_ftab) {         // likelihood pipeline (model variant bit 3), feature form: two chained GEMMs per 8 outputs (bit 4)
        switch (M.lik_nr * 2 + (M.lik_ext ? 1 : 0)) {
        case 8: return launch_dmma_w<4, 24>(h, o, n_iter);
        case 14: return launch_dmma_w<7, 24>(h, o, n_iter);
        case 16: return launch_dmma_w<8, 24>(h, o, n_iter);
        case 9: return launch_dmma_w<4, 26>(h, o, n_iter);
        case 15: return launch_dmma_w<7, 26>(h, o, n_iter);
        case 17: return launch_dmma_w<8, 26>(h, o, n_iter);
        }
    } else if (M.epilogue) {                // likelihood pipeline: operand streamed from L2
        switch (M.lik_nr * 2 + (M.lik_ext ? 1 : 0)) {
        case 8: return launch_dmma_w<4, 8>(h, o, n_iter);
        case 14: return launch_dmma_w<7, 8>(h, o, n_iter);
        case 16: return launch_dmma_w<8, 8>(h, o, n_iter);
        case 9: return launch_dmma_w<4, 10>(h, o, n_iter);           // bound / rescale / transform / prior around the outputs
        case 15: return launch_dmma_w<7, 10>(h, o, n_iter);
        case 17: return launch_dmma_w<8, 10>(h, o, n_iter);
        }
    } else {
        const int mv = (M.has_c2 ? 1 : 0) | (M.frag_ext ? 2 : 0) | (M.has_c3 ? 4 : 0);
#ifdef BFB_NO_HEADLINE_SPLIT
        if (M.frag_nr == 7 && mv == 1) return launch_dmma_w<7, 1>(h, o, n_iter);
#else
        if (M.frag_nr == 7 && mv == 1) return bfb_launch_nuts_dmma_headline(h, o, n_iter);
#endif
#define BFB_CASE(NR_, MV_) if (M.frag_nr == NR_ && mv == MV_) return launch_dmma_w<NR_, MV_>(h, o, n_iter);
        BFB_CASE(4, 0) BFB_CASE(4, 1) BFB_CASE(4, 2) BFB_CASE(4, 3) BFB_CASE(7, 0) BFB_CASE(7, 2) BFB_CASE(7, 3)
        BFB_CASE(8, 0) BFB_CASE(8, 1) BFB_CASE(8, 2) BFB_CASE(8, 3)
        BFB_CASE(4, 5) BFB_CASE(4, 7) BFB_CASE(7, 5) BFB_CASE(7, 7)          // with cubic-3 configs (n <= 28)
#undef BFB_CASE
    }
    bfb_set_error("bfb_launch_nuts_dmma: no kernel instantiation for this model");
    return BFB_ERR_ARG;
}
#endif

#ifndef BFB_DMMA_PART_HEADLINE
__global__ void norminv_fill_kernel(const double *p, int64_t count, double *z, double *z_ref)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    z[i] = bfb_norminv_small(p[i]);
    z_ref[i] = bfb_norminv(p[i]);
}

extern "C" int bfb_norminv_fill(bfb_handle h, const double *p, int64_t count, double *z, double *z_ref)
{
    BFB_REQUIRE(h && p && z && z_ref && count >= 0, BFB_ERR_ARG, "bfb_norminv_fill: bad arguments");
    if (count == 0) return BFB_OK;
    BFB_CUDA(cudaSetDevice(h->device));
    double *dp;
    BFB_CUDA(cudaMalloc(&dp, sizeof(double) * 3 * count));
    BFB_CUDA(cudaMemcpyAsync(dp, p, sizeof(double) * count, cudaMemcpyHostToDevice, h->stream));
    norminv_fill_kernel<<<(unsigned)((count + 255) / 256), 256, 0, h->stream>>>(dp, count, dp + count, dp + 2 * count);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    BFB_CUDA(cudaMemcpyAsync(z, dp + count, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaMemcpyAsync(z_ref, dp + 2 * count, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
    BFB_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(dp);
    return BFB_OK;
}
#endif
