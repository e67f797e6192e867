// bfb_sampler_pair.cu -- NUTS on the FP64 tensor cores with the work of an 8-chain group split by ROLE over a warp pair.
//
// The one-warp kernel (bfb_sampler_dmma.cu) spends ~8 k cycles of a ~20 k-cycle round (two leapfrogs of 8 chains) in the two
// tensor-core evaluations and ~12 k in the NUTS bookkeeping around them, everything latency bound because 4096 chains are one
// warp per scheduler.  Here the two parts run CONCURRENTLY on the same scheduler:
//   * the INTEGRATOR warp (E) owns position, momentum and gradient of the 8 chains and does nothing but kick / drift /
//     two-stage DMMA evaluation (bfb_dmma.cuh), two leaves per round, and publishes every leaf (momentum, logp, energy to a
//     shared-memory ring; position and gradient to a proposal slot in the L2-resident pool);
//   * the TREE warp (T) consumes the leaves one round behind: multinomial weights, U-turn tests, sub-tree merges
//     (nuts.py:134-178), Tree.extend (nuts.py:45-103), the iteration boundary (base_hmc.py:62-85: outputs, dual averaging,
//     windowed Welford metric, momentum draw) -- the state machine of the one-warp kernel minus the evaluations.
// A trajectory never depends on the tree's decisions except for WHEN it stops: the direction of every doubling is a Philox
// draw whose counter is known at the start of the iteration (a doubling of 2^j leaves that continues consumes exactly
// 2^j + 1 draws), so E integrates ahead speculatively -- saving and re-loading the two ends of the trajectory itself -- until
// T tells the chain to restart from a new point (per-chain mailbox: accepted position / gradient, fresh momentum, metric, step,
// draw counter, epoch number).  A leaf carries the epoch it belongs to; T ignores leaves of a finished iteration.  Cost of the
// speculation: one wasted round per chain and iteration.  Synchronisation: shared-memory mbarriers (E -> T "round r
// published", T -> E "round r consumed", T -> E "unit set up"); E runs at most one round ahead of the round T works on.
// Same algorithm, same draw order (SURVEY.md 8a N-RNG), same results as nuts_dmma_kernel: every NUTS test runs on both.
//
// Reference restated here: samplers/hmc_utils/base_hmc.py:62-85, samplers/nuts.py:27-217, hmc_utils/integration.py:28-95,
// hmc_utils/metrics.py:73-91,186-211,333-371, hmc_utils/step_size.py:10-51.
#include "bfb_dmma.cuh"
#include "bfb_nuts_common.cuh"
#include "bfb_nuts_dmma_common.cuh"
#include <cstring>
#include <cstdlib>

#define BFB_STR_(x) #x
#define BFB_STR(x) BFB_STR_(x)
#define BFB_PAIR_NSLOT 16      // proposal slots per chain: the 12 of the one-warp kernel + two rounds of leaves in flight

__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *b, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(b)), "r"(count) : "memory");
}
// release (cta scope): everything this thread -- and, after a __syncwarp, its warp -- wrote before is visible to whoever
// observes the completed phase
__device__ __forceinline__ void mbar_arrive(uint64_t *b)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_addr(b)) : "memory");
}
// acquire: returns once the phase with this parity has completed (the hardware suspends the thread between polls)
__device__ __forceinline__ void mbar_wait(uint64_t *b, unsigned parity)
{
    asm volatile("{\n"
                 ".reg .pred p_;\n"
                 "W_LOOP:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p_, [%0], %1;\n"
                 "@p_ bra W_DONE;\n"
#ifdef BFB_PAIR_SLEEP
                 "nanosleep.u32 " BFB_STR(BFB_PAIR_SLEEP) ";\n"
#endif
                 "bra W_LOOP;\n"
                 "W_DONE:\n"
                 "}" :: "r"(smem_addr(b)), "r"(parity) : "memory");
}

// shared memory of a pair, in doubles (SLOT = NR * 32, element (r, lane) of a vector at r * 32 + lane):
//   E: TL q,p,g | TR q,p,g                                                    6 slots
//   ring: momentum of the leaves [round parity][half]                         4 slots
//   mailbox T -> E: momentum, position, gradient, metric of a restart         4 slots
//   T: PS | PB | TL p | TR p | stack levels (pl, pr, psum) x LS               4 + 3 LS slots
//   T: per-level scalars [5][10][8]                                           400
//   small: leaf scalars, mailbox scalars, slot mail, unit info, mbarriers     144
__host__ __device__ inline int pair_smem_doubles(int NR, int LS) { return (18 + 3 * LS) * NR * 32 + 400 + 144; }

template <int NR, int MV, int NP>
__global__ void __launch_bounds__(64 * NP, 1) nuts_pair_kernel(DevModel M, bfb_sampler_cfg cfg, ChainState st, RunOutDevF out,
                                                               int L, int LS, double *__restrict__ gstack,
                                                               double *__restrict__ gprop, int base_iter, int chunk_iters,
                                                               int n_groups, int n_units, int *__restrict__ queue)
{
    using SH = DmmaShape<NR, MV>;
    constexpr int SLOT = NR * 32;
    extern __shared__ double smem[];
    double *bsm = smem;                          // coefficient operand table
    double *msm = smem + SH::frag_doubles(NP);   // per-dimension tables (dmma_stage_tables)
    if (!SH::LIK) { for (int i = threadIdx.x; i < SH::FRAG_DOUBLES; i += blockDim.x) bsm[i] = M.bfrag[i]; }
    dmma_stage_tables<MV>(M, msm);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, gi = lane >> 2, lg = lane & 3;
    const bool role_T = wib >= NP;
    const int pi = role_T ? wib - NP : wib;
    const int c3x = SH::C3 ? dmma_c3_doubles(NR, M.c3_kt, NP) : 0;
    double *psm = smem + SH::frag_doubles(NP) + SH::MSM_DOUBLES + c3x + (size_t)pi * pair_smem_doubles(NR, LS);
    double *eTL = psm, *eTR = psm + 3 * SLOT, *ringP = psm + 6 * SLOT;
    double *mP0 = psm + 10 * SLOT, *mQ = psm + 11 * SLOT, *mG = psm + 12 * SLOT, *mVAR = psm + 13 * SLOT;
    double *sPS = psm + 14 * SLOT, *sPB = psm + 15 * SLOT, *sTLp = psm + 16 * SLOT, *sTRp = psm + 17 * SLOT, *sST = psm + 18 * SLOT;
    double *ssc = psm + (18 + 3 * LS) * SLOT + gi;       // scalar (field f, level l) of this chain at ssc[(f * 10 + l) * 8]
    double *sml = psm + (18 + 3 * LS) * SLOT + 400;
    double *rec_lp = sml, *rec_E = sml + 32, *mb_step = sml + 64;
    long long *mb_tstart = reinterpret_cast<long long *>(sml + 72);
    int *ints = reinterpret_cast<int *>(sml + 80);
    int *rec_tag = ints, *slotmail = ints + 32;
    int *mail_ep = ints + 64;                 // [round parity][chain]: epoch the chain is in (-1: finished), as of the hand-over of that round
    volatile int *unit_i = ints + 80;         // group | first round E must not compute (never reset: valid when > first round of the unit)
    uint64_t *bars = reinterpret_cast<uint64_t *>(sml + 128);
    uint64_t *bar_full = bars, *bar_done = bars + 2, *bar_unit = bars + 4;
    if (!role_T) {
        if (lane == 0) {
            mbar_init(bar_full, 1); mbar_init(bar_full + 1, 1); mbar_init(bar_done, 1); mbar_init(bar_done + 1, 1); mbar_init(bar_unit, 1);
            unit_i[0] = 0; unit_i[1] = 0;
        }
    }
    __syncthreads();
    const int n = M.n;
    const DmmaConsts K = dmma_consts(M);

#ifdef BFB_PAIR_TIMING     // per-section cycle counters (printed with BFB200_DEBUG=1)
#define TICK(k) { const long long now_ = clock64(); tacc[k] += now_ - tlast; tlast = now_; }
#define DBG_COUNT(v) ++v;
#else
#define TICK(k)
#define DBG_COUNT(v)
#endif
#define VLD(dst, base)  _Pragma("unroll") for (int r_ = 0; r_ < NR; ++r_) dst[r_] = (base)[r_ * 32 + lane];
#define VST(base, src)  _Pragma("unroll") for (int r_ = 0; r_ < NR; ++r_) (base)[r_ * 32 + lane] = src[r_];

    const uint64_t seed = cfg.seed;
    int r = 0;                                 // round counter of the pair (never reset: it indexes the mbarrier phases)
    unsigned unit_no = 0;

    if (!role_T) {
        // =============================================== integrator warp ===============================================
        double q[NR], p[NR], g[NR], var[NR];
#pragma unroll
        for (int k = 0; k < NR; ++k) { q[k] = p[k] = g[k] = 0.; var[k] = 1.; }
        int epoch_seen = 0;
        long long tacc[4] = {0, 0, 0, 0}, tlast = clock64(); (void)tacc; (void)tlast;
        unsigned dbg_rounds = 0; (void)dbg_rounds;
#pragma unroll 1
        for (;;) {
            mbar_wait(bar_unit, unit_no & 1);
            ++unit_no;
            const int group = unit_i[0];
            if (group < 0) break;
            const int r0 = r;
            const int64_t c_raw = (int64_t)group * 8 + gi;
            const int64_t c = c_raw < st.C ? c_raw : st.C - 1;
            const uint64_t chain_id = (uint64_t)(cfg.chain0 + c);
            double *gpr = gprop + (size_t)group * BFB_PAIR_NSLOT * 2 * SLOT;
            bool liveE = false;
            int depthE = 0, ileafE = 0;
            unsigned dir4 = 0;
            double stepE = 0.;
            long long tstart = 0;
            TICK(0)
#pragma unroll 1
            for (;;) {
                if (r >= r0 + 2) mbar_wait(bar_done + (r & 1), (unsigned)((r - 2) >> 1) & 1u);
                {
                    const int stop_at = unit_i[1];
                    if (stop_at > r0 && r >= stop_at) break;
                }
                TICK(1)
                DBG_COUNT(dbg_rounds)
                // ---- mailbox: restart of a chain from the point T accepted ----
                bool restarted = false;
                const int rb = r & 1;
                {
                    const int ep = mail_ep[rb * 8 + gi];
                    restarted = ep >= 0 && ep != epoch_seen;
                    if (__any_sync(BFB_FULL, restarted)) {
                        if (restarted) {
                            VLD(q, mQ) VLD(p, mP0) VLD(g, mG) VLD(var, mVAR)
                            VST(eTL, q) VST(eTL + SLOT, p) VST(eTL + 2 * SLOT, g)
                            VST(eTR, q) VST(eTR + SLOT, p) VST(eTR + 2 * SLOT, g)
                            stepE = mb_step[gi]; tstart = mb_tstart[gi];
                            depthE = 0; ileafE = 0; liveE = true; epoch_seen = ep;
                        }
                    }
                    if (ep < 0) liveE = false;
                }
                // ---- start of a doubling: direction (nuts.py:210), the end of the trajectory it continues from ----
                const bool dstart = liveE && ileafE == 0;
                if (__any_sync(BFB_FULL, dstart)) {
                    const bool newdir = dstart && (depthE & 3) == 0;
                    if (__any_sync(BFB_FULL, newdir)) {
                        // lane lg of the quad draws the direction of doubling depth + lg: its counter is the counter at the start of
                        // the iteration plus the 2^j + 1 draws of every doubling j before it
                        const int dj = depthE + lg;
                        const long long td = tstart + ((1ll << dj) - 1 + dj);
                        const double ud = draw_uniform_ni(seed, chain_id, (uint64_t)td);
                        const unsigned bal = __ballot_sync(BFB_FULL, ud < 0.5);      // log(u) < log(0.5) on the draw grid of bfb_rng.h
                        if (newdir) dir4 = (bal >> (lane & ~3)) & 0xfu;
                    }
                    if (dstart) {
                        const bool right = (dir4 >> (depthE & 3)) & 1u;
                        if (!restarted) {
                            const double *src = right ? eTR : eTL;
                            VLD(q, src) VLD(p, src + SLOT) VLD(g, src + 2 * SLOT)
                        }
                        stepE = right ? fabs(stepE) : -fabs(stepE);
                    }
                }
                const int s0 = slotmail[(rb * 2 + 0) * 8 + gi], s1 = slotmail[(rb * 2 + 1) * 8 + gi];
                const double dt = 0.5 * stepE;
                // ---- two leaves: integration.py:68-95 ----
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    const bool go = liveE && (half == 0 || depthE >= 1);
                    const int ri = rb * 2 + half;
                    if (!__any_sync(BFB_FULL, go)) {
                        if (lg == 0) { rec_tag[ri * 8 + gi] = -1; if (half == 0) rec_tag[(ri + 1) * 8 + gi] = -1; }
                        break;
                    }
                    if (go) {
#pragma unroll
                        for (int k = 0; k < NR; ++k) {
                            p[k] = fma(dt, g[k], p[k]);
                            q[k] = fma(stepE, var[k] * p[k], q[k]);
                        }
                    }
                    double lp, ke2;
                    {
                        double gn[NR];
                        dmma_logp_grad<NR, MV>(bsm, lane, K, q, msm, go, lp, gn,
                                               [&](const double (&gg)[NR]) {
                                                   double s_ = 0.;
#pragma unroll
                                                   for (int k = 0; k < NR; ++k) { const double pn = fma(dt, gg[k], p[k]); s_ = fma(pn, var[k] * pn, s_); }
                                                   return s_;
                                               }, ke2);
                        if (go) {
#pragma unroll
                            for (int k = 0; k < NR; ++k) {
                                g[k] = gn[k];
                                p[k] = fma(dt, gn[k], p[k]);
                            }
                        }
                    }
                    const double Eng = 0.5 * ke2 - lp;
                    if (go) {
                        VST(ringP + ri * SLOT, p)
                        const int sl = half ? s1 : s0;
                        if (sl >= 0) {
                            double *slot = gpr + (size_t)sl * 2 * SLOT;
                            VST(slot, q) VST(slot + SLOT, g)
                        }
                    }
                    if (lg == 0) { rec_lp[ri * 8 + gi] = lp; rec_E[ri * 8 + gi] = Eng; rec_tag[ri * 8 + gi] = go ? epoch_seen : -1; }
                }
                // ---- end of a doubling: keep the new end of the trajectory ----
                if (liveE) {
                    ileafE += (depthE >= 1) ? 2 : 1;
                    if (ileafE == (1 << depthE)) {
                        double *dst = stepE > 0. ? eTR : eTL;
                        VST(dst, q) VST(dst + SLOT, p) VST(dst + 2 * SLOT, g)
                        depthE += 1; ileafE = 0;
                        if (depthE >= L) liveE = false;
                    }
                }
                TICK(2)
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_full + rb);
                ++r;
            }
        }
#ifdef BFB_PAIR_TIMING
        if (lane == 0) {
            atomicAdd(st.tree_total + 12, (unsigned long long)dbg_rounds);
            for (int k_ = 0; k_ < 3; ++k_) atomicAdd(st.tree_total + 13 + k_, (unsigned long long)tacc[k_]);
        }
#endif
        return;
    }

    // ==================================================== tree warp ====================================================
    volatile int *qv = queue;
    volatile int *ring = queue + 2 + n_groups;
    bool first_unit = true;                       // the first unit of a pair is pre-assigned: the groups spread over all SMs
    int epochT = 0;
#pragma unroll 1
    for (;;) {
    int idx = 0, group = 0;
    if (lane == 0) {
        idx = first_unit ? (int)(blockIdx.x + gridDim.x * pi) : atomicAdd(queue, 1);
        if (idx < n_units) { while ((group = ring[idx]) < 0) __nanosleep(1000); }
    }
    first_unit = false;
    idx = __shfl_sync(BFB_FULL, idx, 0);
    if (idx >= n_units) {
        if (lane == 0) { unit_i[0] = -1; mbar_arrive(bar_unit); }
        break;
    }
    group = __shfl_sync(BFB_FULL, group, 0);
    __threadfence();
    const int chunk = qv[2 + group];
    const int it_lo = chunk * chunk_iters;
    const int it_hi = min(out.n_iter, it_lo + chunk_iters);
    const long long t_unit0 = clock64(); (void)t_unit0;
    if (lane == 0) unit_i[0] = group;
    const int64_t c_raw = (int64_t)group * 8 + gi;
    const bool exists = c_raw < st.C;
    const int64_t c = exists ? c_raw : st.C - 1;
    double *gst = gstack + (size_t)group * (size_t)(L - 1 > LS ? L - 1 - LS : 0) * 3 * SLOT;   // deep stack levels (L2 resident)
    double *gpr = gprop + (size_t)group * BFB_PAIR_NSLOT * 2 * SLOT;

    // ---- chain state (adaptation scalars stay in global memory: they are touched once per iteration) ----
    const size_t vb = (size_t)c * M.np;
    double p[NR], var[NR];
    {
        // the starting point = slot 0 of the pool, "the accepted proposal" of the boundary below
        double q0[NR], g0[NR];
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const int j = 4 * k + lg;
            q0[k] = st.q[vb + j]; g0[k] = st.g[vb + j]; var[k] = st.var[vb + j]; p[k] = 0.;
        }
        VST(gpr, q0) VST(gpr + SLOT, g0)
    }
    const uint64_t chain_id = (uint64_t)(cfg.chain0 + c);
    int64_t t = st.t_draw[c];
    const int it0 = base_iter;                 // iterations done before this launch (same for every chain)
    double logp_q = st.logp[c];
    double log_step = st.log_step[c], log_bar = st.log_bar[c];
    double e_step = exp(log_step), e_bar = exp(log_bar);    // refreshed only when dual averaging moves them
    int status = exists ? st.status[c] : 9;
    const int status_in = status;
    unsigned tree_total = 0, dbg_rounds = 0, dbg_merges = 0, dbg_iend = 0; (void)dbg_rounds; (void)dbg_merges; (void)dbg_iend;
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64(); (void)tacc; (void)tlast;
    bool done = (status != 0) || it_lo >= it_hi;
    int it = it_lo;

    // transition state
    double E0 = 0., step = 0., prop_E = 0., prop_lp = 0., acc_sum = 0., maxdE = 0.;
    WT Wtree; Wtree.m = 1.; Wtree.k = 0;
    int depth = 0, ileaf = 0, n_prop = 0, diverging = 0, prop_slot = 0, Rslot = 0;
    unsigned freemask = 0;
    int A0 = -1, A1 = -1, B0 = -1, B1 = -1;        // slots reserved for the leaves of the round T works on / of the next one
    double Rpl[NR], Rps[NR], REp = 0., Rlpp = 0.;
    WT RW; RW.m = 0.; RW.k = 0;
#pragma unroll
    for (int k = 0; k < NR; ++k) Rpl[k] = Rps[k] = 0.;
    bool bnd = !done, fresh = true, ns_dbl = false, first = true;

    auto stack_ptr = [&](int lvl) -> double * {
        return (lvl <= LS) ? (sST + (lvl - 1) * 3 * SLOT) : (gst + (size_t)(lvl - 1 - LS) * 3 * SLOT);
    };
    auto reserve = [&]() -> int {
        if (!freemask) return -1;
        const int s = __ffs(freemask) - 1;
        freemask &= ~(1u << s);
        return s;
    };

#pragma unroll 1
    for (;;) {
        bool newtree = false;
        // ================= iteration boundary: base_hmc.py:62-85, Tree.__init__ nuts.py:27-43 =================
        if (__any_sync(BFB_FULL, bnd)) {
            DBG_COUNT(dbg_iend)
            const bool endp = bnd && !fresh;
            const bool warm_old = (it0 + it) < cfg.n_warmup;            // of the iteration that ends
            const size_t orow = (size_t)c * out.n_iter + it;
            // the accepted proposal (position, gradient) comes from the L2-resident pool: issue the loads first
            double qn[NR], gx[NR];
            {
                const double *slot = gpr + (size_t)prop_slot * 2 * SLOT;
                VLD(qn, slot) VLD(gx, slot + SLOT)
            }
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
            // the mailbox doubles as the scratch of the cooperative part: E reads a chain's lanes only after the epoch moved
            if (bnd) { VST(mVAR, var) VST(mQ, qn) VST(mG, gx) }
            __syncwarp();
            // ---- (2) cooperative, lane j = dimension j, one chain at a time: new sample out, windowed Welford
            //      metric (metrics.py:186-211, 333-371), momentum draw (metrics.py:83-86) ----
            unsigned mask = __ballot_sync(BFB_FULL, bnd);
#pragma unroll 1
            while (mask) {
                const int src = (__ffs(mask) - 1) & ~3;
                mask &= ~(0xfu << src);
                const int64_t c_s = shfl64(c, src), t_s = shfl64(t, src);
                const int it_s = __shfl_sync(BFB_FULL, it, src);
                const int fl = __shfl_sync(BFB_FULL, (endp ? 1 : 0) | (done ? 2 : 0) | (warm_old ? 4 : 0), src);
                const int j = lane, e = (j >> 2) * 32 + src + (j & 3);     // element of a vector slot holding dim j of that chain
                if (fl & 1) {
                    const double qj = (j < 4 * NR) ? mQ[e] : 0.;
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
                        if (upd) mVAR[e] = fgr / fg_n;
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
                    if (j < n) p0j = draw_normal_ni(seed, (uint64_t)(cfg.chain0 + c_s), (uint64_t)(t_s + j)) / sqrt(mVAR[e]);
                    if (j < 4 * NR) mP0[e] = p0j;
                }
            }
            __syncwarp();
            // ---- (3) per chain, predicated: the new state and the empty tree ----
            double p0[NR], part = 0.;
            {
                double vn[NR];
                VLD(vn, mVAR) VLD(p0, mP0)
                if (bnd) {
#pragma unroll
                    for (int k = 0; k < NR; ++k) var[k] = vn[k];
                }
            }
#pragma unroll
            for (int k = 0; k < NR; ++k) part = fma(p0[k], var[k] * p0[k], part);
            const double ke = qsum(part);
            const bool warm_new = (it0 + it) < cfg.n_warmup;
            bool startp = bnd && !done;
            if (startp) {
                t += n;
                E0 = 0.5 * ke - logp_q;
                if (!isfinite(E0)) { status = 2; done = true; startp = false; }
            }
            if (startp) {
                step = warm_new ? e_step : e_bar;
                VST(sTLp, p0) VST(sTRp, p0) VST(sPS, p0)
                freemask = ((1u << BFB_PAIR_NSLOT) - 1u) & ~(1u << prop_slot);
                prop_E = E0; prop_lp = logp_q; Wtree.m = 1.; Wtree.k = 0; acc_sum = 0.; maxdE = 0.;
                depth = 0; n_prop = 0; diverging = 0;
                ns_dbl = true;
                newtree = true;
                epochT += 1;
                if (lg == 0) { mb_step[gi] = step; mb_tstart[gi] = (long long)t; }
            }
            bnd = false; fresh = false;
        }
        TICK(0)
        // ---- slots for the leaves E publishes next; hand the finished round back to E ----
        {
            if (first) { A0 = reserve(); A1 = reserve(); }
            else { A0 = newtree ? -1 : B0; A1 = newtree ? -1 : B1; }      // leaves in flight belong to the finished iteration
            B0 = reserve(); B1 = reserve();
            if (lg == 0) {
                if (first) { slotmail[((r & 1) * 2 + 0) * 8 + gi] = A0; slotmail[((r & 1) * 2 + 1) * 8 + gi] = A1; }
                slotmail[(((r + 1) & 1) * 2 + 0) * 8 + gi] = B0; slotmail[(((r + 1) & 1) * 2 + 1) * 8 + gi] = B1;
                const int ep = done ? -1 : epochT;
                if (first) mail_ep[(r & 1) * 8 + gi] = ep;
                mail_ep[((r + 1) & 1) * 8 + gi] = ep;
            }
            const bool all_done = !__any_sync(BFB_FULL, !done);
            if (all_done && lane == 0) unit_i[1] = r + 1;
            __syncwarp();
            if (lane == 0) mbar_arrive(first ? bar_unit : bar_done + ((r - 1) & 1));
            if (all_done) {
                // E computes exactly one more round: drain it so that the phases of both barriers stay in step
                mbar_wait(bar_full + (r & 1), (unsigned)(r >> 1) & 1u);
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_done + (r & 1));
                ++r;
                break;
            }
            first = false;
        }
        TICK(7)
        const bool live = !done;
        DBG_COUNT(dbg_rounds)
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
                const double *src = right ? sTRp : sTLp;
                double pe[NR];
                VLD(pe, src)
                VST(sPB, pe)
                step = right ? fabs(step) : -fabs(step);
                ileaf = 0;
                ns_dbl = false;
            }
        }
        TICK(1)
        // ================= the two leaves of the round, as published by the integrator =================
        mbar_wait(bar_full + (r & 1), (unsigned)(r >> 1) & 1u);
        TICK(2)
        bool div_now = false, turn = false, did2 = false, adv = false, used0 = false, used1 = false;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            const int ri = (r & 1) * 2 + half;
            const bool go = live && rec_tag[ri * 8 + gi] == epochT && (half == 0 || (!div_now && depth >= 1));
            if (half == 1 && !__any_sync(BFB_FULL, go)) break;
            if (go) { VLD(p, ringP + ri * SLOT) }
            const double lp = rec_lp[ri * 8 + gi], E = rec_E[ri * 8 + gi];
            // ---- leaf: Tree._single_step, nuts.py:105-132 ----
            double dE = E - E0;
            if (isnan(dE)) dE = INFINITY;
            bool div_leaf = false;
            if (go) {
                if (half == 0) adv = true;
                if (fabs(dE) > fabs(maxdE)) maxdE = dE;
                n_prop += 1;
                div_leaf = !(fabs(dE) < cfg.max_change);
                if (half == 1) ileaf += 1;
            }
            const WT wl = wt_from_dE(div_leaf ? 0. : dE);
            const bool okl = go && !div_leaf;
            const int nslot = half ? A1 : A0;
            if (okl) {
                acc_sum += wt_min1(wl);
                if (half) used1 = true; else used0 = true;
            }
            if (div_leaf) { diverging = 1; div_now = true; }
            if (half == 0) {
                if (okl) {
#pragma unroll
                    for (int k = 0; k < NR; ++k) { Rpl[k] = p[k]; Rps[k] = p[k]; }
                    RW = wl; REp = E; Rlpp = lp; Rslot = nslot;
                }
            } else {
                // ---- level-0 merge of the two leaves (nuts.py:134-178 with depth 1: only the full-span U-turn test) ----
                double v0 = 0., v1 = 0.;
#pragma unroll
                for (int k = 0; k < NR; ++k) {
                    const double ps = Rps[k] + p[k];
                    v0 = fma(ps, var[k] * Rpl[k], v0); v1 = fma(ps, var[k] * p[k], v1);
                }
                double z0 = 1., z1 = 1.;
                qsum4(v0, v1, z0, z1, lane);
                const double um = uni(t);
                if (okl) {
                    t += 1;
                    const WT tot = wt_add(RW, wl);
                    if (!wt_select(um, tot, wl)) {               // keep the first leaf as the proposal (nuts.py:164-167)
                        freemask |= 1u << nslot;
                    } else {
                        freemask |= 1u << Rslot;
                        Rslot = nslot; REp = E; Rlpp = lp;
                    }
#pragma unroll
                    for (int k = 0; k < NR; ++k) Rps[k] += p[k];
                    RW = tot;
                    if (v0 <= 0. || v1 <= 0.) turn = true;
                    did2 = true;
                }
            }
        }
        // reserved slots that got no (accepted) leaf go back to the pool
        if (A0 >= 0 && !used0) freemask |= 1u << A0;
        if (A1 >= 0 && !used1) freemask |= 1u << A1;
        TICK(3)
        // ================= merges above level 0: Tree._build_subtree, nuts.py:134-178 =================
        int lvl = 1;
        bool need = did2 && !turn && ((ileaf >> lvl) & 1);
#pragma unroll 1
        while (__any_sync(BFB_FULL, need)) {
            const int lv = need ? lvl : 1;
            DBG_COUNT(dbg_merges)
            double T1pl[NR], T1pr[NR], T1ps[NR];
            if (__any_sync(BFB_FULL, lv > LS)) {              // a deep level somewhere in the warp: generic loads
                const double *sp = stack_ptr(lv);
                VLD(T1pl, sp) VLD(T1pr, sp + SLOT) VLD(T1ps, sp + 2 * SLOT)
            } else {                                          // common case: shared-memory loads
                const double *sp = sST + (lv - 1) * 3 * SLOT;
                VLD(T1pl, sp) VLD(T1pr, sp + SLOT) VLD(T1ps, sp + 2 * SLOT)
            }
            double v0 = 0., v1 = 0., v2 = 0., v3 = 0., v4 = 0., v5 = 0.;
            double ps[NR];
#pragma unroll
            for (int k = 0; k < NR; ++k) {
                ps[k] = T1ps[k] + Rps[k];
                const double vT1pl = var[k] * T1pl[k], vp = var[k] * p[k];
                const double ps1 = T1ps[k] + Rpl[k], ps2 = T1pr[k] + Rps[k];
                v0 = fma(ps[k], vT1pl, v0); v1 = fma(ps[k], vp, v1);
                v2 = fma(ps1, vT1pl, v2); v3 = fma(ps1, var[k] * Rpl[k], v3);
                v4 = fma(ps2, var[k] * T1pr[k], v4); v5 = fma(ps2, vp, v5);
            }
            const bool turning = quad_any_nonpos6(v0, v1, v2, v3, v4, v5, lane);
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
#pragma unroll
                for (int k = 0; k < NR; ++k) { Rpl[k] = T1pl[k]; Rps[k] = ps[k]; }
                RW = tot;
                if (turning) turn = true;
                lvl++;
            }
            need = need && !turn && ((ileaf >> lvl) & 1);
        }
        TICK(4)
        const bool fin = adv && (div_now || turn || (ileaf + 1 == (1 << depth)));
        const bool push = adv && !fin;
        if (__any_sync(BFB_FULL, push)) {
            const int lv = push ? lvl : 1;
            if (__any_sync(BFB_FULL, lv > LS)) {
                double *sp = stack_ptr(lv);
                if (push) { VST(sp, Rpl) VST(sp + SLOT, p) VST(sp + 2 * SLOT, Rps) }
            } else {
                double *sp = sST + (lv - 1) * 3 * SLOT;
                if (push) { VST(sp, Rpl) VST(sp + SLOT, p) VST(sp + 2 * SLOT, Rps) }
            }
            if (push) {
                ssc[lvl * 8] = RW.m; ssc[(10 + lvl) * 8] = (double)RW.k; ssc[(20 + lvl) * 8] = REp; ssc[(30 + lvl) * 8] = Rlpp;
                ssc[(40 + lvl) * 8] = (double)Rslot;
                ileaf += 1;
            }
        }
        TICK(5)
        // ================= end of a doubling: Tree.extend, nuts.py:45-103 =================
        if (__any_sync(BFB_FULL, fin)) {
            const double ue = uni(t);
            const bool right = step > 0.;
            if (fin) {
                double *dst = right ? sTRp : sTLp;
                VST(dst, p)
                depth += 1;
            }
            const bool ok = fin && !div_now && !turn;
            double PS[NR], PB[NR], TLp[NR], TRp[NR];
            VLD(PS, sPS) VLD(PB, sPB) VLD(TLp, sTLp) VLD(TRp, sTRp)
            double v0 = 0., v1 = 0., v2 = 0., v3 = 0., v4 = 0., v5 = 0.;
#pragma unroll
            for (int k = 0; k < NR; ++k) {
                PS[k] += Rps[k];
                const double vp = var[k] * p[k], vRpl = var[k] * Rpl[k], vPB = var[k] * PB[k];
                const double vTL = var[k] * TLp[k], vTR = var[k] * TRp[k];
                v0 = fma(PS[k], vTL, v0); v1 = fma(PS[k], vTR, v1);
                // nuts.py:86-98: self.p_sum is updated in place BEFORE p_sum1 / p_sum2 are formed, so the
                // "old tree" p_sum entering them is already the total (see the oracle, bf_oracle.c tree_extend)
                if (right) {
                    const double ps1 = PS[k] + Rpl[k], ps2 = PB[k] + Rps[k];
                    v2 = fma(ps1, vTL, v2); v3 = fma(ps1, vRpl, v3); v4 = fma(ps2, vPB, v4); v5 = fma(ps2, vp, v5);
                } else {
                    const double ps1 = Rps[k] + PB[k], ps2 = Rpl[k] + PS[k];
                    v2 = fma(ps1, vp, v2); v3 = fma(ps1, vPB, v3); v4 = fma(ps2, vRpl, v4); v5 = fma(ps2, vTR, v5);
                }
            }
            const bool turning = quad_any_nonpos6(v0, v1, v2, v3, v4, v5, lane);
            if (ok) {
                t += 1;
                const WT tot = wt_add(Wtree, RW);
                if (wt_select(ue, Wtree, RW)) {               // nuts.py:81-83 biased progressive: log(u) < size2 - size1
                    freemask |= 1u << prop_slot;
                    prop_slot = Rslot; prop_E = REp; prop_lp = Rlpp;
                } else {
                    freemask |= 1u << Rslot;
                }
                Wtree = tot;
                VST(sPS, PS)
                if (turning) turn = true;
            }
            if (fin) {
                const bool iter_end = div_now || turn || (depth >= cfg.max_treedepth);
                bnd = iter_end;
                ns_dbl = !iter_end;
            }
        }
        TICK(6)
        ++r;
    }

    // ---- persist chain state: position and gradient are those of the accepted proposal ----
    if (exists && status_in == 0) {
        double qf[NR], gf[NR];
        const double *slot = gpr + (size_t)prop_slot * 2 * SLOT;
        VLD(qf, slot) VLD(gf, slot + SLOT)
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const int j = 4 * k + lg;
            st.q[vb + j] = qf[k]; st.g[vb + j] = gf[k]; st.var[vb + j] = var[k];
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
#ifdef BFB_PAIR_TIMING
        atomicAdd(st.tree_total + 1, (unsigned long long)dbg_rounds);
        atomicAdd(st.tree_total + 2, (unsigned long long)dbg_merges);
        atomicAdd(st.tree_total + 3, (unsigned long long)dbg_iend);
        long long tsum = 0;
        for (int k_ = 0; k_ < 7; ++k_) { atomicAdd(st.tree_total + 4 + k_, (unsigned long long)tacc[k_]); tsum += tacc[k_]; }
        atomicAdd(st.tree_total + 11, (unsigned long long)tacc[7]);
#endif
        qv[2 + group] = chunk + 1;
        if ((chunk + 1) * chunk_iters < out.n_iter) {
            const int ti = atomicAdd(queue + 1, 1);
            __threadfence();
            ring[ti] = group;
        }
    }
    }   // unit loop
#undef VLD
#undef VST
}

template <int NR, int MV>
static int launch_pair(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    using SH = DmmaShape<NR, MV>;
    constexpr int SLOT = NR * 32, NP = 4;
    const int L = h->scfg.max_treedepth;
    const int64_t C = h->cs.C;
    const int n_groups = (int)((C + 7) / 8);
    const size_t fixed = sizeof(double) * (SH::frag_doubles(NP) + SH::MSM_DOUBLES + (SH::C3 ? dmma_c3_doubles(NR, h->dm.c3_kt, NP) : 0));
    const size_t cap = 227 * 1024;
    if (fixed + sizeof(double) * NP * pair_smem_doubles(NR, 1) > cap) return 1;          // does not fit
    int LS = L - 1 > 1 ? L - 1 : 1;
    while (LS > 1 && fixed + sizeof(double) * NP * pair_smem_doubles(NR, LS) > cap) --LS;
    if (const char *e = getenv("BFB200_STACK_LEVELS_SMEM")) { int v = atoi(e); if (v >= 1 && v < LS) LS = v; }
    const size_t smem = fixed + sizeof(double) * NP * pair_smem_doubles(NR, LS);
    BFB_CUDA(cudaFuncSetAttribute(nuts_pair_kernel<NR, MV, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    double *gprop;
    int rc;
    if ((rc = gstack_reserve(h, n_groups, L, LS, SLOT, BFB_PAIR_NSLOT, &gprop))) return rc;
    RunOutDevF od;
    od.o = o; od.n_iter = n_iter;
    int blocks = h->sm_count;
    if ((int64_t)blocks > n_groups) blocks = n_groups;
    int chunk_iters, n_units;
    if ((rc = queue_setup(h, n_groups, n_iter, 6, blocks * NP, 0, chunk_iters, n_units))) return rc;
    nuts_pair_kernel<NR, MV, NP><<<blocks, 64 * NP, smem, h->stream>>>(h->dm, h->scfg, h->cs, od, L, LS, h->gstack, gprop,
                                                                       (int)h->iters_done, chunk_iters, n_groups, n_units, h->queue);
    h->launches++;
    BFB_CUDA(cudaGetLastError());
    return BFB_OK;
}

// launches the pair kernel of the model (select_family, bfb_sampler.cu, chose this family): 0 on launch, 1 when its shared memory
// does not fit, < 0 on error
int bfb_launch_nuts_pair(bfb_context *h, const bfb_run_out &o, int n_iter)
{
    const DevModel &M = h->dm;
    const int mv = (M.has_c2 ? 1 : 0) | (M.frag_ext ? 2 : 0);
#define BFB_CASE(NR_, MV_) if (M.frag_nr == NR_ && mv == MV_) return launch_pair<NR_, MV_>(h, o, n_iter);
    BFB_CASE(4, 0) BFB_CASE(4, 1) BFB_CASE(4, 2) BFB_CASE(4, 3) BFB_CASE(7, 0) BFB_CASE(7, 1) BFB_CASE(7, 2) BFB_CASE(7, 3)
    BFB_CASE(8, 0) BFB_CASE(8, 1) BFB_CASE(8, 2) BFB_CASE(8, 3)
#undef BFB_CASE
    bfb_set_error("bfb_launch_nuts_pair: no kernel instantiation for this model");
    return BFB_ERR_ARG;
}
