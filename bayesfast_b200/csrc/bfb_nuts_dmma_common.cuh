// bfb_nuts_dmma_common.cuh -- helpers shared by the tensor-core NUTS kernels (bfb_sampler_dmma.cu, bfb_sampler_pair.cu):
// packed quad reductions of the U-turn tests, one out-of-line instance of the RNG functions and of the dual averaging.
#pragma once
#include "bfb_dmma.cuh"
#include "bfb_nuts_common.cuh"

// per chain: is any of the six sums over its 4 lanes <= 0 ?
__device__ __forceinline__ bool quad_any_nonpos6(double v0, double v1, double v2, double v3, double v4, double v5, int lane)
{
    const bool b0 = lane & 1, b1 = lane & 2;
    double k0 = b0 ? v4 : v0, k1 = b0 ? v5 : v1, k2 = b0 ? 1. : v2, k3 = b0 ? 1. : v3;
    const double s0 = b0 ? v0 : v4, s1 = b0 ? v1 : v5, s2 = b0 ? v2 : 1., s3 = b0 ? v3 : 1.;
    k0 += shx4(s0, 1); k1 += shx4(s1, 1); k2 += shx4(s2, 1); k3 += shx4(s3, 1);
    double m0 = b1 ? k2 : k0, m1 = b1 ? k3 : k1;
    const double t0 = b1 ? k0 : k2, t1 = b1 ? k1 : k3;
    m0 += shx4(t0, 2); m1 += shx4(t1, 2);
    const unsigned bal = __ballot_sync(BFB_FULL, (m0 <= 0.) || (m1 <= 0.));
    return ((bal >> (lane & ~3)) & 0xfu) != 0u;
}

// One instance of Philox and of Phi^-1 in the kernel image instead of one per call site (the code of a round must stay
// small: with one or two warps per scheduler instruction-fetch stalls are not hidden by other warps).  Every draw goes
// through philox_pair_ni, the block of draws 2 blk and 2 blk + 1 of a chain's stream (bfb_rng.h).
static __device__ __noinline__ double2 philox_pair_ni(uint64_t seed, uint64_t chain, uint64_t blk)
{
    double u0, u1;
    const bfb_philox_block b = bfb_philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)chain,
                                                 (uint32_t)(chain >> 32), (uint32_t)seed, (uint32_t)(seed >> 32));
    u0 = bfb_u64_to_uniform((uint64_t)b.v[0] | ((uint64_t)b.v[1] << 32));
    u1 = bfb_u64_to_uniform((uint64_t)b.v[2] | ((uint64_t)b.v[3] << 32));
    return make_double2(u0, u1);
}
static __device__ __noinline__ double draw_uniform_ni(uint64_t seed, uint64_t chain, uint64_t t)
{
    const double2 u = philox_pair_ni(seed, chain, t >> 1);
    return (t & 1) ? u.y : u.x;
}

// Wichura's AS 241 coefficients of bfb_norminv (bfb_rng.h), numerator then denominator, highest power first, for the
// central branch (|p - 0.5| <= 0.425), the tail with r <= 5 and the tail with r > 5
static __constant__ double bfb_as241[3][16] = {
    {2.5090809287301226727e+3, 3.3430575583588128105e+4, 6.7265770927008700853e+4, 4.5921953931549871457e+4,
     1.3731693765509461125e+4, 1.9715909503065514427e+3, 1.3314166789178437745e+2, 3.3871328727963666080e0,
     5.2264952788528545610e+3, 2.8729085735721942674e+4, 3.9307895800092710610e+4, 2.1213794301586595867e+4,
     5.3941960214247511077e+3, 6.8718700749205790830e+2, 4.2313330701600911252e+1, 1.0},
    {7.74545014278341407640e-4, 2.27238449892691845833e-2, 2.41780725177450611770e-1, 1.27045825245236838258e0,
     3.64784832476320460504e0, 5.76949722146069140550e0, 4.63033784615654529590e0, 1.42343711074968357734e0,
     1.05075007164441684324e-9, 5.47593808499534494600e-4, 1.51986665636164571966e-2, 1.48103976427480074590e-1,
     6.89767334985100004550e-1, 1.67638483018380384940e0, 2.05319162663775882187e0, 1.0},
    {2.01033439929228813265e-7, 2.71155556874348757815e-5, 1.24266094738807843860e-3, 2.65321895265761230930e-2,
     2.96560571828504891230e-1, 1.78482653991729133580e0, 5.46378491116411436990e0, 6.65790464350110377720e0,
     2.04426310338993978564e-15, 1.42151175831644588870e-7, 1.84631831751005468180e-5, 7.86869131145613259100e-4,
     1.48753612908506148525e-2, 1.36929880922735805310e-1, 5.99832206555887937690e-1, 1.0}};

// Phi^-1(p) of bfb_norminv, restated for code size: the same operations on the same operands in the same order, so the
// result is bit-identical, but the three branches share one pair of polynomials (coefficients selected from bfb_as241)
// and one division, where bfb_norminv has three of each.  bfb_rng.h stays the stream contract that the oracle compiles.
__device__ __forceinline__ double bfb_norminv_small(double p)
{
    const double q = p - 0.5;
    const bool mid = fabs(q) <= 0.425;
    double x;
    int b = 0;
    if (mid) {
        x = __fma_rn(-q, q, 0.180625);
    } else {
        x = sqrt(-log(q < 0.0 ? p : 1.0 - p));
        b = x <= 5.0 ? 1 : 2;
        x -= b == 1 ? 1.6 : 5.0;
    }
    const double *c = bfb_as241[b];
    double num = c[0], den = c[8];
#pragma unroll
    for (int k = 1; k < 8; ++k) { num = __fma_rn(num, x, c[k]); den = __fma_rn(den, x, c[8 + k]); }
    const double val = (mid ? q * num : num) / den;
    return (!mid && q < 0.0) ? -val : val;
}
static __device__ __noinline__ double draw_normal_ni(uint64_t seed, uint64_t chain, uint64_t t)
{
    const double2 u = philox_pair_ni(seed, chain, t >> 1);
    return bfb_norminv_small((t & 1) ? u.y : u.x);
}
// Nesterov dual averaging of the step size, step_size.py:31-45 -- out of line: pow and exp are ~250 instructions that only
// warm-up iteration boundaries execute, and the hot loop is larger than the instruction cache
static __device__ __noinline__ void dual_average_ni(double cnt, double hbar0, double mu_da, double accept_stat, double log_bar,
                                                    double t0, double target, double gamma, double kk,
                                                    double &hbar, double &log_step, double &log_bar_new, double &e_step, double &e_bar)
{
    const double w = 1. / (cnt + t0);
    hbar = ((1. - w) * hbar0 + w * (target - accept_stat));
    log_step = mu_da - hbar * sqrt(cnt) / gamma;
    const double mk = pow(cnt, -kk);
    log_bar_new = mk * log_step + (1. - mk) * log_bar;
    e_step = exp(log_step); e_bar = exp(log_bar_new);
}
__device__ __forceinline__ int64_t shfl64(int64_t v, int src)
{
    return (int64_t)__shfl_sync(BFB_FULL, (long long)v, src);
}
