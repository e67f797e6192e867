// bfb_gram.cuh -- the FP64 tensor-core Gram tile shared by the surrogate fit (bfb_fit.cu: gram_kernel) and the chain diagnostics
// (bfb_diag.cu: lagsum_kernel).  A CTA of 4 warps (2 x 2) owns one 64 x 64 tile (ti <= tj) of the upper block triangle of a Gram
// A^T B and multiplies two panels of KC rows staged in shared memory with DMMA m8n8k4, 32 x 32 per warp.
#pragma once

#define TS 64          // Gram tile per CTA
#define KC 32          // rows per pipeline stage
#define LDP (TS + 4)   // padded leading dimension of a staged panel: conflict-free DMMA fragment loads (LDP % 16 == 4)

__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// acc += phiI^T phiJ over the KC rows of two panels [KC][LDP].  Warp (wm, wn) owns rows 32 wm + 8 a + (lane >> 2) and columns
// 32 wn + 8 b + 2 (lane & 3) + {0, 1} of the tile in acc[a][b][0..1].
__device__ __forceinline__ void gram_tile_mma(const double *phiI, const double *phiJ, int lane, int wm, int wn,
                                              double (&acc)[4][4][2])
{
#pragma unroll
    for (int kk = 0; kk < KC / 4; ++kk) {
        const int krow = kk * 4 + (lane & 3);
        double af[4], bf[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) af[a] = phiI[krow * LDP + 32 * wm + 8 * a + (lane >> 2)];
#pragma unroll
        for (int b = 0; b < 4; ++b) bf[b] = phiJ[krow * LDP + 32 * wn + 8 * b + (lane >> 2)];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) dmma884(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
    }
}
