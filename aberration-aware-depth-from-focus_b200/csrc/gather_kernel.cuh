// Stand-alone per-pixel PSF gather: the CUDA counterpart of
// deeplens/render_psf.py:76-107 (local_psf_render) for a PSF tensor that already
// lives in HBM ([N,H,W,ks,ks] fp32).  HBM-bound on the PSF read: 4*ks^2 B per pixel
// (484 B at ks = 11) against 12 B of image and 12 B of output.
//
// local_psf_render_kernel is the generic kernel (any ks, any W, any alignment): one warp per 32 pixels, taps staged
// through shared memory with plain coalesced loads, image through L1.  Odd ks in 3..31 run the strip-walking or the
// register-streaming kernel instead (gather_strip_kernel.cuh, gather_coalesced_kernel.cuh).
#pragma once
#include <cuda_runtime.h>

namespace aadff {

constexpr int GATHER_TT = 128;                  // taps staged per chunk
constexpr int GATHER_WARPS = 4;                 // warps per CTA
constexpr int GATHER_MAXC = 4;                  // channels per pass

__global__ void __launch_bounds__(GATHER_WARPS * 32)
local_psf_render_kernel(const float* __restrict__ img, const float* __restrict__ psf, float* __restrict__ out,
                        int N, int C, int H, int W, int ks, int c0, int cn) {
    extern __shared__ float sm_taps[];          // [GATHER_WARPS][32][GATHER_TT+1]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* sp = sm_taps + warp * 32 * (GATHER_TT + 1);
    const int segs = (W + 31) / 32;
    const long long total = (long long)N * H * segs;
    const int kk = ks * ks, r = (ks - 1) / 2;

    for (long long item = (long long)blockIdx.x * GATHER_WARPS + warp; item < total;
         item += (long long)gridDim.x * GATHER_WARPS) {
        const int seg = (int)(item % segs);
        const int h = (int)((item / segs) % H);
        const int n = (int)(item / ((long long)segs * H));
        const int w0 = seg * 32;
        const int w = w0 + lane;
        const int npx = min(32, W - w0);
        const float* tap_base = psf + ((long long)(n * H + h) * W + w0) * kk;
        float acc[GATHER_MAXC] = {0.f, 0.f, 0.f, 0.f};

        for (int t0 = 0; t0 < kk; t0 += GATHER_TT) {
            const int nt = min(GATHER_TT, kk - t0);
            __syncwarp();
            for (int pp = 0; pp < npx; ++pp)
                for (int tt = lane; tt < nt; tt += 32)
                    sp[pp * (GATHER_TT + 1) + tt] = __ldg(tap_base + (long long)pp * kk + t0 + tt);
            __syncwarp();
            if (w < W) {
                int i = t0 / ks, j = t0 - i * ks;
                for (int tt = 0; tt < nt; ++tt) {
                    const float tap = sp[lane * (GATHER_TT + 1) + tt];
                    const int yy = min(max(h + i - r, 0), H - 1);
                    const int xx = min(max(w + j - r, 0), W - 1);
                    const float* px = img + ((long long)(n * C + c0) * H + yy) * W + xx;
#pragma unroll
                    for (int c = 0; c < GATHER_MAXC; ++c)
                        if (c < cn) acc[c] = fmaf(__ldg(px + (long long)c * H * W), tap, acc[c]);
                    if (++j == ks) { j = 0; ++i; }
                }
            }
        }
        if (w < W) {
#pragma unroll
            for (int c = 0; c < GATHER_MAXC; ++c)
                if (c < cn) out[((long long)(n * C + c0 + c) * H + h) * W + w] = acc[c];
        }
    }
}

}  // namespace aadff
