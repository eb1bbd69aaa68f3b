// Fused thin-lens render: the CUDA counterpart of ThinLens.render + ThinLens.coc
// (deeplens/psfnet.py:503-570).  Per output pixel: circle of confusion from depth and focus
// distance -> clipped Gaussian k x k PSF (sigma = coc/2, taps outside the coc radius are zero)
// -> normalise -> gather (deeplens/render_psf.py:76-107).  The reference materialises the
// [N,H,W,k,k] PSF tensor through ~15 elementwise torch kernels; here taps live in registers.
//
// CTA tile = 8 rows x 64 columns, two horizontally adjacent pixels per thread (warp = row, lane j = columns 2j, 2j+1),
// image halo tile in shared memory, planar per channel, DOUBLE-BUFFERED: the halo of the next tile arrives under the
// current tile's arithmetic
//   * as ONE TMA tensor-tile copy (cp.async.bulk.tensor.3d: box = [channels][rows][columns] of the [N*C, H, W] image,
//     issued by one thread, completion on an mbarrier; the box starts at a 16-byte-aligned column) when the tile's halo
//     lies inside the image, and
//   * by per-thread cp.async of the replicate-clamped pixels (render_psf.py:96 pads with mode='replicate', which a
//     TMA box cannot do: it zero-fills out-of-bounds elements) for tiles that touch the image border, or when the
//     image does not meet TMA's 16-byte row-pitch rule (W % 4 != 0).
// The Gaussian is separable: exp(-(dx^2+dy^2)/2s^2) = g(dx) g(dy), so a pixel needs (k+1)/2 exponentials per PSF row
// pair instead of one per tap; the disk mask (dx^2+dy^2 < radius^2) is an integer compare against a per-row limit.
//   * the weights of a PSF row depend on |dy| and |dx| only: for each |dy| the (k+1)/2 weights per pixel are formed
//     once (FMUL + compare/select) and serve the rows -dy and +dy and both signs of dx; the normalising sum is taken
//     from the same (k+1)/2 values -- nothing but LDS and FFMA is left per tap;
//   * per PSF row and channel the thread loads ONE (k+1 [+1 for alignment])-wide window with LDS.64 and both pixels
//     take their k taps from it: (k+3)/2 LDS.64 per 2k FFMA instead of 2k LDS.32.
// ~5 instructions per tap and pixel, against ~9 for one pixel per thread (FMUL + ISETP/FSEL + FADD + 3 FFMA + 3 LDS).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include "ptx_sm100.cuh"

namespace aadff {

constexpr int TL_TILE_H = 8;
constexpr int TL_MAXC = 3;                // channels per launch (RGB); more channels = more passes
constexpr int TL_NT = TL_TILE_H * 32;

struct ThinLensArgs {
    const float* img;     // [N,C,H,W]
    const float* depth;   // [N,H,W] mm (sign as given by the caller)
    const float* foc;     // [N] mm
    float* out;           // [N,C,H,W]
    int N, C, H, W, c0, cn;
    float k1;             // foc_len / fnum
    float foc_len, ps;    // focal length [mm], pixel size [mm]
    float d_lo, d_hi;     // depth clamp: 200, 20000 mm
    int flip;             // 1: depth and foc are negated first (reference: `if (depth < 0).any()`)
    const unsigned char* flip_dev;   // if not null, the decision is read from device memory (see any_negative_kernel):
                                     // the reference's data-dependent branch without a device->host round trip
    int use_tma;          // the tensor map below is valid (W % 4 == 0, 16-byte aligned image)
};

// flag[0] |= any(x < 0)   (the reference's `if (depth < 0).any()`, psfnet.py:504, decided on the device)
__global__ void __launch_bounds__(256) any_negative_kernel(const float* __restrict__ x, long long n, unsigned char* flag) {
    bool neg = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        neg |= (__ldg(x + i) < 0.f);
    if (__syncthreads_or(neg) && threadIdx.x == 0) *flag = 1;     // benign race: every writer stores 1
}

// TMA: one [planes][rows][cols] box of a 3-D tensor map -> shared memory, completion counted on `bar`
__device__ __forceinline__ void tma_load_3d(uint32_t dst_smem, const CUtensorMap* map, int x, int y, int z, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(bar)
        : "memory");
}

constexpr int TL2_TILE_W = 64;
#ifndef AADFF_TL2_MINB
#define AADFF_TL2_MINB 1          // resident CTAs per SM the register allocation aims at
#endif

template <int KS>
struct ThinLens2Cfg {
    static constexpr int R = (KS - 1) / 2;
    static constexpr int HH = TL_TILE_H + KS - 1;
    static constexpr int HW = TL2_TILE_W + KS - 1;
    // TMA rules (measured: a box whose first element is not 16-byte aligned in global memory raises "illegal
    // instruction"): the box starts SH columns left of the halo, at a multiple of 4 floats, and its width is a multiple of 4
    static constexpr int SH = (4 - R % 4) % 4;
    static constexpr int WOFF = SH & 1;                         // LDS.64 windows start at an even float index
    static constexpr int NLD = (WOFF + KS + 1 + 1) / 2;         // float2 loads per window
    static constexpr int BW = (HW + SH + 1 + 3) / 4 * 4;        // one spare column: the last window may read one float past the halo
    static constexpr int CSTRIDE = HH * BW;
    __host__ __device__ static constexpr int BUF_FLOATS(int cn) { return (cn * CSTRIDE + 31) / 32 * 32; }   // 128-byte multiple: TMA destination alignment
    // Two halo buffers (the next tile's copy runs under this tile's arithmetic) while they are small; large kernels keep
    // one buffer: at k = 31 two 29 KB buffers left 3 CTAs per SM and the kernel, which lives on resident warps hiding
    // LDS latency, lost 11 % (measured)
    static constexpr int NBUF = KS <= 15 ? 2 : 1;
    __host__ __device__ static constexpr int SMEM_BYTES(int cn) { return NBUF * BUF_FLOATS(cn) * 4 + 128; }  // barriers in front
};

template <int KS>
__global__ void __launch_bounds__(TL_NT, AADFF_TL2_MINB)
thinlens_render2_kernel(const ThinLensArgs a, const __grid_constant__ CUtensorMap img_map) {
    using Cfg = ThinLens2Cfg<KS>;
    constexpr int R = Cfg::R, HH = Cfg::HH, HW = Cfg::HW, BW = Cfg::BW, SH = Cfg::SH, CSTRIDE = Cfg::CSTRIDE;
    constexpr int WOFF = Cfg::WOFF, NLD = Cfg::NLD;
    extern __shared__ __align__(128) unsigned char tl_smem[];
    float* bufs = reinterpret_cast<float*>(tl_smem + 128);
    const uint32_t bar0 = smem_u32(tl_smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_x = (a.W + TL2_TILE_W - 1) / TL2_TILE_W, tiles_y = (a.H + TL_TILE_H - 1) / TL_TILE_H;
    const int n_tiles = a.N * tiles_x * tiles_y;               // < 2^31 (checked by the host): 32-bit tile arithmetic
    const bool flip = a.flip_dev ? (*a.flip_dev != 0) : (a.flip != 0);
    const int buf_floats = Cfg::BUF_FLOATS(a.cn);

    if (threadIdx.x == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto coords = [&](int tile, int& n, int& h0, int& w0) {
        const int row = tile / tiles_x, tx = tile - row * tiles_x;
        n = row / tiles_y;
        h0 = (row - n * tiles_y) * TL_TILE_H;
        w0 = tx * TL2_TILE_W;
    };
    auto interior = [&](int h0, int w0) {      // the halo lies inside the image (the box's alignment / spare columns may not: unused)
        return a.use_tma && h0 - R >= 0 && w0 - R >= 0 && h0 - R + HH <= a.H && w0 - R + HW <= a.W;
    };
    auto issue_halo = [&](int tile, int b) {
        int n, h0, w0;
        coords(tile, n, h0, w0);
        float* dst = bufs + b * buf_floats;
        if (interior(h0, w0)) {
            if (threadIdx.x == 0) {
                mbar_arrive_expect_tx(bar0 + 8 * b, (uint32_t)(a.cn * CSTRIDE * 4));
                tma_load_3d(smem_u32(dst), &img_map, w0 - R - SH, h0 - R, n * a.C + a.c0, bar0 + 8 * b);
            }
        } else {
            // warp = halo row (stride 8), lane = halo column (stride 32): no index divisions
            const uint32_t d0 = smem_u32(dst) + 4u * (uint32_t)SH;
            const float* plane0 = a.img + (long long)(n * a.C + a.c0) * a.H * a.W;
            const long long plane = (long long)a.H * a.W;
            for (int yy = warp; yy < HH; yy += TL_TILE_H) {
                const int gy = min(max(h0 + yy - R, 0), a.H - 1);                                   // replicate
#pragma unroll
                for (int x0 = 0; x0 < HW; x0 += 32) {
                    const int xx = x0 + lane;
                    if (xx < HW) {
                        const float* src = plane0 + (long long)gy * a.W + min(max(w0 + xx - R, 0), a.W - 1);
                        const uint32_t d = d0 + 4u * (uint32_t)(yy * BW + xx);
                        cp_async4(d, src);
                        if (a.cn > 1) cp_async4(d + 4u * CSTRIDE, src + plane);
                        if (a.cn > 2) cp_async4(d + 8u * CSTRIDE, src + 2 * plane);
                    }
                }
            }
        }
    };

    constexpr bool DB = Cfg::NBUF == 2;
    uint32_t phase = 0;
    int cur = 0;
    if (DB && (int)blockIdx.x < n_tiles) issue_halo(blockIdx.x, 0);
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int n, h0, w0;
        coords(tile, n, h0, w0);
        const int h = h0 + warp, w = w0 + 2 * lane;
        // circle of confusion (ThinLens.coc, psfnet.py:503-511), operation order of the reference
        float cexp[2] = {0.f, 0.f};
        int r2c[2] = {0, 0};
        bool ok[2];
        const float f0 = __ldg(a.foc + n);
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            ok[p] = (h < a.H) && (w + p < a.W);
            if (ok[p]) {
                float d = __ldg(a.depth + ((long long)n * a.H + h) * a.W + w + p);
                float f = f0;
                if (flip) { d = -d; f = -f; }
                d = fminf(fmaxf(d, a.d_lo), a.d_hi);
                float coc = a.k1 * fabsf(d - f);
                coc = __fdiv_rn(coc, d);
                coc = coc * a.foc_len;
                coc = __fdiv_rn(coc, f - a.foc_len);
                const float coc_px = fmaxf(__fdiv_rn(coc, a.ps), 0.1f);
                const float rad = coc_px * 0.5f;
                const float r2 = rad * rad;
                cexp[p] = __fdiv_rn(-0.5f * 1.4426950408889634f, r2);    // exp(-d2/2/r2) = 2^(d2 * cexp)
                r2c[p] = (r2 >= 4096.f) ? 4096 : (int)ceilf(r2);          // d2 < r2 as an integer compare (d2 <= 450)
            }
        }
        if (!DB) issue_halo(tile, 0);
        if (interior(h0, w0)) {
            mbar_wait(bar0 + 8 * cur, (phase >> cur) & 1);
            phase ^= 1u << cur;
        } else {
            cp_async_wait_all();
        }
        __syncthreads();
        if (DB && tile + (int)gridDim.x < n_tiles) issue_halo(tile + gridDim.x, cur ^ 1);

        if (ok[0]) {
            float g[2][R + 1];                                  // g[p][d] = 2^(d^2 cexp): the separable Gaussian factor
#pragma unroll
            for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int d = 0; d <= R; ++d) g[p][d] = exp2f((float)(d * d) * cexp[p]);
            float acc[2][TL_MAXC], wsum[2] = {0.f, 0.f};
#pragma unroll
            for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int c = 0; c < TL_MAXC; ++c) acc[p][c] = 0.f;
            const float* ib = bufs + cur * buf_floats + warp * BW + (SH - WOFF) + 2 * lane;
            // absent channels re-read channel 0 (results discarded at the store): no branches in the tap loop
            const int cs[TL_MAXC] = {0, a.cn > 1 ? CSTRIDE : 0, a.cn > 2 ? 2 * CSTRIDE : 0};
#pragma unroll 1
            for (int da = 0; da <= R; ++da) {
                float wt[2][R + 1];
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    const float gi = exp2f((float)(da * da) * cexp[p]);
                    const int lim = r2c[p] - da * da;           // tap (dy, dx) is inside the disk iff dx^2 < lim
                    float rs = 0.f;
#pragma unroll
                    for (int d = R; d >= 1; --d) {
                        wt[p][d] = (d * d < lim) ? gi * g[p][d] : 0.f;      // psf_mask = (x^2 + y^2 < radius^2)
                        rs += wt[p][d];
                    }
                    wt[p][0] = (0 < lim) ? gi : 0.f;            // g[p][0] = 1
                    rs = fmaf(2.f, rs, wt[p][0]);
                    wsum[p] += (da == 0) ? rs : 2.f * rs;
                }
#pragma unroll
                for (int side = 0; side < 2; ++side) {      // rows -dy and +dy, straight-line
                    if (side == 1 && da == 0) break;
                    const int i = side ? R + da : R - da;
                    const float* prow = ib + i * BW;
#pragma unroll
                    for (int c = 0; c < TL_MAXC; ++c) {
                        const float2* pw = reinterpret_cast<const float2*>(prow + cs[c]);
                        float win[2 * NLD];
#pragma unroll
                        for (int l = 0; l < NLD; ++l) {
                            const float2 v = pw[l];
                            win[2 * l] = v.x;
                            win[2 * l + 1] = v.y;
                        }
#pragma unroll
                        for (int p = 0; p < 2; ++p)
#pragma unroll
                            for (int j = 0; j < KS; ++j)
                                acc[p][c] = fmaf(win[WOFF + p + j], wt[p][j <= R ? R - j : j - R], acc[p][c]);
                    }
                }
            }
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                if (!ok[p]) continue;
                const float inv = __fdiv_rn(1.0f, wsum[p]);     // the centre tap always passes the mask: wsum >= 1
#pragma unroll
                for (int c = 0; c < TL_MAXC; ++c)
                    if (c < a.cn) a.out[((long long)(n * a.C + a.c0 + c) * a.H + h) * a.W + w + p] = acc[p][c] * inv;
            }
        }
        __syncthreads();
        if (DB) cur ^= 1;
    }
}

}  // namespace aadff
