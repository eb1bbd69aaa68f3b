// Backward of the per-pixel PSF gather (local_psf_render, deeplens/render_psf.py:76-107).  With G = grad_out
// [N,C,H,W], P = psf [N,H,W,ks,ks], r = (ks-1)/2 and clamp() the replicate border of the forward:
//
//   dP  [n,h,w,i,j] = sum_c G[n,c,h,w] * img[n,c,clamp(h+i-r),clamp(w+j-r)]
//   dimg[n,c,y,x]   = sum over (h,w,i,j) with clamp(h+i-r) = y, clamp(w+j-r) = x of G[n,c,h,w] * P[n,h,w,i,j]
//
// Both are written exactly once per element, each as one fixed-order sum in one thread: no atomics, so two runs give
// bit-identical gradients.  All indexing of P / dP is 64-bit (P can exceed 2^31 elements).
//
// local_psf_grad_psf_strip_kernel (3 <= ks <= 15, W % 4 == 0, C <= 4) is the forward strip kernel
// (gather_strip_kernel.cuh) with the dataflow reversed.  dP is write-bound: 4 ks^2 B per pixel (484 B at ks = 11)
// against 8 C B of image and gradient read.  A warp walks down a 64-column strip with the same circular ks+1-row image
// halo; lane l owns the pixels (2l, 2l+1) and writes their 2 ks^2 products into the flat run [2l ks^2, (2l+2) ks^2)
// of a shared-memory chunk with STS.64 (lane stride 2 ks^2 floats, ks^2 odd: conflict-free, as the forward's LDS.64).
// Lane 0 then stores the whole strip row -- 64 ks^2 contiguous floats of dP -- with one cp.async.bulk shared->global
// and moves on to the next row in the other slot while the copy drains.
//
// local_psf_grad_img_strip_kernel (3 <= ks <= 15, W % 4 == 0) is the transposed gather for dimg (see below).
//
// The generic pair (runtime ks, any W, any alignment, any C) covers every other case: one thread per dP element, and
// one thread per image pixel that walks the (h,i) x (w,j) preimages of its clamped position.  dP takes the generic
// kernel for C > 4 too: dP sums over all channels and is stored once per strip row, so channel passes would have to
// read back and rewrite dP (doubling its dominant write traffic), and a halo of every channel does not fit.
#pragma once
#include <cuda_runtime.h>
#include "ptx_sm100.cuh"
#include "gather_strip_kernel.cuh"

namespace aadff {

constexpr int GPS_MAXC = 4;                      // channels the strip dP kernel keeps in its halo
constexpr int GPS_SMEM = 232448;                 // opt-in shared memory per block

template <int KS, int CN>
struct GradPsfStripCfg {
    static constexpr int KK = KS * KS;
    static constexpr int HR = KS + 1;
    static constexpr int PITCH = GSW_PX + KS - 1;
    static constexpr int CHUNK_BYTES = GSW_PX * KK * 4;
    static constexpr int HALO_BYTES = ((HR * CN * PITCH * 4 + 127) / 128) * 128;
    // two slots (store of row q drains while row q+1 is computed) unless that leaves fewer than three warps per SM
    static constexpr int SL = (GPS_SMEM / (2 * CHUNK_BYTES + HALO_BYTES) >= 3) ? 2 : 1;
    static constexpr int WARP_BYTES = SL * CHUNK_BYTES + HALO_BYTES;
    static constexpr int NW = (GPS_SMEM / WARP_BYTES < 16) ? GPS_SMEM / WARP_BYTES : 16;
    static constexpr int SMEM_BYTES = NW * WARP_BYTES;
};

template <int KS, int CN>
__global__ void __launch_bounds__(GradPsfStripCfg<KS, CN>::NW * 32, 1)
local_psf_grad_psf_strip_kernel(const float* __restrict__ img, const float* __restrict__ gout, float* __restrict__ dpsf,
                                int N, int H, int W) {
    using Cfg = GradPsfStripCfg<KS, CN>;
    constexpr int KK = Cfg::KK, R = (KS - 1) / 2, HR = Cfg::HR, PITCH = Cfg::PITCH, SL = Cfg::SL, NW = Cfg::NW;
    constexpr int C = CN;
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_chunk = reinterpret_cast<float*>(s_raw + warp * Cfg::WARP_BYTES);
    float* s_halo = reinterpret_cast<float*>(s_raw + warp * Cfg::WARP_BYTES + SL * Cfg::CHUNK_BYTES);
    const uint32_t halo_u32 = smem_u32(s_halo);

    const int nstrips = (W + GSW_PX - 1) / GSW_PX;
    const long long RT = (long long)N * nstrips * H;                    // strip rows in the launch
    const long long TW = (long long)gridDim.x * NW, gw = (long long)blockIdx.x * NW + warp;
    const long long q0 = RT * gw / TW, q1 = RT * (gw + 1) / TW;
    if (q0 >= q1) return;
    const int nq = (int)(q1 - q0);

    int y = (int)(q0 % H), s = (int)((q0 / H) % nstrips), n = (int)(q0 / ((long long)H * nstrips));
    auto issue_halo_row = [&](int r, int hslot) {                       // as the forward: image row clamp(r)
        const int gy = min(max(r, 0), H - 1);
#pragma unroll
        for (int c = 0; c < CN; ++c) {
            const float* src = img + ((long long)(n * C + c) * H + gy) * W;
            const uint32_t dst = halo_u32 + 4u * (uint32_t)((hslot * CN + c) * PITCH);
#pragma unroll
            for (int i0 = 0; i0 < PITCH; i0 += 32) {
                const int i = i0 + lane;
                if (i < PITCH) cp_async4(dst + 4u * i, src + min(max(GSW_PX * s - R + i, 0), W - 1));
            }
        }
    };

    bool fresh = true;
    int hs = 0;
    for (int it = 0; it < nq; ++it) {
        if (fresh) {
            cp_async_wait_group<0>();
#pragma unroll 1
            for (int d = 0; d < KS; ++d) issue_halo_row(y - R + d, d);
            cp_async_commit();
            issue_halo_row(y + R + 1, KS);
            cp_async_commit();
            hs = 0;
            fresh = false;
        }
        const int npx = min(GSW_PX, W - GSW_PX * s);
        const int col = 2 * lane;
        float2 g[CN];
        if (col < npx) {
#pragma unroll
            for (int c = 0; c < CN; ++c)
                g[c] = *reinterpret_cast<const float2*>(gout + ((long long)(n * C + c) * H + y) * W + GSW_PX * s + col);
        }
        const int slot = it % SL;
        if (it >= SL && lane == 0) bulk_wait_read<SL - 1>();           // the store that last used this slot has read it
        cp_async_wait_group<1>();                                       // halo rows y-R .. y+R (this lane's part)
        __syncwarp();

        if (col < npx) {
            float* run = s_chunk + slot * GSW_PX * KK + col * KK;       // flat run [2l ks^2, (2l+2) ks^2)
            float pend0 = 0.f, pend1 = 0.f, first1 = 0.f;               // pairs (e, e+1) of the run, e even
#pragma unroll
            for (int dy = 0; dy < KS; ++dy) {
                int hsl = hs + dy;
                hsl -= (hsl >= HR) ? HR : 0;
                const float2* hrow = reinterpret_cast<const float2*>(s_halo + hsl * CN * PITCH) + lane;
                float win[CN][KS + 1];
#pragma unroll
                for (int c = 0; c < CN; ++c)
#pragma unroll
                    for (int i = 0; i < (KS + 1) / 2; ++i) {
                        const float2 v = hrow[c * (PITCH / 2) + i];
                        win[c][2 * i] = v.x;
                        win[c][2 * i + 1] = v.y;
                    }
#pragma unroll
                for (int dx = 0; dx < KS; ++dx) {
                    float v0 = 0.f, v1 = 0.f;
#pragma unroll
                    for (int c = 0; c < CN; ++c) {
                        v0 = fmaf(g[c].x, win[c][dx], v0);
                        v1 = fmaf(g[c].y, win[c][dx + 1], v1);
                    }
                    const int e0 = dy * KS + dx, e1 = KK + e0;          // compile-time after unrolling
                    if (e0 & 1) *reinterpret_cast<float2*>(run + e0 - 1) = make_float2(pend0, v0);
                    else pend0 = v0;
                    if (e1 == KK) first1 = v1;                          // pairs with the last element of pixel 0
                    else if (e1 & 1) *reinterpret_cast<float2*>(run + e1 - 1) = make_float2(pend1, v1);
                    else pend1 = v1;
                }
            }
            *reinterpret_cast<float2*>(run + KK - 1) = make_float2(pend0, first1);
        }
        fence_proxy_async_smem();                                       // generic-proxy writes -> the bulk copy
        __syncwarp();                                                   // every lane is done with the chunk and row y-R
        if (lane == 0) {
            bulk_s2g(dpsf + ((long long)(n * H + y) * W + GSW_PX * s) * KK, smem_u32(s_chunk + slot * GSW_PX * KK),
                     (uint32_t)npx * (uint32_t)(KK * 4));
            bulk_commit();
        }
        if (++y == H) {
            y = 0;
            fresh = true;
            if (++s == nstrips) { s = 0; ++n; }
        } else {
            issue_halo_row(y + R + 1, hs);
            cp_async_commit();
            hs = (hs + 1 == HR) ? 0 : hs + 1;
        }
    }
    cp_async_wait_group<0>();
    if (lane == 0) bulk_wait_all();
}

// Generic dP: one thread per element of dP (coalesced writes), grid-stride.
__global__ void __launch_bounds__(256)
local_psf_grad_psf_kernel(const float* __restrict__ img, const float* __restrict__ gout, float* __restrict__ dpsf,
                          int N, int C, int H, int W, int ks) {
    const long long kk = (long long)ks * ks, HW = (long long)H * W;
    const long long total = (long long)N * HW * kk;
    const int r = (ks - 1) / 2;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long px = e / kk;
        const int t = (int)(e - px * kk);
        const int i = t / ks, j = t - i * ks;
        const long long n = px / HW;
        const int hw = (int)(px - n * HW);
        const int h = hw / W, w = hw - h * W;
        const long long src = (long long)min(max(h + i - r, 0), H - 1) * W + min(max(w + j - r, 0), W - 1);
        float acc = 0.f;
        for (int c = 0; c < C; ++c) {
            const long long plane = (n * C + c) * HW;
            acc = fmaf(__ldg(gout + plane + hw), __ldg(img + plane + src), acc);
        }
        dpsf[e] = acc;
    }
}

// Generic dimg: one thread per (n, y, x), up to GPS_MAXC channels per pass.  Along each axis the preimages of a target
// y are h = y + r - i for an interior y; the border rows also collect every tap the replicate pad clamped onto them
// (y = 0: h + i - r <= 0, y = H-1: h + i - r >= H-1).  With border != 0 it covers only the pixels of rows 0, H-1 and
// columns 0, W-1 (after the strip dimg kernel, which computes every pixel without those folds).
__device__ __forceinline__ int border_pixels(int H, int W) {
    return (H == 1 ? W : 2 * W) + (H > 2 ? (H - 2) * min(W, 2) : 0);
}
__global__ void __launch_bounds__(256)
local_psf_grad_img_kernel(const float* __restrict__ psf, const float* __restrict__ gout, float* __restrict__ dimg,
                          int N, int C, int H, int W, int ks, int c0, int cn, int border) {
    const long long kk = (long long)ks * ks, HW = (long long)H * W;
    const int per_image = border ? border_pixels(H, W) : H * W;
    const long long total = (long long)N * per_image;
    const int r = (ks - 1) / 2;
    for (long long px = (long long)blockIdx.x * blockDim.x + threadIdx.x; px < total; px += (long long)gridDim.x * blockDim.x) {
        const long long n = px / per_image;
        const int q = (int)(px - n * per_image);
        int y, x;
        if (!border) {
            y = q / W; x = q - y * W;
        } else if (q < W) {
            y = 0; x = q;
        } else if (H > 1 && q < 2 * W) {
            y = H - 1; x = q - W;
        } else {                                                       // columns 0 and W-1 of rows 1 .. H-2
            const int e = q - 2 * W, ncol = min(W, 2);
            y = 1 + e / ncol;
            x = (e % ncol) ? W - 1 : 0;
        }
        const int yx = y * W + x;
        float acc[GPS_MAXC] = {0.f, 0.f, 0.f, 0.f};
        const float* gp = gout + (n * C + c0) * HW;
        for (int i = 0; i < ks; ++i) {
            const int hlo = max(y == 0 ? 0 : y + r - i, 0), hhi = min(y == H - 1 ? H - 1 : y + r - i, H - 1);
            for (int h = hlo; h <= hhi; ++h) {
                for (int j = 0; j < ks; ++j) {
                    const int wlo = max(x == 0 ? 0 : x + r - j, 0), whi = min(x == W - 1 ? W - 1 : x + r - j, W - 1);
                    for (int w = wlo; w <= whi; ++w) {
                        const long long s = (long long)h * W + w;
                        const float p = __ldg(psf + (n * HW + s) * kk + i * ks + j);
#pragma unroll
                        for (int c = 0; c < GPS_MAXC; ++c)
                            if (c < cn) acc[c] = fmaf(__ldg(gp + c * HW + s), p, acc[c]);
                    }
                }
            }
        }
#pragma unroll
        for (int c = 0; c < GPS_MAXC; ++c)
            if (c < cn) dimg[(n * C + c0 + c) * HW + yx] = acc[c];
    }
}

// Strip dimg (3 <= ks <= 15, W % 4 == 0, 16-byte aligned psf): the transposed gather.  A warp owns the 64 target columns
// [x0, x0+64) of a strip and a contiguous run of its target rows [ya, yb]; it walks the SOURCE rows h in
// [ya-r, yb+r] (clipped to the image).  Per source row, lane 0 bulk-copies the PSFs of the columns
// [x0-CP, x0+64+CP) (CP = r rounded up to 4, so that the copy is 16-byte aligned; clipped to the image) -- one
// contiguous run of <= (64+2CP) ks^2 floats -- and all lanes cp.async the matching grad_out row.  Lane l owns the target
// columns x0+l and x0+l+32 and adds, for every tap row i, sum_j G[h][x+r-j] P[h][x+r-j][i][j] into the accumulator of
// target row h+i-r: ks registers per column and channel, shifted down one row per source row.  Lane stride in the
// chunk is ks^2 floats (odd): conflict-free.  The accumulator of row h-r is complete after source h and is written once
// if it is in [ya, yb]; a warp whose run starts mid-strip replays the 2r source rows before ya, so every target row is
// written by exactly one warp, as one fixed-order sum.  Source columns / rows outside the image contribute zero (their
// G is zeroed), so this computes every target without the replicate-border folds; local_psf_grad_img_kernel with
// border = 1 then rewrites rows 0, H-1 and columns 0, W-1.
template <int KS, int CN>
struct GradImgStripCfg {
    static constexpr int KK = KS * KS, R = (KS - 1) / 2;
    static constexpr int CP = (R + 3) & ~3;
    static constexpr int CW = GSW_PX + 2 * CP;                          // chunk columns
    static constexpr int CHUNK_BYTES = CW * KK * 4;                     // multiple of 16
    static constexpr int G_BYTES = ((CN * CW * 4 + 127) / 128) * 128;
    static constexpr int SL = (GPS_SMEM / (2 * (CHUNK_BYTES + G_BYTES) + 16) >= 3) ? 2 : 1;
    static constexpr int WARP_BYTES = SL * (CHUNK_BYTES + G_BYTES);
    static constexpr int NW_ = (GPS_SMEM - 16 * 16) / WARP_BYTES;
    static constexpr int NW = NW_ < 16 ? NW_ : 16;
    static constexpr int SMEM_BYTES = NW * WARP_BYTES + NW * SL * 8;
};

template <int KS, int CN>
__global__ void __launch_bounds__(GradImgStripCfg<KS, CN>::NW * 32, 1)
local_psf_grad_img_strip_kernel(const float* __restrict__ psf, const float* __restrict__ gout, float* __restrict__ dimg,
                                int N, int C, int H, int W, int c0) {
    using Cfg = GradImgStripCfg<KS, CN>;
    constexpr int KK = Cfg::KK, R = Cfg::R, CP = Cfg::CP, CW = Cfg::CW, SL = Cfg::SL, NW = Cfg::NW;
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* s_p = reinterpret_cast<float*>(s_raw + warp * Cfg::WARP_BYTES);                       // [SL][CW][KK]
    float* s_g = reinterpret_cast<float*>(s_raw + warp * Cfg::WARP_BYTES + SL * Cfg::CHUNK_BYTES); // [SL][CN][CW]
    const uint32_t bar0 = smem_u32(s_raw + NW * Cfg::WARP_BYTES) + 8u * (uint32_t)(warp * SL);
    constexpr int GSL = Cfg::G_BYTES / 4;                              // floats per G slot

    const int nstrips = (W + GSW_PX - 1) / GSW_PX;
    const long long RT = (long long)N * nstrips * H;
    const long long TW = (long long)gridDim.x * NW, gw = (long long)blockIdx.x * NW + warp;
    const long long q0 = RT * gw / TW, q1 = RT * (gw + 1) / TW;
    if (q0 >= q1) return;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < SL; ++s) mbar_init(bar0 + 8u * s, 1);
        fence_mbar_init();
    }
    __syncwarp();

    int ip = 0, it = 0;                                                // chunks issued / consumed by this warp
    for (long long q = q0; q < q1;) {
        const int ya = (int)(q % H), s = (int)((q / H) % nstrips), n = (int)(q / ((long long)H * nstrips));
        const int yb = (int)min((long long)H - 1, ya + (q1 - q) - 1);
        q += yb - ya + 1;
        const int x0 = GSW_PX * s;
        const int wlo = max(0, x0 - CP), whi = min(W, x0 + GSW_PX + CP);       // multiples of 4
        const int mlo = wlo - (x0 - CP), mhi = whi - (x0 - CP);
        const int hs0 = max(0, ya - R), he = min(H - 1, yb + R), nsrc = he - hs0 + 1;
        if (mlo > 0 || mhi < CW) {                                     // image edge: columns never copied read as 0
            for (int sl = 0; sl < SL; ++sl) {
                for (int m = 0; m < CW; ++m) {
                    if (m >= mlo && m < mhi) continue;
                    for (int e = lane; e < KK; e += 32) s_p[(sl * CW + m) * KK + e] = 0.f;
                    if (lane < CN) s_g[sl * GSL + lane * CW + m] = 0.f;
                }
            }
            __syncwarp();
        }
        auto issue = [&](int k) {                                      // source row hs0 + k; one cp.async group always
            if (k < nsrc) {
                const int h = hs0 + k, slot = ip % SL;
                if (lane == 0) {
                    const uint32_t bytes = (uint32_t)(whi - wlo) * (uint32_t)(KK * 4);
                    mbar_arrive_expect_tx(bar0 + 8u * slot, bytes);
                    bulk_g2s(smem_u32(s_p + (slot * CW + mlo) * KK), psf + ((long long)(n * H + h) * W + wlo) * KK,
                             bytes, bar0 + 8u * slot);
                }
                const uint32_t gdst = smem_u32(s_g + slot * GSL);
#pragma unroll
                for (int c = 0; c < CN; ++c) {
                    const float* src = gout + ((long long)(n * C + c0 + c) * H + h) * W + (x0 - CP);
                    for (int m = mlo + lane; m < mhi; m += 32) cp_async4(gdst + 4u * (uint32_t)(c * CW + m), src + m);
                }
                ++ip;
            }
            cp_async_commit();
        };
#pragma unroll
        for (int k = 0; k < SL; ++k) issue(k);

        float acc[KS][2][CN];
#pragma unroll
        for (int i = 0; i < KS; ++i)
#pragma unroll
            for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int c = 0; c < CN; ++c) acc[i][p][c] = 0.f;
        auto store = [&](int v, const float (&a)[2][CN]) {
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                const int x = x0 + lane + 32 * p;
                if (x < W) {
#pragma unroll
                    for (int c = 0; c < CN; ++c) dimg[((long long)(n * C + c0 + c) * H + v) * W + x] = a[p][c];
                }
            }
        };
#pragma unroll 1
        for (int k = 0; k < nsrc; ++k) {
            const int slot = it % SL;
            cp_async_wait_group<SL - 1>();                             // this lane's part of grad_out row k
            mbar_wait(bar0 + 8u * slot, (uint32_t)((it / SL) & 1));
            __syncwarp();                                              // ... every lane's part
            const float* P = s_p + slot * CW * KK;
            const float* G = s_g + slot * GSL;
#pragma unroll
            for (int j = 0; j < KS; ++j) {
                float g[2][CN];
                int m[2];
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    m[p] = lane + 32 * p + CP + R - j;                 // source column x + r - j, chunk-relative
#pragma unroll
                    for (int c = 0; c < CN; ++c) g[p][c] = G[c * CW + m[p]];
                }
#pragma unroll
                for (int i = 0; i < KS; ++i)
#pragma unroll
                    for (int p = 0; p < 2; ++p) {
                        const float t = P[m[p] * KK + i * KS + j];
#pragma unroll
                        for (int c = 0; c < CN; ++c) acc[i][p][c] = fmaf(g[p][c], t, acc[i][p][c]);
                    }
            }
            const int v = hs0 + k - R;                                 // target row complete after this source row
            if (v >= ya && v <= yb) store(v, acc[0]);
#pragma unroll
            for (int i = 0; i < KS - 1; ++i)
#pragma unroll
                for (int p = 0; p < 2; ++p)
#pragma unroll
                    for (int c = 0; c < CN; ++c) acc[i][p][c] = acc[i + 1][p][c];
#pragma unroll
            for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int c = 0; c < CN; ++c) acc[KS - 1][p][c] = 0.f;
            ++it;
            __syncwarp();                                              // every lane is done with this slot
            issue(k + SL);
        }
        // rows whose remaining sources lie below the image: slot i holds target row he + 1 - r + i
#pragma unroll
        for (int i = 0; i < KS - 1; ++i) {
            const int v = he + 1 - R + i;
            if (v >= ya && v <= yb) store(v, acc[i]);
        }
    }
    cp_async_wait_group<0>();
}

}  // namespace aadff
