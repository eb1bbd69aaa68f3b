// Backward of the focal-stack render (aadff_render_stack_backward_f32): gradients of
//   out[n,c,s,h,w] = sum_{i,j} img[n,c,clamp(h+i-r),clamp(w+j-r)] * P[n,s,h,w,i,j],
//   P = MLP(x_w, y_h, depth2z(depth[n,h,w]), depth2z(foc[n,s]))
// for the image, the depth map, the focus distances and the MLP's weights and biases, given an arbitrary upstream
// gradient G in the forward's (n, c, s, h, w) element strides.
//
// The work runs in bands of whole image rows of one (image, slice), in (n, s, band) order; a band holds at most
// MG_CHUNK pixels, so the workspace is bounded whatever N*S*H*W is.  Per band:
//   1. rg_probe_kernel writes the band's (x, y, z, foc_z) probes with the forward's own coord_x / coord_y / depth_to_z;
//   2. (dimg) the PSFs of the band in the forward's mode (aadff_psfnet_pred_tc_f32), then rg_grad_img_band_kernel adds
//      every (source pixel of the band, tap) pair into the target pixel it lands on, replicate-border folds included;
//   3. (ddepth, dfoc, dW, db) mlp_fp32_store_kernel recomputes the band in fp32, rg_head_kernel forms dP from the image
//      taps and G and turns it into dZ of the head (dP never reaches HBM), the MLP backward chain of
//      mlp_grad_kernel.cuh runs down to dX, and rg_depth_focus_kernel turns dX columns 2 and 3 into ddepth and dfoc.
// Every output element has one writer per band and the bands are added in a fixed order: no atomics, two calls are
// bit-identical.
#pragma once
#include <cuda_runtime.h>
#include "render_args.h"
#include "train_kernels.cuh"

namespace aadff {

// probes [rows * W][4] of rows [b0, b0 + rows) of image n, slice s: the values the forward kernels compute
__global__ void __launch_bounds__(256)
rg_probe_kernel(const float* __restrict__ depth, const float* __restrict__ foc, int n, int s, int S, int H, int W,
                int b0, int valid, float d_min, float d_range, float step_x, float step_y, float* __restrict__ probes) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= valid) return;
    const int h = b0 + p / W, w = p % W;
    float4 o;
    o.x = coord_x(w, W, step_x);
    o.y = coord_y(h, H, step_y);
    o.z = depth_to_z(__ldg(depth + ((long long)n * H + h) * W + w), d_min, d_range);
    o.w = depth_to_z(__ldg(foc + (long long)n * S + s), d_min, d_range);
    reinterpret_cast<float4*>(probes)[p] = o;
}

// The transposed gather of one band: dimg[n,c,y,x] += sum over the sources (h, w) of rows [b0, b1) and taps (i, j)
// with clamp(h+i-r) = y, clamp(w+j-r) = x of G[n,c,s,h,w] * P[(h-b0) W + w][i ks + j], one thread per target pixel of
// rows [max(0, b0-r), min(H, b1+r)).  Along each axis the sources of an interior target y are h = y + r - i; the border
// rows also collect every tap the replicate pad clamped onto them (as local_psf_grad_img_kernel).  Every (source, tap)
// pair belongs to exactly one band, so the bands need no halo.  All channels in one launch, four per pass.
__global__ void __launch_bounds__(256)
rg_grad_img_band_kernel(const float* __restrict__ psf, const float* __restrict__ gout, long long os_n, long long os_c,
                        long long os_s, long long os_h, long long os_w, float* __restrict__ dimg, int n, int s, int C,
                        int H, int W, int ks, int b0, int b1) {
    const int r = (ks - 1) / 2, kk = ks * ks;
    const int y0 = max(0, b0 - r), y1 = min(H, b1 + r);
    const long long npx = (long long)(y1 - y0) * W;
    const long long HW = (long long)H * W;
    const float* gb = gout + n * os_n + s * os_s;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < npx; q += (long long)gridDim.x * blockDim.x) {
        const int y = y0 + (int)(q / W), x = (int)(q % W);
        for (int c0 = 0; c0 < C; c0 += 4) {
            const int cn = min(4, C - c0);
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int i = 0; i < ks; ++i) {
                const int hlo = max(y == 0 ? 0 : y + r - i, b0), hhi = min(y == H - 1 ? H - 1 : y + r - i, b1 - 1);
                for (int h = hlo; h <= hhi; ++h) {
                    for (int j = 0; j < ks; ++j) {
                        const int wlo = max(x == 0 ? 0 : x + r - j, 0), whi = min(x == W - 1 ? W - 1 : x + r - j, W - 1);
                        for (int w = wlo; w <= whi; ++w) {
                            const float p = __ldg(psf + ((long long)(h - b0) * W + w) * kk + i * ks + j);
                            const float* g = gb + h * os_h + w * os_w;
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                if (c < cn) acc[c] = fmaf(__ldg(g + (c0 + c) * os_c), p, acc[c]);
                        }
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < cn) dimg[((long long)n * C + c0 + c) * HW + (long long)y * W + x] += acc[c];
        }
    }
}

// dP[t] = sum_c G[n,c,s,h,w] img[n,c,clamp(h+i-r),clamp(w+j-r)] of tap t = i ks + j of pixel (h, w), channels in order
__device__ __forceinline__ float rg_dpsf(const float* __restrict__ img, const float* __restrict__ g, long long os_c,
                                         long long plane, int C, int H, int W, int h, int w, int ks, int t) {
    const int r = (ks - 1) / 2, i = t / ks, j = t - i * ks;
    const long long src = (long long)min(max(h + i - r, 0), H - 1) * W + min(max(w + j - r, 0), W - 1);
    float acc = 0.f;
    for (int c = 0; c < C; ++c) acc = fmaf(__ldg(g + c * os_c), __ldg(img + c * plane + src), acc);
    return acc;
}

// dZ of the head for the pixels of one band, one warp per pixel: dP from the image taps and G (rg_dpsf), then the
// formula of mlp_head_backward_kernel (head_dz) with s and S from mlp_fp32_store_kernel.  Rows past `valid` get dZ = 0.
__global__ void __launch_bounds__(256)
rg_head_kernel(const float* __restrict__ s_buf, int lds, const float* __restrict__ ssum, const float* __restrict__ img,
               const float* __restrict__ gout, long long os_n, long long os_c, long long os_s, long long os_h,
               long long os_w, int n, int s, int C, int H, int W, int ks, int b0, int valid, int cp,
               float* __restrict__ dz, int ldz) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= cp) return;
    float* dr = dz + (size_t)warp * ldz;
    if (warp >= valid) {
        for (int j = lane; j < ldz; j += 32) dr[j] = 0.f;
        return;
    }
    const int kk = ks * ks, h = b0 + warp / W, w = warp % W;
    const long long plane = (long long)H * W;
    const float* im = img + (long long)n * C * plane;
    const float* g = gout + n * os_n + s * os_s + h * os_h + w * os_w;
    const float* sr = s_buf + (size_t)warp * lds;
    const float S = ssum[warp];
    const float denom = fmaxf(S, 1e-12f);
    float gp = 0.f;
    for (int t = lane; t < kk; t += 32) gp = fmaf(rg_dpsf(im, g, os_c, plane, C, H, W, h, w, ks, t), sr[t] / denom, gp);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gp += __shfl_xor_sync(0xffffffffu, gp, o);
    for (int t = lane; t < ldz; t += 32)
        dr[t] = t < kk ? head_dz(sr[t], rg_dpsf(im, g, os_c, plane, C, H, W, h, w, ks, t), gp, S, denom) : 0.f;
}

constexpr int RG_DF_NT = 1024;

// d depth2z(d) / dd = 1 / d_range where 0 <= (d - d_min) / d_range <= 1 (torch.clamp passes the gradient on both
// bounds), 0 elsewhere -- NaN, invalid (0) and out-of-range depths included
__device__ __forceinline__ bool rg_z_inside(float d, float d_min, float d_range) {
    const float z = __fdiv_rn(d - d_min, d_range);
    return z >= 0.f && z <= 1.f;
}

// dX [valid][4] of one band -> ddepth (written by slice 0, added by later slices) and dfoc.  dfoc[n,s] accumulates the
// raw sum of dX[., 3] over the bands of (n, s), each band's sum a fixed-order tree; the last band scales it by the
// clamp rule of foc[n,s].  One block per band.
__global__ void __launch_bounds__(RG_DF_NT)
rg_depth_focus_kernel(const float* __restrict__ dx, const float* __restrict__ depth, const float* __restrict__ foc,
                      float* __restrict__ grad_depth, float* __restrict__ grad_foc, int n, int s, int S, int H, int W,
                      int b0, int valid, float d_min, float d_range, int first_band, int last_band) {
    __shared__ float red[RG_DF_NT];
    const int t = threadIdx.x;
    const long long base = ((long long)n * H + b0) * W;
    float acc = 0.f;
    for (int p = t; p < valid; p += RG_DF_NT) {
        if (grad_depth) {
            const float gd = rg_z_inside(__ldg(depth + base + p), d_min, d_range) ? __fdiv_rn(dx[p * 4 + 2], d_range) : 0.f;
            grad_depth[base + p] = s == 0 ? gd : grad_depth[base + p] + gd;
        }
        acc += dx[p * 4 + 3];
    }
    if (!grad_foc) return;
    red[t] = acc;
    __syncthreads();
    for (int o = RG_DF_NT / 2; o > 0; o >>= 1) {
        if (t < o) red[t] += red[t + o];
        __syncthreads();
    }
    if (t == 0) {
        float* gf = grad_foc + (long long)n * S + s;
        float v = first_band ? red[0] : *gf + red[0];
        if (last_band) v = rg_z_inside(__ldg(foc + (long long)n * S + s), d_min, d_range) ? __fdiv_rn(v, d_range) : 0.f;
        *gf = v;
    }
}

}  // namespace aadff
