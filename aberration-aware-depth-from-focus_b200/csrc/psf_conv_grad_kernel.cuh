// Backward of the PSF-map convolution (psf_conv_kernel.cuh: render_psf / render_psf_map).  With G = grad_out,
// K = the PSF of a cell, p = (ks-1)/2 and refl() the reflect pad of the forward:
//
//   dimg[b,c,y,x]           = sum over (h,i) with refl(h+i-p) = y, (w,j) with refl(w+j-p) = x, (h,w) inside a cell,
//                             of G[b,c,h,w] * K[c][cell(h,w)][ks-1-i][ks-1-j]
//   dK[c][cell][ks-1-i][ks-1-j] = sum_b sum_{(h,w) in cell} G[b,c,h,w] * img[b,c,refl(h+i-p),refl(w+j-p)]
//
// Every element is one fixed-order sum in one thread or one warp (no atomics): two runs give bit-identical gradients.
//
// psf_conv_grad_img_kernel: one thread per image pixel.  Along each axis a padded position u in [-p, n-1+p] reflects to
// y when u = y, u = -y (1 <= y <= p) or u = 2(n-1) - y (n-1-p <= y <= n-2); each preimage u has the sources
// h = u + p - i.  The cell of each source row / column of the CTA's 32 x 64 tile comes from a table in shared memory.
// psf_conv_grad_psf_kernel (stage 1): one CTA per (image, channel, cell, 32 x 64 tile) as the forward's tiling; the
// ks^2 correlation of the gradient tile with the reflect-padded image tile is split over (row group, tap row i,
// 8-column group) threads, each sliding a register window as the forward does, then summed in a fixed order into one
// ks^2 partial per tile of the caller's workspace.  psf_conv_grad_reduce_kernel (stage 2): one warp per PSF element
// sums that element's partials over all images and tiles of its cell.
#pragma once
#include <cuda_runtime.h>
#include "psf_conv_kernel.cuh"

namespace aadff {

constexpr int PCG_TH = 32, PCG_TW = 64;          // image tile of the dimg kernel

__device__ __forceinline__ int cell_of(int v, const int* bounds, int grid) {     // -1: beyond the last bound
    if (v < bounds[0] || v >= bounds[grid]) return -1;
    int g = 0;
    while (v >= bounds[g + 1]) ++g;
    return g;
}

__global__ void __launch_bounds__(PC_NT) psf_conv_grad_img_kernel(const PsfConvArgs a, const float* __restrict__ gout,
                                                                  float* __restrict__ dimg, int ks) {
    const int p = (ks - 1) / 2;
    __shared__ int s_rc[PCG_TH + 31 - 1], s_cc[PCG_TW + 31 - 1];      // cell of source row / column (or -1)
    const int tiles_y = (a.H + PCG_TH - 1) / PCG_TH, tiles_x = (a.W + PCG_TW - 1) / PCG_TW;
    const long long per_plane = (long long)tiles_y * tiles_x;
    const long long n_tiles = per_plane * a.B * a.C;
    const int Kw = a.grid * ks;                                        // row pitch of the PSF map
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const long long bc = t / per_plane;
        const int rem = (int)(t % per_plane);
        const int y0 = (rem / tiles_x) * PCG_TH, x0 = (rem % tiles_x) * PCG_TW;
        const int c = (int)(bc % a.C);
        __syncthreads();                                               // previous tile done with the tables
        for (int e = threadIdx.x; e < PCG_TH + 2 * p; e += PC_NT) {
            const int h = y0 - p + e;
            s_rc[e] = (h >= 0 && h < a.H) ? cell_of(h, a.hb, a.grid) : -1;
        }
        for (int e = threadIdx.x; e < PCG_TW + 2 * p; e += PC_NT) {
            const int w = x0 - p + e;
            s_cc[e] = (w >= 0 && w < a.W) ? cell_of(w, a.wb, a.grid) : -1;
        }
        __syncthreads();
        const float* gp = gout + bc * a.H * a.W;
        const float* kp = a.psf_map + (long long)c * Kw * Kw;
        for (int q = threadIdx.x; q < PCG_TH * PCG_TW; q += PC_NT) {
            const int y = y0 + q / PCG_TW, x = x0 + q % PCG_TW;
            if (y >= a.H || x >= a.W) continue;
            int uy[3], ux[3], ny = 0, nx = 0;
            uy[ny++] = y;
            if (y >= 1 && y <= p) uy[ny++] = -y;
            if (y <= a.H - 2 && y >= a.H - 1 - p) uy[ny++] = 2 * (a.H - 1) - y;
            ux[nx++] = x;
            if (x >= 1 && x <= p) ux[nx++] = -x;
            if (x <= a.W - 2 && x >= a.W - 1 - p) ux[nx++] = 2 * (a.W - 1) - x;
            float acc = 0.f;
            for (int ay = 0; ay < ny; ++ay)
                for (int i = 0; i < ks; ++i) {
                    const int h = uy[ay] + p - i;
                    if (h < 0 || h >= a.H) continue;
                    const int gi = s_rc[h - (y0 - p)];
                    if (gi < 0) continue;
                    const float* grow = gp + (long long)h * a.W;
                    const float* krow = kp + (long long)(gi * ks + ks - 1 - i) * Kw + ks - 1;
                    for (int ax = 0; ax < nx; ++ax)
                        for (int j = 0; j < ks; ++j) {
                            const int w = ux[ax] + p - j;
                            if (w < 0 || w >= a.W) continue;
                            const int gj = s_cc[w - (x0 - p)];
                            if (gj < 0) continue;
                            acc = fmaf(__ldg(grow + w), __ldg(krow + gj * ks - j), acc);
                        }
                }
            dimg[bc * a.H * a.W + (long long)y * a.W + x] = acc;
        }
    }
}

template <int KS>
struct PsfConvGradCfg {
    static constexpr int HH = PC_TILE_H + KS - 1, HW = PC_TILE_W + KS - 1, PITCH = HW | 1;
    static constexpr int WG = PC_TILE_W / PC_PX;                        // 8-column groups
    static constexpr int NG = (PC_NT / (WG * KS)) > 0 ? PC_NT / (WG * KS) : 1;     // row groups
    static constexpr int TILE_FLOATS = HH * PITCH + PC_TILE_H * PC_TILE_W;
    static constexpr int PART_FLOATS = NG * WG * KS * KS;
    static constexpr int SMEM_FLOATS = TILE_FLOATS > PART_FLOATS ? TILE_FLOATS : PART_FLOATS;
};

// work[((c * grid^2 + cell) * B + b) * tiles_per_cell + tile][ks^2], tap order (i, j) of the forward's flipped PSF
template <int KS>
__global__ void __launch_bounds__(PC_NT) psf_conv_grad_psf_kernel(const PsfConvArgs a, const float* __restrict__ gout,
                                                                  float* __restrict__ work) {
    using Cfg = PsfConvGradCfg<KS>;
    constexpr int P = (KS - 1) / 2, KK = KS * KS, HW = Cfg::HW, PITCH = Cfg::PITCH, WG = Cfg::WG, NG = Cfg::NG;
    __shared__ float s_buf[Cfg::SMEM_FLOATS];
    float* s_img = s_buf;
    float* s_g = s_buf + Cfg::HH * PITCH;
    float* s_part = s_buf;                                             // reused after the correlation
    const int tiles_y = (a.max_ch + PC_TILE_H - 1) / PC_TILE_H, tiles_x = (a.max_cw + PC_TILE_W - 1) / PC_TILE_W;
    const int tpc = tiles_y * tiles_x;
    const int G2 = a.grid * a.grid;
    const long long n_tiles = (long long)a.C * G2 * a.B * tpc;
    const int wg = threadIdx.x % WG, ti = (threadIdx.x / WG) % KS, hg = threadIdx.x / (WG * KS);
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int tile = (int)(t % tpc);
        const int b = (int)((t / tpc) % a.B);
        const int cell = (int)((t / ((long long)tpc * a.B)) % G2);
        const int c = (int)(t / ((long long)tpc * a.B * G2));
        const int gi = cell / a.grid, gj = cell % a.grid;
        const int h_lo = a.hb[gi], h_hi = a.hb[gi + 1], w_lo = a.wb[gj], w_hi = a.wb[gj + 1];
        const int h0 = h_lo + (tile / tiles_x) * PC_TILE_H, w0 = w_lo + (tile % tiles_x) * PC_TILE_W;
        const bool live = h0 < h_hi && w0 < w_hi;                      // this cell may be smaller than the largest
        const long long bc = (long long)b * a.C + c;
        __syncthreads();                                               // previous tile done with smem
        if (live) {
            const float* plane = a.img + bc * a.H * a.W;
            for (int i = threadIdx.x; i < Cfg::HH * HW; i += PC_NT) {
                const int yy = i / HW, xx = i - yy * HW;
                s_img[yy * PITCH + xx] = __ldg(plane + (long long)reflect_index(h0 + yy - P, a.H) * a.W +
                                               reflect_index(w0 + xx - P, a.W));
            }
            const float* gp = gout + bc * a.H * a.W;
            for (int i = threadIdx.x; i < PC_TILE_H * PC_TILE_W; i += PC_NT) {
                const int h = h0 + i / PC_TILE_W, w = w0 + i % PC_TILE_W;
                s_g[i] = (h < h_hi && w < w_hi) ? __ldg(gp + (long long)h * a.W + w) : 0.f;
            }
        }
        __syncthreads();
        float acc[KS];
#pragma unroll
        for (int j = 0; j < KS; ++j) acc[j] = 0.f;
        if (live && hg < NG) {
#pragma unroll 1
            for (int h = hg; h < PC_TILE_H; h += NG) {
                float g[PC_PX], v[PC_PX + KS - 1];
#pragma unroll
                for (int q = 0; q < PC_PX; ++q) g[q] = s_g[h * PC_TILE_W + wg * PC_PX + q];
#pragma unroll
                for (int u = 0; u < PC_PX + KS - 1; ++u) v[u] = s_img[(h + ti) * PITCH + wg * PC_PX + u];
#pragma unroll
                for (int j = 0; j < KS; ++j)
#pragma unroll
                    for (int q = 0; q < PC_PX; ++q) acc[j] = fmaf(g[q], v[q + j], acc[j]);
            }
        }
        __syncthreads();                                               // the tile buffers become s_part
        if (hg < NG) {
#pragma unroll
            for (int j = 0; j < KS; ++j) s_part[(hg * WG + wg) * KK + ti * KS + j] = acc[j];
        }
        __syncthreads();
        float* wout = work + t * KK;
        for (int e = threadIdx.x; e < KK; e += PC_NT) {
            float s = 0.f;
            for (int g = 0; g < NG * WG; ++g) s += s_part[g * KK + e];
            wout[e] = s;
        }
    }
}

// grad_psf_map[c][gi*ks + ks-1-i][gj*ks + ks-1-j] = sum over the cell's B * tpc partials of tap (i, j); one warp each
__global__ void __launch_bounds__(256) psf_conv_grad_reduce_kernel(const float* __restrict__ work, float* __restrict__ dpsf,
                                                                   int C, int grid, int ks, long long parts) {
    const int kk = ks * ks, G2 = grid * grid;
    const long long n_out = (long long)C * G2 * kk;
    const int lane = threadIdx.x & 31;
    for (long long o = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; o < n_out;
         o += ((long long)gridDim.x * blockDim.x) >> 5) {
        const int e = (int)(o % kk);
        const long long cc = o / kk;                                   // c * G2 + cell
        const float* src = work + cc * parts * kk + e;
        float s = 0.f;
        for (long long q = lane; q < parts; q += 32) s += __ldg(src + q * kk);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0) {
            const int c = (int)(cc / G2), cell = (int)(cc % G2), gi = cell / grid, gj = cell % grid;
            const int i = e / ks, j = e % ks;
            dpsf[((long long)c * grid * ks + gi * ks + (ks - 1 - i)) * (grid * ks) + gj * ks + (ks - 1 - j)] = s;
        }
    }
}

}  // namespace aadff
