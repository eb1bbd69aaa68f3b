// Device-side input preparation for the focal-stack simulator: what the reference's Dataset classes do on the CPU per
// sample after decoding the files (dff/dataset.py:43-52 Matterport3D, :190-205 Middlebury, :252-272 AutoAgument's
// colour jitter and flips):
//
//   aif   = ToTensor(cvtColor(img, BGR2RGB) / 255.)        uint8 [H,W,3] BGR  ->  float [3,h,w] RGB in [0,1]
//           (+ AutoAgument colour jitter  clip(0.5 + contrast*(x - 0.5) + brightness, 0, 1)  and horizontal/vertical flips)
//           Resize((h,w), antialias=True)                  torchvision / ATen _upsample_bilinear2d_aa: triangle filter
//                                                          whose support scales with the down-sampling factor
//   depth = ToTensor(depth_png / div)                      uint16 [H,W] -> float [1,h,w] metres  (div 4000 / 1000)
//           Resize(..., antialias=True)  (Matterport3D)  or  cv.resize(..., INTER_LINEAR)  (Middlebury)
//
// One thread per output pixel; the separable filter weights are evaluated on the fly (a 1280x1024 -> 640x480 resize
// touches 5 x 5 inputs per output).  HBM traffic: 5 B per input pixel + 16 B per output pixel.  The spline rotation of
// AutoAgument (scipy.ndimage.rotate, order 3) needs a global prefilter pass: spline_rotate_kernel.cuh produces rotated
// full-resolution fp32 planes, which this kernel resizes through its `fsrc` source.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace aadff {

struct PreprocessArgs {
    const uint8_t* bgr;       // [B,H,W,3] or null
    const uint16_t* depth;    // [B,H,W] or null
    float* aif_out;           // [B,3,h,w]
    float* depth_out;         // [B,1,h,w]
    const float* jitter;      // [B,2] (contrast, brightness), contrast < 0 = none; or null
    const uint8_t* flips;     // [B] bit 0: horizontal (np.flip axis 1), bit 1: vertical (axis 0); or null
    int B, H, W, h, w;
    float depth_div;
    // alternative source: fp32 planes [B,P,H,W] at full resolution (RGB planes first, then depth) that already carry
    // jitter / flips / rotation (spline_rotate_kernel.cuh); aif_out / depth_out say which outputs are wanted
    const float* fsrc;
    int fsrc_planes, fsrc_depth_plane;
};

// ATen's antialiased linear filter along one axis: window [lo, lo+n) of input samples and normalisation for output i
__device__ __forceinline__ void aa_window(int i, int in, int out, int& lo, int& n, float& center, float& invscale) {
    const float scale = (float)in / (float)out;
    const float support = scale >= 1.f ? scale : 1.f;
    invscale = scale >= 1.f ? 1.f / scale : 1.f;
    center = scale * ((float)i + 0.5f);
    lo = max(0, (int)(center - support + 0.5f));
    n = min(in, (int)(center + support + 0.5f)) - lo;
}
__device__ __forceinline__ float aa_weight(int j, int lo, float center, float invscale) {
    return fmaxf(0.f, 1.f - fabsf(((float)(j + lo) - center + 0.5f) * invscale));
}

constexpr int PP_MAXW = 12;      // filter taps per axis kept in registers (down-scaling factors up to ~5.5); beyond: recomputed

// grid = (chunks of output pixels, image): a block works on ONE image, so the whole per-value arithmetic of the image --
// /255 and the colour jitter, both evaluated in double like the reference's numpy code and then rounded to fp32 as its
// astype('float32') does -- is a 256-entry table in shared memory: per tap and channel one byte load, one LDS, one FFMA.
// FSRC: read the fp32 planes `fsrc` instead of the decoded uint8 / uint16 arrays.  CV2: resize the depth like
// cv2.resize INTER_LINEAR instead of the antialiased filter (a template parameter so that its double-precision
// coordinate arithmetic costs the antialias instantiation no registers)
template <bool FSRC, bool CV2>
__global__ void __launch_bounds__(256) preprocess_rgbd_kernel(const PreprocessArgs a) {
    __shared__ float lut[256];
    const int b = blockIdx.y;
    {
        double con = -1.0, bri = 0.0;
        if (a.jitter) { con = (double)a.jitter[2 * b]; bri = (double)a.jitter[2 * b + 1]; }
        double v = (double)threadIdx.x / 255.0;
        if (con >= 0.0) v = fmin(fmax(0.5 + con * (v - 0.5) + bri, 0.0), 1.0);
        lut[threadIdx.x] = (float)v;
    }
    __syncthreads();
    const long long total = (long long)a.h * a.w;
    for (long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (long long)gridDim.x * blockDim.x) {
        const int ox = (int)(id % a.w), oy = (int)(id / a.w);
        const int fl = (a.flips && !FSRC) ? a.flips[b] : 0;
        const bool flx = fl & 1, fly = fl & 2;
        const long long fplane = (long long)a.H * a.W;
        const float* fs = FSRC ? a.fsrc + (long long)b * a.fsrc_planes * fplane : nullptr;
        int ylo, yn, xlo, xn;
        float yc, yinv, xc, xinv;
        aa_window(oy, a.H, a.h, ylo, yn, yc, yinv);
        aa_window(ox, a.W, a.w, xlo, xn, xc, xinv);
        float wysum = 0.f, wxsum = 0.f;
        for (int j = 0; j < yn; ++j) wysum += aa_weight(j, ylo, yc, yinv);
        for (int j = 0; j < xn; ++j) wxsum += aa_weight(j, xlo, xc, xinv);
        // normalised column weights, evaluated once per output pixel (ATen divides every weight by the window's sum)
        float wxs[PP_MAXW];
#pragma unroll
        for (int j = 0; j < PP_MAXW; ++j) wxs[j] = (j < xn) ? aa_weight(j, xlo, xc, xinv) / wxsum : 0.f;
        auto wx_of = [&](int j) { return (xn <= PP_MAXW) ? wxs[j] : aa_weight(j, xlo, xc, xinv) / wxsum; };
        if (a.aif_out) {
            float acc[3] = {0.f, 0.f, 0.f};
            for (int jy = 0; jy < yn; ++jy) {
                const float wy = aa_weight(jy, ylo, yc, yinv) / wysum;
                const int sy = fly ? a.H - 1 - (ylo + jy) : ylo + jy;             // the flip precedes the resize
                const uint8_t* row = a.bgr + ((long long)b * a.H + sy) * a.W * 3;
                const float* frow = fs + (long long)sy * a.W;
                float racc[3] = {0.f, 0.f, 0.f};
                auto tap = [&](int jx, float wx) {
                    const int sx = flx ? a.W - 1 - (xlo + jx) : xlo + jx;
                    if (FSRC) {
#pragma unroll
                        for (int c = 0; c < 3; ++c) racc[c] = fmaf(wx, frow[c * fplane + sx], racc[c]);
                    } else {
                        const uint8_t* px = row + sx * 3;
#pragma unroll
                        for (int c = 0; c < 3; ++c) racc[c] = fmaf(wx, lut[px[2 - c]], racc[c]);   // BGR -> RGB, /255, jitter
                    }
                };
                if (xn <= PP_MAXW) {
#pragma unroll
                    for (int jx = 0; jx < PP_MAXW; ++jx)
                        if (jx < xn) tap(jx, wxs[jx]);
                } else {
                    for (int jx = 0; jx < xn; ++jx) tap(jx, wx_of(jx));
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[c] = fmaf(wy, racc[c], acc[c]);
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) a.aif_out[(((long long)b * 3 + c) * a.h + oy) * a.w + ox] = acc[c];
        }
        if (a.depth_out) {
            const uint16_t* dp = a.depth + (long long)b * a.H * a.W;
            const float* fd = fs + (long long)a.fsrc_depth_plane * fplane;
            auto at = [&](int sy, int sx) {
                if (FSRC) return fd[(long long)sy * a.W + sx];
                sy = fly ? a.H - 1 - sy : sy;
                sx = flx ? a.W - 1 - sx : sx;
                return (float)dp[(long long)sy * a.W + sx] / a.depth_div;
            };
            float v = 0.f;
            if (!CV2) {
                for (int jy = 0; jy < yn; ++jy) {
                    const float wy = aa_weight(jy, ylo, yc, yinv) / wysum;
                    float r = 0.f;
                    for (int jx = 0; jx < xn; ++jx) r = fmaf(wx_of(jx), at(ylo + jy, xlo + jx), r);
                    v = fmaf(wy, r, v);
                }
            } else {
                // cv2.resize INTER_LINEAR on float64 depth (Middlebury): source coordinate (dst + 0.5) * scale - 0.5, its
                // floor and its fraction in double as OpenCV computes them, clamped at the borders; only the fraction
                // is rounded to fp32.  An fp32 coordinate has steps of 2.4e-4 px at 2964 columns: millimetres of depth
                // across a hard depth edge.
                const double cy = ((double)oy + 0.5) * ((double)a.H / (double)a.h) - 0.5;
                const double cx = ((double)ox + 0.5) * ((double)a.W / (double)a.w) - 0.5;
                const double y0 = floor(cy), x0 = floor(cx);
                int sy = (int)y0, sx = (int)x0;
                float fy = (float)(cy - y0), fx = (float)(cx - x0);
                if (sy < 0) { sy = 0; fy = 0.f; }
                if (sy >= a.H - 1) { sy = a.H - 1; fy = 0.f; }
                if (sx < 0) { sx = 0; fx = 0.f; }
                if (sx >= a.W - 1) { sx = a.W - 1; fx = 0.f; }
                const int sy1 = min(sy + 1, a.H - 1), sx1 = min(sx + 1, a.W - 1);
                const float top = at(sy, sx) * (1.f - fx) + at(sy, sx1) * fx, bot = at(sy1, sx) * (1.f - fx) + at(sy1, sx1) * fx;
                v = top * (1.f - fy) + bot * fy;
            }
            a.depth_out[((long long)b * a.h + oy) * a.w + ox] = v;
        }
    }
}

}  // namespace aadff
