// Backward of the PSFNet MLP (aadff_psfnet_backward_f32): gradients of psf = MLP(inp) for the weights, the biases and
// the probes, given an arbitrary upstream gradient dL/dpsf [M, kk].  fp32 on CUDA cores.
//
// Nothing from the forward is kept.  The probes are processed in chunks of MG_CHUNK; per chunk
//   1. mlp_fp32_store_kernel recomputes the activations with mlp_fp32_kernel's arithmetic (the same f32_tile calls,
//      the same ReLU and sigmoid expressions, the same order of the L1 sum), so the ReLU masks and the sigmoid outputs
//      differentiated through are exactly those of the forward that produced psf;
//   2. mlp_head_backward_kernel: dZ of the head, one warp per probe (the formula of train_head_kernel, head_dz);
//   3. per layer, from the head down: dW_l = dZ_l^T A_l and db_l = colsum(dZ_l) as partial sums over slices of
//      MG_SLICE probes, then mlp_grad_reduce_kernel adds the slices in slice order to the running total of the earlier
//      chunks (every element has one writer and a fixed-order sum: no atomics, bit-reproducible);
//      dA_{l-1} = (dZ_l W_l) masked by A_l > 0, and for layer 0 dX = dZ_0 W_0.
// Activations and dZ are stored probe-major ([probe][feature]): the weight-gradient GEMM then reads both operands along
// their contiguous dimension, and only the dZ operand of dA has to be transposed on its way into shared memory.
#pragma once
#include <cuda_runtime.h>
#include "mlp_fp32_kernel.cuh"
#include "train_kernels.cuh"

namespace aadff {

constexpr int MG_CHUNK = 16384;   // probes per chunk (bounds the workspace whatever M is)
constexpr int MG_SLICE = 256;     // probes per partial sum of dW / db
constexpr int MG_BM = 128, MG_BN = 128, MG_BK = 16, MG_NT = 256;   // GEMM: 128 x 128 tile, 8 x 8 outputs per thread
constexpr int MG_APAD = 4;        // row padding of the transposed A tile (keeps float4 alignment)

struct MlpActs {
    float* act[MAX_LAYERS];   // act[l] = input of layer l, [cp][k[l]], l >= 1 (layer 0's input is the probes)
    float* s;                 // sigmoid outputs of the head, [cp][lds]
    float* ssum;              // the forward's L1 sum of s, [cp]
    int lds;
    int cp;                   // probes in this chunk, padded to a multiple of F32_TP
};

// mlp_fp32_kernel<false> for probes [m0, m0 + cp) (zeros past M), writing every layer's input and the head's sigmoid
// outputs and L1 sum instead of the normalised PSF.  The arithmetic is the forward's, operation for operation.
__global__ void __launch_bounds__(F32_NT, 1)
mlp_fp32_store_kernel(Fp32Net net, const float* __restrict__ probes, long long m0, long long M, MlpActs acts) {
    extern __shared__ __align__(16) float sm[];
    float* buf0 = sm;
    float* buf1 = sm + 256 * F32_TP;
    float* red = sm + 2 * 256 * F32_TP;
    float* wbuf = red + 4 * F32_TP * 5;
    const int t = threadIdx.x;
    const int fg = t >> 3, pg = t & 7;
    const int gp = t & 63, part = t >> 6;
    const int kk = net.kk;

    for (int base = blockIdx.x * F32_TP; base < acts.cp; base += gridDim.x * F32_TP) {
        if (t < F32_TP) {
            const long long id = m0 + base + t;
            float o[4] = {0.f, 0.f, 0.f, 0.f};
            if (id < M) {
#pragma unroll
                for (int c = 0; c < 4; ++c) o[c] = __ldg(probes + id * 4 + c);
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) buf0[c * F32_TP + t] = o[c];
        }
        __syncthreads();

        float* in = buf0;
        float* ob = buf1;
        for (int l = 0; l < net.n_layers - 1; ++l) {
            const int f0 = fg * 8;
            float acc[8][8];
            f32_tile(net.wt[l], net.bias[l], net.k[l], net.npad[l], 0, net.npad[l], f0, in, pg, wbuf, acc);
            if (f0 < net.npad[l]) {
#pragma unroll
                for (int a = 0; a < 8; ++a) {
#pragma unroll
                    for (int p = 0; p < 8; ++p) acc[a][p] = fmaxf(acc[a][p], 0.f);
                    *reinterpret_cast<float4*>(ob + (f0 + a) * F32_TP + pg * 4) =
                        make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
                    *reinterpret_cast<float4*>(ob + (f0 + a) * F32_TP + 32 + pg * 4) =
                        make_float4(acc[a][4], acc[a][5], acc[a][6], acc[a][7]);
                }
                float* dst = acts.act[l + 1];
                const int K = net.npad[l];
#pragma unroll
                for (int p = 0; p < 8; ++p) {
                    float* row = dst + (size_t)(base + (p < 4 ? pg * 4 + p : 32 + pg * 4 + p - 4)) * K + f0;
                    *reinterpret_cast<float4*>(row) = make_float4(acc[0][p], acc[1][p], acc[2][p], acc[3][p]);
                    *reinterpret_cast<float4*>(row + 4) = make_float4(acc[4][p], acc[5][p], acc[6][p], acc[7][p]);
                }
            }
            __syncthreads();
            float* tmp = in; in = ob; ob = tmp;
        }

        const int L = net.n_layers - 1;
        const int gid = base + gp;
        float ssum = 0.f;
        for (int nb = 0; nb < net.npad[L]; nb += 256) {
            const int f0 = nb + fg * 8;
            float acc[8][8];
            f32_tile(net.wt[L], net.bias[L], net.k[L], net.npad[L], nb, min(256, net.npad[L] - nb), fg * 8, in, pg, wbuf, acc);
            if (f0 < net.npad[L]) {
#pragma unroll
                for (int a = 0; a < 8; ++a) {
                    float v[8];
#pragma unroll
                    for (int p = 0; p < 8; ++p) v[p] = 1.0f / (1.0f + expf(-acc[a][p]));
                    *reinterpret_cast<float4*>(ob + (fg * 8 + a) * F32_TP + pg * 4) = make_float4(v[0], v[1], v[2], v[3]);
                    *reinterpret_cast<float4*>(ob + (fg * 8 + a) * F32_TP + 32 + pg * 4) =
                        make_float4(v[4], v[5], v[6], v[7]);
                }
            }
            __syncthreads();
            const int nt = min(256, kk - nb);
            for (int tl = part; tl < nt; tl += 4) {
                const float s = ob[tl * F32_TP + gp];
                ssum += s;
                acts.s[(size_t)gid * acts.lds + nb + tl] = s;
            }
            __syncthreads();
        }
        red[(part * F32_TP + gp) * 5] = ssum;
        __syncthreads();
        if (part == 0) {
            float tot = 0.f;
#pragma unroll
            for (int q = 0; q < 4; ++q) tot += red[(q * F32_TP + gp) * 5];
            acts.ssum[gid] = tot;
        }
        __syncthreads();
    }
}

// dL/dz of the head for p = s / max(S, 1e-12): one warp per probe of the chunk (rows past `valid` get dZ = 0, so they
// add nothing to any gradient).  g = dL/dp is the caller's [M, kk], rows m0 ... ; dz is [cp][ldz], its padding columns
// zeroed.
__global__ void __launch_bounds__(256)
mlp_head_backward_kernel(const float* __restrict__ s_buf, int lds, const float* __restrict__ ssum,
                         const float* __restrict__ g, long long m0, int valid, int cp, int kk, float* __restrict__ dz,
                         int ldz) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= cp) return;
    float* dr = dz + (size_t)warp * ldz;
    if (warp >= valid) {
        for (int j = lane; j < ldz; j += 32) dr[j] = 0.f;
        return;
    }
    const float* sr = s_buf + (size_t)warp * lds;
    const float* gr = g + (m0 + warp) * kk;
    const float S = ssum[warp];
    const float denom = fmaxf(S, 1e-12f);
    float gp = 0.f;
    for (int j = lane; j < kk; j += 32) gp = fmaf(__ldg(gr + j), sr[j] / denom, gp);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gp += __shfl_xor_sync(0xffffffffu, gp, o);
    for (int j = lane; j < ldz; j += 32) dr[j] = j < kk ? head_dz(sr[j], __ldg(gr + j), gp, S, denom) : 0.f;
}

__device__ __forceinline__ void mg_cp_async16(uint32_t dst, const void* src, bool valid) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0) : "memory");
}

enum MgEpilogue { MG_PLAIN = 0, MG_RELU_MASK = 1 };

// C(i, j) = sum_{k < K} A(i, k) B(k, j) for i < M, j < N; fp32, 8 x 8 outputs per thread, operand tiles of MG_BK
// k-rows double-buffered in shared memory.
//   A: A_T ? A[i * lda + k] (k contiguous: dZ as the left operand of dA, transposed through registers)
//          : A[k * lda + i] (i contiguous: dZ^T of dW, streamed with cp.async)
//   B: B[k * ldb + j], streamed with cp.async.
// lda (when !A_T), ldb and ldc are multiples of 4, rows of 16-byte-aligned operands hold at least round4(M) / round4(N)
// floats.  Past K and past M / N the operand tiles are zero-filled.
//   MG_PLAIN:     C[i * ldc + j] = acc
//   MG_RELU_MASK: C[i * ldc + j] = mask[i * ldc + j] > 0 ? acc : 0   (backward through the ReLU whose output is mask)
// blockIdx.z = probe slice (the dW partial sums): A and B advance by z * slice_k k-rows, C by z * c_slice, K is cut to
// the slice.
template <bool A_T, int EPI>
__global__ void __launch_bounds__(MG_NT, 2)
mlp_grad_gemm_kernel(const float* __restrict__ A, long long lda, const float* __restrict__ B, long long ldb,
                     float* __restrict__ C, long long ldc, int M, int N, int K, int slice_k, long long c_slice,
                     const float* __restrict__ mask) {
    __shared__ __align__(16) float As[2][MG_BK][MG_BM + MG_APAD];
    __shared__ __align__(16) float Bs[2][MG_BK][MG_BN];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int i0 = blockIdx.y * MG_BM, j0 = blockIdx.x * MG_BN;
    if (slice_k > 0) {
        const int z = blockIdx.z;
        A += A_T ? (long long)z * slice_k : (long long)z * slice_k * lda;
        B += (long long)z * slice_k * ldb;
        C += z * c_slice;
        K = min(slice_k, K - z * slice_k);
    }
    float acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
    const int nkt = (K + MG_BK - 1) / MG_BK;
    float4 ra[2];                                                 // A_T: the next A tile, on its way through registers
    auto issue = [&](int kt, int buf) {
        const int k0 = kt * MG_BK;
#pragma unroll
        for (int r = 0; r < 2; ++r) {                             // B: 16 rows x 32 float4
            const int e = t + r * MG_NT, kr = e >> 5, c4 = e & 31;
            const bool ok = k0 + kr < K && j0 + c4 * 4 < N;
            mg_cp_async16(smem_u32(&Bs[buf][kr][c4 * 4]), ok ? B + (long long)(k0 + kr) * ldb + j0 + c4 * 4 : B, ok);
        }
        if (!A_T) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int e = t + r * MG_NT, kr = e >> 5, c4 = e & 31;
                const bool ok = k0 + kr < K && i0 + c4 * 4 < M;
                mg_cp_async16(smem_u32(&As[buf][kr][c4 * 4]), ok ? A + (long long)(k0 + kr) * lda + i0 + c4 * 4 : A, ok);
            }
        } else {
#pragma unroll
            for (int r = 0; r < 2; ++r) {                         // 128 rows x 4 float4 along k
                const int e = t + r * MG_NT, row = e >> 2, kq = (e & 3) * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (i0 + row < M && k0 + kq < K) {
                    v = __ldg(reinterpret_cast<const float4*>(A + (long long)(i0 + row) * lda + k0 + kq));
                    if (k0 + kq + 1 >= K) v.y = 0.f;
                    if (k0 + kq + 2 >= K) v.z = 0.f;
                    if (k0 + kq + 3 >= K) v.w = 0.f;
                }
                ra[r] = v;
            }
        }
        f32_cp_commit();
    };
    auto stash = [&](int buf) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int e = t + r * MG_NT, row = e >> 2, kq = (e & 3) * 4;
            As[buf][kq + 0][row] = ra[r].x;
            As[buf][kq + 1][row] = ra[r].y;
            As[buf][kq + 2][row] = ra[r].z;
            As[buf][kq + 3][row] = ra[r].w;
        }
    };
    if (nkt > 0) {
        issue(0, 0);
        if (A_T) stash(0);
    }
    for (int kt = 0; kt < nkt; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nkt) {
            issue(kt + 1, buf ^ 1);
            f32_cp_wait<1>();
        } else {
            f32_cp_wait<0>();
        }
        __syncthreads();                                          // tile kt has landed
#pragma unroll
        for (int k = 0; k < MG_BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
            const float x[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float y[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(x[a], y[b], acc[a][b]);
        }
        __syncthreads();                                          // buffer buf may be refilled
        if (A_T && kt + 1 < nkt) stash(buf ^ 1);
    }
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int i = i0 + (a < 4 ? ty * 4 + a : 64 + ty * 4 + a - 4);
        if (i >= M) continue;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int j = j0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + b - 4);
            if (j >= N) continue;
            float c = acc[a][b];
            if (EPI == MG_RELU_MASK) c = __ldg(mask + (long long)i * ldc + j) > 0.f ? c : 0.f;
            C[(long long)i * ldc + j] = c;
        }
    }
}

// Partial bias gradients: part[z][n] = sum of dZ[p][n] over the probes p of slice z, in probe order.
__global__ void __launch_bounds__(256)
mlp_colsum_kernel(const float* __restrict__ dz, int ldz, int N, int valid, float* __restrict__ part) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x, z = blockIdx.y;
    if (n >= N) return;
    const int p1 = min(valid, (z + 1) * MG_SLICE);
    float s = 0.f;
    for (int p = z * MG_SLICE; p < p1; ++p) s += __ldg(dz + (size_t)p * ldz + n);
    part[(size_t)z * N + n] = s;
}

// out[e] = (first chunk ? 0 : out[e]) + part[0][e] + part[1][e] + ... + part[slices-1][e], left to right
__global__ void __launch_bounds__(256)
mlp_grad_reduce_kernel(const float* __restrict__ part, long long n, int slices, float* __restrict__ out, int first) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        float acc = first ? 0.f : out[e];
        for (int z = 0; z < slices; ++z) acc += part[(size_t)z * n + e];
        out[e] = acc;
    }
}

}  // namespace aadff
