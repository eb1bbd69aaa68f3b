// PSFNet fitting step on the device: forward + MSE loss + backward + AdamW for MLP(4, ks^2, 256, n) --
// the optimisation half of PSFNet.train_psfnet (deeplens/psfnet.py:79-132: psfnet(inp) -> nn.MSELoss ->
// backward -> torch.optim.AdamW.step), in fp32 on CUDA cores.  The ray-traced training targets
// (get_training_data, psfnet.py:135-170) stay with the reference: the caller hands in (inp [M,4], psf [M,ks^2]).
//
// The reference's batch is 128 probes: 0.44 GFLOP per step spread over ~35 dependent operators, i.e. a launch-bound
// chain (eager PyTorch: ~100 launches).  Here the chain is 3 small kernels per layer and direction plus one head
// kernel and ONE AdamW kernel over a contiguous parameter buffer, captured once in a CUDA graph and replayed per
// step (aadff_api.cu: aadff_trainer_step).
#pragma once
#include <cuda_runtime.h>

namespace aadff {

constexpr int TG_TILE = 32;      // C tile (TG_TILE x TG_TILE), 256 threads, 2 x 2 outputs per thread
constexpr int TG_K = 32;
constexpr int TG_NT = 256;

enum TgEpilogue { TG_BIAS_RELU = 0, TG_BIAS = 1, TG_RELU_MASK = 2, TG_PLAIN = 3 };

// C[i][j] = sum_k A(i,k) * B(k,j) with arbitrary element strides (covers X W^T, dZ W and dZ^T X), fp32.
//   TG_BIAS_RELU : C = relu(C + bias[j])          (hidden layer forward)
//   TG_BIAS      : C = C + bias[j]                (head pre-activation)
//   TG_RELU_MASK : C = mask[i][j] > 0 ? C : 0     (backward through the ReLU that produced `mask` = the activation)
//   TG_PLAIN     : C                              (weight gradient)
template <int EPI>
__global__ void __launch_bounds__(TG_NT)
train_gemm_kernel(const float* __restrict__ A, long long sa_i, long long sa_k, const float* __restrict__ B, long long sb_k,
                  long long sb_j, float* __restrict__ C, int M, int N, int K, const float* __restrict__ aux) {
    __shared__ float sA[TG_K][TG_TILE + 1], sB[TG_K][TG_TILE + 1];
    const int i0 = blockIdx.y * TG_TILE, j0 = blockIdx.x * TG_TILE;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;           // 16 x 16 threads, 2 x 2 outputs each
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    constexpr int PER = TG_K * TG_TILE / TG_NT;                       // operand elements per thread and K tile (4)
    // the K tile after the current one is fetched into registers while the current one is multiplied: these GEMMs are
    // a dependent chain of small launches, so the global-load latency per K tile is what they cost
    float pa[PER], pb[PER];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int r = 0; r < PER; ++r) {
            const int e = threadIdx.x + r * TG_NT;
            int ka, ia, kb, jb;               // the fast-running index follows the contiguous direction of each operand
            if (sa_k == 1) { ka = e % TG_K; ia = e / TG_K; } else { ia = e % TG_TILE; ka = e / TG_TILE; }
            if (sb_j == 1) { jb = e % TG_TILE; kb = e / TG_TILE; } else { kb = e % TG_K; jb = e / TG_K; }
            pa[r] = (i0 + ia < M && k0 + ka < K) ? __ldg(A + (i0 + ia) * sa_i + (k0 + ka) * sa_k) : 0.f;
            pb[r] = (j0 + jb < N && k0 + kb < K) ? __ldg(B + (k0 + kb) * sb_k + (j0 + jb) * sb_j) : 0.f;
        }
    };
    auto stash = [&]() {
#pragma unroll
        for (int r = 0; r < PER; ++r) {
            const int e = threadIdx.x + r * TG_NT;
            int ka, ia, kb, jb;
            if (sa_k == 1) { ka = e % TG_K; ia = e / TG_K; } else { ia = e % TG_TILE; ka = e / TG_TILE; }
            if (sb_j == 1) { jb = e % TG_TILE; kb = e / TG_TILE; } else { kb = e % TG_K; jb = e / TG_K; }
            sA[ka][ia] = pa[r];
            sB[kb][jb] = pb[r];
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < K; k0 += TG_K) {
        stash();
        __syncthreads();
        if (k0 + TG_K < K) fetch(k0 + TG_K);
#pragma unroll
        for (int k = 0; k < TG_K; ++k) {
            const float a0 = sA[k][ty], a1 = sA[k][ty + 16], b0 = sB[k][tx], b1 = sB[k][tx + 16];
            acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
            acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
            if (i >= M || j >= N) continue;
            float c = acc[u][v];
            if (EPI == TG_BIAS_RELU) c = fmaxf(c + __ldg(aux + j), 0.f);
            if (EPI == TG_BIAS) c = c + __ldg(aux + j);
            if (EPI == TG_RELU_MASK) c = (__ldg(aux + (long long)i * N + j) > 0.f) ? c : 0.f;
            C[(long long)i * N + j] = c;
        }
}

// db[j] = sum_i dZ[i][j]   (one thread per column; M is a few hundred)
__global__ void __launch_bounds__(256) train_colsum_kernel(const float* __restrict__ dZ, float* __restrict__ db, int M, int N) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    float s = 0.f;
    for (int i = 0; i < M; ++i) s += __ldg(dZ + (long long)i * N + j);
    db[j] = s;
}

// dL/dz_j of the head s = sigmoid(z), p = s / max(S, 1e-12), S = sum s, from g = dL/dp_j and gp = sum_i g_i p_i:
//   dL/ds_j = (g_j - gp) / S,   dL/dz_j = dL/ds_j * s_j (1 - s_j);
// for S below the clamp the denominator is constant: no normalisation gradient (F.normalize's clamp_min).
__device__ __forceinline__ float head_dz(float s, float g, float gp, float S, float denom) {
    const float ds = (S > 1e-12f) ? (g - gp) / denom : g / denom;
    return ds * s * (1.0f - s);
}

// Head: z -> s = sigmoid(z) -> p = s / max(sum|s|, 1e-12) (psfnet_arch.py:39-46) -> loss += sum (p - t)^2 / (M*kk)
// -> dZ = dL/dz (head_dz).  One warp per probe, g = dL/dp = 2 (p - t) / (M*kk).
__global__ void __launch_bounds__(256)
train_head_kernel(const float* __restrict__ z, const float* __restrict__ target, float* __restrict__ p_out,
                  float* __restrict__ dZ, float* __restrict__ loss, int M, int kk) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= M) return;
    const float* zr = z + (long long)warp * kk;
    const float* tr = target + (long long)warp * kk;
    float S = 0.f;
    for (int j = lane; j < kk; j += 32) S += 1.0f / (1.0f + expf(-zr[j]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) S += __shfl_xor_sync(0xffffffffu, S, o);
    const float denom = fmaxf(S, 1e-12f);
    const float scale = 2.0f / ((float)M * (float)kk);
    float gp = 0.f, l = 0.f;
    for (int j = lane; j < kk; j += 32) {
        const float s = 1.0f / (1.0f + expf(-zr[j]));
        const float p = s / denom, d = p - tr[j];
        p_out[(long long)warp * kk + j] = p;
        l = fmaf(d, d, l);
        gp = fmaf(scale * d, p, gp);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        gp += __shfl_xor_sync(0xffffffffu, gp, o);
        l += __shfl_xor_sync(0xffffffffu, l, o);
    }
    for (int j = lane; j < kk; j += 32) {
        const float s = 1.0f / (1.0f + expf(-zr[j]));
        const float g = scale * (s / denom - tr[j]);
        dZ[(long long)warp * kk + j] = head_dz(s, g, gp, S, denom);
    }
    if (lane == 0) atomicAdd(loss, l / ((float)M * (float)kk));
}

struct AdamHyper {        // written by train_hyper_kernel before every replay of the graph
    float lr, beta1, beta2, eps, weight_decay;
    float bias_correction1, bias_correction2_sqrt;
};

__global__ void train_hyper_kernel(AdamHyper* h, AdamHyper v, float* loss) {
    *h = v;
    *loss = 0.f;
}

// torch.optim.AdamW (single-tensor path): p *= 1 - lr*wd; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
// p -= (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
__global__ void __launch_bounds__(256)
train_adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                   long long n, const AdamHyper* __restrict__ hp) {
    const AdamHyper h = *hp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i];
        float pi = p[i] * (1.0f - h.lr * h.weight_decay);
        const float mi = m[i] + (1.0f - h.beta1) * (gi - m[i]);          // exp_avg.lerp_(grad, 1 - beta1)
        const float vi = h.beta2 * v[i] + (1.0f - h.beta2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) / h.bias_correction2_sqrt + h.eps;
        p[i] = pi - (h.lr / h.bias_correction1) * (mi / denom);
    }
}

}  // namespace aadff
