// C-ABI of libaadff.so (declared in include/aadff.h): handle management, weight pre-packing,
// launch configuration and error reporting for the sm_100a kernels in this directory.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/aadff.h"
#include "fused_tc_kernel.cuh"
#include "fused_fast2_kernel.cuh"
#include "gather_kernel.cuh"
#include "gather_coalesced_kernel.cuh"
#include "gather_strip_kernel.cuh"
#include "mlp_fp32_kernel.cuh"
#include "thinlens_kernel.cuh"
#include "focus_kernel.cuh"
#include "psf_conv_kernel.cuh"
#include "train_kernels.cuh"
#include "preprocess_kernel.cuh"
#include "spline_rotate_kernel.cuh"
#include "econ_calib.h"

using namespace aadff;

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};
std::atomic<int> g_desc_swap{0};
std::atomic<int> g_dbg_flags{0};
std::atomic<unsigned long long*> g_trace{nullptr};

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

// Template switch of the register-streaming gather: odd ks in 3..31, cn in {1, 3}.
template <int KS, int CN>
void launch_gc(int grid, cudaStream_t st, const float* img, const float* psf, float* out, int N, int C, int H, int W,
               int c0) {
    constexpr int smem = GatherCfg<KS>::SMEM_FLOATS(CN) * (int)sizeof(float);      // <= 69.6 KB (ks = 31, 3 channels)
    if (smem > 48 * 1024)      // the attribute is per device: set it on every launch (a host-side table write)
        cudaFuncSetAttribute(local_psf_coalesced_kernel<KS, CN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    local_psf_coalesced_kernel<KS, CN><<<grid, GC_WARPS * 32, smem, st>>>(img, psf, out, N, C, H, W, c0);
}
template <int KS>
bool launch_gc_ks(int ks, int cn, int grid, cudaStream_t st, const float* img, const float* psf, float* out, int N, int C,
                  int H, int W, int c0) {
    if constexpr (KS > 31) {
        return false;
    } else {
        if (ks == KS) {
            if (cn == 3) launch_gc<KS, 3>(grid, st, img, psf, out, N, C, H, W, c0);
            else launch_gc<KS, 1>(grid, st, img, psf, out, N, C, H, W, c0);
            return true;
        }
        return launch_gc_ks<KS + 2>(ks, cn, grid, st, img, psf, out, N, C, H, W, c0);
    }
}
bool launch_gather_coalesced(int ks, int cn, int grid, cudaStream_t st, const float* img, const float* psf, float* out,
                             int N, int C, int H, int W, int c0) {
    return launch_gc_ks<3>(ks, cn, grid, st, img, psf, out, N, C, H, W, c0);
}

// Strip-walking gather (gather_strip_kernel.cuh), ks <= 15: slots per warp (SL) / warps per CTA (NW) / strip width
// (SPX: 32, 64, or 64 U taken in U passes) chosen so that the PSF slots and the per-warp halo rings fill the 227 KB of shared memory.
// Plans are ordered widest strip first: the memory system likes long contiguous requests (ks = 7: 12.5 KB chunks reach
// 0.79 of the HBM peak, 25 KB 0.84, 50 KB 0.88), but a strip width that does not divide W wastes the narrower last
// strip (a chunk costs its latency, whatever its width): the first plan whose strips cover W with <= 10 % of padding
// runs.  Debug flags 1024 / 4096 force plan 1 / 2 (A/B timing).
struct StripShape { int SL, NW, SPX; };
template <int KS> struct StripPlan;
template <> struct StripPlan<3>  { static constexpr StripShape P[3] = {{2, 7, 256}, {2, 12, 128}, {4, 16, 64}}; };
template <> struct StripPlan<5>  { static constexpr StripShape P[3] = {{1, 5, 256}, {2, 6, 128}, {2, 12, 64}}; };
template <> struct StripPlan<7>  { static constexpr StripShape P[3] = {{1, 3, 256}, {1, 6, 128}, {1, 11, 64}}; };
template <> struct StripPlan<9>  { static constexpr StripShape P[3] = {{1, 3, 128}, {1, 7, 64}, {2, 4, 64}}; };
template <> struct StripPlan<11> { static constexpr StripShape P[3] = {{1, 5, 64}, {2, 3, 64}, {2, 3, 64}}; };
template <> struct StripPlan<13> { static constexpr StripShape P[3] = {{2, 2, 64}, {1, 4, 64}, {1, 4, 64}}; };
template <> struct StripPlan<15> { static constexpr StripShape P[3] = {{1, 3, 64}, {3, 1, 64}, {3, 1, 64}}; };
// Beyond 15 a 64-column chunk plus its halo ring fits only twice (measured 0.61 / 0.63 of the HBM peak at ks = 17 / 19
// against 0.72 / 0.78 for the register-streaming kernel), and 32-column strips (sixteen lanes of each warp idle, three
// or four warps) are bound by the warps' own arithmetic: 0.58 / 0.48 / 0.49 / 0.35 at ks = 17 / 19 / 21 / 23.
constexpr int STRIP_MAX_KS = 15;

template <int KS, int CN, int SL, int NW, int SPX>
void launch_gs(int sms, cudaStream_t st, const float* img, const float* psf, float* out, int N, int C, int H, int W,
               int c0) {
    constexpr int smem = StripCfg<KS, CN, SPX>::SMEM_BYTES(SL, NW);
    static_assert(smem <= 232448, "strip gather: shared memory plan does not fit");
    if (smem > 48 * 1024)      // per-device attribute: set on every launch that needs the opt-in
        cudaFuncSetAttribute(local_psf_strip_kernel<KS, CN, SL, NW, SPX>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const long long rows = (long long)N * ((W + SPX - 1) / SPX) * H;
    const int grid = (int)std::min<long long>((rows + NW - 1) / NW, sms);
    local_psf_strip_kernel<KS, CN, SL, NW, SPX><<<grid, NW * 32, smem, st>>>(img, psf, out, N, C, H, W, c0);
}
template <int KS, int I>
void launch_gs_plan(int cn, int sms, cudaStream_t st, const float* img, const float* psf, float* out, int N, int C, int H,
                    int W, int c0) {
    constexpr StripShape S = StripPlan<KS>::P[I];
    if (cn == 3) launch_gs<KS, 3, S.SL, S.NW, S.SPX>(sms, st, img, psf, out, N, C, H, W, c0);
    else launch_gs<KS, 1, S.SL, S.NW, S.SPX>(sms, st, img, psf, out, N, C, H, W, c0);
}
template <int KS>
bool launch_gs_ks(int ks, int cn, int plan, int sms, cudaStream_t st, const float* img, const float* psf, float* out,
                  int N, int C, int H, int W, int c0) {
    if constexpr (KS > STRIP_MAX_KS) {
        return false;
    } else {
        if (ks == KS) {
            if (plan < 0) {                                    // automatic: widest strips that cover W with <= 10 % padding
                plan = 2;
                for (int i = 0; i < 3; ++i) {
                    const int spx = StripPlan<KS>::P[i].SPX;
                    if ((long long)((W + spx - 1) / spx) * spx * 10 <= (long long)W * 11 || spx <= GSW_PX) { plan = i; break; }
                }
            }
            if (plan == 1) launch_gs_plan<KS, 1>(cn, sms, st, img, psf, out, N, C, H, W, c0);
            else if (plan == 2) launch_gs_plan<KS, 2>(cn, sms, st, img, psf, out, N, C, H, W, c0);
            else launch_gs_plan<KS, 0>(cn, sms, st, img, psf, out, N, C, H, W, c0);
            return true;
        }
        return launch_gs_ks<KS + 2>(ks, cn, plan, sms, st, img, psf, out, N, C, H, W, c0);
    }
}

template <int KS>
bool launch_psf_conv(int ks, int grid, cudaStream_t st, const PsfConvArgs& a) {
    if constexpr (KS > 31) {
        return false;
    } else {
        if (ks == KS) {
            psf_conv_kernel<KS><<<grid, PC_NT, 0, st>>>(a);
            return true;
        }
        return launch_psf_conv<KS + 2>(ks, grid, st, a);
    }
}

template <int KS>
bool launch_thinlens(int ks, int grid, int smem, cudaStream_t st, const ThinLensArgs& a, const CUtensorMap& map) {
    if constexpr (KS > 31) {
        return false;
    } else {
        if (ks == KS) {
            if (smem > 48 * 1024)      // per-device attribute
                cudaFuncSetAttribute(thinlens_render_kernel<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            thinlens_render_kernel<KS><<<grid, TL_NT, smem, st>>>(a, map);
            return true;
        }
        return launch_thinlens<KS + 2>(ks, grid, smem, st, a, map);
    }
}
// two pixels per thread (thinlens_render2_kernel): tile geometry by kernel size
template <int KS>
bool thinlens2_geometry(int ks, int cn, int* box_w, int* box_h, int* smem) {
    if constexpr (KS > 31) {
        return false;
    } else {
        if (ks == KS) {
            *box_w = ThinLens2Cfg<KS>::BW;
            *box_h = ThinLens2Cfg<KS>::HH;
            *smem = ThinLens2Cfg<KS>::SMEM_BYTES(cn);
            return true;
        }
        return thinlens2_geometry<KS + 2>(ks, cn, box_w, box_h, smem);
    }
}
template <int KS>
bool launch_thinlens2(int ks, int grid, int smem, cudaStream_t st, const ThinLensArgs& a, const CUtensorMap& map) {
    if constexpr (KS > 31) {
        return false;
    } else {
        if (ks == KS) {
            if (smem > 48 * 1024)      // per-device attribute
                cudaFuncSetAttribute(thinlens_render2_kernel<KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            thinlens_render2_kernel<KS><<<grid, TL_NT, smem, st>>>(a, map);
            return true;
        }
        return launch_thinlens2<KS + 2>(ks, grid, smem, st, a, map);
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// [planes][H][W] fp32 image as a 3-D tensor map with a [box_c][box_h][box_w] box; false if TMA's rules are not met
bool make_image_map(CUtensorMap* map, const float* img, long long planes, int H, int W, int box_w, int box_h, int box_c) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc || (W % 4) != 0 || (reinterpret_cast<uintptr_t>(img) % 16) != 0 || box_w > 256 || box_h > 256 || box_c > 256)
        return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes};
    const cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_c};
    const cuuint32_t estr[3] = {1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(img), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            return fail(AADFF_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));      \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

template <typename T>
int upload(const std::vector<T>& h, T** d) {
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(d), h.size() * sizeof(T)));
    CUDA_TRY(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return AADFF_OK;
}

// W rows [n0, n0+N) x all K -> K/32 slabs, each (hi, lo), canonical no-swizzle K-major layout:
// half index inside a slab = (k/8) * (N*8) + n*8 + (k%8)
// (for the calibrated econ weights W already holds fp16 values: hi = W exactly, lo = 0 and never loaded)
void pack_group(const float* W, int out_f, int in_f, int n0, int N, std::vector<__half>& dst) {
    for (int kc = 0; kc < in_f / TC_SLAB_K; ++kc) {
        for (int part = 0; part < 2; ++part) {
            const size_t base = dst.size();
            dst.resize(base + (size_t)N * TC_SLAB_K);
            for (int k = 0; k < TC_SLAB_K; ++k) {
                for (int n = 0; n < N; ++n) {
                    const int row = n0 + n, col = kc * TC_SLAB_K + k;
                    const float w = (row < out_f) ? W[(size_t)row * in_f + col] : 0.0f;
                    const __half hi = __float2half_rn(w);
                    const __half v = part == 0 ? hi : __float2half_rn(w - __half2float(hi));
                    dst[base + (size_t)(k / 8) * (N * 8) + (size_t)n * 8 + (k % 8)] = v;
                }
            }
        }
    }
}

// Bias slab of a hidden group: B[n][k], k < 16, canonical K-major layout; k = 0 holds fp16(b_n), k = 1 the fp16
// remainder.  Multiplied by the constant A operand (ones in K columns 0 and 1) it starts the accumulator at b_n.
void pack_bias_slab(const float* bias, int N, std::vector<__half>& dst) {
    const size_t base = dst.size();
    dst.resize(base + (size_t)N * 16, __float2half_rn(0.f));
    for (int n = 0; n < N; ++n) {
        const __half hi = __float2half_rn(bias[n]);
        dst[base + (size_t)n * 8 + 0] = hi;
        dst[base + (size_t)n * 8 + 1] = __float2half_rn(bias[n] - __half2float(hi));
    }
}

}  // namespace

struct aadff_psfnet {
    int device = 0, ks = 0, kk = 0, n_layers = 0;
    int num_sms = 0, smem_optin = 0;
    // fp32 (CUDA-core) path
    Fp32Net f32{};
    std::vector<float*> owned;
    // tcgen05 path
    bool tc_ok = false;
    std::string tc_why;
    uint8_t* d_wpack = nullptr;
    float* d_bias_tc = nullptr;
    float* d_w0b0 = nullptr;
    TcGroup groups[TC_MAX_GROUPS]{};
    // econ mode, 2-term groups: calibrated fp16 weights (econ_calib.h), built on the first AADFF_MODE_ECON launch
    // (the calibration is a host pass of a few hundred ms that parity / fast / fp32 users should not pay for)
    uint32_t w_off_econ[TC_MAX_GROUPS]{};
    uint8_t* d_wpack_econ = nullptr;        // main pack followed by the calibrated slabs
    size_t pack_bytes = 0;
    bool econ_ready = false;
    std::mutex econ_mu;
    std::vector<std::vector<float>> host_w, host_b;   // fp32 copy of the state_dict (calibration input)
    std::vector<int> host_dims;
    int n_groups = 0, n_hidden = 0, n_bias = 0, head_bias0 = 0;
    // host-call workspace
    cudaStream_t ws_stream = nullptr, ws_copy_stream = nullptr;
    std::vector<cudaEvent_t> ws_events;
    float* ws = nullptr;
    size_t ws_bytes = 0;
};

// ------------------------------------------------------------------------------------------ PSFNet fitting (f3)
struct aadff_trainer {
    int device = 0, n_layers = 0, batch = 0, kk = 0;
    std::vector<int> dims;
    std::vector<size_t> w_off, b_off;          // float offsets into params / grads
    size_t n_params = 0;
    float *params = nullptr, *grads = nullptr, *m = nullptr, *v = nullptr;
    std::vector<float*> act;                   // act[l] = input of layer l, [batch, dims[l]]
    float *z = nullptr, *p = nullptr, *target = nullptr, *loss = nullptr;
    std::vector<float*> dz;                    // dz[l] = dL/d(pre-activation of layer l), [batch, dims[l+1]]: one buffer per
                                               // layer, because dW_l (side branch of the graph) reads dz[l] while the main
                                               // branch already produces dz[l-1], dz[l-2], ...
    AdamHyper* hyper = nullptr;
    AdamHyper host_hyper{};
    long long step = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaStream_t cap_stream = nullptr;
    cudaStream_t side[2] = {nullptr, nullptr};  // capture-time fork targets (created before the capture begins)
    std::vector<cudaEvent_t> evs;
};

static void trainer_free(aadff_trainer* t) {
    if (!t) return;
    DeviceGuard guard(t->device);
    if (t->exec) cudaGraphExecDestroy(t->exec);
    if (t->graph) cudaGraphDestroy(t->graph);
    if (t->cap_stream) cudaStreamDestroy(t->cap_stream);
    for (cudaEvent_t ev : t->evs) cudaEventDestroy(ev);
    for (int i = 0; i < 2; ++i) if (t->side[i]) cudaStreamDestroy(t->side[i]);
    for (float* a : t->act) cudaFree(a);
    cudaFree(t->params); cudaFree(t->grads); cudaFree(t->m); cudaFree(t->v);
    cudaFree(t->z); cudaFree(t->p); cudaFree(t->target);
    for (float* d : t->dz) cudaFree(d);
    cudaFree(t->loss); cudaFree(t->hyper);
    delete t;
}

template <int EPI>
static void tg_launch(cudaStream_t st, const float* A, long long sa_i, long long sa_k, const float* B, long long sb_k,
                      long long sb_j, float* C, int M, int N, int K, const float* aux) {
    dim3 grid((N + TG_TILE - 1) / TG_TILE, (M + TG_TILE - 1) / TG_TILE);
    train_gemm_kernel<EPI><<<grid, TG_NT, 0, st>>>(A, sa_i, sa_k, B, sb_k, sb_j, C, M, N, K, aux);
}

// the whole step (forward, loss, backward, AdamW): recorded once into a CUDA graph.  Only the dX chain of the backward
// pass is serial; the weight gradients dW_l = dZ_l^T X_l and the bias gradients (column sums of dZ_l) hang off it, so they
// are recorded on two side streams (forked / joined with events: parallel branches of the graph) -- the critical path
// shrinks from 3 L + ... to L launches of the backward pass.
static int trainer_record(aadff_trainer* t, cudaStream_t st) {
    const int L = t->n_layers, M = t->batch;
    cudaStream_t* side = t->side;
    size_t next_ev = 0;
    auto new_event = [&]() { return t->evs[next_ev++]; };      // L + 2 events, created before the capture began
    for (int l = 0; l < L; ++l) {
        const int K = t->dims[l], N = t->dims[l + 1];
        const float* W = t->params + t->w_off[l];
        const float* b = t->params + t->b_off[l];
        if (l < L - 1) tg_launch<TG_BIAS_RELU>(st, t->act[l], K, 1, W, 1, K, t->act[l + 1], M, N, K, b);
        else tg_launch<TG_BIAS>(st, t->act[l], K, 1, W, 1, K, t->z, M, N, K, b);
    }
    train_head_kernel<<<(M * 32 + 255) / 256, 256, 0, st>>>(t->z, t->target, t->p, t->dz[L - 1], t->loss, M, t->kk);
    for (int l = L - 1; l >= 0; --l) {
        const int K = t->dims[l], N = t->dims[l + 1];
        const float* W = t->params + t->w_off[l];
        const float* dZ = t->dz[l];
        cudaEvent_t ready = new_event();                                                                    // dZ_l exists
        cudaEventRecord(ready, st);
        cudaStreamWaitEvent(side[0], ready, 0);
        cudaStreamWaitEvent(side[1], ready, 0);
        tg_launch<TG_PLAIN>(side[0], dZ, 1, N, t->act[l], K, 1, t->grads + t->w_off[l], N, K, M, nullptr);  // dW = dZ^T X
        train_colsum_kernel<<<(N + 255) / 256, 256, 0, side[1]>>>(dZ, t->grads + t->b_off[l], M, N);
        if (l > 0) tg_launch<TG_RELU_MASK>(st, dZ, N, 1, W, K, 1, t->dz[l - 1], M, K, N, t->act[l]);        // dX = dZ W, masked
    }
    for (int i = 0; i < 2; ++i) {                                                                           // join
        cudaEvent_t done = new_event();
        cudaEventRecord(done, side[i]);
        cudaStreamWaitEvent(st, done, 0);
    }
    train_adamw_kernel<<<(int)std::min<size_t>((t->n_params + 255) / 256, 1184), 256, 0, st>>>(
        t->params, t->grads, t->m, t->v, (long long)t->n_params, t->hyper);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(AADFF_E_CUDA, std::string("trainer_record: ") + cudaGetErrorString(e));
    return AADFF_OK;
}


extern "C" {

int aadff_version(void) { return AADFF_VERSION; }
const char* aadff_last_error(void) { return g_err.c_str(); }
int64_t aadff_launch_count(void) { return g_launches.load(); }
int aadff_debug_set_desc_swap(int swap) {
    g_desc_swap.store(swap ? 1 : 0);
    return AADFF_OK;
}

int aadff_debug_set_trace(void* device_buffer) {
    g_trace.store(static_cast<unsigned long long*>(device_buffer));
    return AADFF_OK;
}
int aadff_debug_trace_entries(void) { return TC_TRACE_N; }
int aadff_debug_set_flags(int flags) {
    g_dbg_flags.store(flags);
    return AADFF_OK;
}

int aadff_psfnet_create(const float* const* weights, const float* const* biases, const int* dims, int n_layers,
                        int ks, int device, aadff_psfnet_t* out) {
    if (!weights || !biases || !dims || !out) return fail(AADFF_E_INVALID, "null argument");
    if (n_layers < 2 || n_layers > MAX_LAYERS) return fail(AADFF_E_INVALID, "n_layers must be in [2,16]");
    if (ks < 1 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "kernel size must be odd and positive");
    if (dims[0] != 4 || dims[n_layers] != ks * ks)
        return fail(AADFF_E_INVALID, "dims must start with 4 and end with ks*ks");
    for (int l = 0; l < n_layers; ++l) {
        if (!weights[l] || !biases[l]) return fail(AADFF_E_INVALID, "null layer pointer");
        if (dims[l + 1] < 1 || (l + 1 < n_layers && (dims[l + 1] > 256 || dims[l + 1] % 8)))
            return fail(AADFF_E_INVALID, "hidden widths must be multiples of 8 and <= 256");
    }
    DeviceGuard guard(device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select CUDA device " + std::to_string(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(AADFF_E_CUDA, "libaadff is built for sm_100a only; device is sm_" + std::to_string(prop.major) +
                                      std::to_string(prop.minor));

    aadff_psfnet* h = new aadff_psfnet();
    h->device = device;
    h->ks = ks;
    h->kk = ks * ks;
    h->n_layers = n_layers;
    h->num_sms = prop.multiProcessorCount;
    h->smem_optin = (int)prop.sharedMemPerBlockOptin;

    // ---- fp32 path: W^T [K][npad], bias [npad]
    h->f32.n_layers = n_layers;
    h->f32.kk = h->kk;
    for (int l = 0; l < n_layers; ++l) {
        const int K = dims[l], Nf = dims[l + 1], npad = (Nf + 7) / 8 * 8;
        std::vector<float> wt((size_t)K * npad, 0.f), b(npad, 0.f);
        for (int n = 0; n < Nf; ++n) {
            b[n] = biases[l][n];
            for (int k = 0; k < K; ++k) wt[(size_t)k * npad + n] = weights[l][(size_t)n * K + k];
        }
        float *dw = nullptr, *db = nullptr;
        int rc = upload(wt, &dw);
        if (rc) { aadff_psfnet_destroy(h); return rc; }
        h->owned.push_back(dw);
        rc = upload(b, &db);
        if (rc) { aadff_psfnet_destroy(h); return rc; }
        h->owned.push_back(db);
        h->f32.wt[l] = dw;
        h->f32.bias[l] = db;
        h->f32.k[l] = K;
        h->f32.npad[l] = npad;
    }
#define CREATE_TRY(expr)                                                                         \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            aadff_psfnet_destroy(h);                                                             \
            return fail(AADFF_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));       \
        }                                                                                        \
    } while (0)
    CREATE_TRY(cudaFuncSetAttribute(mlp_fp32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, F32_SMEM));
    CREATE_TRY(cudaFuncSetAttribute(mlp_fp32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, F32_SMEM));

    // ---- tcgen05 path: needs the PSFNet architecture 4 -> 64 -> 256 -> 256 x n -> ks^2
    h->tc_ok = true;
    if (n_layers < 3 || dims[1] != 64) { h->tc_ok = false; h->tc_why = "first hidden width must be 64"; }
    for (int l = 2; l < n_layers && h->tc_ok; ++l)
        if (dims[l] != TC_HID) { h->tc_ok = false; h->tc_why = "hidden width must be 256"; }
    if (ks > TC_MAX_KS) { h->tc_ok = false; h->tc_why = "kernel size > 31"; }
    const int nh_pad = (h->kk + 15) / 16 * 16;
    const int n_head_blocks = (nh_pad + 255) / 256;
    if (h->tc_ok && (n_layers - 2) + n_head_blocks > TC_MAX_GROUPS) { h->tc_ok = false; h->tc_why = "too many layers"; }
    if (h->tc_ok) {
        std::vector<__half> pack;
        std::vector<float> bias_tc;
        int gi = 0;
        for (int l = 1; l < n_layers - 1; ++l, ++gi) {      // L1 .. L(n-2): hidden MMA layers
            TcGroup& g = h->groups[gi];
            g.w_off = (uint32_t)(pack.size() * sizeof(__half));
            g.K = (uint16_t)dims[l];
            g.N = TC_HID;
            g.terms = 3;
            g.bias_off = (uint16_t)bias_tc.size();
            g.new_a = 1;
            g.tap0 = 0;
            pack_bias_slab(biases[l], TC_HID, pack);        // first slab of every hidden group
            pack_group(weights[l], dims[l + 1], dims[l], 0, TC_HID, pack);
            bias_tc.insert(bias_tc.end(), biases[l], biases[l] + TC_HID);
        }
        h->n_hidden = gi;
        const int L = n_layers - 1;
        const int head_bias0 = (int)bias_tc.size();
        h->head_bias0 = head_bias0;
        bias_tc.resize(head_bias0 + nh_pad, 0.f);
        // head bias is stored pre-scaled by -log2(e): the kernel evaluates exp(-(acc+b)) as ex2(fma(acc,-log2e,b'))
        for (int n = 0; n < h->kk; ++n) bias_tc[head_bias0 + n] = -1.4426950408889634f * biases[L][n];
        for (int b = 0; b < n_head_blocks; ++b, ++gi) {
            TcGroup& g = h->groups[gi];
            const int N = std::min(256, nh_pad - 256 * b);
            g.w_off = (uint32_t)(pack.size() * sizeof(__half));
            g.K = TC_HID;
            g.N = (uint16_t)N;
            g.terms = 3;
            g.bias_off = (uint16_t)(head_bias0 + 256 * b);
            g.new_a = (b == 0);
            g.tap0 = (uint16_t)(256 * b);
            pack_group(weights[L], h->kk, TC_HID, 256 * b, N, pack);
        }
        h->n_groups = gi;
        h->n_bias = (int)bias_tc.size();
        // econ mode needs the fp32 weights again (lazy calibration, ensure_econ below)
        h->host_dims.assign(dims, dims + n_layers + 1);
        for (int l = 0; l < n_layers; ++l) {
            h->host_w.emplace_back(weights[l], weights[l] + (size_t)dims[l] * dims[l + 1]);
            h->host_b.emplace_back(biases[l], biases[l] + dims[l + 1]);
        }
        h->pack_bytes = pack.size() * sizeof(__half);
        std::vector<float> w0b0(320);
        std::memcpy(w0b0.data(), weights[0], 256 * sizeof(float));
        std::memcpy(w0b0.data() + 256, biases[0], 64 * sizeof(float));
        __half* dp = nullptr;
        int rc = upload(pack, &dp);
        if (rc) { aadff_psfnet_destroy(h); return rc; }
        h->d_wpack = reinterpret_cast<uint8_t*>(dp);
        rc = upload(bias_tc, &h->d_bias_tc);
        if (rc) { aadff_psfnet_destroy(h); return rc; }
        rc = upload(w0b0, &h->d_w0b0);
        if (rc) { aadff_psfnet_destroy(h); return rc; }
        const int so = h->smem_optin;
        const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<true, false, 0>, attr, so));
#define AADFF_SET_ATTR(U)                                                                        \
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, false, U>, attr, so));   \
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, false, U, true>, attr, so));   \
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, true, U>, attr, so));
        AADFF_SET_ATTR(0) AADFF_SET_ATTR(1) AADFF_SET_ATTR(3) AADFF_SET_ATTR(13) AADFF_SET_ATTR(12) AADFF_SET_ATTR(15)
#undef AADFF_SET_ATTR
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, false, 14>, attr, so));      // econ8: no cluster variant
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, true, 14>, attr, so));
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<true, false, 0, false, true>, attr, so));
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, false, 12, false, true>, attr, so));
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, false, 13, false, true>, attr, so));
        CREATE_TRY(cudaFuncSetAttribute(fused_psfnet_render_kernel<false, false, 14, false, true>, attr, so));
    }
#undef CREATE_TRY
    *out = h;
    return AADFF_OK;
}

int aadff_psfnet_destroy(aadff_psfnet_t h) {
    if (!h) return AADFF_OK;
    DeviceGuard guard(h->device);
    for (float* p : h->owned) cudaFree(p);
    cudaFree(h->d_wpack);
    cudaFree(h->d_wpack_econ);
    cudaFree(h->d_bias_tc);
    cudaFree(h->d_w0b0);
    cudaFree(h->ws);
    if (h->ws_stream) cudaStreamDestroy(h->ws_stream);
    if (h->ws_copy_stream) cudaStreamDestroy(h->ws_copy_stream);
    for (cudaEvent_t e : h->ws_events) cudaEventDestroy(e);
    delete h;
    return AADFF_OK;
}

// First AADFF_MODE_ECON launch on a handle: calibrate the fp16 rounding of the 2-term layers on the host
// (econ_calib.h), pack them and place them behind a copy of the main pack.  Synchronous, once per handle.
static int ensure_econ(aadff_psfnet_t h) {
    std::lock_guard<std::mutex> lock(h->econ_mu);
    if (h->econ_ready) return AADFF_OK;
    const int n_layers = h->n_layers, L = n_layers - 1;
    std::vector<const float*> W(n_layers), B(n_layers);
    for (int l = 0; l < n_layers; ++l) { W[l] = h->host_w[l].data(); B[l] = h->host_b[l].data(); }
    std::vector<std::vector<float>> wq;
    calibrate_econ(W.data(), B.data(), h->host_dims.data(), n_layers, TC_ECON_FIRST_LAYER, wq);
    std::vector<__half> pack;
    for (int g2 = 0; g2 < h->n_groups; ++g2) {
        const bool hidden = g2 < h->n_hidden;
        const int l = hidden ? g2 + 1 : L;
        h->w_off_econ[g2] = h->groups[g2].w_off;                  // plain rounding unless calibrated
        if (l < TC_ECON_FIRST_LAYER || wq[l].empty()) continue;
        h->w_off_econ[g2] = (uint32_t)(h->pack_bytes + pack.size() * sizeof(__half));
        if (hidden) {
            pack_bias_slab(B[l], TC_HID, pack);
            pack_group(wq[l].data(), h->host_dims[l + 1], h->host_dims[l], 0, TC_HID, pack);
        } else {
            pack_group(wq[l].data(), h->kk, TC_HID, h->groups[g2].tap0, h->groups[g2].N, pack);
        }
    }
    uint8_t* d = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d), h->pack_bytes + pack.size() * sizeof(__half)));
    cudaError_t e = cudaMemcpy(d, h->d_wpack, h->pack_bytes, cudaMemcpyDeviceToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d + h->pack_bytes, pack.data(), pack.size() * sizeof(__half), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(d);
        return fail(AADFF_E_CUDA, std::string("econ weight upload: ") + cudaGetErrorString(e));
    }
    h->d_wpack_econ = d;
    h->econ_ready = true;
    return AADFF_OK;
}

// AADFF_MODE_FAST with two tiles in flight per CTA (fused_fast2_kernel.cuh).  Built, bit-identical to the one-tile kernel
// and measured SLOWER (0.80-0.91x, profiles/NOTES_r02.md: the second tile's activations leave a 64 KB weight ring, too
// shallow to cover the L2 latency at fast mode's 64 B/clk per SM), so it only runs when debug flag 32 asks for it.
// Returns 1 if the launch does not qualify (flag not set, several head blocks, shared-memory budget).
static int launch_fast2(aadff_psfnet_t h, const RenderArgs& ra, cudaStream_t st, long long tile_row0, long long tile_row1) {
    if (!h->tc_ok || h->n_groups != h->n_hidden + 1 || !(g_dbg_flags.load() & 32)) return 1;
    F2Params P{};
    P.ra = ra;
    P.wpack = h->d_wpack;
    P.bias = h->d_bias_tc;
    P.w0b0 = h->d_w0b0;
    P.n_groups = h->n_groups;
    P.n_hidden = h->n_hidden;
    P.n_bias = h->n_bias;
    P.bias_skip = h->head_bias0;
    P.kk = h->kk;
    for (int i = 0; i < h->n_groups; ++i) { P.g[i] = h->groups[i]; P.g[i].terms = 1; }
    P.tiles_x = (ra.W + TC_TILE_W - 1) / TC_TILE_W;
    P.tiles_y = (ra.H + TC_TILE_H - 1) / TC_TILE_H;
    P.n_tiles = (long long)P.tiles_x * P.tiles_y * ra.N * ra.S;
    if (tile_row1 >= 0) {
        P.tile0 = tile_row0 * P.tiles_x;
        P.n_tiles = (tile_row1 - tile_row0) * P.tiles_x;
        if (P.n_tiles <= 0) return AADFF_OK;
    }
    P.halo_pitch = TC_TILE_W + ra.ks - 1;
    P.halo_bytes = (uint32_t)(TC_TILE_H + ra.ks - 1) * P.halo_pitch * 16;
    const uint32_t bias_bytes = (uint32_t)(h->n_bias - h->head_bias0) * 4;
    P.off_stage = 2 * TC_A_PART_BYTES;
    P.off_bias = P.off_stage + F2_STAGES * TC_STAGE_BYTES;
    P.off_w0 = P.off_bias + bias_bytes;
    P.off_halo = (P.off_w0 + 320 * 4 + 15u) & ~15u;
    P.off_red = P.off_halo + 2 * P.halo_bytes;
    P.off_bar = P.off_red + 2 * TC_M * 5 * 4;
    P.off_ones = (P.off_bar + TC_BAR_BYTES + 15u) & ~15u;
    P.off_bslab = P.off_ones + 2 * TC_A_LBO;
    const uint32_t smem = P.off_bslab + 2 * TC_BSLAB_BYTES;
    if (smem > (uint32_t)h->smem_optin) return 1;
    const long long units = (P.n_tiles + 1) / 2;
    const int grid = (int)std::min<long long>(units, h->num_sms);
    cudaFuncSetAttribute(fused_fast2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin);
    fused_fast2_kernel<<<grid, TC_NT, smem, st>>>(P);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

static int launch_tc(aadff_psfnet_t h, RenderArgs ra, int mode, cudaStream_t st, long long tile_row0 = 0,
                     long long tile_row1 = -1, const float* probes = nullptr, float* psf_out = nullptr,
                     long long n_probes = 0) {
    if (!h->tc_ok) return fail(AADFF_E_UNSUPPORTED, "tensor-core path unavailable: " + h->tc_why + " (use AADFF_MODE_FP32)");
    const bool econ_like = (mode == AADFF_MODE_ECON || mode == AADFF_MODE_ECON8);
    if (econ_like) {
        const int rc = ensure_econ(h);
        if (rc) return rc;
    }
    if (mode == AADFF_MODE_FAST && probes == nullptr && g_trace.load() == nullptr) {
        const int rc = launch_fast2(h, ra, st, tile_row0, tile_row1);
        if (rc <= 0) return rc;                                   // launched (0) or failed (< 0); 1 = not eligible
    }
    TcParams P{};
    P.ra = ra;
    P.wpack = econ_like ? h->d_wpack_econ : h->d_wpack;
    P.bias = h->d_bias_tc;
    P.w0b0 = h->d_w0b0;
    P.n_groups = h->n_groups;
    P.n_hidden = h->n_hidden;
    P.n_bias = h->n_bias;
    P.bias_skip = h->head_bias0;                               // hidden biases live in the bias slabs
    P.kk = h->kk;
    // debug flags bits 16..19: first two-term group of AADFF_MODE_ECON for this launch (0 = the shipped pattern, L5 =
    // group 4; later groups trade speed for accuracy -- tests/gpu_econ_certificate.py sweeps it; runs the generic kernel)
    const int econ_first_dbg = (g_dbg_flags.load() >> 16) & 15;
    const int econ_first = (econ_first_dbg > TC_ECON_FIRST_GROUP) ? econ_first_dbg : TC_ECON_FIRST_GROUP;
    for (int i = 0; i < h->n_groups; ++i) {
        P.g[i] = h->groups[i];
        const bool hidden = i < h->n_hidden;
        P.g[i].terms = (mode == AADFF_MODE_FAST) ? 1
                       : (mode == AADFF_MODE_MIXED && i >= TC_MIXED_FIRST_GROUP) ? 1
                       : (mode == AADFF_MODE_ECON && i >= econ_first) ? 2              // L5.. and the head: fp16 weights
                       : (mode == AADFF_MODE_ECON8 && i >= TC_ECON8_FIRST_GROUP) ? 2   // L8, L9 and the head
                       : 3;
        if (econ_like && P.g[i].terms == 2 && !(g_dbg_flags.load() & 256))
            P.g[i].w_off = h->w_off_econ[i];                   // calibrated rounding (debug flag 256: plain rounding)
        (void)hidden;
    }
    P.tiles_x = (ra.W + TC_TILE_W - 1) / TC_TILE_W;
    P.tiles_y = (ra.H + TC_TILE_H - 1) / TC_TILE_H;
    P.n_tiles = (long long)P.tiles_x * P.tiles_y * ra.N * ra.S;
    if (tile_row1 >= 0) {                                      // a contiguous run of tile rows of the flattened stack
        P.tile0 = tile_row0 * P.tiles_x;
        P.n_tiles = (tile_row1 - tile_row0) * P.tiles_x;
        if (P.n_tiles <= 0) return AADFF_OK;
    }
    if (probes != nullptr) {                                   // pred mode: 128 probes per tile, no image
        P.probes = probes;
        P.psf_out = psf_out;
        P.n_probes = n_probes;
        P.n_tiles = (n_probes + TC_M - 1) / TC_M;
    }
    P.trace = g_trace.load();
    P.dbg = (uint32_t)g_dbg_flags.load();
    // shared-memory carve-up
    uint32_t halo_bytes = (uint32_t)(TC_TILE_H + ra.ks - 1) * TC_HALO_PITCH * 16;          // float4 per pixel
    if (probes != nullptr) halo_bytes = std::max<uint32_t>(halo_bytes, 8 * 32 * 9 * 4);        // pred mode: the store staging lives there
    const uint32_t bias_bytes = (uint32_t)(h->n_bias - h->head_bias0) * 4;                 // head bias only
    const uint32_t ones_bytes = 2 * TC_A_LBO;                                              // constant A operand of the bias slabs
    const uint32_t bslab_bytes = 2 * TC_BSLAB_BYTES;                                        // bias-slab slot + its block of zeros
    const uint32_t fixed = 2 * TC_A_PART_BYTES + bias_bytes + 320 * 4 + halo_bytes + TC_M * 5 * 4 + TC_BAR_BYTES + ones_bytes +
                           bslab_bytes + 16;
    int stages = 4;
    while (stages >= 2 && fixed + (uint32_t)stages * TC_STAGE_BYTES > (uint32_t)h->smem_optin) --stages;
    if (stages < 2) return fail(AADFF_E_UNSUPPORTED, "shared memory budget exceeded for this kernel size / channel count");
    bool any_lo = false;
    for (int i = 0; i < h->n_groups; ++i) any_lo |= (P.g[i].terms >= 2);
    P.off_stage = 2 * TC_A_PART_BYTES;
    P.off_bias = P.off_stage + stages * TC_STAGE_BYTES;
    P.off_w0 = P.off_bias + bias_bytes;
    P.off_halo = P.off_w0 + 320 * 4;
    P.off_red = P.off_halo + halo_bytes;
    P.off_bar = P.off_red + TC_M * 5 * 4;
    P.off_ones = (P.off_bar + TC_BAR_BYTES + 15u) & ~15u;
    P.off_bslab = P.off_ones + ones_bytes;
    const uint32_t smem = P.off_bslab + bslab_bytes;
    // no layer needs lo operands (fast mode): the A_lo region doubles the ring to 128 KB, organised as four
    // 32 KB stages (two packed K=32 slabs each) so that every issue iteration queues four MMAs
    P.kslab = (!any_lo && stages == 4) ? 2 : 1;
    P.n_stages = (P.kslab == 2) ? 4 : stages;
    int grid = (int)std::min<long long>(P.n_tiles, h->num_sms);
    // kernel specialisation (fused_tc_kernel.cuh, template UNI): pattern 3 = all groups three-term (parity), 1 = all
    // single-term with the long ring (fast), 2 = econ, 5 = mixed, 0 = per-group terms at run time; +10 when the ring has
    // four stages and every group consumes a multiple of four of them (ring position of a K-step = compile-time)
    bool all3 = true, all1 = true, econ_pat = true, econ8_pat = true, mixed_pat = true, aligned = (P.n_stages == 4 && P.kslab == 1);
    for (int i = 0; i < h->n_groups; ++i) {
        const int t = P.g[i].terms;
        all3 &= (t == 3);
        all1 &= (t == 1);
        econ_pat &= (t == (i < TC_ECON_FIRST_GROUP ? 3 : 2));
        econ8_pat &= (t == (i < TC_ECON8_FIRST_GROUP ? 3 : 2));
        mixed_pat &= (t == (i < TC_MIXED_FIRST_GROUP ? 3 : 1));
        aligned &= (((P.g[i].K / TC_SLAB_K) * (t == 3 ? 2 : 1)) % 4 == 0);
    }
    static_assert(TC_ECON_FIRST_GROUP == TC_ECON_FIRST_LAYER - 1, "group g holds layer g + 1");
    int uni = 0;
    if (all3 && P.kslab == 1) uni = aligned ? 13 : 3;
    else if (all1 && P.kslab == 2) uni = 1;
    else if (econ_pat && aligned) uni = 12;
    else if (econ8_pat && aligned && h->n_groups > TC_ECON8_FIRST_GROUP) uni = 14;
    else if (mixed_pat && aligned) uni = 15;
    // 2-CTA clusters sharing the weight stream by multicast (fused_tc_kernel.cuh, CL2).  Built, bit-exact, and measured
    // NOT to pay (profiles/NOTES_r02.md: -7 % at c2, +-1 % where power-capped), so it is off unless debug flag 8 asks for it.
    const bool cl2 = P.probes == nullptr && P.trace == nullptr && uni != 0 && uni != 14 && (P.dbg & 8u) && h->num_sms >= 2;
    // A operands in tensor memory (fused_tc_kernel.cuh, TA): render launches of the 2-/3-term specialisations with one
    // head block of N <= 192 (ks <= 13) and at least two hidden layers, 4-stage ring.  Its shared memory holds no
    // activations: ring, raw head values of the tile being gathered, two halo slots.  Debug flag 1 << 20 keeps such
    // launches on the shared-memory path (equality tests, A/B timing).
    bool all2 = true;
    for (int i = 0; i < h->n_groups; ++i) all2 &= (P.g[i].terms >= 2);
    const uint32_t head_n = h->groups[h->n_hidden].N;
    uint32_t smem_launch = smem;
    const bool ta = P.probes == nullptr && !cl2 && !(P.dbg & (1u << 20)) && h->n_groups == h->n_hidden + 1 &&
                    h->n_hidden >= 2 && head_n <= (uint32_t)TC_TA_L1_COL && P.kslab == 1 && P.n_stages == 4 && all2 &&
                    (uni == 12 || uni == 13 || uni == 14 || P.trace != nullptr);
    if (ta) {
        const uint32_t stg_bytes = ((head_n + 31u) & ~31u) * TC_M * 4;      // the gather reads 32-column blocks
        P.halo_bytes = halo_bytes;
        P.off_stage = 0;
        P.off_stg = 4 * TC_STAGE_BYTES;
        P.off_bias = P.off_stg + stg_bytes;
        P.off_w0 = P.off_bias + bias_bytes;
        P.off_halo = (P.off_w0 + 320 * 4 + 15u) & ~15u;
        P.off_red = P.off_halo + 2 * halo_bytes;
        P.off_bar = P.off_red + TC_M * 5 * 4;
        P.off_ones = (P.off_bar + TC_BAR_BYTES + 15u) & ~15u;
        P.off_bslab = P.off_ones + ones_bytes;
        smem_launch = P.off_bslab + bslab_bytes;
        if (smem_launch > (uint32_t)h->smem_optin) return fail(AADFF_E_UNSUPPORTED, "shared memory budget exceeded (TA)");
    }
    if (cl2) {
        grid = (int)std::min<long long>((P.n_tiles + 1) & ~1ll, (long long)(h->num_sms & ~1));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(TC_NT);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute la[1];
        la[0].id = cudaLaunchAttributeClusterDimension;
        la[0].val.clusterDim.x = 2; la[0].val.clusterDim.y = 1; la[0].val.clusterDim.z = 1;
        cfg.attrs = la;
        cfg.numAttrs = 1;
        cudaError_t le = cudaSuccess;
        switch (uni) {
            case 1: le = cudaLaunchKernelEx(&cfg, fused_psfnet_render_kernel<false, false, 1, true>, P); break;
            case 3: le = cudaLaunchKernelEx(&cfg, fused_psfnet_render_kernel<false, false, 3, true>, P); break;
            case 13: le = cudaLaunchKernelEx(&cfg, fused_psfnet_render_kernel<false, false, 13, true>, P); break;
            case 12: le = cudaLaunchKernelEx(&cfg, fused_psfnet_render_kernel<false, false, 12, true>, P); break;
            default: le = cudaLaunchKernelEx(&cfg, fused_psfnet_render_kernel<false, false, 15, true>, P); break;
        }
        if (le != cudaSuccess) return fail(AADFF_E_CUDA, std::string("cluster launch: ") + cudaGetErrorString(le));
    } else if (P.trace != nullptr && P.probes == nullptr) {
        if (ta) fused_psfnet_render_kernel<true, false, 0, false, true><<<grid, TC_NT, smem_launch, st>>>(P);
        else fused_psfnet_render_kernel<true, false, 0><<<grid, TC_NT, smem, st>>>(P);
    } else if (ta) {
        switch (uni) {
            case 12: fused_psfnet_render_kernel<false, false, 12, false, true><<<grid, TC_NT, smem_launch, st>>>(P); break;
            case 13: fused_psfnet_render_kernel<false, false, 13, false, true><<<grid, TC_NT, smem_launch, st>>>(P); break;
            default: fused_psfnet_render_kernel<false, false, 14, false, true><<<grid, TC_NT, smem_launch, st>>>(P); break;
        }
    } else {
#define AADFF_LAUNCH(U)                                                                                   \
        case U:                                                                                           \
            if (P.probes != nullptr) fused_psfnet_render_kernel<false, true, U><<<grid, TC_NT, smem, st>>>(P);   \
            else fused_psfnet_render_kernel<false, false, U><<<grid, TC_NT, smem, st>>>(P);               \
            break;
        switch (uni) {
            AADFF_LAUNCH(1) AADFF_LAUNCH(3) AADFF_LAUNCH(13) AADFF_LAUNCH(12) AADFF_LAUNCH(14) AADFF_LAUNCH(15)
            default:
                if (P.probes != nullptr) fused_psfnet_render_kernel<false, true, 0><<<grid, TC_NT, smem, st>>>(P);
                else fused_psfnet_render_kernel<false, false, 0><<<grid, TC_NT, smem, st>>>(P);
        }
#undef AADFF_LAUNCH
    }
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

static int render_stack_impl(aadff_psfnet_t h, const float* img, const float* depth, const float* foc, int foc_stride,
                             float* out, const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                             float d_max, int mode, void* stream, long long tile_row0 = 0, long long tile_row1 = -1);

int aadff_tile_row_height(void) { return TC_TILE_H; }
int aadff_econ_first_group(void) { return TC_ECON_FIRST_GROUP; }

int aadff_render_stack_rows_f32(aadff_psfnet_t h, const float* img, const float* depth, const float* foc, float* out,
                                const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                                float d_max, int mode, int64_t tile_row_begin, int64_t tile_row_end, void* stream) {
    const long long total = (long long)N * S * ((H + TC_TILE_H - 1) / TC_TILE_H);
    if (tile_row_begin < 0 || tile_row_end < tile_row_begin || tile_row_end > total)
        return fail(AADFF_E_INVALID, "tile-row range outside [0, N*S*ceil(H/8)]");
    return render_stack_impl(h, img, depth, foc, S, out, out_strides, N, C, S, H, W, d_min, d_max, mode, stream,
                             tile_row_begin, tile_row_end);
}

int aadff_render_stack_f32(aadff_psfnet_t h, const float* img, const float* depth, const float* foc, float* out,
                           const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                           float d_max, int mode, void* stream) {
    return render_stack_impl(h, img, depth, foc, S, out, out_strides, N, C, S, H, W, d_min, d_max, mode, stream);
}

static int render_stack_impl(aadff_psfnet_t h, const float* img, const float* depth, const float* foc, int foc_stride,
                             float* out, const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                             float d_max, int mode, void* stream, long long tile_row0, long long tile_row1) {
    if (!h || !img || !depth || !foc || !out || !out_strides) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || S < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (mode < 0 || mode > 5) return fail(AADFF_E_INVALID, "unknown mode");
    if (d_max == d_min) return fail(AADFF_E_INVALID, "d_max == d_min");
    if (N == 0) return AADFF_OK;
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    RenderArgs ra{};
    ra.img = img; ra.depth = depth; ra.foc = foc; ra.out = out;
    ra.os_n = out_strides[0]; ra.os_c = out_strides[1]; ra.os_s = out_strides[2];
    ra.os_h = out_strides[3]; ra.os_w = out_strides[4];
    ra.N = N; ra.S = S; ra.H = H; ra.W = W; ra.ks = h->ks; ra.Ctot = C;
    ra.foc_stride = foc_stride;
    ra.d_min = d_min;
    ra.d_range = d_max - d_min;
    ra.step_x = (W > 1) ? (1.0f - (-1.0f)) / (float)(W - 1) : 0.f;
    ra.step_y = (H > 1) ? (-1.0f - 1.0f) / (float)(H - 1) : 0.f;
    for (int c0 = 0; c0 < C; c0 += 4) {          // PSFs are shared by all channels; > 4 channels -> several passes
        ra.c0 = c0;
        ra.C = std::min(4, C - c0);
        if (mode == AADFF_MODE_FP32) {
            long long M0 = 0, M = (long long)N * S * H * W;
            if (tile_row1 >= 0) {                    // tile row R = (image*S + slice)*tiles_y + ty  ->  flat pixel rows
                const long long tiles_y = (H + TC_TILE_H - 1) / TC_TILE_H;
                auto flat_row = [&](long long R) { return (R / tiles_y) * H + std::min<long long>((R % tiles_y) * TC_TILE_H, H); };
                M0 = flat_row(tile_row0) * W;
                M = flat_row(tile_row1) * W;
            }
            if (M > M0) {
                const int grid = (int)std::min<long long>((M - M0 + F32_TP - 1) / F32_TP, (long long)h->num_sms * 8);
                mlp_fp32_kernel<true><<<grid, F32_NT, F32_SMEM, st>>>(h->f32, ra, nullptr, nullptr, M0, M);
                g_launches.fetch_add(1);
                CUDA_TRY(cudaGetLastError());
            }
        } else {
            int rc = launch_tc(h, ra, mode, st, tile_row0, tile_row1);
            if (rc) return rc;
        }
    }
    return AADFF_OK;
}

int aadff_render_stack_host_f32(aadff_psfnet_t h, const float* img, const float* depth, const float* foc,
                                float* out, int N, int C, int S, int H, int W, float d_min, float d_max, int mode) {
    if (!h || !img || !depth || !foc || !out) return fail(AADFF_E_INVALID, "null argument");
    if (N < 1 || C < 1 || S < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    const size_t n_img = (size_t)N * C * H * W, n_dep = (size_t)N * H * W, n_foc = (size_t)N * S;
    const size_t n_out = n_img * S;
    auto up = [](size_t n) { return (n + 63) / 64 * 64; };
    const size_t need = (up(n_img) + up(n_dep) + up(n_foc) + up(n_out)) * sizeof(float);
    if (!h->ws_stream) CUDA_TRY(cudaStreamCreateWithFlags(&h->ws_stream, cudaStreamNonBlocking));
    if (need > h->ws_bytes) {
        if (h->ws) CUDA_TRY(cudaFree(h->ws));
        h->ws = nullptr;
        h->ws_bytes = 0;
        CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&h->ws), need));
        h->ws_bytes = need;
    }
    float* d_img = h->ws;
    float* d_dep = d_img + up(n_img);
    float* d_foc = d_dep + up(n_dep);
    float* d_out = d_foc + up(n_foc);
    cudaStream_t st = h->ws_stream;
    CUDA_TRY(cudaMemcpyAsync(d_img, img, n_img * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_dep, depth, n_dep * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_foc, foc, n_foc * sizeof(float), cudaMemcpyHostToDevice, st));
    const int64_t strides[5] = {(int64_t)C * S * H * W, (int64_t)S * H * W, (int64_t)H * W, W, 1};
    // One launch per focal slice; the device->host copy of slice s runs on a second stream while the kernel of
    // slice s+1 computes, so only the last slice's copy is exposed.  (A slice is C planes of H*W floats, S*H*W
    // apart, per image: one 2-D copy per image.)
    if (!h->ws_copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&h->ws_copy_stream, cudaStreamNonBlocking));
    if (h->ws_events.size() < (size_t)S) {
        const size_t old = h->ws_events.size();
        h->ws_events.resize(S);
        for (size_t i = old; i < (size_t)S; ++i) CUDA_TRY(cudaEventCreateWithFlags(&h->ws_events[i], cudaEventDisableTiming));
    }
    const size_t plane = (size_t)H * W * sizeof(float);
    for (int s = 0; s < S; ++s) {
        int rc = render_stack_impl(h, d_img, d_dep, d_foc + s, S, d_out + (size_t)s * H * W, strides, N, C, 1, H, W, d_min,
                                   d_max, mode, st);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(h->ws_events[s], st));
        CUDA_TRY(cudaStreamWaitEvent(h->ws_copy_stream, h->ws_events[s], 0));
        for (int n = 0; n < N; ++n) {
            const size_t off = ((size_t)n * C * S + s) * H * W;
            CUDA_TRY(cudaMemcpy2DAsync(out + off, (size_t)S * plane, d_out + off, (size_t)S * plane, plane, C,
                                       cudaMemcpyDeviceToHost, h->ws_copy_stream));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(h->ws_copy_stream));
    CUDA_TRY(cudaStreamSynchronize(st));
    return AADFF_OK;
}

int aadff_psfnet_pred_f32(aadff_psfnet_t h, const float* inp, float* psf, int64_t M, void* stream) {
    if (!h || !inp || !psf) return fail(AADFF_E_INVALID, "null argument");
    if (M < 0) return fail(AADFF_E_INVALID, "negative M");
    if (M == 0) return AADFF_OK;
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    RenderArgs ra{};
    ra.ks = h->ks;
    const int grid = (int)std::min<long long>((M + F32_TP - 1) / F32_TP, (long long)h->num_sms * 8);
    mlp_fp32_kernel<false><<<grid, F32_NT, F32_SMEM, static_cast<cudaStream_t>(stream)>>>(h->f32, ra, inp, psf, 0, M);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_psfnet_pred_tc_f32(aadff_psfnet_t h, const float* inp, float* psf, int64_t M, int mode, void* stream) {
    if (!h || !inp || !psf) return fail(AADFF_E_INVALID, "null argument");
    if (M < 0) return fail(AADFF_E_INVALID, "negative M");
    if (mode == AADFF_MODE_FP32) return aadff_psfnet_pred_f32(h, inp, psf, M, stream);
    if (mode < 0 || mode > 5) return fail(AADFF_E_INVALID, "unknown mode");
    if (reinterpret_cast<uintptr_t>(inp) % 16) return fail(AADFF_E_INVALID, "inp must be 16-byte aligned");
    if (M == 0) return AADFF_OK;
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    RenderArgs ra{};
    ra.ks = h->ks; ra.N = 1; ra.S = 1; ra.H = 1; ra.W = 1; ra.C = 1; ra.Ctot = 1;
    return launch_tc(h, ra, mode, static_cast<cudaStream_t>(stream), 0, -1, inp, psf, (long long)M);
}

int aadff_local_psf_render_f32(const float* img, const float* psf, float* out, int N, int C, int H, int W, int ks,
                               void* stream) {
    if (!img || !psf || !out) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "kernel size must be odd and positive");
    if (N == 0) return AADFF_OK;
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int dbg = g_dbg_flags.load();
    if (ks >= 3 && ks <= STRIP_MAX_KS && !(dbg & (128 | 512)) && W % 4 == 0 && reinterpret_cast<uintptr_t>(psf) % 16 == 0 &&
        reinterpret_cast<uintptr_t>(out) % 8 == 0 && (long long)N * H * ((W + 31) / 32) < (1ll << 40)) {
        // strip-walking kernel (gather_strip_kernel.cuh): bulk-copied PSF rows, per-warp pipelines
        int c0 = 0;
        while (c0 < C) {
            const int cn = (C - c0 >= 3) ? 3 : 1;
            if (!launch_gs_ks<3>(ks, cn, (dbg & 1024) ? 1 : (dbg & 4096) ? 2 : (dbg & 8192) ? 0 : -1, sms, st, img, psf, out, N, C, H, W, c0))
                return fail(AADFF_E_INVALID, "unsupported kernel size");
            g_launches.fetch_add(1);
            CUDA_TRY(cudaGetLastError());
            c0 += cn;
        }
        return AADFF_OK;
    }
    if (ks >= 3 && ks <= 31 && !(g_dbg_flags.load() & 128)) {
        // register-streaming kernel (gather_coalesced_kernel.cuh): any W, any alignment
        const long long tiles = (long long)N * ((H + GC_WARPS - 1) / GC_WARPS) * ((W + GC_TW - 1) / GC_TW);
        if (tiles >= (1ll << 31)) return fail(AADFF_E_INVALID, "image batch too large for one launch");
        const int grid = (int)std::min<long long>(tiles, sms);
        int c0 = 0;
        while (c0 < C) {
            const int cn = (C - c0 >= 3) ? 3 : 1;
            if (!launch_gather_coalesced(ks, cn, grid, st, img, psf, out, N, C, H, W, c0))
                return fail(AADFF_E_INVALID, "unsupported kernel size");
            g_launches.fetch_add(1);
            CUDA_TRY(cudaGetLastError());
            c0 += cn;
        }
        return AADFF_OK;
    }
    const int kk = ks * ks;
    int P = 32;
    while (P > 4 && P * kk * 4 > GS_BUF_BYTES) P >>= 1;
    const bool stream_ok = (W % 4 == 0) && (reinterpret_cast<uintptr_t>(psf) % 16 == 0) && (P * kk * 4 <= GS_BUF_BYTES);
    if (stream_ok) {
        // HBM-streaming path: cp.async.bulk PSF chunks, smem halo tile.  One 16 KB chunk buffer per warp, 8 warps.
        // (Two buffers per warp only fit with 6 warps and measured 20 % slower: the kernel is limited by the
        //  arithmetic/latency of its 8 warps, not by exposed copy latency -- debug flag 64 selects that variant.)
        const int nbuf = (P == 32 && (g_dbg_flags.load() & 64)) ? 2 : 1;
        const int nw = (nbuf == 2) ? GS_TILE_H_2BUF : GS_TILE_H_1BUF;
        const int buf_bytes = (P * kk * 4 + 127) / 128 * 128;
        const int HH = nw + ks - 1, pitch = (GS_TILE_W + ks - 1) | 1;
        const int smem = nw * nbuf * buf_bytes + GS_MAXC * HH * pitch * 4 + 16 * nw;
        if (smem > 48 * 1024) {    // per-device attribute: set on every launch that needs the opt-in
            if (nw == GS_TILE_H_1BUF)
                CUDA_TRY(cudaFuncSetAttribute(local_psf_stream_kernel<GS_TILE_H_1BUF>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            else
                CUDA_TRY(cudaFuncSetAttribute(local_psf_stream_kernel<GS_TILE_H_2BUF>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        }
        const long long tiles = (long long)N * ((H + nw - 1) / nw) * ((W + GS_TILE_W - 1) / GS_TILE_W);
        const int grid = (int)std::min<long long>(tiles, sms);
        for (int c0 = 0; c0 < C; c0 += GS_MAXC) {
            const int cn = std::min(GS_MAXC, C - c0);
            if (nw == GS_TILE_H_1BUF)
                local_psf_stream_kernel<GS_TILE_H_1BUF><<<grid, nw * 32, smem, st>>>(img, psf, out, N, C, H, W, ks, c0, cn,
                                                                                   P, nbuf, buf_bytes);
            else
                local_psf_stream_kernel<GS_TILE_H_2BUF><<<grid, nw * 32, smem, st>>>(img, psf, out, N, C, H, W, ks, c0, cn,
                                                                                   P, nbuf, buf_bytes);
            g_launches.fetch_add(1);
            CUDA_TRY(cudaGetLastError());
        }
        return AADFF_OK;
    }
    const int smem = GATHER_WARPS * 32 * (GATHER_TT + 1) * (int)sizeof(float);
    if (smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(local_psf_render_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const long long items = (long long)N * H * ((W + 31) / 32);
    const int grid = (int)std::min<long long>((items + GATHER_WARPS - 1) / GATHER_WARPS, (long long)sms * 3);
    for (int c0 = 0; c0 < C; c0 += GATHER_MAXC) {
        local_psf_render_kernel<<<grid, GATHER_WARPS * 32, smem, st>>>(img, psf, out, N, C, H, W, ks, c0,
                                                                       std::min(GATHER_MAXC, C - c0));
        g_launches.fetch_add(1);
        CUDA_TRY(cudaGetLastError());
    }
    return AADFF_OK;
}

int aadff_any_negative_f32(const float* x, int64_t n, unsigned char* flag_dev, void* stream) {
    if (!x || !flag_dev || n < 0) return fail(AADFF_E_INVALID, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemsetAsync(flag_dev, 0, 1, st));
    if (n == 0) return AADFF_OK;
    const int grid = (int)std::min<long long>((n + 255) / 256, 592);
    any_negative_kernel<<<grid, 256, 0, st>>>(x, (long long)n, flag_dev);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_thinlens_render_f32(const float* img, const float* depth, const float* foc, float* out, int N, int C, int H,
                              int W, int ks, float foc_len, float fnum, float pixel_size, float d_lo, float d_hi,
                              int flip_sign, const unsigned char* flip_sign_dev, void* stream) {
    if (!img || !depth || !foc || !out) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "kernel size must be odd and positive");
    if (!(fnum > 0.f) || !(pixel_size > 0.f) || !(d_hi > d_lo)) return fail(AADFF_E_INVALID, "bad lens parameters");
    if (N == 0) return AADFF_OK;
    int dev = 0, sms = 0, optin = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    ThinLensArgs a{};
    a.img = img; a.depth = depth; a.foc = foc; a.out = out;
    a.N = N; a.C = C; a.H = H; a.W = W;
    a.k1 = (float)((double)foc_len / (double)fnum);
    a.foc_len = foc_len; a.ps = pixel_size; a.d_lo = d_lo; a.d_hi = d_hi; a.flip = flip_sign ? 1 : 0;
    a.flip_dev = flip_sign_dev;
    if (ks > 31) return fail(AADFF_E_UNSUPPORTED, "thin-lens kernel sizes above 31 are not built");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool two_px = !(g_dbg_flags.load() & 2048);        // 2048: the one-pixel-per-thread kernel (A/B timing)
    const int tl_r = (ks - 1) / 2, tl_sh = (4 - tl_r % 4) % 4;
    const int tile_w = two_px ? TL2_TILE_W : TL_TILE_W;
    const long long tiles = (long long)N * ((H + TL_TILE_H - 1) / TL_TILE_H) * ((W + tile_w - 1) / tile_w);
    if (tiles >= (1ll << 31)) return fail(AADFF_E_INVALID, "image batch too large for one launch");
    const int grid = (int)std::min<long long>(tiles, (long long)sms * 4);
    for (int c0 = 0; c0 < C; c0 += TL_MAXC) {
        a.c0 = c0;
        a.cn = std::min(TL_MAXC, C - c0);
        int HH = TL_TILE_H + ks - 1, BW = (TL_TILE_W + ks - 1 + tl_sh + 3) / 4 * 4;      // = ThinLensCfg<ks>::HH, BW
        int smem = (ks <= 15 ? 2 : 1) * ((a.cn * HH * BW + 31) / 32 * 32) * 4 + 128;      // = ThinLensCfg<ks>::SMEM_BYTES(cn)
        if (two_px && !thinlens2_geometry<1>(ks, a.cn, &BW, &HH, &smem)) return fail(AADFF_E_INVALID, "unsupported kernel size");
        if (smem > optin) return fail(AADFF_E_UNSUPPORTED, "kernel size too large for the shared-memory halo tile");
        // the image halo of interior tiles arrives as one TMA box [cn][HH][BW] of the [N*C, H, W] tensor
        CUtensorMap map;
        std::memset(&map, 0, sizeof(map));
        a.use_tma = make_image_map(&map, img, (long long)N * C, H, W, BW, HH, a.cn) && !(g_dbg_flags.load() & 16);
        const bool launched = two_px ? launch_thinlens2<1>(ks, grid, smem, st, a, map) : launch_thinlens<1>(ks, grid, smem, st, a, map);
        if (!launched) return fail(AADFF_E_INVALID, "unsupported kernel size");
        g_launches.fetch_add(1);
        CUDA_TRY(cudaGetLastError());
    }
    return AADFF_OK;
}

int aadff_render_psf_map_f32(const float* img, const float* psf_map, float* out, int B, int C, int H, int W, int ks,
                             int grid, const int* row_bounds, const int* col_bounds, void* stream) {
    if (!img || !psf_map || !out || !row_bounds || !col_bounds) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || ks > 31 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "PSF kernel size should be odd (and <= 31)");
    if (grid < 1 || grid > PC_MAX_GRID) return fail(AADFF_E_INVALID, "grid must be in [1, 32]");
    if ((ks - 1) / 2 >= H || (ks - 1) / 2 >= W) return fail(AADFF_E_INVALID, "reflect padding needs (ks-1)/2 < H, W");
    if (B == 0) return AADFF_OK;
    PsfConvArgs a{};
    a.img = img; a.psf_map = psf_map; a.out = out;
    a.B = B; a.C = C; a.H = H; a.W = W; a.grid = grid;
    for (int i = 0; i <= grid; ++i) { a.hb[i] = row_bounds[i]; a.wb[i] = col_bounds[i]; }
    if (a.hb[0] != 0 || a.wb[0] != 0 || a.hb[grid] > H || a.wb[grid] > W) return fail(AADFF_E_INVALID, "bad patch bounds");
    for (int i = 0; i < grid; ++i) {
        if (a.hb[i + 1] < a.hb[i] || a.wb[i + 1] < a.wb[i]) return fail(AADFF_E_INVALID, "patch bounds must ascend");
        a.max_ch = std::max(a.max_ch, a.hb[i + 1] - a.hb[i]);
        a.max_cw = std::max(a.max_cw, a.wb[i + 1] - a.wb[i]);
    }
    if (a.max_ch == 0 || a.max_cw == 0) return AADFF_OK;
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const long long tiles = (long long)B * C * grid * grid * ((a.max_ch + PC_TILE_H - 1) / PC_TILE_H) *
                            ((a.max_cw + PC_TILE_W - 1) / PC_TILE_W);
    const int nblk = (int)std::min<long long>(tiles, (long long)sms * 8);
    if (!launch_psf_conv<1>(ks, nblk, static_cast<cudaStream_t>(stream), a)) return fail(AADFF_E_INVALID, "unsupported kernel size");
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_preprocess_rgbd_u8(const uint8_t* bgr, const uint16_t* depth, float* aif_out, float* depth_out, int B, int H, int W,
                             int h, int w, float depth_div, int depth_mode, const float* jitter, const uint8_t* flips,
                             void* stream) {
    if ((!bgr && !depth) || (bgr && !aif_out) || (depth && !depth_out)) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || H < 1 || W < 1 || h < 1 || w < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (depth && !(depth_div > 0.f)) return fail(AADFF_E_INVALID, "depth divisor must be positive");
    if (depth_mode != 0 && depth_mode != 1) return fail(AADFF_E_INVALID, "depth_mode must be 0 (antialias) or 1 (cv2 linear)");
    if (B == 0) return AADFF_OK;
    PreprocessArgs a{};
    a.bgr = bgr; a.depth = depth; a.aif_out = bgr ? aif_out : nullptr; a.depth_out = depth ? depth_out : nullptr;
    a.jitter = jitter; a.flips = flips;
    a.B = B; a.H = H; a.W = W; a.h = h; a.w = w; a.depth_div = depth_div; a.depth_mode = depth_mode;
    const long long per_image = (long long)h * w;
    const dim3 grid((unsigned)std::min<long long>((per_image + 255) / 256, 148 * 16), (unsigned)B);
    if (B > 65535) return fail(AADFF_E_INVALID, "batch too large for one launch");
    preprocess_rgbd_kernel<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_prepare_planes_u8(const uint8_t* bgr, const uint16_t* depth, float* planes, int B, int H, int W, float depth_div,
                            const float* jitter, const uint8_t* flips, void* stream) {
    if ((!bgr && !depth) || !planes) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (depth && !(depth_div > 0.f)) return fail(AADFF_E_INVALID, "depth divisor must be positive");
    if (B > 65535) return fail(AADFF_E_INVALID, "batch too large for one launch");
    if (B == 0) return AADFF_OK;
    PlanesArgs a{};
    a.bgr = bgr; a.depth = depth; a.planes = planes; a.jitter = jitter; a.flips = flips;
    a.B = B; a.H = H; a.W = W; a.P = (bgr ? 3 : 0) + (depth ? 1 : 0); a.depth_div = depth_div;
    const dim3 grid((unsigned)std::min<long long>(((long long)H * W + 255) / 256, 148 * 8), (unsigned)B);
    prepare_planes_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_spline_affine_f32(const float* planes, float* work, float* out, int B, int P, int H, int W, const double* xform,
                            int clamp_plane, void* stream) {
    if (!planes || !work || !out || !xform) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || P < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (clamp_plane >= P) return fail(AADFF_E_INVALID, "clamp_plane out of range");
    if (B > 65535) return fail(AADFF_E_INVALID, "batch too large for one launch");
    if (B == 0) return AADFF_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n = (long long)B * P * H * W;
    float* tmp = work;                 // prefiltered along W
    float* coef = work + n;            // ... and along H
    const unsigned blocks = (unsigned)std::min<long long>((n + 255) / 256, 148 * 16);
    spline_prefilter_kernel<1><<<blocks, 256, 0, st>>>(planes, tmp, (long long)B * P, H, W);
    spline_prefilter_kernel<0><<<blocks, 256, 0, st>>>(tmp, coef, (long long)B * P, H, W);
    AffineArgs a{};
    a.coef = coef; a.raw = planes; a.out = out; a.xform = xform; a.B = B; a.P = P; a.H = H; a.W = W; a.clamp_plane = clamp_plane;
    const dim3 grid((unsigned)std::min<long long>(((long long)H * W + 255) / 256, 148 * 8), (unsigned)B);
    spline_affine_kernel<<<grid, 256, 0, st>>>(a);
    g_launches.fetch_add(3);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_resize_planes_f32(const float* planes, float* aif_out, float* depth_out, int B, int P, int H, int W, int h, int w,
                            int depth_mode, void* stream) {
    if (!planes || (!aif_out && !depth_out)) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || H < 1 || W < 1 || h < 1 || w < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (P != (aif_out ? 3 : 0) + (depth_out ? 1 : 0)) return fail(AADFF_E_INVALID, "P must be 3 (image), 1 (depth) or 4 (both)");
    if (depth_mode != 0 && depth_mode != 1) return fail(AADFF_E_INVALID, "depth_mode must be 0 (antialias) or 1 (cv2 linear)");
    if (B > 65535) return fail(AADFF_E_INVALID, "batch too large for one launch");
    if (B == 0) return AADFF_OK;
    PreprocessArgs a{};
    a.aif_out = aif_out; a.depth_out = depth_out; a.fsrc = planes; a.fsrc_planes = P; a.fsrc_depth_plane = P - 1;
    a.B = B; a.H = H; a.W = W; a.h = h; a.w = w; a.depth_div = 1.f; a.depth_mode = depth_mode;
    const long long per_image = (long long)h * w;
    const dim3 grid((unsigned)std::min<long long>((per_image + 255) / 256, 148 * 16), (unsigned)B);
    preprocess_rgbd_kernel<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

int aadff_select_focus_f32(const float* depth_m, int B, int64_t HW, int num, float* out, void* stream) {
    if (!depth_m || !out) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || HW < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (num <= 3) return fail(AADFF_E_INVALID, "Focal stack size is too small");   // the reference asserts num > 3
    if (B == 0) return AADFF_OK;
    select_focus_kernel<<<B, FOCUS_NT, 0, static_cast<cudaStream_t>(stream)>>>(depth_m, (long long)HW, num, out);
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}


int aadff_trainer_create(const float* const* weights, const float* const* biases, const int* dims, int n_layers,
                         int batch, float beta1, float beta2, float eps, float weight_decay, int device,
                         aadff_trainer_t* out) {
    if (!weights || !biases || !dims || !out) return fail(AADFF_E_INVALID, "null argument");
    if (n_layers < 1 || n_layers > MAX_LAYERS || batch < 1) return fail(AADFF_E_INVALID, "bad n_layers / batch");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select CUDA device " + std::to_string(device));
    aadff_trainer* t = new aadff_trainer();
    t->device = device; t->n_layers = n_layers; t->batch = batch; t->kk = dims[n_layers];
    t->dims.assign(dims, dims + n_layers + 1);
    t->host_hyper.beta1 = beta1; t->host_hyper.beta2 = beta2; t->host_hyper.eps = eps; t->host_hyper.weight_decay = weight_decay;
    size_t off = 0;
    int wmax = 0;
    for (int l = 0; l < n_layers; ++l) {
        t->w_off.push_back(off); off += (size_t)dims[l] * dims[l + 1];
        t->b_off.push_back(off); off += (size_t)dims[l + 1];
        wmax = std::max(wmax, std::max(dims[l], dims[l + 1]));
    }
    t->n_params = off;
#define TR_TRY(expr)                                                                             \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            trainer_free(t);                                                                     \
            return fail(AADFF_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));       \
        }                                                                                        \
    } while (0)
    auto dalloc = [&](float** p, size_t n) { return cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(float)); };
    TR_TRY(dalloc(&t->params, off)); TR_TRY(dalloc(&t->grads, off)); TR_TRY(dalloc(&t->m, off)); TR_TRY(dalloc(&t->v, off));
    TR_TRY(cudaMemset(t->m, 0, off * sizeof(float))); TR_TRY(cudaMemset(t->v, 0, off * sizeof(float)));
    for (int l = 0; l < n_layers; ++l) {
        if (!weights[l] || !biases[l]) { trainer_free(t); return fail(AADFF_E_INVALID, "null layer pointer"); }
        TR_TRY(cudaMemcpy(t->params + t->w_off[l], weights[l], (size_t)dims[l] * dims[l + 1] * sizeof(float), cudaMemcpyHostToDevice));
        TR_TRY(cudaMemcpy(t->params + t->b_off[l], biases[l], (size_t)dims[l + 1] * sizeof(float), cudaMemcpyHostToDevice));
        float* a = nullptr;
        TR_TRY(dalloc(&a, (size_t)batch * dims[l]));
        t->act.push_back(a);
    }
    TR_TRY(dalloc(&t->z, (size_t)batch * t->kk)); TR_TRY(dalloc(&t->p, (size_t)batch * t->kk));
    TR_TRY(dalloc(&t->target, (size_t)batch * t->kk));
    for (int l = 0; l < n_layers; ++l) {
        float* d = nullptr;
        TR_TRY(dalloc(&d, (size_t)batch * dims[l + 1]));
        t->dz.push_back(d);
    }
    (void)wmax;
    TR_TRY(dalloc(&t->loss, 1));
    TR_TRY(cudaMalloc(reinterpret_cast<void**>(&t->hyper), sizeof(AdamHyper)));
    TR_TRY(cudaStreamCreateWithFlags(&t->cap_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) TR_TRY(cudaStreamCreateWithFlags(&t->side[i], cudaStreamNonBlocking));
    for (int i = 0; i < n_layers + 2; ++i) {
        cudaEvent_t ev = nullptr;
        TR_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        t->evs.push_back(ev);
    }
    TR_TRY(cudaStreamBeginCapture(t->cap_stream, cudaStreamCaptureModeThreadLocal));
    const int rc = trainer_record(t, t->cap_stream);
    cudaError_t ce = cudaStreamEndCapture(t->cap_stream, &t->graph);
    if (rc != AADFF_OK || ce != cudaSuccess) { trainer_free(t); return rc ? rc : fail(AADFF_E_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce)); }
    TR_TRY(cudaGraphInstantiate(&t->exec, t->graph, 0));
#undef TR_TRY
    *out = t;
    return AADFF_OK;
}

int aadff_trainer_destroy(aadff_trainer_t t) {
    trainer_free(t);
    return AADFF_OK;
}

int aadff_trainer_step(aadff_trainer_t t, const float* inp, const float* target, float lr, float* loss_out, void* stream) {
    if (!t || !inp || !target) return fail(AADFF_E_INVALID, "null argument");
    DeviceGuard guard(t->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t M = (size_t)t->batch;
    CUDA_TRY(cudaMemcpyAsync(t->act[0], inp, M * t->dims[0] * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(t->target, target, M * t->kk * sizeof(float), cudaMemcpyDeviceToDevice, st));
    t->step += 1;
    AdamHyper h = t->host_hyper;
    h.lr = lr;
    h.bias_correction1 = (float)(1.0 - std::pow((double)h.beta1, (double)t->step));
    h.bias_correction2_sqrt = (float)std::sqrt(1.0 - std::pow((double)h.beta2, (double)t->step));
    train_hyper_kernel<<<1, 1, 0, st>>>(t->hyper, h, t->loss);
    CUDA_TRY(cudaGraphLaunch(t->exec, st));
    g_launches.fetch_add(2 + 3 * t->n_layers * 2);
    if (loss_out) CUDA_TRY(cudaMemcpyAsync(loss_out, t->loss, sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

// which: 0 = parameters, 1 = gradients of the last step, 2 = the last step's predicted PSFs (p into weights[0], [batch, kk])
int aadff_trainer_read(aadff_trainer_t t, int which, float* const* weights, float* const* biases, void* stream) {
    if (!t || !weights) return fail(AADFF_E_INVALID, "null argument");
    DeviceGuard guard(t->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaStreamSynchronize(st));
    if (which == 2) {
        CUDA_TRY(cudaMemcpy(weights[0], t->p, (size_t)t->batch * t->kk * sizeof(float), cudaMemcpyDeviceToHost));
        return AADFF_OK;
    }
    if (which != 0 && which != 1) return fail(AADFF_E_INVALID, "which must be 0, 1 or 2");
    if (!biases) return fail(AADFF_E_INVALID, "null argument");
    const float* src = which == 0 ? t->params : t->grads;
    for (int l = 0; l < t->n_layers; ++l) {
        CUDA_TRY(cudaMemcpy(weights[l], src + t->w_off[l], (size_t)t->dims[l] * t->dims[l + 1] * sizeof(float), cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(biases[l], src + t->b_off[l], (size_t)t->dims[l + 1] * sizeof(float), cudaMemcpyDeviceToHost));
    }
    return AADFF_OK;
}

int aadff_debug_umma_gemm(const float* A, const float* B, float* D, int K, int N, int device) {
    if (!A || !B || !D) return fail(AADFF_E_INVALID, "null argument");
    if (K < 32 || K > 256 || K % 32 || N < 16 || N > 256 || N % 16) return fail(AADFF_E_INVALID, "bad K/N");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    std::vector<__half> pack_all, pack_hi;
    pack_group(B, N, K, 0, N, pack_all);                 // (hi, lo) per slab; keep the hi slabs only
    for (int kc = 0; kc < K / TC_SLAB_K; ++kc)
        pack_hi.insert(pack_hi.end(), pack_all.begin() + (size_t)(2 * kc) * N * TC_SLAB_K,
                       pack_all.begin() + (size_t)(2 * kc + 1) * N * TC_SLAB_K);
    float *dA = nullptr, *dD = nullptr;
    __half* dB = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dA), (size_t)128 * K * 4));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dD), (size_t)128 * N * 4));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dB), pack_hi.size() * 2));
    CUDA_TRY(cudaMemcpy(dA, A, (size_t)128 * K * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(dB, pack_hi.data(), pack_hi.size() * 2, cudaMemcpyHostToDevice));
    const int smem = TC_A_PART_BYTES + 131072 + 64;
    CUDA_TRY(cudaFuncSetAttribute(debug_umma_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    debug_umma_gemm_kernel<<<1, 128, smem>>>(dA, reinterpret_cast<const uint8_t*>(dB), dD, K, N,
                                             (uint32_t)g_desc_swap.load());
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(D, dD, (size_t)128 * N * 4, cudaMemcpyDeviceToHost));
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
    return AADFF_OK;
}


int aadff_debug_econ_round(const float* W, int N, int K, const float* A, int NC, float* out) {
    if (!W || !A || !out || N < 1 || K < 1 || NC < 1) return fail(AADFF_E_INVALID, "bad args");
    std::vector<float> a(A, A + (size_t)NC * K), q;
    if (!gptq_round_fp16(W, N, K, a, NC, q)) return fail(AADFF_E_INVALID, "activation covariance is not positive definite");
    std::memcpy(out, q.data(), q.size() * sizeof(float));
    return AADFF_OK;
}

int aadff_debug_mma_timing(const int* mmas_per_commit, int n_patterns, int reps, int N, int epi_load,
                           uint64_t* out_cycles, int device) {
    if (!mmas_per_commit || !out_cycles || n_patterns < 1 || n_patterns > 16) return fail(AADFF_E_INVALID, "bad args");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    int* d_m = nullptr;
    unsigned long long* d_out = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_m), n_patterns * sizeof(int)));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_out), 64 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemcpy(d_m, mmas_per_commit, n_patterns * sizeof(int), cudaMemcpyHostToDevice));
    uint8_t* d_src = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_src), 65536));
    CUDA_TRY(cudaMemset(d_src, 0, 65536));
    CUDA_TRY(cudaMemset(d_out, 0, 64 * sizeof(unsigned long long)));
    const int smem = TC_A_PART_BYTES + 65536 + 128;
    CUDA_TRY(cudaFuncSetAttribute(debug_mma_timing_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    debug_mma_timing_kernel<<<1, 128, smem>>>(d_out, n_patterns, d_m, reps, N, epi_load, d_src);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(out_cycles, d_out, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    cudaFree(d_src);
    cudaFree(d_m);
    cudaFree(d_out);
    return AADFF_OK;
}

}  // extern "C"
