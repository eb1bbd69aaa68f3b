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
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/aadff.h"
#include "fused_tc_kernel.cuh"
#include "gather_kernel.cuh"
#include "gather_coalesced_kernel.cuh"
#include "gather_strip_kernel.cuh"
#include "mlp_fp32_kernel.cuh"
#include "thinlens_kernel.cuh"
#include "focus_kernel.cuh"
#include "psf_conv_kernel.cuh"
#include "psf_grad_kernel.cuh"
#include "psf_conv_grad_kernel.cuh"
#include "train_kernels.cuh"
#include "mlp_grad_kernel.cuh"
#include "render_grad_kernel.cuh"
#include "preprocess_kernel.cuh"
#include "spline_rotate_kernel.cuh"
#include "econ_calib.h"

using namespace aadff;

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};
std::atomic<int> g_dbg_flags{0};
std::atomic<unsigned long long*> g_trace{nullptr};

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess)                                                                  \
            return fail(AADFF_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));      \
    } while (0)

// Bits of aadff_debug_set_flags (include/aadff.h documents them): cross-check paths that keep results valid, all read
// on the host.
constexpr int DBG_THINLENS_NO_TMA = 16;
constexpr int DBG_ECON_PLAIN_ROUNDING = 256;
constexpr int DBG_NO_STRIP_GATHER = 512;
constexpr int DBG_STRIP_PLAN1 = 1024, DBG_STRIP_PLAN2 = 4096, DBG_STRIP_PLAN0 = 8192;
constexpr int DBG_SMEM_A_OPERANDS = 1 << 20;

template <int V> constexpr std::integral_constant<int, V> ic{};

// f(ic<KS>) for the odd KS in [LO, HI] equal to ks; returns f's status code
template <int LO, int HI, class F>
int with_odd_ks(int ks, F&& f) {
    if constexpr (LO > HI) return fail(AADFF_E_INVALID, "unsupported kernel size");
    else return ks == LO ? f(ic<LO>) : with_odd_ks<LO + 2, HI>(ks, std::forward<F>(f));
}

int counted_launch() {
    g_launches.fetch_add(1);
    CUDA_TRY(cudaGetLastError());
    return AADFF_OK;
}

// One counted launch.  The dynamic-shared-memory opt-in is a per-device attribute, so it is set on every launch that
// needs it (a host-side table write).
template <class... P, class... A>
int launch(void (*kernel)(P...), dim3 grid, int block, int smem, cudaStream_t st, A... args) {
    if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kernel<<<grid, block, smem, st>>>(args...);
    return counted_launch();
}

// SM count (and opt-in shared memory per block) of the current device
int device_sms(int& sms, int* optin = nullptr) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (optin) CUDA_TRY(cudaDeviceGetAttribute(optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    return AADFF_OK;
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

// index into StripPlan<KS>::P: forced by a debug flag, else the widest strips that cover W with <= 10 % padding
int strip_plan(const StripShape (&plans)[3], int W, int dbg) {
    if (dbg & DBG_STRIP_PLAN1) return 1;
    if (dbg & DBG_STRIP_PLAN2) return 2;
    if (dbg & DBG_STRIP_PLAN0) return 0;
    for (int i = 0; i < 3; ++i) {
        const int spx = plans[i].SPX;
        if ((long long)((W + spx - 1) / spx) * spx * 10 <= (long long)W * 11 || spx <= GSW_PX) return i;
    }
    return 2;
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

// Every specialisation of the fused kernel that launch_tc runs.  aadff_psfnet_create sets their shared-memory opt-in,
// launch_tc picks one by <TRACE, PRED, UNI, TA> (fused_tc_kernel.cuh).
using FusedKernel = void (*)(TcParams);
struct FusedVariant { bool trace, pred; int uni; bool ta; FusedKernel fn; };
#define FUSED(TR, PR, U, TA) {TR, PR, U, TA, fused_psfnet_render_kernel<TR, PR, U, TA>}
const FusedVariant FUSED_VARIANTS[] = {
    FUSED(true, false, 0, false), FUSED(true, false, 0, true),                       // traced render
    FUSED(false, false, 0, false), FUSED(false, true, 0, false),                      // render / pred, by UNI
    FUSED(false, false, 1, false), FUSED(false, true, 1, false),
    FUSED(false, false, 3, false), FUSED(false, true, 3, false),
    FUSED(false, false, 12, false), FUSED(false, true, 12, false),
    FUSED(false, false, 13, false), FUSED(false, true, 13, false),
    FUSED(false, false, 14, false), FUSED(false, true, 14, false),
    FUSED(false, false, 15, false), FUSED(false, true, 15, false),
    FUSED(false, false, 12, true), FUSED(false, false, 13, true), FUSED(false, false, 14, true),   // render, TA
};
#undef FUSED

// Arithmetic of each mode: the layer groups from `first` on take `terms` MMA terms, the groups before three.  um is
// the kernel specialisation of that pattern (UNI % 10 in fused_tc_kernel.cuh).
struct TermPattern { int mode, first, terms, um; };
constexpr TermPattern TERM_PATTERNS[] = {
    {AADFF_MODE_PARITY, TC_MAX_GROUPS, 3, 3},           // no group reduced
    {AADFF_MODE_FAST, 0, 1, 1},
    {AADFF_MODE_ECON, TC_ECON_FIRST_GROUP, 2, 2},       // L5.. and the head: fp16 weights
    {AADFF_MODE_ECON8, TC_ECON8_FIRST_GROUP, 2, 4},     // L8, L9 and the head
    {AADFF_MODE_MIXED, TC_MIXED_FIRST_GROUP, 1, 5},
};
static_assert(TC_ECON_FIRST_GROUP == TC_ECON_FIRST_LAYER - 1, "group g holds layer g + 1");

// Shared-memory carve-up of the fused kernel into P's offsets; returns its size.  A operands in shared memory: both
// A parts (hi, lo), `stages` ring stages, one halo slot.  In tensor memory (ta): the ring, the raw head values of the
// tile being gathered (stg_bytes), two halo slots.
uint32_t carve_smem(TcParams& P, bool ta, int stages, uint32_t stg_bytes, uint32_t bias_bytes, uint32_t halo_bytes) {
    P.off_stage = ta ? 0 : 2 * TC_A_PART_BYTES;
    P.off_stg = P.off_stage + stages * TC_STAGE_BYTES;
    P.off_bias = P.off_stg + stg_bytes;
    P.off_w0 = P.off_bias + bias_bytes;
    P.off_halo = (P.off_w0 + 320 * 4 + 15u) & ~15u;
    P.off_red = P.off_halo + (ta ? 2 : 1) * halo_bytes;
    P.off_bar = P.off_red + TC_M * 5 * 4;
    P.off_ones = (P.off_bar + TC_BAR_BYTES + 15u) & ~15u;      // constant A operand of the bias slabs
    P.off_bslab = P.off_ones + 2 * TC_A_LBO;
    return P.off_bslab + 2 * TC_BSLAB_BYTES;                     // bias-slab slot + its block of zeros
}

}  // namespace

struct aadff_psfnet {
    int device = 0, ks = 0, kk = 0, n_layers = 0;
    int num_sms = 0, smem_optin = 0;
    // fp32 (CUDA-core) path
    Fp32Net f32{};
    const float* w_row[MAX_LAYERS]{};       // W [N][K] row-major fp32: the right operand of dZ W in the backward
    std::vector<int> dims;
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
        std::vector<float> wr(weights[l], weights[l] + (size_t)Nf * K);
        float* dr = nullptr;
        rc = upload(wr, &dr);
        if (rc) { aadff_psfnet_destroy(h); return rc; }
        h->owned.push_back(dr);
        h->w_row[l] = dr;
    }
    h->dims.assign(dims, dims + n_layers + 1);
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
        for (const FusedVariant& v : FUSED_VARIANTS)
            CREATE_TRY(cudaFuncSetAttribute(v.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_optin));
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

static int launch_tc(aadff_psfnet_t h, RenderArgs ra, int mode, cudaStream_t st, long long tile_row0 = 0,
                     long long tile_row1 = -1, const float* probes = nullptr, float* psf_out = nullptr,
                     long long n_probes = 0) {
    if (!h->tc_ok) return fail(AADFF_E_UNSUPPORTED, "tensor-core path unavailable: " + h->tc_why + " (use AADFF_MODE_FP32)");
    const bool econ_like = (mode == AADFF_MODE_ECON || mode == AADFF_MODE_ECON8);
    if (econ_like) {
        const int rc = ensure_econ(h);
        if (rc) return rc;
    }
    const int dbg = g_dbg_flags.load();
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
    TermPattern tp = TERM_PATTERNS[0];
    for (const TermPattern& p : TERM_PATTERNS)
        if (p.mode == mode) tp = p;
    if (tp.first >= h->n_groups) tp = TERM_PATTERNS[0];       // no group reduced: the network runs as in parity mode
    bool any_lo = false, all2 = true, aligned = true;
    for (int i = 0; i < h->n_groups; ++i) {
        P.g[i] = h->groups[i];
        const int t = i >= tp.first ? tp.terms : 3;
        P.g[i].terms = t;
        if (econ_like && t == 2 && !(dbg & DBG_ECON_PLAIN_ROUNDING))
            P.g[i].w_off = h->w_off_econ[i];                   // calibrated rounding
        any_lo |= t >= 2;
        all2 &= t >= 2;
        aligned &= ((P.g[i].K / TC_SLAB_K) * (t == 3 ? 2 : 1)) % 4 == 0;
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
    uint32_t halo_bytes = (uint32_t)(TC_TILE_H + ra.ks - 1) * TC_HALO_PITCH * 16;          // float4 per pixel
    if (probes != nullptr) halo_bytes = std::max<uint32_t>(halo_bytes, 8 * 32 * 9 * 4);        // pred mode: the store staging lives there
    const uint32_t bias_bytes = (uint32_t)(h->n_bias - h->head_bias0) * 4;                 // head bias only
    // the deepest weight ring (4..2 stages of 16 KB) that fits, 16 bytes held back for the alignment of the carve-up
    int stages = 4;
    uint32_t smem = 0;
    while (stages >= 2 && (smem = carve_smem(P, false, stages, 0, bias_bytes, halo_bytes)) + 16 > (uint32_t)h->smem_optin)
        --stages;
    if (stages < 2) return fail(AADFF_E_UNSUPPORTED, "shared memory budget exceeded for this kernel size / channel count");
    // no layer needs lo operands (fast mode): the A_lo region doubles the ring to 128 KB, organised as four
    // 32 KB stages (two packed K=32 slabs each) so that every issue iteration queues four MMAs
    P.kslab = (!any_lo && stages == 4) ? 2 : 1;
    P.n_stages = (P.kslab == 2) ? 4 : stages;
    // UNI (fused_tc_kernel.cuh): the specialisation of this launch's term pattern, 0 = per-group terms at run time.
    // +10 when the ring has four stages and every group consumes a multiple of four of them (ring position of a K-step
    // = compile-time); the fast pattern needs the long ring, the reduced ones the aligned ring.
    aligned &= P.n_stages == 4 && P.kslab == 1;
    int um = 0;
    for (const TermPattern& p : TERM_PATTERNS)
        if (p.first == tp.first && p.terms == tp.terms) um = p.um;
    const int uni = um == 3 ? (aligned ? 13 : 3) : um == 1 ? (P.kslab == 2 ? 1 : 0) : aligned ? 10 + um : 0;
    // A operands in tensor memory (fused_tc_kernel.cuh, TA): render launches of the 2-/3-term specialisations with one
    // head block of N <= 192 (ks <= 13) and at least two hidden layers, 4-stage ring.  Its shared memory holds no
    // activations: ring, raw head values of the tile being gathered, two halo slots.  Debug flag 1 << 20 keeps such
    // launches on the shared-memory path (equality tests, A/B timing).
    const uint32_t head_n = h->groups[h->n_hidden].N;
    const bool trace = P.trace != nullptr && P.probes == nullptr;
    const bool ta = P.probes == nullptr && !(dbg & DBG_SMEM_A_OPERANDS) && h->n_groups == h->n_hidden + 1 &&
                    h->n_hidden >= 2 && head_n <= (uint32_t)TC_TA_L1_COL && P.kslab == 1 && P.n_stages == 4 && all2 &&
                    (uni == 12 || uni == 13 || uni == 14 || P.trace != nullptr);
    if (ta) {
        const uint32_t stg_bytes = ((head_n + 31u) & ~31u) * TC_M * 4;      // the gather reads 32-column blocks
        P.halo_bytes = halo_bytes;
        smem = carve_smem(P, true, 4, stg_bytes, bias_bytes, halo_bytes);
        if (smem > (uint32_t)h->smem_optin) return fail(AADFF_E_UNSUPPORTED, "shared memory budget exceeded (TA)");
    }
    FusedKernel kernel = nullptr;
    for (const FusedVariant& v : FUSED_VARIANTS)
        if (v.trace == trace && v.pred == (probes != nullptr) && v.uni == (trace ? 0 : uni) && v.ta == ta) kernel = v.fn;
    if (!kernel) return fail(AADFF_E_UNSUPPORTED, "fused kernel specialisation not built");
    const int grid = (int)std::min<long long>(P.n_tiles, h->num_sms);
    kernel<<<grid, TC_NT, smem, st>>>(P);
    return counted_launch();
}

static int render_stack_impl(aadff_psfnet_t h, const float* img, const float* depth, const float* foc, int foc_stride,
                             float* out, const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                             float d_max, int mode, void* stream, long long tile_row0 = 0,
                             long long tile_row1 = -1) {
    if (!h || !img || !depth || !foc || !out || !out_strides) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || S < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (mode < 0 || mode > AADFF_MODE_ECON8) return fail(AADFF_E_INVALID, "unknown mode");
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
                if (int rc = counted_launch()) return rc;
            }
        } else {
            int rc = launch_tc(h, ra, mode, st, tile_row0, tile_row1);
            if (rc) return rc;
        }
    }
    return AADFF_OK;
}

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
    return counted_launch();
}

int aadff_psfnet_pred_tc_f32(aadff_psfnet_t h, const float* inp, float* psf, int64_t M, int mode, void* stream) {
    if (!h || !inp || !psf) return fail(AADFF_E_INVALID, "null argument");
    if (M < 0) return fail(AADFF_E_INVALID, "negative M");
    if (mode == AADFF_MODE_FP32) return aadff_psfnet_pred_f32(h, inp, psf, M, stream);
    if (mode < 0 || mode > AADFF_MODE_ECON8) return fail(AADFF_E_INVALID, "unknown mode");
    if (reinterpret_cast<uintptr_t>(inp) % 16) return fail(AADFF_E_INVALID, "inp must be 16-byte aligned");
    if (M == 0) return AADFF_OK;
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    RenderArgs ra{};
    ra.ks = h->ks; ra.N = 1; ra.S = 1; ra.H = 1; ra.W = 1; ra.C = 1; ra.Ctot = 1;
    return launch_tc(h, ra, mode, static_cast<cudaStream_t>(stream), 0, -1, inp, psf, (long long)M);
}

}  // extern "C"

// Workspace of aadff_psfnet_backward_f32 for chunks of cp probes: float offsets of each buffer (256-byte aligned).
struct MlpGradLayout {
    int cp = 0, lds = 0, ldz = 0, slices = 0;
    size_t act[MAX_LAYERS]{}, s = 0, ssum = 0, dz[2]{}, part_w = 0, part_b = 0, floats = 0;
};

static MlpGradLayout mlp_grad_layout(const aadff_psfnet* h, long long M) {
    MlpGradLayout g;
    g.cp = (int)std::min<long long>((M + F32_TP - 1) / F32_TP * F32_TP, MG_CHUNK);
    g.slices = (g.cp + MG_SLICE - 1) / MG_SLICE;
    g.lds = (h->kk + 3) / 4 * 4;
    g.ldz = g.lds;
    size_t max_w = 0, max_n = 0;
    for (int l = 0; l < h->n_layers; ++l) {
        g.ldz = std::max(g.ldz, (h->dims[l + 1] + 3) / 4 * 4);
        max_w = std::max(max_w, (size_t)h->dims[l] * h->dims[l + 1]);
        max_n = std::max(max_n, (size_t)h->dims[l + 1]);
    }
    size_t off = 0;
    auto take = [&](size_t n) { const size_t o = off; off += (n + 63) / 64 * 64; return o; };
    for (int l = 1; l < h->n_layers; ++l) g.act[l] = take((size_t)g.cp * h->dims[l]);
    g.s = take((size_t)g.cp * g.lds);
    g.ssum = take((size_t)g.cp);
    g.dz[0] = take((size_t)g.cp * g.ldz);
    g.dz[1] = take((size_t)g.cp * g.ldz);
    g.part_w = take((size_t)g.slices * max_w);
    g.part_b = take((size_t)g.slices * max_n);
    g.floats = off;
    return g;
}

static int grid_blocks(long long n, long long per, long long cap) { return (int)std::min<long long>((n + per - 1) / per, cap); }

// One chunk of the MLP backward below the head, shared by aadff_psfnet_backward_f32 and
// aadff_render_stack_backward_f32.  dZ of the head is in ws + g.dz[0], acts holds the chunk's recomputed activations
// and inp its probes [valid][4].  From the head down to layer `lowest`: each requested dW_l / db_l (partial sums over
// MG_SLICE probes, added to the running total of the earlier chunks unless `first`) and, when grad_inp is not NULL,
// dX = dZ_0 W_0 into grad_inp [valid][4].
static int mlp_backward_layers(const aadff_psfnet* h, const MlpGradLayout& g, float* ws, const MlpActs& acts,
                               const float* inp, int valid, int cp, int lowest, int first, float* const* grad_weights,
                               float* const* grad_biases, float* grad_inp, cudaStream_t st) {
    auto dW = [&](int l) { return grad_weights ? grad_weights[l] : nullptr; };
    auto dB = [&](int l) { return grad_biases ? grad_biases[l] : nullptr; };
    float* part_w = ws + g.part_w;
    float* part_b = ws + g.part_b;
    const int slices = (valid + MG_SLICE - 1) / MG_SLICE;
    int cur = 0;                                     // dz[cur] holds dZ of the layer being processed
    float* dz = ws + g.dz[cur];
    for (int l = h->n_layers - 1; l >= lowest; --l) {
        const int K = h->dims[l], N = h->dims[l + 1], ldz = (N + 3) / 4 * 4;
        const float* act = l ? acts.act[l] : inp;
        if (dW(l)) {                                 // dW_l = dZ_l^T A_l, one partial per probe slice
            const long long n = (long long)N * K;
            if (int rc = launch(mlp_grad_gemm_kernel<false, MG_PLAIN>,
                                dim3((K + MG_BN - 1) / MG_BN, (N + MG_BM - 1) / MG_BM, slices), MG_NT, 0, st,
                                (const float*)dz, (long long)ldz, act, (long long)K, part_w, (long long)K, N, K, valid,
                                MG_SLICE, n, (const float*)nullptr))
                return rc;
            if (int rc = launch(mlp_grad_reduce_kernel, grid_blocks(n, 256, (long long)h->num_sms * 8), 256, 0, st,
                                (const float*)part_w, n, slices, dW(l), first))
                return rc;
        }
        if (dB(l)) {                                 // db_l = column sums of dZ_l, one partial per probe slice
            if (int rc = launch(mlp_colsum_kernel, dim3((N + 255) / 256, slices), 256, 0, st, (const float*)dz, ldz, N,
                                valid, part_b))
                return rc;
            if (int rc = launch(mlp_grad_reduce_kernel, grid_blocks(N, 256, (long long)h->num_sms * 8), 256, 0, st,
                                (const float*)part_b, (long long)N, slices, dB(l), first))
                return rc;
        }
        if (l > lowest) {                            // dZ_{l-1} = (dZ_l W_l) masked by A_l > 0
            float* dz_next = ws + g.dz[cur ^ 1];
            if (int rc = launch(mlp_grad_gemm_kernel<true, MG_RELU_MASK>,
                                dim3((K + MG_BN - 1) / MG_BN, (cp + MG_BM - 1) / MG_BM, 1), MG_NT, 0, st,
                                (const float*)dz, (long long)ldz, h->w_row[l], (long long)K, dz_next, (long long)K,
                                cp, K, N, 0, 0ll, (const float*)acts.act[l]))
                return rc;
            cur ^= 1;
            dz = dz_next;
        } else if (l == 0 && grad_inp) {             // dX = dZ_0 W_0, rows of this chunk
            if (int rc = launch(mlp_grad_gemm_kernel<true, MG_PLAIN>,
                                dim3((K + MG_BN - 1) / MG_BN, (valid + MG_BM - 1) / MG_BM, 1), MG_NT, 0, st,
                                (const float*)dz, (long long)ldz, h->w_row[0], (long long)K, grad_inp, (long long)K,
                                valid, K, N, 0, 0ll, (const float*)nullptr))
                return rc;
        }
    }
    return AADFF_OK;
}

extern "C" {

int64_t aadff_psfnet_backward_work_bytes(aadff_psfnet_t h, int64_t M) {
    if (M < 0) return fail(AADFF_E_INVALID, "M must be >= 0");
    if (!h) return fail(AADFF_E_INVALID, "net is NULL");
    if (M == 0) return 0;
    return (int64_t)(mlp_grad_layout(h, M).floats * sizeof(float));
}

int aadff_psfnet_backward_f32(aadff_psfnet_t h, const float* inp, const float* grad_psf, float* grad_inp,
                              float* const* grad_weights, float* const* grad_biases, void* work, int64_t work_bytes,
                              int64_t M, void* stream) {
    // the checks that need no handle first: they are testable without a device
    if (M < 0) return fail(AADFF_E_INVALID, "M must be >= 0");
    if (!inp) return fail(AADFF_E_INVALID, "inp is NULL");
    if (!grad_psf) return fail(AADFF_E_INVALID, "grad_psf is NULL");
    if (reinterpret_cast<uintptr_t>(inp) % 16) return fail(AADFF_E_INVALID, "inp must be 16-byte aligned");
    if (!grad_inp && !grad_weights && !grad_biases)
        return fail(AADFF_E_INVALID, "no output requested: grad_inp, grad_weights and grad_biases are all NULL");
    if (!h) return fail(AADFF_E_INVALID, "net is NULL");
    const int L = h->n_layers;
    int lowest = grad_inp ? 0 : L;                   // the lowest layer whose dZ is needed
    for (int l = 0; l < L; ++l)
        if ((grad_weights && grad_weights[l]) || (grad_biases && grad_biases[l])) lowest = std::min(lowest, l);
    if (lowest == L)
        return fail(AADFF_E_INVALID, "no output requested: grad_inp and every grad_weights / grad_biases entry are NULL");
    const MlpGradLayout g = mlp_grad_layout(h, M);
    if (M > 0 && !work) return fail(AADFF_E_INVALID, "work is NULL");
    if (M > 0 && work_bytes < (int64_t)(g.floats * sizeof(float)))
        return fail(AADFF_E_INVALID, "work_bytes is smaller than aadff_psfnet_backward_work_bytes(net, M)");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto dW = [&](int l) { return grad_weights ? grad_weights[l] : nullptr; };
    auto dB = [&](int l) { return grad_biases ? grad_biases[l] : nullptr; };
    if (M == 0) {                                    // no probe: the parameter gradients are 0
        for (int l = 0; l < L; ++l) {
            if (dW(l)) CUDA_TRY(cudaMemsetAsync(dW(l), 0, (size_t)h->dims[l] * h->dims[l + 1] * sizeof(float), st));
            if (dB(l)) CUDA_TRY(cudaMemsetAsync(dB(l), 0, (size_t)h->dims[l + 1] * sizeof(float), st));
        }
        return AADFF_OK;
    }
    float* ws = static_cast<float*>(work);
    MlpActs acts{};
    for (int l = 1; l < L; ++l) acts.act[l] = ws + g.act[l];
    acts.s = ws + g.s;
    acts.ssum = ws + g.ssum;
    acts.lds = g.lds;
    auto blocks = grid_blocks;
    for (long long m0 = 0; m0 < M; m0 += MG_CHUNK) {
        const int valid = (int)std::min<long long>(MG_CHUNK, M - m0);
        const int cp = (valid + F32_TP - 1) / F32_TP * F32_TP;
        const int first = m0 == 0;
        acts.cp = cp;
        if (int rc = launch(mlp_fp32_store_kernel, blocks(cp, F32_TP, (long long)h->num_sms * 8), F32_NT, F32_SMEM, st,
                            h->f32, inp, m0, (long long)M, acts))
            return rc;
        float* dz = ws + g.dz[0];
        if (int rc = launch(mlp_head_backward_kernel, blocks(cp, 8, 1ll << 30), 256, 0, st, (const float*)acts.s, g.lds,
                            (const float*)acts.ssum, grad_psf, m0, valid, cp, h->kk, dz, (h->kk + 3) / 4 * 4))
            return rc;
        if (int rc = mlp_backward_layers(h, g, ws, acts, inp + m0 * 4, valid, cp, lowest, first, grad_weights, grad_biases,
                                         grad_inp ? grad_inp + m0 * h->dims[0] : nullptr, st))
            return rc;
    }
    return AADFF_OK;
}

}  // extern "C"

// Workspace of aadff_render_stack_backward_f32 for bands of rows * W pixels: the band's probes, its PSFs (for dimg),
// dX, then the MLP backward's buffers for one chunk of that size (float offsets, 256-byte aligned).
struct RenderGradLayout {
    int rows = 0;
    size_t probes = 0, psf = 0, dx = 0, mlp = 0, floats = 0;
    MlpGradLayout g;
};

static RenderGradLayout render_grad_layout(const aadff_psfnet* h, int H, int W) {
    RenderGradLayout r;
    r.rows = std::min(H, MG_CHUNK / W);
    const size_t px = (size_t)r.rows * W;
    size_t off = 0;
    auto take = [&](size_t n) { const size_t o = off; off += (n + 63) / 64 * 64; return o; };
    r.probes = take(px * 4);
    r.psf = take(px * h->kk);
    r.dx = take(px * 4);
    r.mlp = off;
    r.g = mlp_grad_layout(h, (long long)px);
    r.floats = off + r.g.floats;
    return r;
}

extern "C" {

int64_t aadff_render_stack_backward_work_bytes(aadff_psfnet_t h, int H, int W) {
    if (H < 1 || W < 1) return fail(AADFF_E_INVALID, "H and W must be >= 1");
    if (W > MG_CHUNK) return fail(AADFF_E_INVALID, "W must be <= 16384");
    if (!h) return fail(AADFF_E_INVALID, "net is NULL");
    return (int64_t)(render_grad_layout(h, H, W).floats * sizeof(float));
}

int aadff_render_stack_backward_f32(aadff_psfnet_t h, const float* img, const float* depth, const float* foc,
                                    const float* grad_out, const int64_t grad_out_strides[5], float* grad_img,
                                    float* grad_depth, float* grad_foc, float* const* grad_weights,
                                    float* const* grad_biases, int N, int C, int S, int H, int W, float d_min,
                                    float d_max, int mode, void* work, int64_t work_bytes, void* stream) {
    // the checks that need no handle first: they are testable without a device
    if (N < 0) return fail(AADFF_E_INVALID, "N must be >= 0");
    if (C < 1) return fail(AADFF_E_INVALID, "C must be >= 1");
    if (S < 1) return fail(AADFF_E_INVALID, "S must be >= 1");
    if (H < 1 || W < 1) return fail(AADFF_E_INVALID, "H and W must be >= 1");
    if (W > MG_CHUNK) return fail(AADFF_E_INVALID, "W must be <= 16384");
    if (mode < 0 || mode > AADFF_MODE_ECON8) return fail(AADFF_E_INVALID, "mode is unknown");
    if (!(d_max != d_min)) return fail(AADFF_E_INVALID, "d_max must differ from d_min");
    if (!img) return fail(AADFF_E_INVALID, "img is NULL");
    if (!depth) return fail(AADFF_E_INVALID, "depth is NULL");
    if (!foc) return fail(AADFF_E_INVALID, "foc is NULL");
    if (!grad_out) return fail(AADFF_E_INVALID, "grad_out is NULL");
    if (!grad_out_strides) return fail(AADFF_E_INVALID, "grad_out_strides is NULL");
    if (!grad_img && !grad_depth && !grad_foc && !grad_weights && !grad_biases)
        return fail(AADFF_E_INVALID,
                    "no output requested: grad_img, grad_depth, grad_foc, grad_weights and grad_biases are all NULL");
    // the band buffers inside `work` sit at multiples of 256 bytes from it (float4 probes, tensor-core pred input)
    if (reinterpret_cast<uintptr_t>(work) % 256) return fail(AADFF_E_INVALID, "work must be 256-byte aligned");
    if (!h) return fail(AADFF_E_INVALID, "net is NULL");
    const int L = h->n_layers;
    int lowest = (grad_depth || grad_foc) ? 0 : L;   // the lowest layer whose dZ is needed (L: no MLP backward)
    for (int l = 0; l < L; ++l)
        if ((grad_weights && grad_weights[l]) || (grad_biases && grad_biases[l])) lowest = std::min(lowest, l);
    if (lowest == L && !grad_img)
        return fail(AADFF_E_INVALID, "no output requested: grad_img, grad_depth, grad_foc and every grad_weights / "
                                     "grad_biases entry are NULL");
    const RenderGradLayout rl = render_grad_layout(h, H, W);
    if (N > 0 && !work) return fail(AADFF_E_INVALID, "work is NULL");
    if (N > 0 && work_bytes < (int64_t)(rl.floats * sizeof(float)))
        return fail(AADFF_E_INVALID, "work_bytes is smaller than aadff_render_stack_backward_work_bytes(net, H, W)");
    DeviceGuard guard(h->device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select device");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto dW = [&](int l) { return grad_weights ? grad_weights[l] : nullptr; };
    auto dB = [&](int l) { return grad_biases ? grad_biases[l] : nullptr; };
    if (N == 0) {                                    // no pixel: the parameter gradients are 0
        for (int l = 0; l < L; ++l) {
            if (dW(l)) CUDA_TRY(cudaMemsetAsync(dW(l), 0, (size_t)h->dims[l] * h->dims[l + 1] * sizeof(float), st));
            if (dB(l)) CUDA_TRY(cudaMemsetAsync(dB(l), 0, (size_t)h->dims[l + 1] * sizeof(float), st));
        }
        return AADFF_OK;
    }
    const int64_t* os = grad_out_strides;
    const float d_range = d_max - d_min;
    const float step_x = (W > 1) ? (1.0f - (-1.0f)) / (float)(W - 1) : 0.f;      // as render_stack_impl
    const float step_y = (H > 1) ? (-1.0f - 1.0f) / (float)(H - 1) : 0.f;
    const int r = (h->ks - 1) / 2;
    float* ws = static_cast<float*>(work);
    float* probes = ws + rl.probes;
    float* psf = ws + rl.psf;
    float* dx = ws + rl.dx;
    float* mws = ws + rl.mlp;
    MlpActs acts{};
    for (int l = 1; l < L; ++l) acts.act[l] = mws + rl.g.act[l];
    acts.s = mws + rl.g.s;
    acts.ssum = mws + rl.g.ssum;
    acts.lds = rl.g.lds;
    if (grad_img) CUDA_TRY(cudaMemsetAsync(grad_img, 0, (size_t)N * C * H * W * sizeof(float), st));
    const long long cap = (long long)h->num_sms * 8;
    int first = 1;                                   // first band of the whole call (dW / db start from 0)
    for (int n = 0; n < N; ++n)
        for (int s = 0; s < S; ++s)
            for (int b0 = 0; b0 < H; b0 += rl.rows) {
                const int b1 = std::min(H, b0 + rl.rows), valid = (b1 - b0) * W;
                const int cp = (valid + F32_TP - 1) / F32_TP * F32_TP;
                if (int rc = launch(rg_probe_kernel, grid_blocks(valid, 256, 1ll << 30), 256, 0, st, depth, foc, n, s, S,
                                    H, W, b0, valid, d_min, d_range, step_x, step_y, probes))
                    return rc;
                if (grad_img) {                      // PSFs in the forward's mode, then the transposed gather
                    if (int rc = aadff_psfnet_pred_tc_f32(h, probes, psf, valid, mode, st)) return rc;
                    const long long targets = (long long)(std::min(H, b1 + r) - std::max(0, b0 - r)) * W;
                    if (int rc = launch(rg_grad_img_band_kernel, grid_blocks(targets, 256, cap), 256, 0, st,
                                        (const float*)psf, grad_out, (long long)os[0], (long long)os[1], (long long)os[2],
                                        (long long)os[3], (long long)os[4], grad_img, n, s, C, H, W, h->ks, b0, b1))
                        return rc;
                }
                if (lowest == L) continue;
                acts.cp = cp;
                if (int rc = launch(mlp_fp32_store_kernel, grid_blocks(cp, F32_TP, cap), F32_NT, F32_SMEM, st, h->f32,
                                    (const float*)probes, 0ll, (long long)valid, acts))
                    return rc;
                if (int rc = launch(rg_head_kernel, grid_blocks(cp, 8, 1ll << 30), 256, 0, st, (const float*)acts.s,
                                    rl.g.lds, (const float*)acts.ssum, img, grad_out, (long long)os[0], (long long)os[1],
                                    (long long)os[2], (long long)os[3], (long long)os[4], n, s, C, H, W, h->ks, b0,
                                    valid, cp, mws + rl.g.dz[0], (h->kk + 3) / 4 * 4))
                    return rc;
                const bool need_dx = grad_depth || grad_foc;
                if (int rc = mlp_backward_layers(h, rl.g, mws, acts, probes, valid, cp, lowest, first, grad_weights,
                                                 grad_biases, need_dx ? dx : nullptr, st))
                    return rc;
                if (need_dx)
                    if (int rc = launch(rg_depth_focus_kernel, 1, RG_DF_NT, 0, st, (const float*)dx, depth, foc,
                                        grad_depth, grad_foc, n, s, S, H, W, b0, valid, d_min, d_range, (int)(b0 == 0),
                                        (int)(b1 == H)))
                        return rc;
                first = 0;
            }
    return AADFF_OK;
}

int aadff_local_psf_render_f32(const float* img, const float* psf, float* out, int N, int C, int H, int W, int ks,
                               void* stream) {
    if (!img || !psf || !out) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "kernel size must be odd and positive");
    if (N == 0) return AADFF_OK;
    int sms = 0;
    if (int rc = device_sms(sms)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int dbg = g_dbg_flags.load();
    if (ks >= 3 && ks <= STRIP_MAX_KS && !(dbg & DBG_NO_STRIP_GATHER) && W % 4 == 0 && reinterpret_cast<uintptr_t>(psf) % 16 == 0 &&
        reinterpret_cast<uintptr_t>(out) % 8 == 0 && (long long)N * H * ((W + 31) / 32) < (1ll << 40)) {
        // strip-walking kernel (gather_strip_kernel.cuh): bulk-copied PSF rows, per-warp pipelines
        for (int c0 = 0; c0 < C;) {
            const int cn = (C - c0 >= 3) ? 3 : 1;
            const int rc = with_odd_ks<3, STRIP_MAX_KS>(ks, [&](auto ks_c) {
                constexpr int KS = decltype(ks_c)::value;
                auto run = [&](auto plan_c, auto cn_c) {
                    constexpr StripShape S = StripPlan<KS>::P[decltype(plan_c)::value];
                    constexpr int CN = decltype(cn_c)::value;
                    constexpr int smem = StripCfg<KS, CN, S.SPX>::SMEM_BYTES(S.SL, S.NW);
                    static_assert(smem <= 232448, "strip gather: shared memory plan does not fit");
                    const long long rows = (long long)N * ((W + S.SPX - 1) / S.SPX) * H;
                    return launch(local_psf_strip_kernel<KS, CN, S.SL, S.NW, S.SPX>,
                                  (int)std::min<long long>((rows + S.NW - 1) / S.NW, sms), S.NW * 32, smem, st, img, psf,
                                  out, N, C, H, W, c0);
                };
                auto run_plan = [&](auto plan_c) { return cn == 3 ? run(plan_c, ic<3>) : run(plan_c, ic<1>); };
                const int plan = strip_plan(StripPlan<KS>::P, W, dbg);
                return plan == 1 ? run_plan(ic<1>) : plan == 2 ? run_plan(ic<2>) : run_plan(ic<0>);
            });
            if (rc) return rc;
            c0 += cn;
        }
        return AADFF_OK;
    }
    if (ks >= 3 && ks <= 31) {
        // register-streaming kernel (gather_coalesced_kernel.cuh): any W, any alignment
        const long long tiles = (long long)N * ((H + GC_WARPS - 1) / GC_WARPS) * ((W + GC_TW - 1) / GC_TW);
        if (tiles >= (1ll << 31)) return fail(AADFF_E_INVALID, "image batch too large for one launch");
        const int grid = (int)std::min<long long>(tiles, sms);
        for (int c0 = 0; c0 < C;) {
            const int cn = (C - c0 >= 3) ? 3 : 1;
            const int rc = with_odd_ks<3, 31>(ks, [&](auto ks_c) {
                constexpr int KS = decltype(ks_c)::value;
                auto run = [&](auto cn_c) {
                    constexpr int CN = decltype(cn_c)::value;
                    constexpr int smem = GatherCfg<KS>::SMEM_FLOATS(CN) * (int)sizeof(float);   // <= 69.6 KB (ks = 31, 3 channels)
                    return launch(local_psf_coalesced_kernel<KS, CN>, grid, GC_WARPS * 32, smem, st, img, psf, out, N, C, H,
                                  W, c0);
                };
                return cn == 3 ? run(ic<3>) : run(ic<1>);
            });
            if (rc) return rc;
            c0 += cn;
        }
        return AADFF_OK;
    }
    // any other kernel size (1, or above 31): the generic kernel (gather_kernel.cuh)
    const int smem = GATHER_WARPS * 32 * (GATHER_TT + 1) * (int)sizeof(float);
    const long long items = (long long)N * H * ((W + 31) / 32);
    const int grid = (int)std::min<long long>((items + GATHER_WARPS - 1) / GATHER_WARPS, (long long)sms * 3);
    for (int c0 = 0; c0 < C; c0 += GATHER_MAXC)
        if (int rc = launch(local_psf_render_kernel, grid, GATHER_WARPS * 32, smem, st, img, psf, out, N, C, H, W, ks, c0,
                            std::min(GATHER_MAXC, C - c0)))
            return rc;
    return AADFF_OK;
}

int aadff_local_psf_render_backward_f32(const float* img, const float* psf, const float* grad_out, float* grad_img,
                                        float* grad_psf, int N, int C, int H, int W, int ks, void* stream) {
    if (!img || !psf || !grad_out || (!grad_img && !grad_psf)) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "kernel size must be odd and positive");
    if (N == 0) return AADFF_OK;
    int sms = 0;
    if (int rc = device_sms(sms)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (grad_psf) {
        // the forward strip kernel's conditions (aadff_local_psf_render_f32), and all channels in one halo
        int rc;
        if (ks >= 3 && ks <= STRIP_MAX_KS && C <= GPS_MAXC && W % 4 == 0 &&
            reinterpret_cast<uintptr_t>(grad_psf) % 16 == 0 && reinterpret_cast<uintptr_t>(grad_out) % 8 == 0 &&
            (long long)N * H * ((W + 31) / 32) < (1ll << 40)) {
            rc = with_odd_ks<3, STRIP_MAX_KS>(ks, [&](auto ks_c) {
                constexpr int KS = decltype(ks_c)::value;
                auto run = [&](auto cn_c) {
                    constexpr int CN = decltype(cn_c)::value;
                    using Cfg = GradPsfStripCfg<KS, CN>;
                    static_assert(Cfg::SMEM_BYTES <= GPS_SMEM && Cfg::NW >= 1, "strip dP: shared memory plan does not fit");
                    const long long rows = (long long)N * ((W + GSW_PX - 1) / GSW_PX) * H;
                    return launch(local_psf_grad_psf_strip_kernel<KS, CN>,
                                  (int)std::min<long long>((rows + Cfg::NW - 1) / Cfg::NW, sms), Cfg::NW * 32,
                                  Cfg::SMEM_BYTES, st, img, grad_out, grad_psf, N, H, W);
                };
                switch (C) {
                    case 1: return run(ic<1>);
                    case 2: return run(ic<2>);
                    case 3: return run(ic<3>);
                    case 4: return run(ic<4>);
                    default: return fail(AADFF_E_INVALID, "unsupported kernel size");
                }
            });
        } else {
            const long long total = (long long)N * H * W * ks * ks;
            rc = launch(local_psf_grad_psf_kernel, (int)std::min<long long>((total + 255) / 256, (long long)sms * 16), 256, 0,
                        st, img, grad_out, grad_psf, N, C, H, W, ks);
        }
        if (rc) return rc;
    }
    if (grad_img) {
        const bool strip = ks >= 3 && ks <= STRIP_MAX_KS && W % 4 == 0 && reinterpret_cast<uintptr_t>(psf) % 16 == 0 &&
                           (long long)N * H * ((W + 31) / 32) < (1ll << 40);
        // strip kernel: every pixel without the replicate folds, then rows 0, H-1 and columns 0, W-1 again with them
        const long long px = (long long)N * (strip ? std::min<long long>((long long)H * W, 2ll * (H + W)) : (long long)H * W);
        const int grid = (int)std::min<long long>((px + 255) / 256, (long long)sms * 8);
        for (int c0 = 0; c0 < C;) {
            const int cn = strip ? ((C - c0 >= 3) ? 3 : 1) : std::min(GPS_MAXC, C - c0);
            if (strip) {
                const int rc = with_odd_ks<3, STRIP_MAX_KS>(ks, [&](auto ks_c) {
                    constexpr int KS = decltype(ks_c)::value;
                    auto run = [&](auto cn_c) {
                        using Cfg = GradImgStripCfg<KS, decltype(cn_c)::value>;
                        static_assert(Cfg::SMEM_BYTES <= GPS_SMEM && Cfg::NW >= 1, "strip dimg: shared memory plan does not fit");
                        const long long rows = (long long)N * ((W + GSW_PX - 1) / GSW_PX) * H;
                        return launch(local_psf_grad_img_strip_kernel<KS, decltype(cn_c)::value>,
                                      (int)std::min<long long>((rows + Cfg::NW - 1) / Cfg::NW, sms), Cfg::NW * 32,
                                      Cfg::SMEM_BYTES, st, psf, grad_out, grad_img, N, C, H, W, c0);
                    };
                    return cn == 3 ? run(ic<3>) : run(ic<1>);
                });
                if (rc) return rc;
            }
            if (int rc = launch(local_psf_grad_img_kernel, grid, 256, 0, st, psf, grad_out, grad_img, N, C, H, W, ks, c0, cn,
                                strip ? 1 : 0))
                return rc;
            c0 += cn;
        }
    }
    return AADFF_OK;
}

int aadff_any_negative_f32(const float* x, int64_t n, unsigned char* flag_dev, void* stream) {
    if (!x || !flag_dev || n < 0) return fail(AADFF_E_INVALID, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemsetAsync(flag_dev, 0, 1, st));
    if (n == 0) return AADFF_OK;
    return launch(any_negative_kernel, (int)std::min<long long>((n + 255) / 256, 592), 256, 0, st, x, (long long)n, flag_dev);
}

int aadff_thinlens_render_f32(const float* img, const float* depth, const float* foc, float* out, int N, int C, int H,
                              int W, int ks, float foc_len, float fnum, float pixel_size, float d_lo, float d_hi,
                              int flip_sign, const unsigned char* flip_sign_dev, void* stream) {
    if (!img || !depth || !foc || !out) return fail(AADFF_E_INVALID, "null argument");
    if (N < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "kernel size must be odd and positive");
    if (!(fnum > 0.f) || !(pixel_size > 0.f) || !(d_hi > d_lo)) return fail(AADFF_E_INVALID, "bad lens parameters");
    if (N == 0) return AADFF_OK;
    int sms = 0, optin = 0;
    if (int rc = device_sms(sms, &optin)) return rc;
    ThinLensArgs a{};
    a.img = img; a.depth = depth; a.foc = foc; a.out = out;
    a.N = N; a.C = C; a.H = H; a.W = W;
    a.k1 = (float)((double)foc_len / (double)fnum);
    a.foc_len = foc_len; a.ps = pixel_size; a.d_lo = d_lo; a.d_hi = d_hi; a.flip = flip_sign ? 1 : 0;
    a.flip_dev = flip_sign_dev;
    if (ks > 31) return fail(AADFF_E_UNSUPPORTED, "thin-lens kernel sizes above 31 are not built");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long tiles = (long long)N * ((H + TL_TILE_H - 1) / TL_TILE_H) * ((W + TL2_TILE_W - 1) / TL2_TILE_W);
    if (tiles >= (1ll << 31)) return fail(AADFF_E_INVALID, "image batch too large for one launch");
    const int grid = (int)std::min<long long>(tiles, (long long)sms * 4);
    for (int c0 = 0; c0 < C; c0 += TL_MAXC) {
        a.c0 = c0;
        a.cn = std::min(TL_MAXC, C - c0);
        const int rc = with_odd_ks<1, 31>(ks, [&](auto ks_c) {
            using Cfg = ThinLens2Cfg<decltype(ks_c)::value>;
            const int smem = Cfg::SMEM_BYTES(a.cn);
            if (smem > optin) return fail(AADFF_E_UNSUPPORTED, "kernel size too large for the shared-memory halo tile");
            // the image halo of interior tiles arrives as one TMA box [cn][HH][BW] of the [N*C, H, W] tensor
            CUtensorMap map;
            std::memset(&map, 0, sizeof(map));
            a.use_tma = make_image_map(&map, img, (long long)N * C, H, W, Cfg::BW, Cfg::HH, a.cn) &&
                        !(g_dbg_flags.load() & DBG_THINLENS_NO_TMA);
            return launch(thinlens_render2_kernel<decltype(ks_c)::value>, grid, TL_NT, smem, st, a, map);
        });
        if (rc) return rc;
    }
    return AADFF_OK;
}

}  // extern "C"

// Argument checks shared by aadff_render_psf_map_f32 and its backward (no device call); fills a.
static int psf_map_args(PsfConvArgs& a, int B, int C, int H, int W, int ks, int grid, const int* row_bounds,
                        const int* col_bounds) {
    if (B < 0 || C < 1 || H < 1 || W < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (ks < 1 || ks > 31 || (ks % 2) == 0) return fail(AADFF_E_INVALID, "PSF kernel size should be odd (and <= 31)");
    if (grid < 1 || grid > PC_MAX_GRID) return fail(AADFF_E_INVALID, "grid must be in [1, 32]");
    if ((ks - 1) / 2 >= H || (ks - 1) / 2 >= W) return fail(AADFF_E_INVALID, "reflect padding needs (ks-1)/2 < H, W");
    a.B = B; a.C = C; a.H = H; a.W = W; a.grid = grid;
    a.max_ch = a.max_cw = 0;
    for (int i = 0; i <= grid; ++i) { a.hb[i] = row_bounds[i]; a.wb[i] = col_bounds[i]; }
    if (a.hb[0] != 0 || a.wb[0] != 0 || a.hb[grid] > H || a.wb[grid] > W) return fail(AADFF_E_INVALID, "bad patch bounds");
    for (int i = 0; i < grid; ++i) {
        if (a.hb[i + 1] < a.hb[i] || a.wb[i + 1] < a.wb[i]) return fail(AADFF_E_INVALID, "patch bounds must ascend");
        a.max_ch = std::max(a.max_ch, a.hb[i + 1] - a.hb[i]);
        a.max_cw = std::max(a.max_cw, a.wb[i + 1] - a.wb[i]);
    }
    return AADFF_OK;
}

extern "C" {

int aadff_render_psf_map_f32(const float* img, const float* psf_map, float* out, int B, int C, int H, int W, int ks,
                             int grid, const int* row_bounds, const int* col_bounds, void* stream) {
    if (!img || !psf_map || !out || !row_bounds || !col_bounds) return fail(AADFF_E_INVALID, "null argument");
    PsfConvArgs a{};
    if (int rc = psf_map_args(a, B, C, H, W, ks, grid, row_bounds, col_bounds)) return rc;
    if (B == 0) return AADFF_OK;
    a.img = img; a.psf_map = psf_map; a.out = out;
    if (a.max_ch == 0 || a.max_cw == 0) return AADFF_OK;
    int sms = 0;
    if (int rc = device_sms(sms)) return rc;
    const long long tiles = (long long)B * C * grid * grid * ((a.max_ch + PC_TILE_H - 1) / PC_TILE_H) *
                            ((a.max_cw + PC_TILE_W - 1) / PC_TILE_W);
    const int nblk = (int)std::min<long long>(tiles, (long long)sms * 8);
    return with_odd_ks<1, 31>(ks, [&](auto ks_c) {
        return launch(psf_conv_kernel<decltype(ks_c)::value>, nblk, PC_NT, 0, static_cast<cudaStream_t>(stream), a);
    });
}

// Stage-1 partials of the PSF-map gradient: one ks^2 vector per (channel, cell, image, tile of the largest cell).
static long long psf_map_grad_parts(const PsfConvArgs& a) {
    return (long long)a.B * ((a.max_ch + PC_TILE_H - 1) / PC_TILE_H) * ((a.max_cw + PC_TILE_W - 1) / PC_TILE_W);
}

int64_t aadff_render_psf_map_backward_work_bytes(int B, int C, int H, int W, int ks, int grid, const int* row_bounds,
                                                 const int* col_bounds) {
    if (!row_bounds || !col_bounds) return fail(AADFF_E_INVALID, "null argument");
    PsfConvArgs a{};
    if (int rc = psf_map_args(a, B, C, H, W, ks, grid, row_bounds, col_bounds)) return rc;
    return (int64_t)C * grid * grid * psf_map_grad_parts(a) * ks * ks * (int64_t)sizeof(float);
}

int aadff_render_psf_map_backward_f32(const float* img, const float* psf_map, const float* grad_out, float* grad_img,
                                      float* grad_psf_map, void* work, int64_t work_bytes, int B, int C, int H, int W,
                                      int ks, int grid, const int* row_bounds, const int* col_bounds, void* stream) {
    if (!img || !psf_map || !grad_out || !row_bounds || !col_bounds || (!grad_img && !grad_psf_map) ||
        (grad_psf_map && !work))
        return fail(AADFF_E_INVALID, "null argument");
    PsfConvArgs a{};
    if (int rc = psf_map_args(a, B, C, H, W, ks, grid, row_bounds, col_bounds)) return rc;
    const int64_t need = (int64_t)C * grid * grid * psf_map_grad_parts(a) * ks * ks * (int64_t)sizeof(float);
    if (grad_psf_map && work_bytes < need) return fail(AADFF_E_INVALID, "workspace too small");
    a.img = img; a.psf_map = psf_map; a.out = nullptr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t psf_bytes = (size_t)C * grid * ks * grid * ks * sizeof(float);
    if (B == 0 || a.max_ch == 0 || a.max_cw == 0) {                   // no pixel inside a cell: both gradients are 0
        if (grad_img) CUDA_TRY(cudaMemsetAsync(grad_img, 0, (size_t)B * C * H * W * sizeof(float), st));
        if (grad_psf_map) CUDA_TRY(cudaMemsetAsync(grad_psf_map, 0, psf_bytes, st));
        return AADFF_OK;
    }
    int sms = 0;
    if (int rc = device_sms(sms)) return rc;
    if (grad_img) {
        const long long tiles = (long long)B * C * ((H + PCG_TH - 1) / PCG_TH) * ((W + PCG_TW - 1) / PCG_TW);
        if (int rc = launch(psf_conv_grad_img_kernel, (int)std::min<long long>(tiles, (long long)sms * 8), PC_NT, 0, st, a,
                            grad_out, grad_img, ks))
            return rc;
    }
    if (grad_psf_map) {
        const long long parts = psf_map_grad_parts(a), tiles = (long long)C * grid * grid * parts;
        float* ws = static_cast<float*>(work);
        if (int rc = with_odd_ks<1, 31>(ks, [&](auto ks_c) {
                return launch(psf_conv_grad_psf_kernel<decltype(ks_c)::value>,
                              (int)std::min<long long>(tiles, (long long)sms * 8), PC_NT, 0, st, a, grad_out, ws);
            }))
            return rc;
        const long long warps = (long long)C * grid * grid * ks * ks;
        return launch(psf_conv_grad_reduce_kernel, (int)std::min<long long>((warps + 7) / 8, (long long)sms * 16), 256, 0,
                      st, ws, grad_psf_map, C, grid, ks, parts);
    }
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
    a.B = B; a.H = H; a.W = W; a.h = h; a.w = w; a.depth_div = depth_div;
    const long long per_image = (long long)h * w;
    const dim3 grid((unsigned)std::min<long long>((per_image + 255) / 256, 148 * 16), (unsigned)B);
    if (B > 65535) return fail(AADFF_E_INVALID, "batch too large for one launch");
    return launch(depth_mode == 1 ? preprocess_rgbd_kernel<false, true> : preprocess_rgbd_kernel<false, false>, grid, 256, 0,
                  static_cast<cudaStream_t>(stream), a);
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
    return launch(prepare_planes_kernel, grid, 256, 0, static_cast<cudaStream_t>(stream), a);
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
    if (int rc = launch(spline_prefilter_kernel<1>, blocks, 256, 0, st, planes, tmp, (long long)B * P, H, W)) return rc;
    if (int rc = launch(spline_prefilter_kernel<0>, blocks, 256, 0, st, tmp, coef, (long long)B * P, H, W)) return rc;
    AffineArgs a{};
    a.coef = coef; a.raw = planes; a.out = out; a.xform = xform; a.B = B; a.P = P; a.H = H; a.W = W; a.clamp_plane = clamp_plane;
    const dim3 grid((unsigned)std::min<long long>(((long long)H * W + 255) / 256, 148 * 8), (unsigned)B);
    return launch(spline_affine_kernel, grid, 256, 0, st, a);
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
    a.B = B; a.H = H; a.W = W; a.h = h; a.w = w; a.depth_div = 1.f;
    const long long per_image = (long long)h * w;
    const dim3 grid((unsigned)std::min<long long>((per_image + 255) / 256, 148 * 16), (unsigned)B);
    return launch(depth_mode == 1 ? preprocess_rgbd_kernel<true, true> : preprocess_rgbd_kernel<true, false>, grid, 256, 0,
                  static_cast<cudaStream_t>(stream), a);
}

int aadff_select_focus_f32(const float* depth_m, int B, int64_t HW, int num, float* out, void* stream) {
    if (!depth_m || !out) return fail(AADFF_E_INVALID, "null argument");
    if (B < 0 || HW < 1) return fail(AADFF_E_INVALID, "bad shape");
    if (num <= 3) return fail(AADFF_E_INVALID, "Focal stack size is too small");   // the reference asserts num > 3
    if (B == 0) return AADFF_OK;
    return launch(select_focus_kernel, B, FOCUS_NT, 0, static_cast<cudaStream_t>(stream), depth_m, (long long)HW, num, out);
}


int aadff_trainer_create(const float* const* weights, const float* const* biases, const int* dims, int n_layers,
                         int batch, float beta1, float beta2, float eps, float weight_decay, int device,
                         aadff_trainer_t* out) {
    if (!weights || !biases || !dims || !out) return fail(AADFF_E_INVALID, "null argument");
    if (n_layers < 1 || n_layers > MAX_LAYERS || batch < 1) return fail(AADFF_E_INVALID, "bad n_layers / batch");
    // aadff_psfnet_create's dims rules, except that any kk >= 1 goes (the trainer takes no kernel size): every step
    // copies batch * dims[0] floats from an input documented as [batch, 4]
    if (dims[0] != 4) return fail(AADFF_E_INVALID, "dims must start with 4");
    for (int l = 0; l < n_layers; ++l) {
        if (!weights[l] || !biases[l]) return fail(AADFF_E_INVALID, "null layer pointer");
        if (l + 1 < n_layers && (dims[l + 1] < 8 || dims[l + 1] > 256 || dims[l + 1] % 8))
            return fail(AADFF_E_INVALID, "hidden widths must be multiples of 8 and <= 256");
    }
    if (dims[n_layers] < 1) return fail(AADFF_E_INVALID, "dims must end with kk >= 1");
    // the ranges torch.optim.AdamW accepts
    if (!(beta1 >= 0.f && beta1 < 1.f)) return fail(AADFF_E_INVALID, "beta1 must be in [0, 1)");
    if (!(beta2 >= 0.f && beta2 < 1.f)) return fail(AADFF_E_INVALID, "beta2 must be in [0, 1)");
    if (!(eps >= 0.f && std::isfinite(eps))) return fail(AADFF_E_INVALID, "eps must be finite and >= 0");
    if (!(weight_decay >= 0.f && std::isfinite(weight_decay)))
        return fail(AADFF_E_INVALID, "weight_decay must be finite and >= 0");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(AADFF_E_CUDA, "cannot select CUDA device " + std::to_string(device));
    aadff_trainer* t = new aadff_trainer();
    t->device = device; t->n_layers = n_layers; t->batch = batch; t->kk = dims[n_layers];
    t->dims.assign(dims, dims + n_layers + 1);
    t->host_hyper.beta1 = beta1; t->host_hyper.beta2 = beta2; t->host_hyper.eps = eps; t->host_hyper.weight_decay = weight_decay;
    size_t off = 0;
    for (int l = 0; l < n_layers; ++l) {
        t->w_off.push_back(off); off += (size_t)dims[l] * dims[l + 1];
        t->b_off.push_back(off); off += (size_t)dims[l + 1];
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
    // the scalar first: its check needs no handle, so it is testable without a device or a trainer
    if (!(lr >= 0.f && std::isfinite(lr))) return fail(AADFF_E_INVALID, "lr must be finite and >= 0");
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
    if (int rc = launch(debug_umma_gemm_kernel, 1, 128, TC_A_PART_BYTES + 131072 + 64, nullptr, dA,
                        reinterpret_cast<const uint8_t*>(dB), dD, K, N))
        return rc;
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

}  // extern "C"
