// Fused PSFNet + per-pixel PSF render for sm_100a (tcgen05 / TMEM / bulk-async copies).
//
// Replaces, for one focal stack, the reference's
//   PSFNet.render  (deeplens/psfnet.py:393-441)  -> MLP.forward (deeplens/psfnet_arch.py:24-47)
//   -> local_psf_render (deeplens/render_psf.py:76-107), called S times and stacked
//   (2_aber_aware_dff_aif.py:108-114).
// The per-pixel k x k PSFs exist only in tensor memory and registers.
//
// Work unit: a tile of 8 x 16 = 128 output pixels of one (image, slice); MMA M = 128, one
// TMEM lane per pixel.  A persistent CTA (one per SM) walks tiles round-robin.
//
//   warps 0-7   epilogue/compute (256 threads, two warps per TMEM lane quadrant):
//               layer 0 (4->64) in fp32 FFMA, per-layer epilogue (TMEM -> ReLU + fp16 hi/lo split in
//               the conversions -> K-major smem operand for the next layer; the hidden-layer bias is
//               put into the accumulator by a K=16 "bias slab" MMA), and the head epilogue
//               (sigmoid -> k x k gather from the smem halo tile -> normalise -> store)
//   warp 8      weight producer: streams pre-packed fp16 weight slabs L2 -> smem ring
//               (cp.async.bulk + mbarrier complete_tx), also owns TMEM alloc/dealloc
//   warp 9      MMA issuer: converged warp, an elected lane issues tcgen05.mma (kind::f16,
//               M128 x N<=256 x K16); accumulators ping-pong between TMEM columns [0,256), [256,512)
//   (the two single-thread roles are the highest warp ids on purpose, see TC_WARP_PRODUCER)
//
// Precision: fp16 operands cannot hold the activations/weights to the 1e-4 image tolerance
// (SURVEY.md 7.3), so in parity mode every product is evaluated as
//   A*W ~= Ah*Wh + Al*Wh + Ah*Wl   (Ah = fp16(A), Al = fp16(A - Ah), same for W)
// with fp32 accumulation in TMEM: three tcgen05.mma per K-step.  "terms" is per layer, so
// fast (1-term), econ and mixed modes are the same kernel source; the template parameter UNI
// compiles one variant per arithmetic pattern (see the kernel's comment).
//
// Intra-tile pipelining: the epilogue of layer l hands its output to the MMA warp in 32/64-column
// chunks (a_ready[j]); the MMAs of layer l+1 for K-chunk j start as soon as chunk j is in smem and
// write the *other* accumulator, so the tensor pipe idles only for the first chunk of each epilogue.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include "ptx_sm100.cuh"
#include "render_args.h"

namespace aadff {

constexpr int TC_TILE_H = 8;
constexpr int TC_TILE_W = 16;
constexpr int TC_M = TC_TILE_H * TC_TILE_W;           // 128 pixels = MMA M
constexpr int TC_HALO_PITCH = 48;                     // floats; 48 % 32 == 16 -> 2 tile rows/warp conflict-free
constexpr int TC_HID = 256;
constexpr int TC_SLAB_K = 32;                         // K columns per weight slab (2 MMA K-steps)
constexpr int TC_STAGE_BYTES = TC_HID * TC_SLAB_K * 2;  // 16 KB
constexpr int TC_A_PART_BYTES = TC_M * TC_HID * 2;    // 64 KB: one fp16 [128 x 256] operand
constexpr int TC_A_LBO = TC_M * 16;                   // 2048 B between K-adjacent core matrices of A
constexpr int TC_EPI_WARPS = 8;
constexpr int TC_EPI_THREADS = TC_EPI_WARPS * 32;
constexpr int TC_NT = 64 + TC_EPI_THREADS;            // 320 threads
constexpr int TC_MAX_GROUPS = 16;
constexpr int TC_MAX_STAGES = 8;        // 4 in the stage area (+ 4 in the A_lo region when no layer needs lo parts)
constexpr int TC_MAX_KS = 31;
constexpr int TC_MAX_C = 4;
constexpr int TC_BAR_BYTES = 256;        // mbarriers (2*8 + 8 + 2 + 2 + 2) * 8 B + TMEM slot
constexpr int TC_BSLAB_BYTES = TC_HID * 16;   // K-group 0 of a bias slab (the only non-zero part): 4 KB
constexpr int TC_TRACE_N = 4096;         // trace entries per role
constexpr int TC_MIXED_FIRST_GROUP = 3;  // mixed: groups 0..2 (L1..L3) three terms, one term after
constexpr int TC_ECON_FIRST_GROUP = 4;   // econ: groups 0..3 (L1..L4) three terms, L5.. and the head two (econ_calib.h)
constexpr int TC_ECON8_FIRST_GROUP = 7;  // econ8: groups 0..6 (L1..L7) three terms, L8, L9 and the head two -- the earliest
                                         // start whose adversarial worst case stays under 1e-4 (DESIGN.md section 5)
// TA (A operands in tensor memory): L1's A (K = 64) is written by layer 0 into the last 64 columns of the head's
// accumulator buffer, behind the head's N <= 192 columns; its hand-off uses a_ready barriers 5 and 6, which the 3-term
// barrier map leaves unused, so that layer 0 of the next tile may arrive before the head has consumed barriers 0 and 1
constexpr int TC_TA_L1_COL = TC_HID - 64;
constexpr int TC_TA_L1_BAR = 5;

struct TcGroup {            // one accumulation group: one layer, or one <=256-column block of the head
    uint32_t w_off;         // byte offset of its first slab in the packed weights
    uint16_t K;             // 64 or 256
    uint16_t N;             // MMA N: multiple of 16, <= 256
    uint16_t terms;         // 3 = hi*hi + lo*hi + hi*lo, 2 = hi*hi + lo*hi (fp16 weights), 1 = hi*hi only
    uint16_t bias_off;      // float offset into the bias table
    uint16_t new_a;         // 1: consumes a freshly produced A operand (wait a_ready), 0: reuses it
    uint16_t tap0;          // head blocks: first tap (output feature) of the block
};

struct TcParams {
    RenderArgs ra;
    const uint8_t* wpack;   // fp16 slabs, consumption order
    const float* bias;      // L1..L9 biases then the padded head bias
    const float* w0b0;      // W0 [64][4] then b0 [64]
    TcGroup g[TC_MAX_GROUPS];
    int n_groups, n_hidden; // n_hidden = 9 (L1..L9); the rest are head blocks
    int n_bias, n_stages, kk;
    int bias_skip;          // floats of the bias table that never go to shared memory: the hidden layers' biases are added
                            // by the tensor core (first slab of every hidden group = a K=16 "bias slab", see below)
    int kslab;              // packed K=32 slabs per ring stage: 1 (any 3-term layer) or 2 (fast mode, 32 KB stages)
    int tiles_x, tiles_y;
    long long n_tiles;      // tiles of this launch ...
    long long tile0;        // ... starting at this index of the flattened (image, slice, tile row, tile column) list:
                            // a launch may cover any contiguous run of tile rows (multi-GPU partition, sharding.py)
    // shared-memory byte offsets
    uint32_t off_stage, off_bias, off_w0, off_halo, off_red, off_bar, off_ones;
    uint32_t off_bslab;     // bias-slab slot: [256 x 8] halves (K columns 0..7) + a shared [256 x 8] block of zeros (K 8..15)
    uint32_t off_stg;       // TA: raw head accumulator of the tile being gathered, [head columns / 4][128 rows] float4
    uint32_t halo_bytes;    // TA: one of the two halo slots (tile t is gathered while tile t+1's halo is fetched)
    // pred mode (kernel instantiated with PRED = true): probes [M,4] in, L1-normalised PSFs [M, ks*ks] out
    const float* probes;
    float* psf_out;
    long long n_probes;
    unsigned long long* trace;  // optional [4 roles][TC_TRACE_N] event log of CTA 0 (nullptr = off)
};

// Event trace (debug): role 0 producer, 1 MMA issuer, 2 epilogue warp e=0, 3 epilogue warp e=7.
// Entry = (event code << 40) | (clock64 & 0xFFFFFFFFFF); only CTA 0 records, first TC_TRACE_N events.
template <bool ON>
struct TcTrace {
    unsigned long long* p;
    int n;
    __device__ __forceinline__ void init(unsigned long long* base, int role) {
        if (ON) {
            p = (base != nullptr && blockIdx.x == 0) ? base + role * TC_TRACE_N : nullptr;
            n = 0;
        }
    }
    __device__ __forceinline__ void ev(unsigned code) {
        if (ON) {
            if (p != nullptr && n < TC_TRACE_N)
                p[n++] = ((unsigned long long)code << 40) | ((unsigned long long)clock64() & 0xFFFFFFFFFFull);
        }
    }
};

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

// fp16x2(max(a,0), max(b,0)) in one instruction (F2FP.RELU): ReLU costs nothing where only the hi part is needed
__device__ __forceinline__ uint32_t pack_half2_relu(float a, float b) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));   // upper half <- first source
    return r;
}

// hi half of the ReLU'd split with round-toward-zero: hi <= max(a, 0), so that the remainder a - hi is >= 0 for a > 0
// and < 0 exactly when a < 0 (hi = 0) -- a second cvt.relu then yields lo without an explicit max().  The pair
// (hi, lo) carries 21 bits instead of the 22 of a round-to-nearest split; both are far below the 1e-4 budget.
__device__ __forceinline__ uint32_t pack_half2_relu_rz(float a, float b) {
    uint32_t r;
    asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}

// v[8] (fp32) -> fp16 hi (and lo = fp16(v - hi)) -> one 16-byte row of a K-major core matrix
__device__ __forceinline__ void store_split8(const float (&v)[8], uint32_t addr_hi, uint32_t addr_lo, bool need_lo) {
    uint32_t h[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) h[u] = pack_half2(v[2 * u], v[2 * u + 1]);
    st_shared_v4(addr_hi, h[0], h[1], h[2], h[3]);
    if (need_lo) {
        uint32_t l[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float2 f = __half22float2(*reinterpret_cast<__half2*>(&h[u]));
            l[u] = pack_half2(v[2 * u] - f.x, v[2 * u + 1] - f.y);
        }
        st_shared_v4(addr_lo, l[0], l[1], l[2], l[3]);
    }
}

// 8 accumulator columns -> ReLU, fp16 hi/lo split -> one 16-byte operand row (K-group `kg`)
// (the bias is already in the accumulator: it was put there by the group's bias-slab MMA)
__device__ __forceinline__ void epi_group8(const uint32_t* acc, uint32_t a_hi, uint32_t a_lo,
                                           uint32_t kg, uint32_t a_row, bool need_lo) {
    if (!need_lo) {                          // single-term consumer: ReLU folded into the conversion
        uint32_t h[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) h[u] = pack_half2_relu(__uint_as_float(acc[2 * u]), __uint_as_float(acc[2 * u + 1]));
        st_shared_v4(a_hi + kg * TC_A_LBO + a_row, h[0], h[1], h[2], h[3]);
        return;
    }
    // hi/lo consumer: hi = rz(relu(a)), lo = rn(relu(a - hi))
    uint32_t h[4], l[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float a0 = __uint_as_float(acc[2 * u]), a1 = __uint_as_float(acc[2 * u + 1]);
        h[u] = pack_half2_relu_rz(a0, a1);
        const float2 f = __half22float2(*reinterpret_cast<__half2*>(&h[u]));
        l[u] = pack_half2_relu(a0 - f.x, a1 - f.y);
    }
    const uint32_t off = kg * TC_A_LBO + a_row;
    st_shared_v4(a_hi + off, h[0], h[1], h[2], h[3]);
    st_shared_v4(a_lo + off, l[0], l[1], l[2], l[3]);
}

// TA: one K=16 step of a tensor-memory A operand, written over the 16 accumulator columns it was made from:
// 8 columns of fp16x2 hi, then 8 of lo (the same conversions as epi_group8 with need_lo)
__device__ __forceinline__ void epi_ta16(const uint32_t* acc, uint32_t taddr) {
    uint32_t o[16];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const float a0 = __uint_as_float(acc[2 * u]), a1 = __uint_as_float(acc[2 * u + 1]);
        o[u] = pack_half2_relu_rz(a0, a1);
        const float2 f = __half22float2(*reinterpret_cast<__half2*>(&o[u]));
        o[8 + u] = pack_half2_relu(a0 - f.x, a1 - f.y);
    }
    tmem_st16(taddr, o);
}

// TA: the same for 16 fp32 values from registers (layer 0; the conversions of store_split8 with need_lo)
__device__ __forceinline__ void split_ta16(const float (&v)[16], uint32_t taddr) {
    uint32_t o[16];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        o[u] = pack_half2(v[2 * u], v[2 * u + 1]);
        const float2 f = __half22float2(*reinterpret_cast<__half2*>(&o[u]));
        o[8 + u] = pack_half2(v[2 * u] - f.x, v[2 * u + 1] - f.y);
    }
    tmem_st16(taddr, o);
}

// Warp roles.  The hardware warp arbiter favours the HIGHEST warp id on a scheduler, so the two
// single-thread roles that must react quickly (weight producer, MMA issuer) are the LAST warps of
// the CTA; with low ids they were starved by the ALU-heavy epilogue warps sharing their scheduler
// (measured: ~250 cycles per tcgen05.mma issue, tensor pipe 50 % busy -- profiles/r01_*).
constexpr int TC_WARP_PRODUCER = TC_EPI_WARPS;       // warp 8
constexpr int TC_WARP_MMA = TC_EPI_WARPS + 1;        // warp 9

// UNI specialises the kernel on the arithmetic of the whole network so that the mode-dependent branches disappear
// from the issuing warps (whose instruction streams are the critical path).  UNI % 10 = pattern: 3 = every group three
// terms, kslab 1 (parity); 1 = every group a single term, kslab 2 (fast with the 128 KB ring); 2 = econ (three terms for
// the first TC_ECON_FIRST_GROUP groups, two after); 5 = mixed (three terms for the first TC_MIXED_FIRST_GROUP groups,
// one after); 0 = per-group terms at run time (short rings, the traced build).  UNI >= 10 ("aligned"): the ring has four
// stages and every group consumes a multiple of four, so the ring stage of a K-step is a compile-time constant too.
//
// TA: the activations never touch shared memory.  Each layer's epilogue turns its accumulator into the next layer's A
// operand in the same TMEM columns (epi_ta16), and the MMAs read A from tensor memory.  A group's A therefore lives in
// the other accumulator buffer, so before a group's first MMA the MMA warp also waits for the previous group's
// accumulator: every MMA that read the A in its destination buffer has retired.  Layer 0 of tile t+1 runs under tile
// t's head MMAs, and tile t's head values are copied raw to shared memory (off_stg) so that its sigmoid / gather runs
// after tile t+1's L1 epilogue, under L2's MMAs.  Render kernels with one head block of N <= 192, at least two hidden
// layers and only 2-/3-term groups (host-checked).
template <bool TRACE, bool PRED, int UNI, bool TA = false>
__global__ void __launch_bounds__(TC_NT, 1) fused_psfnet_render_kernel(const __grid_constant__ TcParams P) {
    static_assert(!(TA && PRED), "tensor-memory A operands exist for the render kernels only");
    constexpr int UM = UNI % 10;
    const long long my_iters = (P.n_tiles > blockIdx.x) ? (P.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    constexpr bool ALIGNED = UNI >= 10;
    const int kslab_c = (UM == 3 || UM == 2 || UM == 4 || UM == 5) ? 1 : UM == 1 ? 2 : P.kslab;
    auto terms_of = [&](int gi) -> int {
        return UM == 3 ? 3 : UM == 1 ? 1 : UM == 2 ? (gi < TC_ECON_FIRST_GROUP ? 3 : 2)
                                         : UM == 4 ? (gi < TC_ECON8_FIRST_GROUP ? 3 : 2)
                                         : UM == 5 ? (gi < TC_MIXED_FIRST_GROUP ? 3 : 1) : (int)P.g[gi].terms;
    };
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const RenderArgs& ra = P.ra;

    const uint32_t a_hi = sbase, a_lo = sbase + TC_A_PART_BYTES;
    const uint32_t stage0 = sbase + P.off_stage;
    // ring stage s: first four in the stage area, the rest (fast mode only) in the unused A_lo region
    const int stage_bytes = kslab_c * TC_STAGE_BYTES, stages_in_area = 4 / kslab_c;
    auto stage_addr = [&](int st) {
        return st < stages_in_area ? stage0 + st * stage_bytes : a_lo + (st - stages_in_area) * stage_bytes;
    };
    float* s_bias = reinterpret_cast<float*>(smem + P.off_bias);
    float* s_w0 = reinterpret_cast<float*>(smem + P.off_w0);
    float4* s_halo = reinterpret_cast<float4*>(smem + P.off_halo);   // [HH][48] pixels, channels in .xyzw
    float* s_red = reinterpret_cast<float*>(smem + P.off_red);
    const uint32_t bar0 = sbase + P.off_bar;
    auto bar_full = [&](int s) { return bar0 + 8u * s; };
    auto bar_empty = [&](int s) { return bar0 + 8u * (TC_MAX_STAGES + s); };
    auto bar_aready = [&](int j) { return bar0 + 8u * (2 * TC_MAX_STAGES + j); };
    auto bar_accfull = [&](int b) { return bar0 + 8u * (2 * TC_MAX_STAGES + 8 + b); };
    auto bar_accfree = [&](int b) { return bar0 + 8u * (2 * TC_MAX_STAGES + 10 + b); };
    auto bar_bfull = [&]() { return bar0 + 8u * (2 * TC_MAX_STAGES + 12); };      // bias-slab slot filled / consumed
    auto bar_bempty = [&]() { return bar0 + 8u * (2 * TC_MAX_STAGES + 13); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + P.off_bar + 8 * (2 * TC_MAX_STAGES + 14));
    static_assert(8 * (2 * TC_MAX_STAGES + 14) + 4 <= TC_BAR_BYTES, "barrier area too small");

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_MAX_STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 1); }
        // one per 32-column A chunk.  3-term modes produce chunks 0 and 1 in 16-column steps by all 8 warps
        // (short first hand-off); every other chunk is written by the 4 warps of one column half.
        // Fast mode (kslab 2) hands over 64-column chunks written by all 8 warps.
        for (int j = 0; j < 8; ++j)
            // 3-term modes: barrier 0, 1 = 32-column chunks 0, 1 (all 8 warps, 16-column steps); barrier 2 = chunks
            // 2+3 and barrier 4 = chunks 4..7 (the MMA warp is slower than the epilogue by then, so it only
            // checks at K-steps 0, 1, 2 and 4: every spared wait is ~90 cycles of idle tensor pipe)
            mbar_init(bar_aready(j), (kslab_c == 2 || j < 4 || (TA && (j == TC_TA_L1_BAR || j == TC_TA_L1_BAR + 1)))
                                         ? TC_EPI_WARPS : 2 * TC_EPI_WARPS);
        for (int b = 0; b < 2; ++b) { mbar_init(bar_accfull(b), 1); mbar_init(bar_accfree(b), TC_EPI_WARPS); }
        mbar_init(bar_bfull(), 1);
        mbar_init(bar_bempty(), 1);
        fence_mbar_init();
    }
    for (int i = threadIdx.x; i < P.n_bias - P.bias_skip; i += TC_NT) s_bias[i] = __ldg(P.bias + P.bias_skip + i);
    // constant A operand of the bias slabs: [128 rows x K=16], columns 0 and 1 = 1.0, so that one MMA with the
    // slab B[n][0] = fp16(b_n), B[n][1] = fp16(b_n - B[n][0]) starts the accumulator at the layer's bias
    for (int i = threadIdx.x; i < 2 * TC_M; i += TC_NT) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (i < TC_M) v.x = 0x3C003C00u;                      // halves (1.0, 1.0) in K columns 0, 1
        *reinterpret_cast<uint4*>(smem + P.off_ones + (i < TC_M ? 0 : TC_A_LBO) + (i % TC_M) * 16) = v;
    }
    for (int i = threadIdx.x; i < TC_BSLAB_BYTES / 16; i += TC_NT)            // K columns 8..15 of every bias slab: zeros
        *reinterpret_cast<uint4*>(smem + P.off_bslab + TC_BSLAB_BYTES + i * 16) = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
    for (int i = threadIdx.x; i < 320; i += TC_NT) s_w0[i] = __ldg(P.w0b0 + i);
    if (warp == TC_WARP_PRODUCER) tmem_alloc<512>(smem_u32(const_cast<uint32_t*>(tmem_slot)));
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == TC_WARP_PRODUCER) {
        // =========================================================== weight producer (converged warp)
        int stage = 0;
        uint32_t phase = 0, bphase = 0;
        TcTrace<TRACE> tr; tr.init(lane == 0 ? P.trace : nullptr, 0);
        for (long long iter = 0; iter < my_iters; ++iter) {
            for (int gi = 0; gi < P.n_groups; ++gi) {
                const uint32_t bytes = (uint32_t)P.g[gi].N * (TC_SLAB_K * 2);
                const int nparts = (terms_of(gi) == 3) ? 2 : 1;
                const uint8_t* src = P.wpack + P.g[gi].w_off;
                const int kslab = kslab_c;
                const int nit = P.g[gi].K / (TC_SLAB_K * kslab);
                if (gi < P.n_hidden) {
                    // bias slab: only its K-group 0 (N x 8 halves, 4 KB) is copied, into a dedicated slot (not a ring
                    // stage: every group then consumes a multiple of four stages and the ring position of a K-step is
                    // a compile-time constant in the specialised kernels)
                    mbar_wait(bar_bempty(), bphase ^ 1);
                    if (elect_one_sync()) {
                        mbar_arrive_expect_tx(bar_bfull(), TC_BSLAB_BYTES);
                        bulk_g2s(sbase + P.off_bslab, src, TC_BSLAB_BYTES, bar_bfull());
                    }
                    __syncwarp();
                    bphase ^= 1;
                    src += (uint32_t)P.g[gi].N * 32;             // the packed slab also carries its (all-zero) K-group 1
                }
                for (int it = 0; it < nit; ++it) {
                    // 3-term groups, 4-stage ring: the hi and the lo slab of a K-slab complete ONE barrier (the hi
                    // stage's), so the MMA warp pays one barrier wait per K-slab; the lo stage's own barrier is not used in
                    // that round (the MMA warp keeps one phase bit per stage barrier)
                    uint32_t pair_bar = 0;
                    for (int part = 0; part < nparts; ++part) {
                        mbar_wait(bar_empty(stage), phase ^ 1);
                        tr.ev(0x100 + gi);                       // stage load issued
                        if (part == 0) pair_bar = bar_full(stage);
                        if (elect_one_sync()) {
                            if (nparts == 2 && P.n_stages >= 4) {
                                if (part == 0) mbar_arrive_expect_tx(pair_bar, 2 * bytes);
                                bulk_g2s(stage_addr(stage), src + (size_t)(it * 2 + part) * bytes, bytes, pair_bar);
                            } else {
                                mbar_arrive_expect_tx(bar_full(stage), bytes * kslab);
                                for (int hs = 0; hs < kslab; ++hs)
                                    bulk_g2s(stage_addr(stage) + hs * TC_STAGE_BYTES,
                                             src + (size_t)((it * kslab + hs) * 2 + part) * bytes, bytes, bar_full(stage));
                            }
                        }
                        __syncwarp();
                        if (++stage == P.n_stages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == TC_WARP_MMA) {
        // =========================================================== MMA issuer (converged warp, elected lane)
        int stage = 0;
        uint32_t fbits = 0, aphase = 0, frphase = 0;      // bit s / j / b = parity to wait for next on that barrier
        uint32_t bphase = 0;                               // bias-slab slot
        uint32_t afbits = 0;                               // TA: bit b = parity of accfull(b) to wait for next
        uint32_t gcount = 0;
        TcTrace<TRACE> tr; tr.init(lane == 0 ? P.trace : nullptr, 1);
        // descriptors: everything but the 14-bit start-address field (16-byte units) is loop invariant
        const uint64_t da_hi = umma_smem_desc(a_hi, TC_A_LBO, 128);
        const uint64_t da_lo = umma_smem_desc(a_lo, TC_A_LBO, 128);
        const uint64_t da_ones = umma_smem_desc(sbase + P.off_ones, TC_A_LBO, 128);
        constexpr uint32_t KSTEP_A = (2 * TC_A_LBO) >> 4;            // one K=16 step of A
        constexpr uint32_t STAGE_STEP = TC_STAGE_BYTES >> 4;
        for (long long iter = 0; iter < my_iters; ++iter) {
            for (int gi = 0; gi < P.n_groups; ++gi) {
                const uint32_t gN = P.g[gi].N;
                const bool three = terms_of(gi) == 3;        // Ah*Wh + Al*Wh + Ah*Wl
                const bool use_al = terms_of(gi) >= 2;       // 2 terms: Ah*Wh + Al*Wh (weights rounded to fp16)
                const bool new_a = P.g[gi].new_a != 0;
                const uint32_t buf = gcount & 1;
                if (gcount >= 2) {           // the epilogue must have drained group gcount-2
                    mbar_wait(bar_accfree(buf), (frphase >> buf) & 1);
                    frphase ^= 1u << buf;
                }
                if (TA && gcount >= 1) {     // write-after-read: the MMAs of group gcount-1 read their A from buffer `buf`
                    mbar_wait(bar_accfull(buf ^ 1), (afbits >> (buf ^ 1)) & 1);
                    afbits ^= 1u << (buf ^ 1);
                }
                tc_fence_after_sync();
                tr.ev(0x200 + gi);                               // group start (accumulator free)
                const uint32_t d_tmem = tmem_base + buf * 256;
                // TA: this group's A = the previous group's accumulator, converted in place (L1: layer 0's, see TC_TA_L1_COL)
                const uint32_t a_tmem = tmem_base + (buf ^ 1) * 256 + (gi == 0 ? TC_TA_L1_COL : 0);
                const int abar0 = (TA && gi == 0) ? TC_TA_L1_BAR : 0;
                const uint32_t idesc = umma_idesc_f16_f32(TC_M, gN);
                const uint32_t kstep_b = (2 * gN * 16) >> 4;     // one K=16 step of B: 2 * LBO_B
                const uint64_t db0 = umma_smem_desc(stage0, gN * 16, 128);
                // Issue loop, software-pipelined by one step: the barrier waits of step it+1 (~90 cycles each even
                // when already complete) are performed after the MMAs of step it are queued and BEFORE the commit
                // that drains the pipe, so they overlap MMA execution instead of idling the tensor pipe.
                const int kslab = kslab_c;
                const int nit = P.g[gi].K / (TC_SLAB_K * kslab);
                const bool has_bias = gi < P.n_hidden;
                if (has_bias) {
                    // accumulator := bias (one MMA, constant A operand): needs no activations, so it is issued before
                    // the first a_ready wait and runs inside the hand-off bubble between two layers
                    mbar_wait(bar_bfull(), bphase);
                    bphase ^= 1;
                    tc_fence_after_sync();
                    if (elect_one_sync()) {
                        // B = [256 x 16]: K-group 0 in the slot, K-group 1 = the block of zeros behind it (LBO = 4 KB)
                        umma_f16_ss(d_tmem, da_ones, umma_smem_desc(sbase + P.off_bslab, TC_BSLAB_BYTES, 128), idesc, 0);
                        umma_commit(bar_bempty());
                    }
                    __syncwarp();
                }
                bool pre_waited = false;
                // One K-step of the group as a lambda so that the common K = 256 case can be unrolled with a compile-time
                // `it` (accumulate flag, A-chunk barrier map, operand offsets become constants in the issuing warp)
                auto kstep = [&](const int it) {
                    const int kc = it * kslab;                   // first K=32 slab of this step
                    const uint64_t ah = da_hi + (uint32_t)kc * (2 * KSTEP_A);
                    const uint64_t al = da_lo + (uint32_t)kc * (2 * KSTEP_A);
                    // one MMA with the hi (lo = false) or lo part of A's K=16 step k16 of this slab
                    auto mma_a = [&](bool lo, int k16, uint64_t b, uint32_t acc) {
                        if constexpr (TA) umma_f16_ts(d_tmem, a_tmem + (uint32_t)(kc * 32 + k16 * 16 + (lo ? 8 : 0)), b, idesc, acc);
                        else umma_f16_ss(d_tmem, (lo ? al : ah) + (uint32_t)k16 * KSTEP_A, b, idesc, acc);
                    };
                    if (ALIGNED) stage = (three ? 2 * it : it) & 3;   // groups start at ring position 0 (host-checked)
                    if (!pre_waited) {
                        tr.ev(0x500 + kc);
                        { mbar_wait(bar_full(stage), (fbits >> stage) & 1); fbits ^= 1u << stage; }      // hi weight stage (prefetched long ago)
                        tr.ev(0x600 + kc);
                        // A chunk: 64 columns per barrier in fast mode; barriers 0, 1, 2 (= chunks 2+3), 4 (= 4..7) else
                        if (new_a && (kslab == 2 || it < 3 || it == 4)) {
                            mbar_wait(bar_aready(abar0 + it), (aphase >> (abar0 + it)) & 1);
                            aphase ^= 1u << (abar0 + it);
                            tr.ev(0x400 + kc);
                        }
                    }
                    tc_fence_after_sync();
                    const int hi_stage = stage;
                    const bool last = (it + 1 == nit);
                    auto next_stage = [&](int st) { return ALIGNED ? ((st + 1) & 3) : (st + 1 == P.n_stages ? 0 : st + 1); };
                    if (use_al) {
                        // ---- 2-/3-term groups (kslab == 1): ONE elected block per K-slab -- every extra elect / syncwarp /
                        //      barrier probe in this warp delays the next MMA (its instruction stream is the critical path)
                        stage = next_stage(stage);
                        const bool merged = three && (ALIGNED || P.n_stages >= 4);       // lo bytes arrived with the pair barrier
                        if (elect_one_sync()) {
                            const uint64_t db = (db0 & ~0x3FFFull) | ((stage_addr(hi_stage) & 0x3FFFFu) >> 4);
                            mma_a(false, 0, db, has_bias || it != 0);
                            mma_a(false, 1, db + kstep_b, 1);
                            mma_a(true, 0, db, 1);
                            mma_a(true, 1, db + kstep_b, 1);
                            if (!three) {
                                if (last) umma_commit(bar_accfull(buf));
                                umma_commit(bar_empty(hi_stage));
                            } else {
                                umma_commit(bar_empty(hi_stage));       // release the hi stage early (64 KB ring)
                                if (merged) {
                                    const uint64_t dl = (db0 & ~0x3FFFull) | ((stage_addr(stage) & 0x3FFFFu) >> 4);
                                    mma_a(false, 0, dl, 1);              // Ah*Wl
                                    mma_a(false, 1, dl + kstep_b, 1);
                                    if (last) umma_commit(bar_accfull(buf));
                                    umma_commit(bar_empty(stage));
                                }
                            }
                        }
                        __syncwarp();
                        if (three) {
                            if (!merged) {
                                // short ring (large kernel sizes): one barrier per stage, so that the hi MMAs above run
                                // while the lo slab is still loading
                                { mbar_wait(bar_full(stage), (fbits >> stage) & 1); fbits ^= 1u << stage; }
                                tc_fence_after_sync();
                                if (elect_one_sync()) {
                                    const uint64_t dl = (db0 & ~0x3FFFull) | ((stage_addr(stage) & 0x3FFFFu) >> 4);
                                    mma_a(false, 0, dl, 1);
                                    mma_a(false, 1, dl + kstep_b, 1);
                                    if (last) umma_commit(bar_accfull(buf));
                                    umma_commit(bar_empty(stage));
                                }
                                __syncwarp();
                            }
                            stage = next_stage(stage);
                        }
                        return;
                    }
                    // ---- 1-term groups (fast / the tail of mixed)
                    if (elect_one_sync()) {
                        const uint64_t db = (db0 & ~0x3FFFull) | ((stage_addr(hi_stage) & 0x3FFFFu) >> 4);
                        mma_a(false, 0, db, has_bias || it != 0);
                        mma_a(false, 1, db + kstep_b, 1);
                        if (kslab == 2) {
                            mma_a(false, 2, db + STAGE_STEP, 1);
                            mma_a(false, 3, db + STAGE_STEP + kstep_b, 1);
                        }
                    }
                    __syncwarp();
                    stage = next_stage(stage);
                    // ---- waits of the next step, while the MMAs above execute (before the commit that drains the pipe)
                    pre_waited = false;
                    if (it + 1 < nit) {
                        tr.ev(0x500 + kc + kslab);
                        { mbar_wait(bar_full(stage), (fbits >> stage) & 1); fbits ^= 1u << stage; }
                        if (new_a && (kslab == 2 || it + 1 < 3 || it + 1 == 4)) {     // same barrier map as above
                            mbar_wait(bar_aready(abar0 + it + 1), (aphase >> (abar0 + it + 1)) & 1);
                            aphase ^= 1u << (abar0 + it + 1);
                        }
                        tr.ev(0x400 + kc + kslab);
                        pre_waited = true;
                    }
                    // ---- now the draining commit(s)
                    if (elect_one_sync()) {
                        if (last) umma_commit(bar_accfull(buf));
                        umma_commit(bar_empty(hi_stage));
                    }
                    __syncwarp();
                };
                if (nit == 8) {
#pragma unroll
                    for (int it = 0; it < 8; ++it) kstep(it);
                } else if (nit == 4) {
#pragma unroll
                    for (int it = 0; it < 4; ++it) kstep(it);
                } else {
                    for (int it = 0; it < nit; ++it) kstep(it);
                }
                tr.ev(0x700 + gi);                               // group fully issued
                ++gcount;
            }
        }
    } else {
        // =========================================================== epilogue / compute warps 0..7
        const int e = warp;                     // 0..7
        const int q = warp & 3;                 // TMEM lane quadrant this warp may access
        const int hh = e >> 2;                  // which half of the columns this warp takes
        const int et = e * 32 + lane;           // 0..255
        const int row = q * 32 + lane;          // pixel within the tile = TMEM lane = MMA row
        const int ty = row >> 4, tx = row & 15;
        const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
        const int ks = ra.ks, r = (ks - 1) / 2, kk = P.kk;
        const int HH = TC_TILE_H + ks - 1, HW = TC_TILE_W + ks - 1;
        const int tiles_xy = P.tiles_x * P.tiles_y;
        const uint32_t a_row = (uint32_t)row * 16;
        uint32_t afphase = 0;
        unsigned long long gcount = 0;
        TcTrace<TRACE> tr; tr.init((lane == 0 && (e == 0 || e == 7)) ? P.trace : nullptr, e == 0 ? 2 : 3);
        const float NEG_LOG2E = -1.4426950408889634f;
        const bool fine = kslab_c == 1;         // 16-column first hand-offs (3-term modes)
        // pred mode: one head block of <= 128 columns -> its values fit in registers until the row sum is known
        const bool pred_one_block = PRED && (P.n_groups - P.n_hidden == 1) && (P.g[P.n_hidden].N <= 128);

        // tile -> (image n, slice s, tile origin); depth / focus of this thread's pixel are fetched
        // one tile ahead so that layer 0 (the head of the serial chain) never waits on HBM
        auto tile_coords = [&](long long tile, int& n, int& s, int& h0, int& w0) {
            const long long gt = tile + P.tile0;
            const int txy = (int)(gt % tiles_xy);
            const long long ns = gt / tiles_xy;
            s = (int)(ns % ra.S);
            n = (int)(ns / ra.S);
            h0 = (txy / P.tiles_x) * TC_TILE_H;
            w0 = (txy % P.tiles_x) * TC_TILE_W;
        };
        float4 nx_in = make_float4(0.f, 0.f, 0.f, 0.f);   // pred mode: the probe (x, y, z, foc_z) of this row
        auto fetch_dz = [&](long long tile, float& d, float& f) {
            if (tile < P.n_tiles) {
                if constexpr (PRED) {
                    const long long m = tile * TC_M + row;
                    nx_in = (m < P.n_probes) ? __ldg(reinterpret_cast<const float4*>(P.probes) + m)
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
                } else {
                    int n, s, h0, w0;
                    tile_coords(tile, n, s, h0, w0);
                    const int hc = min(h0 + ty, ra.H - 1), wc = min(w0 + tx, ra.W - 1);
                    d = __ldg(ra.depth + ((long long)n * ra.H + hc) * ra.W + wc);
                    f = __ldg(ra.foc + (long long)n * ra.foc_stride + s);
                }
            }
        };
        float nx_depth = 0.f, nx_foc = 0.f;
        fetch_dz(blockIdx.x, nx_depth, nx_foc);

        // ---- layer 0 (4 -> 64) in fp32 for tile `t`: (x, y, z, foc_z) -> 64 features -> A operand of L1.
        //      Runs one tile AHEAD: right after the previous tile's last head block has retired (the A buffer is
        //      free again) and BEFORE that tile's gather, so the L1 MMAs of tile t overlap the gather of tile t-1.
        //      TA: L1's A goes to columns [TC_TA_L1_COL, +64) of accumulator buffer `ta_buf` (the previous tile's head).
        auto layer0 = [&](long long t, uint32_t ta_buf) {
            float x, y, z, fz;
            if constexpr (PRED) {
                x = nx_in.x; y = nx_in.y; z = nx_in.z; fz = nx_in.w;
            } else {
                int n, s, h0, w0;
                tile_coords(t, n, s, h0, w0);
                x = coord_x(min(w0 + tx, ra.W - 1), ra.W, ra.step_x);
                y = coord_y(min(h0 + ty, ra.H - 1), ra.H, ra.step_y);
                z = depth_to_z(nx_depth, ra.d_min, ra.d_range);
                fz = depth_to_z(nx_foc, ra.d_min, ra.d_range);
            }
            if constexpr (TA) {
                // K=16 steps hh and 2 + hh of L1's A: the features of the fine shared-memory hand-off below
#pragma unroll
                for (int st = 0; st < 2; ++st) {
                    const int k16 = 2 * st + hh;
                    float v[16];
#pragma unroll
                    for (int u = 0; u < 16; ++u) {
                        const int f = k16 * 16 + u;
                        const float4 wv = *reinterpret_cast<const float4*>(s_w0 + f * 4);
                        float a = s_w0[256 + f];
                        a = fmaf(wv.x, x, a); a = fmaf(wv.y, y, a); a = fmaf(wv.z, z, a); a = fmaf(wv.w, fz, a);
                        v[u] = fmaxf(a, 0.f);
                    }
                    split_ta16(v, t_lane + ta_buf * 256 + TC_TA_L1_COL + k16 * 16);
                }
                tmem_st_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) { mbar_arrive(bar_aready(TC_TA_L1_BAR)); mbar_arrive(bar_aready(TC_TA_L1_BAR + 1)); }
                return;
            }
            const bool need_lo = terms_of(0) >= 2;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                // K-group (8 features) computed in this step: a contiguous quarter in fast mode, half of
                // chunk 0 and half of chunk 1 when the chunks are shared by all warps (fine hand-off)
                const int kg = fine ? ((i >> 1) * 4 + 2 * hh + (i & 1)) : (hh * 4 + i);
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int f = kg * 8 + u;
                    const float4 wv = *reinterpret_cast<const float4*>(s_w0 + f * 4);
                    float a = s_w0[256 + f];
                    a = fmaf(wv.x, x, a); a = fmaf(wv.y, y, a); a = fmaf(wv.z, z, a); a = fmaf(wv.w, fz, a);
                    v[u] = fmaxf(a, 0.f);
                }
                const uint32_t off = (uint32_t)kg * TC_A_LBO + a_row;
                store_split8(v, a_hi + off, a_lo + off, need_lo);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                if (fine) { mbar_arrive(bar_aready(0)); mbar_arrive(bar_aready(1)); }
                else mbar_arrive(bar_aready(0));
            }
        };
        if (my_iters > 0) layer0(blockIdx.x, 1u);

        // ---- 32 head columns of this thread's pixel, taps tap_first.. (bias_c: their -log2(e) * bias): sigmoid, gather
        //      from the halo tile (render_psf.py:103-105), accumulated into ssum / cacc
        auto gather32 = [&](const uint32_t (&rr)[32], int tap_first, const float* bias_c, const float4* hbase, float& ssum,
                            float (&cacc)[TC_MAX_C]) {
            int i = tap_first / ks, j = tap_first - i * ks;
            int off = i * TC_HALO_PITCH + j;
            const int nvalid = kk - tap_first;     // >= 32 for every group but the padded last one
            if (nvalid >= 32) {
                // branch-free so that the MUFU / LDS latencies of different taps overlap
#pragma unroll
                for (int u = 0; u < 32; ++u) {
                    const float sg = rcp_approx(1.0f + ex2_approx(fmaf(__uint_as_float(rr[u]), NEG_LOG2E, bias_c[u])));
                    const float4 px = hbase[off];
                    ssum += sg;
                    cacc[0] = fmaf(sg, px.x, cacc[0]);
                    cacc[1] = fmaf(sg, px.y, cacc[1]);
                    cacc[2] = fmaf(sg, px.z, cacc[2]);
                    cacc[3] = fmaf(sg, px.w, cacc[3]);
                    ++off;
                    if (++j == ks) { j = 0; off += TC_HALO_PITCH - ks; }
                }
            } else {
#pragma unroll
                for (int u = 0; u < 32; ++u) {
                    const bool ok = u < nvalid;    // padding columns contribute nothing and read slot 0
                    float sg = rcp_approx(1.0f + ex2_approx(fmaf(__uint_as_float(rr[u]), NEG_LOG2E, bias_c[u])));
                    sg = ok ? sg : 0.f;
                    const float4 px = hbase[ok ? off : 0];
                    ssum += sg;
                    cacc[0] = fmaf(sg, px.x, cacc[0]);
                    cacc[1] = fmaf(sg, px.y, cacc[1]);
                    cacc[2] = fmaf(sg, px.z, cacc[2]);
                    cacc[3] = fmaf(sg, px.w, cacc[3]);
                    ++off;
                    if (++j == ks) { j = 0; off += TC_HALO_PITCH - ks; }
                }
            }
        };
        // ---- combine the two column-halves of each pixel, normalise (F.normalize p=1), store
        auto store_px = [&](float ssum, const float (&cacc)[TC_MAX_C], int n, int s, int h, int w, bool valid) {
            if (hh == 1) {
                s_red[row * 5 + 0] = ssum;
#pragma unroll
                for (int c = 0; c < TC_MAX_C; ++c) s_red[row * 5 + 1 + c] = cacc[c];
            }
            tr.ev(0xD00);                                // gather done
            named_bar_sync(2 + q, 64);
            if (hh == 0 && valid) {
                const float inv = 1.0f / fmaxf(ssum + s_red[row * 5], 1e-12f);
                float* o = ra.out + n * ra.os_n + ra.c0 * ra.os_c + s * ra.os_s + h * ra.os_h + w * ra.os_w;
#pragma unroll
                for (int c = 0; c < TC_MAX_C; ++c)
                    if (c < ra.C) o[c * ra.os_c] = (cacc[c] + s_red[row * 5 + 1 + c]) * inv;
            }
        };

        // ---- TA: gather of this CTA's tile number `piter` from its raw head values (off_stg) and its halo slot
        const int halo_f4 = (int)(P.halo_bytes / 16);
        auto gather_ta = [&](long long piter) {
            int pn, ps, h0, w0;
            tile_coords(blockIdx.x + piter * gridDim.x, pn, ps, h0, w0);
            float ssum = 0.f, cacc[TC_MAX_C] = {0.f, 0.f, 0.f, 0.f};
            const float4* hbase = s_halo + (piter & 1) * halo_f4 + ty * TC_HALO_PITCH + tx;
            const float4* stg = reinterpret_cast<const float4*>(smem + P.off_stg) + row;
            const int gi = P.n_hidden;
            const float* bias = s_bias + (P.g[gi].bias_off - P.bias_skip);
#pragma unroll 1
            for (int c32 = hh * 32; c32 < P.g[gi].N; c32 += 64) {
                uint32_t rr[32];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float4 v = stg[(c32 / 4 + k) * TC_M];
                    rr[4 * k] = __float_as_uint(v.x); rr[4 * k + 1] = __float_as_uint(v.y);
                    rr[4 * k + 2] = __float_as_uint(v.z); rr[4 * k + 3] = __float_as_uint(v.w);
                }
                gather32(rr, P.g[gi].tap0 + c32, bias + c32, hbase, ssum, cacc);
            }
            store_px(ssum, cacc, pn, ps, h0 + ty, w0 + tx, (h0 + ty < ra.H) && (w0 + tx < ra.W));
        };

        long long tile = blockIdx.x;
        for (long long iter = 0; iter < my_iters; ++iter, tile += gridDim.x) {
            int n = 0, s = 0, h0 = 0, w0 = 0;
            if constexpr (!PRED) tile_coords(tile, n, s, h0, w0);
            const int h = h0 + ty, w = w0 + tx;
            const long long m_row = tile * TC_M + row;      // pred mode: probe index of this thread's row
            const bool valid = PRED ? (m_row < P.n_probes) : ((h < ra.H) && (w < ra.W));
            tr.ev(0x800);                                // tile start (its layer 0 is already done)
            fetch_dz(tile + gridDim.x, nx_depth, nx_foc);    // depth / focus of the next tile, used by layer0 below

            // The halo tile (replicate-clamped, render_psf.py:96) is only needed by the gather at the end of the
            // tile: its pixels are fetched one per thread per hidden layer -- the global loads are issued before
            // the accumulator wait and stored to smem after the layer's epilogue, so they cost no time.
            // (TA: two halo slots; the slot of this tile was last read by the gather of tile iter-2, which every
            // thread finished before the "halo tile complete" barrier of tile iter-1)
            if (!TA) named_bar_sync(1, TC_EPI_THREADS);  // previous tile's gather is done with halo/red
            float4* const s_halo_t = s_halo + (TA ? (int)(iter & 1) * halo_f4 : 0);
            const float* img_n = ra.img + ((long long)n * ra.Ctot + ra.c0) * ra.H * ra.W;
            const long long cstride = (long long)ra.H * ra.W;
            auto halo_fetch = [&](int idx, float4& v) -> int {       // returns the smem slot or -1
                if (PRED || idx >= HH * HW) return -1;
                const int yy = idx / HW, xx = idx - yy * HW;
                const int gy = min(max(h0 + yy - r, 0), ra.H - 1), gx = min(max(w0 + xx - r, 0), ra.W - 1);
                const float* px = img_n + (long long)gy * ra.W + gx;
                v.x = __ldg(px);
                v.y = ra.C > 1 ? __ldg(px + cstride) : 0.f;
                v.z = ra.C > 2 ? __ldg(px + 2 * cstride) : 0.f;
                v.w = ra.C > 3 ? __ldg(px + 3 * cstride) : 0.f;
                return yy * TC_HALO_PITCH + xx;
            };

            // ---- hidden layers L1..L9: accumulator -> bias, ReLU, split -> A operand of the next layer.
            //      TMEM reads are software-pipelined one 32-column chunk ahead of the arithmetic.
            for (int gi = 0; gi < P.n_hidden; ++gi) {
                const int buf = (int)(gcount & 1);
                float4 hv = make_float4(0.f, 0.f, 0.f, 0.f);
                const int hslot = halo_fetch(gi * TC_EPI_THREADS + et, hv);
                tr.ev(0xA00 + gi);                           // start waiting for accumulator gi
                mbar_wait(bar_accfull(buf), (afphase >> buf) & 1);
                afphase ^= 1u << buf;
                tc_fence_after_sync();
                tr.ev(0xB00 + gi);                           // accumulator gi complete
                const bool need_lo = terms_of(gi + 1) >= 2;
                const uint32_t t_acc = t_lane + buf * 256;
                uint32_t rr[2][32], rf[2][16];
                if constexpr (TA) {
                    // the same column map and hand-offs, converted in place: 16 accumulator columns -> one K=16 step of
                    // the next layer's A (8 columns hi, 8 lo); only this thread's lane is read and written
                    tmem_ld16(t_acc + hh * 16, rf[0]);
                    tmem_ld16(t_acc + 32 + hh * 16, rf[1]);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        tmem_ld_wait();
                        if (j < 3) tmem_ld32(t_acc + (j + 1) * 64 + hh * 32, rr[(j + 1) & 1]);
                        if (j == 0) {
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                epi_ta16(rf[c], t_acc + c * 32 + hh * 16);
                                tmem_st_wait();
                                tc_fence_before_sync();
                                __syncwarp();
                                if (lane == 0) mbar_arrive(bar_aready(c));
                            }
                        } else {
                            const int col = j * 64 + hh * 32;
                            epi_ta16(&rr[j & 1][0], t_acc + col);
                            epi_ta16(&rr[j & 1][16], t_acc + col + 16);
                            tmem_st_wait();
                            tc_fence_before_sync();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(bar_aready(j == 1 ? 2 : 4));
                        }
                        tr.ev(0xC00 + j);
                    }
                } else {
                    if (fine) {
                        tmem_ld16(t_acc + hh * 16, rf[0]);          // my 16 columns of chunk 0 ...
                        tmem_ld16(t_acc + 32 + hh * 16, rf[1]);     // ... and of chunk 1
                    } else {
                        tmem_ld32(t_acc + hh * 32, rr[0]);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        tmem_ld_wait();
                        if (j < 3) tmem_ld32(t_acc + (j + 1) * 64 + hh * 32, rr[(j + 1) & 1]);
                        if (j == 0 && fine) {
#pragma unroll
                            for (int c = 0; c < 2; ++c) {
                                const int col = c * 32 + hh * 16;
#pragma unroll
                                for (int i = 0; i < 2; ++i)
                                    epi_group8(&rf[c][i * 8], a_hi, a_lo, col / 8 + i, a_row, need_lo);
                                fence_proxy_async_smem();
                                __syncwarp();
                                if (lane == 0) mbar_arrive(bar_aready(c));
                            }
                        } else {
                            const int col = j * 64 + hh * 32;
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                epi_group8(&rr[j & 1][i * 8], a_hi, a_lo, col / 8 + i, a_row, need_lo);
                            fence_proxy_async_smem();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(bar_aready(fine ? (j == 1 ? 2 : 4) : j));
                        }
                        tr.ev(0xC00 + j);                        // columns of 64-group j handed to the MMA warp
                    }
                }
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_accfree(buf));
                if (hslot >= 0) s_halo_t[hslot] = hv;
                ++gcount;
                if constexpr (TA) {
                    if (gi == 0 && iter > 0) gather_ta(iter - 1);       // under L2's MMAs
                    if (gi == P.n_hidden - 1 && iter + 1 < my_iters) {
                        // under the head's MMAs: the last MMA that read the columns layer 0 writes (L9's) has retired
                        layer0(tile + gridDim.x, (uint32_t)(gcount & 1));
                        tr.ev(0x900);
                    }
                }
            }
            for (int idx = P.n_hidden * TC_EPI_THREADS + et; !PRED && idx < HH * HW; idx += TC_EPI_THREADS) {   // remainder
                float4 hv;
                const int hslot = halo_fetch(idx, hv);
                s_halo_t[hslot] = hv;
            }
            named_bar_sync(1, TC_EPI_THREADS);           // halo tile complete (all warps stored their share)

            if constexpr (TA) {
                // ---- head: raw accumulator -> off_stg, buffer released at once; sigmoid and gather follow tile
                //      t+1's L1 epilogue (gather_ta).  Each thread later reads back only what it wrote here.
                const int buf = (int)(gcount & 1), gi = P.n_hidden;
                tr.ev(0xA00 + gi);
                mbar_wait(bar_accfull(buf), (afphase >> buf) & 1);
                afphase ^= 1u << buf;
                tc_fence_after_sync();
                tr.ev(0xB00 + gi);
                float4* stg = reinterpret_cast<float4*>(smem + P.off_stg) + row;
#pragma unroll 1
                for (int c32 = hh * 32; c32 < P.g[gi].N; c32 += 64) {
                    uint32_t rr[32];
                    tmem_ld32(t_lane + buf * 256 + c32, rr);
                    tmem_ld_wait();
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        stg[(c32 / 4 + k) * TC_M] = make_float4(__uint_as_float(rr[4 * k]), __uint_as_float(rr[4 * k + 1]),
                                                                __uint_as_float(rr[4 * k + 2]), __uint_as_float(rr[4 * k + 3]));
                }
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_accfree(buf));
                ++gcount;
                continue;
            }

            // ---- head blocks: sigmoid, gather from the halo tile (render_psf.py:103-105)
            //      The bias table holds -log2(e) * bias for the head, so exp(-(acc + b)) is one FFMA + EX2.
            float ssum = 0.f, cacc[TC_MAX_C] = {0.f, 0.f, 0.f, 0.f};
            const float4* hbase = s_halo_t + ty * TC_HALO_PITCH + tx;
            for (int gi = P.n_hidden; gi < P.n_groups; ++gi) {
                const int buf = (int)(gcount & 1);
                tr.ev(0xA00 + gi);
                mbar_wait(bar_accfull(buf), (afphase >> buf) & 1);
                afphase ^= 1u << buf;
                tc_fence_after_sync();
                tr.ev(0xB00 + gi);
                if (gi == P.n_groups - 1 && iter + 1 < my_iters) {
                    layer0(tile + gridDim.x, 0u);        // every MMA that read this tile's A operand has retired
                    tr.ev(0x900);
                }
                const int gN = P.g[gi].N, gtap0 = P.g[gi].tap0;
                const float* bias = s_bias + (P.g[gi].bias_off - P.bias_skip);
                if constexpr (PRED) {
                    if (pred_one_block) {
                        // ---- pred with a single head block of <= 128 columns (ks <= 11): the thread's <= 64 sigmoid values stay in
                        // registers until the row sum is known, then go out NORMALISED and COALESCED.  (Storing each
                        // thread's own row directly makes every store instruction touch 32 rows = 32 sectors, and
                        // the rescale pass re-reads and re-writes them the same way: the stores, not the MMAs, set
                        // the pace -- 184 Mprobes/s against 440 Mpix*slices/s for the render.)  Eight columns at a
                        // time are transposed through the (unused in pred mode) halo area: [32 rows][8 + 1] floats
                        // per warp, then lane = (row % 4, column) writes 4 rows x 32 B per instruction.
                        float keep[2][32];
#pragma unroll
                        for (int ci = 0; ci < 2; ++ci) {
                            const int c32 = hh * 32 + ci * 64;
                            if (c32 < gN) {
                                uint32_t rr[32];
                                tmem_ld32(t_lane + buf * 256 + c32, rr);
                                const int nvalid = kk - (gtap0 + c32);
                                tmem_ld_wait();
#pragma unroll
                                for (int u = 0; u < 32; ++u) {
                                    float sg = rcp_approx(1.0f + ex2_approx(fmaf(__uint_as_float(rr[u]), NEG_LOG2E, bias[c32 + u])));
                                    sg = (u < nvalid) ? sg : 0.f;
                                    keep[ci][u] = sg;
                                    ssum += sg;
                                }
                            } else {
#pragma unroll
                                for (int u = 0; u < 32; ++u) keep[ci][u] = 0.f;
                            }
                        }
                        tc_fence_before_sync();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar_accfree(buf));
                        ++gcount;
                        s_red[row * 5 + hh] = ssum;
                        named_bar_sync(2 + q, 64);
                        const float inv = 1.0f / fmaxf(s_red[row * 5] + s_red[row * 5 + 1], 1e-12f);
                        float* stg = reinterpret_cast<float*>(s_halo) + e * (32 * 9);
                        const long long row0 = tile * TC_M + q * 32;            // first probe of this warp's 32 rows
                        const int rsub = lane >> 3, csub = lane & 7;
#pragma unroll
                        for (int ci = 0; ci < 2; ++ci) {
#pragma unroll
                            for (int pc = 0; pc < 4; ++pc) {
                                const int c0 = gtap0 + hh * 32 + ci * 64 + pc * 8;
                                if (c0 >= kk) continue;                          // warp-uniform
#pragma unroll
                                for (int j = 0; j < 8; ++j) stg[lane * 9 + j] = keep[ci][pc * 8 + j] * inv;
                                __syncwarp();
#pragma unroll
                                for (int rb = 0; rb < 8; ++rb) {
                                    const int rloc = rb * 4 + rsub;
                                    const float v = stg[rloc * 9 + csub];
                                    if (row0 + rloc < P.n_probes && c0 + csub < kk)
                                        P.psf_out[(row0 + rloc) * kk + c0 + csub] = v;
                                }
                                __syncwarp();
                            }
                        }
                        continue;
                    }
                }
#pragma unroll 1
                for (int c32 = hh * 32; c32 < gN; c32 += 64) {
                    uint32_t rr[32];
                    tmem_ld32(t_lane + buf * 256 + c32, rr);
                    const int tap_first = gtap0 + c32;
                    tmem_ld_wait();
                    if constexpr (PRED) {
                        // several head blocks (ks >= 13): the un-normalised sigmoid values go out now -- transposed
                        // through the halo area like above, so that a store instruction covers 4 rows x 32 B instead
                        // of 32 rows -- and are rescaled below
                        const int nvalid = kk - tap_first;
                        float sgv[32];
#pragma unroll
                        for (int u = 0; u < 32; ++u) {
                            float sg = rcp_approx(1.0f + ex2_approx(fmaf(__uint_as_float(rr[u]), NEG_LOG2E, bias[c32 + u])));
                            sg = (u < nvalid) ? sg : 0.f;
                            sgv[u] = sg;
                            ssum += sg;
                        }
                        float* stg = reinterpret_cast<float*>(s_halo) + e * (32 * 9);
                        const long long row0 = tile * TC_M + q * 32;
                        const int rsub = lane >> 3, csub = lane & 7;
#pragma unroll
                        for (int pc = 0; pc < 4; ++pc) {
                            const int c0 = tap_first + pc * 8;
                            if (c0 >= kk) continue;                              // warp-uniform
#pragma unroll
                            for (int j = 0; j < 8; ++j) stg[lane * 9 + j] = sgv[pc * 8 + j];
                            __syncwarp();
#pragma unroll
                            for (int rb = 0; rb < 8; ++rb) {
                                const int rloc = rb * 4 + rsub;
                                const float v = stg[rloc * 9 + csub];
                                if (row0 + rloc < P.n_probes && c0 + csub < kk) P.psf_out[(row0 + rloc) * kk + c0 + csub] = v;
                            }
                            __syncwarp();
                        }
                    } else {
                        gather32(rr, tap_first, bias + c32, hbase, ssum, cacc);
                    }
                }
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_accfree(buf));
                ++gcount;
            }
            if constexpr (PRED) {
                if (pred_one_block) continue;                          // normalised and stored above
                // ---- exchange the partial sums of the two column halves, then rescale what this thread wrote
                s_red[row * 5 + hh] = ssum;
                named_bar_sync(2 + q, 64);
                // (the barrier also orders the two warps' global stores of this quadrant's rows before the re-read)
                // each of the two warps rescales sixteen of the quadrant's rows, lanes along the taps: coalesced
                for (int rloc = hh * 16; rloc < hh * 16 + 16; ++rloc) {
                    const long long grow = tile * TC_M + q * 32 + rloc;
                    if (grow >= P.n_probes) break;
                    const float inv = 1.0f / fmaxf(s_red[(q * 32 + rloc) * 5] + s_red[(q * 32 + rloc) * 5 + 1], 1e-12f);
                    float* orow = P.psf_out + grow * kk;
                    for (int t = lane; t < kk; t += 32) orow[t] *= inv;
                }
                continue;
            }
            store_px(ssum, cacc, n, s, h, w, valid);
        }
        if constexpr (TA) {
            if (my_iters > 0) gather_ta(my_iters - 1);
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == TC_WARP_PRODUCER) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------
// Debug / unit-test kernel: D[128 x N] = A[128 x K] * B[N x K]^T with the exact operand
// layouts, descriptors and TMEM read-back used above (single CTA, single MMA term).
// bpack is B pre-packed by the host packer as K/32 slabs of [N x 32].
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128, 1)
debug_umma_gemm_kernel(const float* __restrict__ A, const uint8_t* __restrict__ bpack, float* __restrict__ D,
                       int K, int N) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t a_hi = sbase;                               // [K/8][128][8] fp16
    const uint32_t b_sm = sbase + TC_A_PART_BYTES;             // K/32 slabs of N*64 bytes
    const uint32_t bar = sbase + TC_A_PART_BYTES + 131072;
    volatile uint32_t* slot = reinterpret_cast<volatile uint32_t*>(smem + TC_A_PART_BYTES + 131072 + 16);
    if (threadIdx.x == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc<256>(smem_u32(const_cast<uint32_t*>(slot)));
    // A -> fp16 K-major canonical layout
    const int row = threadIdx.x;
    for (int kg = 0; kg < K / 8; ++kg) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = A[(size_t)row * K + kg * 8 + u];
        store_split8(v, a_hi + kg * TC_A_LBO + row * 16, 0, false);
    }
    const int bbytes = (K / 32) * N * 64;
    for (int i = threadIdx.x * 16; i < bbytes; i += 128 * 16)
        *reinterpret_cast<uint4*>(smem + TC_A_PART_BYTES + i) = *reinterpret_cast<const uint4*>(bpack + i);
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *slot;
    if (threadIdx.x == 0) {
        const uint32_t idesc = umma_idesc_f16_f32(128, N);
        const uint32_t lbo_b = (uint32_t)N * 16;
        for (int ks16 = 0; ks16 < K / 16; ++ks16) {
            const uint32_t slab = b_sm + (ks16 / 2) * (N * 64);
            umma_f16_ss(tmem_base, umma_smem_desc(a_hi + ks16 * 2 * TC_A_LBO, TC_A_LBO, 128),
                        umma_smem_desc(slab + (ks16 & 1) * 2 * lbo_b, lbo_b, 128), idesc, ks16 > 0);
        }
        umma_commit(bar);
    }
    __syncwarp();
    mbar_wait(bar, 0);
    tc_fence_after_sync();
    for (int c0 = 0; c0 < N; c0 += 32) {
        uint32_t rr[32];
        tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + c0, rr);
        tmem_ld_wait();
        for (int u = 0; u < 32; ++u)
            if (c0 + u < N) D[(size_t)row * N + c0 + u] = __uint_as_float(rr[u]);
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<256>(tmem_base);
}

}  // namespace aadff
