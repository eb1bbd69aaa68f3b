/* aadff.h -- C ABI of libaadff.so: B200 (sm_100a) aberrated focal-stack synthesis.
 *
 * The reference (singer-yang/Aberration-Aware-Depth-from-Focus) is pure Python/PyTorch and has
 * no FFI of its own; this header is the boundary a maintainer binds underneath the unchanged
 * Python surface.  Each entry point names the reference interface it replaces (file:line
 * relative to the reference repository).  See INTEGRATION.md for the ctypes binding.
 *
 * Conventions: plain pointers and sizes only (no torch / C++ types); every function returns
 * 0 on success or a negative AADFF_E_* code, with a human-readable message available from
 * aadff_last_error() (thread-local).  Device-pointer entry points are asynchronous and
 * stream-ordered on `stream` (a CUstream / cudaStream_t passed as void*; NULL = legacy default
 * stream); they never allocate, never synchronise and never touch the inputs.  All tensors are
 * fp32 and dense ("contiguous") unless strides are given.  There is no CPU fallback: on a
 * machine without an sm_100 device every compute call fails with AADFF_E_CUDA.
 */
#ifndef AADFF_H_
#define AADFF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AADFF_VERSION 200

#define AADFF_OK 0
#define AADFF_E_INVALID (-1)      /* bad argument (null pointer, shape, kernel size ...) */
#define AADFF_E_CUDA (-2)         /* CUDA runtime error, message has the cudaError string */
#define AADFF_E_UNSUPPORTED (-3)  /* valid request this build cannot serve on the chosen mode */

/* Arithmetic of the PSFNet MLP (deeplens/psfnet_arch.py:24-47) inside the fused kernel.      */
#define AADFF_MODE_PARITY 0 /* tcgen05, fp16 hi/lo split operands, 3 MMA terms: <=1e-4 vs fp32 reference */
#define AADFF_MODE_FAST 1   /* tcgen05, single fp16 term: max-abs <= 3e-2 on noise images, see DESIGN.md */
#define AADFF_MODE_FP32 2   /* CUDA-core fp32 FFMA, operation-for-operation with the reference          */
#define AADFF_MODE_MIXED 3  /* tcgen05, 3 terms for the first three MMA layers, 1 term afterwards        */
/* (The first AADFF_MODE_ECON call on a handle runs the weight calibration on the host and uploads the result: that one
 *  call allocates and synchronises -- make it outside CUDA-graph capture, e.g. as the usual warm-up call.)            */
#define AADFF_MODE_ECON 4   /* tcgen05, 3 terms for L1-L4, 2 terms (Ah*Wh + Al*Wh) for L5.. and the head on fp16 weights
                               whose rounding is calibrated at create time to minimise the layer's output error over
                               the network's input box (csrc/econ_calib.h): 21 % fewer MMAs, max-abs 2e-5 .. 4e-5   */
#define AADFF_MODE_ECON8 5  /* like AADFF_MODE_ECON but two terms only for L8, L9 and the head: the earliest start whose
                             * worst case over ANY [0,1] image (half the L1 distance of the PSFs) stays under 1e-4 on the
                             * shipped checkpoint (7.5e-5; parity 5.6e-5, econ 2.0e-4) -- 9.5 % fewer MMAs than parity    */

typedef struct aadff_psfnet* aadff_psfnet_t;

int aadff_version(void);
const char* aadff_last_error(void);

/* Replaces PSFNet.init_net + PSFNet.load_net (deeplens/psfnet.py:44-76): takes the state_dict
 * of MLP(4, ks*ks, 256, hidden_layers) as HOST pointers -- weights[l] is `net.{2l}.weight`
 * ([dims[l+1], dims[l]] row-major), biases[l] is `net.{2l}.bias` -- and uploads them to
 * `device` pre-packed for the kernels (fp16 hi/lo K-major slabs for tcgen05, W^T for fp32).
 * dims has n_layers+1 entries and must be {4, 64, 256, ..., 256, ks*ks}.                       */
int aadff_psfnet_create(const float* const* weights, const float* const* biases, const int* dims, int n_layers,
                        int ks, int device, aadff_psfnet_t* out);
int aadff_psfnet_destroy(aadff_psfnet_t net);

/* Replaces the slice loop of the training scripts (2_aber_aware_dff_aif.py:108-114,166-176):
 * S calls of PSFNet.render (deeplens/psfnet.py:393-441, which calls MLP.forward
 * deeplens/psfnet_arch.py:44-47 and local_psf_render deeplens/render_psf.py:76-107) and the
 * torch.stack, as ONE launch.  S = 1 with strides {C*H*W, H*W, 0, W, 1} is PSFNet.render itself.
 *   img    [N,C,H,W]  all-in-focus image, device
 *   depth  [N,H,W]    depth in mm, <= 0 (0 = invalid), device
 *   foc    [N,S]      focus distance per image and slice in mm, < 0, device
 *   out               device; element strides for (n, c, s, h, w) in out_strides
 *   d_min, d_max      PSFNet.d_min / d_max (-200, -20000)  (deeplens/psfnet.py:32-33)          */
int aadff_render_stack_f32(aadff_psfnet_t net, const float* img, const float* depth, const float* foc, float* out,
                           const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                           float d_max, int mode, void* stream);

/* The same for a contiguous run of TILE ROWS -- the unit of the multi-GPU partition (SURVEY.md 8e: "shard by image,
 * slice and/or row band"; the reference itself renders on one device, 2_aber_aware_dff_aif.py:108-114).  A tile row is
 * aadff_tile_row_height() (= 8) image rows of one (image, slice); tile rows are numbered in (image, slice, row) order,
 * R = (n*S + s)*ceil(H/8) + h/8, and the call renders rows [tile_row_begin, tile_row_end) into `out` (same strides
 * and base pointer as the full call; everything else is left untouched).  Results are bit-identical to the full call. */
int aadff_render_stack_rows_f32(aadff_psfnet_t net, const float* img, const float* depth, const float* foc, float* out,
                                const int64_t out_strides[5], int N, int C, int S, int H, int W, float d_min,
                                float d_max, int mode, int64_t tile_row_begin, int64_t tile_row_end, void* stream);
int aadff_tile_row_height(void);
/* First tensor-core layer group (0 = L1) that AADFF_MODE_ECON evaluates with two MMA terms (bench bookkeeping). */
int aadff_econ_first_group(void);

/* Same operation with HOST buffers (out is dense [N,C,S,H,W]): copies in, renders, copies
 * out and synchronises, using a workspace and a stream owned by the handle.  This is the call
 * the end-to-end benchmark times.                                                              */
int aadff_render_stack_host_f32(aadff_psfnet_t net, const float* img, const float* depth, const float* foc,
                                float* out, int N, int C, int S, int H, int W, float d_min, float d_max, int mode);

/* Replaces PSFNet.pred (deeplens/psfnet.py:375-390) for arbitrary probes:
 *   inp [M,4] (x, y, z, foc_z) -> psf [M, ks*ks], L1-normalised; fp32 arithmetic; device ptrs. */
int aadff_psfnet_pred_f32(aadff_psfnet_t net, const float* inp, float* psf, int64_t M, void* stream);
/* The same on the tensor-core path (the fused kernel with the gather replaced by a PSF store); `mode` as for
 * aadff_render_stack_f32 (AADFF_MODE_FP32 forwards to the call above).  inp must be 16-byte aligned.          */
int aadff_psfnet_pred_tc_f32(aadff_psfnet_t net, const float* inp, float* psf, int64_t M, int mode, void* stream);

/* Replaces local_psf_render (deeplens/render_psf.py:76-107) for a PSF tensor in memory:
 *   img [N,C,H,W], psf [N,H,W,ks,ks] -> out [N,C,H,W]; device pointers.                        */
int aadff_local_psf_render_f32(const float* img, const float* psf, float* out, int N, int C, int H, int W, int ks,
                               void* stream);
/* Backward of aadff_local_psf_render_f32: grad_out [N,C,H,W] -> grad_img [N,C,H,W] and/or grad_psf [N,H,W,ks,ks]
 * (either may be NULL, not both; img, psf, grad_out must not be).  Outputs are overwritten, not accumulated; no
 * atomics, so two calls give bit-identical results; stream-ordered, no allocation, CUDA-graph capturable.          */
int aadff_local_psf_render_backward_f32(const float* img, const float* psf, const float* grad_out, float* grad_img,
                                        float* grad_psf, int N, int C, int H, int W, int ks, void* stream);

/* Replaces ThinLens.render + ThinLens.coc (deeplens/psfnet.py:503-570), the thin-lens baseline of the paper:
 * circle of confusion -> clipped Gaussian PSF (sigma = coc/2) -> normalise -> per-pixel gather, fused (no PSF
 * tensor in memory).  img [N,C,H,W], depth [N,H,W] mm, foc [N] mm, out [N,C,H,W]; device pointers.
 * pixel_size = sensor_size[0] / sensor_res[0] [mm]; d_lo/d_hi = 200 / 20000 mm (ThinLens.d_min / d_max);
 * flip_sign = 1 negates depth and foc first, which is what the reference does when any depth is negative
 * (psfnet.py:504).  If flip_sign_dev is not NULL the decision is read from that device byte instead (written by
 * aadff_any_negative_f32 earlier on the same stream), so the data-dependent branch costs no host synchronisation. */
int aadff_thinlens_render_f32(const float* img, const float* depth, const float* foc, float* out, int N, int C, int H,
                              int W, int ks, float foc_len, float fnum, float pixel_size, float d_lo, float d_hi,
                              int flip_sign, const unsigned char* flip_sign_dev, void* stream);
/* flag_dev[0] = any(x[i] < 0), i < n; device pointers, stream-ordered.                                          */
int aadff_any_negative_f32(const float* x, int64_t n, unsigned char* flag_dev, void* stream);

/* Replaces render_psf (deeplens/render_psf.py:12-28; grid = 1, psf_map = [C,ks,ks], bounds {0,H} / {0,W}) and
 * render_psf_map (deeplens/render_psf.py:31-73; psf_map = [C, grid*ks, grid*ks], one PSF per image patch): true
 * convolution (the PSF is flipped) on the reflect-padded image, per channel.  row_bounds / col_bounds are HOST arrays of
 * grid+1 ascending patch limits (the reference's int(i/grid*H), int(j/grid*W)); rows/columns beyond the last limit are
 * left untouched, as in the reference.  ks odd, <= 31; grid <= 32; img, psf_map, out are device pointers.        */
int aadff_render_psf_map_f32(const float* img, const float* psf_map, float* out, int B, int C, int H, int W, int ks,
                             int grid, const int* row_bounds, const int* col_bounds, void* stream);
/* Backward of aadff_render_psf_map_f32 (same arguments): grad_out [B,C,H,W] -> grad_img [B,C,H,W] and/or
 * grad_psf_map [C, grid*ks, grid*ks] (either may be NULL, not both).  `work` is device memory of at least
 * aadff_render_psf_map_backward_work_bytes(...) bytes (needed only when grad_psf_map != NULL; the library allocates
 * nothing).  Outputs are overwritten; deterministic; stream-ordered, CUDA-graph capturable.  The size query returns
 * a negative AADFF_E_* code for arguments the backward would reject.                                             */
int64_t aadff_render_psf_map_backward_work_bytes(int B, int C, int H, int W, int ks, int grid, const int* row_bounds,
                                                 const int* col_bounds);
int aadff_render_psf_map_backward_f32(const float* img, const float* psf_map, const float* grad_out, float* grad_img,
                                      float* grad_psf_map, void* work, int64_t work_bytes, int B, int C, int H, int W,
                                      int ks, int grid, const int* row_bounds, const int* col_bounds, void* stream);

/* Replaces the per-sample CPU work of the reference's Dataset classes after file decoding (dff/dataset.py:43-52
 * Matterport3D, :190-205 Middlebury; AutoAgument's colour jitter and flips :259-272): BGR uint8 -> RGB float / 255
 * (-> clip(0.5 + contrast*(x-0.5) + brightness, 0, 1) -> flips) -> torchvision Resize((h,w), antialias=True), and
 * uint16 depth / depth_div (-> flips) -> the same resize (depth_mode 0) or cv2.resize INTER_LINEAR (depth_mode 1).
 *   bgr [B,H,W,3] uint8, depth [B,H,W] uint16 (either may be NULL), aif_out [B,3,h,w], depth_out [B,1,h,w] fp32;
 *   jitter [B,2] = (contrast, brightness) per image, contrast < 0 = no jitter, or NULL; flips [B]: bit 0 horizontal,
 *   bit 1 vertical, or NULL.  Device pointers, stream-ordered.  AutoAgument's spline rotation: the three calls below. */
int aadff_preprocess_rgbd_u8(const uint8_t* bgr, const uint16_t* depth, float* aif_out, float* depth_out, int B, int H, int W,
                             int h, int w, float depth_div, int depth_mode, const float* jitter, const uint8_t* flips,
                             void* stream);

/* AutoAgument's rotation (dff/dataset.py:275-284: scipy.ndimage.rotate(x, degree, reshape=False), i.e. order-3 spline
 * interpolation, mode 'constant', cval 0, with prefilter) between the flips and the resize, in three stream-ordered steps
 * on fp32 planes [B,P,H,W] at full resolution (P = 3 RGB planes if bgr, + 1 depth plane if depth, in that order):
 *   aadff_prepare_planes_u8   decoded arrays -> planes with /255, colour jitter, flips (arguments as above);
 *   aadff_spline_affine_f32   scipy.ndimage.affine_transform(order=3, mode='constant', cval=0, prefilter=True) per
 *       plane: xform [B,6] doubles (device) = m00, m01, m10, m11, off0, off1 with input (row, col) = M (output row,
 *       col) + off -- for a rotation by `degree` M = [[cos, sin], [-sin, cos]], off = centre - M centre, centre =
 *       ((H-1)/2, (W-1)/2); a sample whose m00 is NaN is copied unchanged.  work holds 2*B*P*H*W floats.  Plane
 *       clamp_plane (the depth plane; -1 = none) is clamped at 0 afterwards (`depth[depth<0] = 0`);
 *   aadff_resize_planes_f32   planes -> aif_out [B,3,h,w] / depth_out [B,1,h,w] (either may be NULL; P must match),
 *       the same resize as aadff_preprocess_rgbd_u8.                                                             */
int aadff_prepare_planes_u8(const uint8_t* bgr, const uint16_t* depth, float* planes, int B, int H, int W, float depth_div,
                            const float* jitter, const uint8_t* flips, void* stream);
int aadff_spline_affine_f32(const float* planes, float* work, float* out, int B, int P, int H, int W, const double* xform,
                            int clamp_plane, void* stream);
int aadff_resize_planes_f32(const float* planes, float* aif_out, float* depth_out, int B, int P, int H, int W, int h, int w,
                            int depth_mode, void* stream);

/* Replaces select_focus_dist(depth, num, mode='linear') (dff/utils.py:4-51), the producer of foc_dist in the
 * training loop: per image the minimum over valid (> 0) depths and the maximum depth, then `num` (> 3) focus
 * distances linearly between them, ascending.  depth_m [B, HW] (metres, any unit really), out [B, num]; device.
 * An image without a single valid depth yields NaN in all its `num` entries (the reference raises on it; its
 * training loop skips such batches, 2_aber_aware_dff_aif.py:103-105).                                      */
int aadff_select_focus_f32(const float* depth_m, int B, int64_t HW, int num, float* out, void* stream);

/* Replaces the optimisation half of PSFNet.train_psfnet (deeplens/psfnet.py:79-132): `psfnet(inp)` ->
 * nn.MSELoss()(pred, psf) -> loss.backward() -> torch.optim.AdamW.step(), fp32, for MLP(4, ks*ks, 256, n) -- the
 * training targets (ray-traced PSFs, psfnet.py:135-170) stay with the caller.  The trainer owns a device copy of the
 * parameters (weights/biases as for aadff_psfnet_create, HOST pointers), their AdamW state and the activations of
 * one batch of `batch` probes; one step is a CUDA graph replay (3 kernels per layer and direction + head + AdamW).
 * dims = [4, hidden widths (multiples of 8, <= 256), kk >= 1], 1 to 16 layers; 0 <= beta1, beta2 < 1; eps and
 * weight_decay finite and >= 0 (as torch.optim.AdamW): anything else is AADFF_E_INVALID, checked before any device work.
 *   aadff_trainer_step: inp [batch,4], target [batch,ks*ks] device pointers; lr = this step's learning rate, finite
 *     and >= 0 (the reference drives it with CosineAnnealingLR); loss_out = optional DEVICE scalar receiving the MSE loss of the
 *     forward pass that preceded the update.  Stream-ordered, no synchronisation.
 *   aadff_trainer_read: which = 0 parameters / 1 gradients of the last step into HOST arrays shaped like the
 *     create call's; which = 2: the last step's predicted PSFs [batch, ks*ks] into weights[0].  Synchronises.   */
typedef struct aadff_trainer* aadff_trainer_t;
int aadff_trainer_create(const float* const* weights, const float* const* biases, const int* dims, int n_layers,
                         int batch, float beta1, float beta2, float eps, float weight_decay, int device,
                         aadff_trainer_t* out);
int aadff_trainer_step(aadff_trainer_t t, const float* inp, const float* target, float lr, float* loss_out, void* stream);
int aadff_trainer_read(aadff_trainer_t t, int which, float* const* weights, float* const* biases, void* stream);
int aadff_trainer_destroy(aadff_trainer_t t);

/* Number of kernels launched by this library in the calling process (bench bookkeeping).      */
int64_t aadff_launch_count(void);

/* Test hooks (used by tests/ only): a single-tile tcgen05 GEMM through the same operand
 * packing, descriptors and TMEM read-back as the fused kernel (host pointers, synchronous),
 * and the descriptor-convention probe it controls.                                            */
int aadff_debug_umma_gemm(const float* A, const float* B, float* D, int K, int N, int device);
int aadff_debug_set_desc_swap(int swap);
/* Event trace of CTA 0 of the fused kernel: device buffer of 4 * aadff_debug_trace_entries()
 * uint64 (zero-filled by the caller), NULL switches tracing off.  See tests/gpu_trace.py.    */
int aadff_debug_set_trace(void* device_buffer);
int aadff_debug_trace_entries(void);
/* Debug switches, 0 restores normal operation.  What-if timing of the fused kernel (results become invalid):
 * 1 = skip the weight copies.  16 = aadff_thinlens_render_f32 fetches every halo tile with clamped cp.async instead of
 * TMA tensor tiles for interior tiles (results unchanged).  Cross-check paths (results stay valid): 256 =
 * AADFF_MODE_ECON with plainly rounded fp16 weights instead of the calibrated ones, 512 = aadff_local_psf_render_f32
 * through the register-streaming kernel also where the strip-walking kernel would run (ks <= 15, W % 4 == 0);
 * 8192 / 1024 / 4096 = the strip-walking kernel with its shared-memory plan 0 / 1 / 2 forced (default: the widest
 * strips that divide W well).  Bits 16..19 (value g > 4): AADFF_MODE_ECON starts its two-term evaluation at layer group
 * g instead of 4 (L5) -- accuracy / speed sweep, generic kernel.  1 << 20 = the fused kernel keeps its A operands in
 * shared memory also where it would keep them in tensor memory (results unchanged).                                 */
int aadff_debug_set_flags(int flags);
/* Host-only: the output-error-calibrated fp16 rounding used by AADFF_MODE_ECON (csrc/econ_calib.h) for one layer.
 * W [N][K], A [NC][K] = sample input activations of the layer, out [N][K] = fp16-representable values.  No GPU. */
int aadff_debug_econ_round(const float* W, int N, int K, const float* A, int NC, float* out);
/* Issue-cost microbenchmark of tcgen05.mma / tcgen05.commit (see tests/gpu_diag.py mma_timing);
 * epi_load: low 16 bits = competing TMEM reads, bit 16 = competing bulk copies into smem, bit 17 =
 * competing st.shared stream.  out_cycles must hold 64 entries.                                   */
int aadff_debug_mma_timing(const int* mmas_per_commit, int n_patterns, int reps, int N, int epi_load,
                           uint64_t* out_cycles, int device);

#ifdef __cplusplus
}
#endif
#endif /* AADFF_H_ */
