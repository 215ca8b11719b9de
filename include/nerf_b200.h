/*
 * nerf_b200.h -- C-ABI of the B200-native vanilla-NeRF volume-rendering hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  The reference (nerficg) has no FFI for this path: every
 * stage is a chain of ATen ops issued from Python.  Each entry point below replaces the ATen
 * chain of one reference function; the reference-side binding is the ctypes stub shown in
 * INTEGRATION.md (nerficg_b200/_lib.py is the real one).  Citations are relative to the
 * reference checkout (/root/reference).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; plain C types only.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it, allocates
 *     nothing, creates no threads or streams, and is re-entrant per device.
 *   - return value 0 = success; negative = error, message via nerf_last_error().
 *   - sm_100 only: there is no CPU path and no fallback (nerf_device_check()).
 *   - "samples" of a pass are ordered ray-major: sample e = ray * S + i.
 *   - an MLP output is packed as float4 (r, g, b, sigma) per sample ("rgbsigma").
 */
#ifndef NERF_B200_H
#define NERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NERF_ABI_VERSION 1

/* fixed architecture handled by the CUDA path (configs/nerf_lego.yaml MODEL section,
 * src/Methods/NeRF/Model.py:86-96): 8 layers x 256, skip before layer 5, 1 colour layer,
 * L=10 / L=4 frequencies, input appended, ReLU.  Anything else is rejected by the host. */
#define NERF_N_PARAM_TENSORS 24
#define NERF_TILE 128 /* samples per MMA tile */

int nerf_abi_version(void);
const char* nerf_last_error(void);
/* 0 if `device` is an sm_100 GPU, negative otherwise (no fallback path exists). */
int nerf_device_check(int device);

/* ---- parameter layout ---------------------------------------------------------------
 * One NeRFBlock (src/Methods/NeRF/Model.py:35-54) is a flat fp32 buffer; tensor t of the
 * torch registration order (initial_layers.{0..7}.0.{weight,bias}, feature_layer.*,
 * density_layer.*, color_layers.0.*, color_layers.2.*) starts at offsets[t] floats and
 * keeps torch's row-major (out, in) layout.  Starts are padded to 4 floats. */
int nerf_param_layout(int64_t* offsets /*[24]*/, int64_t* sizes /*[24]*/, int64_t* total);

/* ---- K1: stratified sampling -- generate_samples, src/Methods/NeRF/utils.py:57-75 ----
 * z[n_rays][n_samples]; u = uniform noise of the same shape (torch.rand) or NULL for the
 * deterministic linspace. */
int nerf_sample_stratified(float* z, const float* u, int n_rays, int n_samples, float near_plane, float far_plane,
                           void* stream);

/* ---- K2: inverse-CDF importance sampling + merge -------------------------------------
 * generate_samples_from_pdf (src/Methods/NeRF/utils.py:78-109) followed by
 * sort(cat(z_coarse, z_fine)) (src/Methods/NeRF/Renderer.py:70).
 * z_coarse, w_coarse: [n_rays][n_coarse]; u: [n_rays][n_fine] or NULL (linspace(0,1,n_fine));
 * z_merged: [n_rays][n_coarse+n_fine] ascending; z_fine (optional, may be NULL): the
 * unsorted fine samples, exported for stage parity tests. */
int nerf_sample_importance(float* z_merged, float* z_fine, const float* z_coarse, const float* w_coarse, const float* u,
                           int n_rays, int n_coarse, int n_fine, void* stream);

/* ---- K5: alpha compositing forward -- integrate_samples, src/Methods/NeRF/utils.py:112-136
 * z [n][S], rgbsigma [n][S][4], dirs [n][3] (un-normalised), background [3] or NULL.
 * Outputs rgb [n][3], depth [n], alpha [n], weights [n][S] (NULL to skip). */
int nerf_composite_forward(float* rgb, float* depth, float* alpha, float* weights, const float* z,
                           const float* rgbsigma, const float* dirs, const float* background, int n_rays, int n_samples,
                           void* stream);

/* ---- K6: alpha compositing backward (autograd of integrate_samples; SURVEY.md A.9) ----
 * Upstream grads g_rgb [n][3] (required), g_depth [n], g_alpha [n] (NULL = zero).
 * d_rgbsigma [n][S][4] receives (dL/dr, dL/dg, dL/db, dL/dsigma) times grad_scale.
 * relu_mask != 0 zeroes dL/dsigma where sigma <= 0 (folds the density ReLU of
 * src/Methods/NeRF/Model.py:77 so the 1e10 last-interval term never leaves fp32). */
int nerf_composite_backward(float* d_rgbsigma, const float* z, const float* rgbsigma, const float* dirs,
                            const float* background, const float* g_rgb, const float* g_depth, const float* g_alpha,
                            int n_rays, int n_samples, int relu_mask, float grad_scale, void* stream);

/* ---- weight images for the tensor-core MLP ---------------------------------------------
 * Converts one block's flat fp32 parameters into fp16 forward and fp16 transposed
 * (backward) UMMA operand images (128B-swizzled K-major panels).  `packed` needs
 * nerf_mlp_packed_bytes() bytes, 1024-byte aligned. */
size_t nerf_mlp_packed_bytes(void);
int nerf_mlp_pack(void* packed, const float* params, int with_backward, void* stream);

/* ---- K3: fused encoding + MLP forward -- FrequencyEncoding + NeRFBlock.forward ---------
 * (src/Methods/NeRF/utils.py:32-36, src/Methods/NeRF/Model.py:59-83) applied to the
 * sample positions origins + dirs * z (src/Methods/NeRF/Renderer.py:54,75).
 * origins/dirs/viewdirs [n_rays][3], z [n_rays][S], noise [n_rays*S] already scaled by the
 * noise std, or NULL.  rgbsigma [n_rays*S][4].  `stash` (NULL for inference) receives the
 * activations the backward needs; it needs nerf_mlp_stash_bytes(n_rays*S) bytes, 1024-aligned. */
size_t nerf_mlp_stash_bytes(int64_t n_samples);
int nerf_mlp_forward(float* rgbsigma, void* stash, const void* packed, const float* params, const float* origins,
                     const float* dirs, const float* viewdirs, const float* z, const float* noise, int n_rays,
                     int n_samples, void* stream);

/* ---- K4: MLP backward (autograd of NeRFBlock.forward w.r.t. its parameters) ------------
 * d_rgbsigma [n_rays*S][4] = grad_scale * dL/d(r,g,b,sigma_raw) (from K6 with relu_mask=1).
 * Gradients are ACCUMULATED into `grads` (flat fp32, layout of nerf_param_layout) after
 * division by grad_scale.  `workspace` needs nerf_mlp_backward_workspace_bytes(n) bytes. */
size_t nerf_mlp_backward_workspace_bytes(int64_t n_samples);
int nerf_mlp_backward(float* grads, const float* d_rgbsigma, const float* rgbsigma, const void* stash, void* workspace,
                      const void* packed, const float* params, int n_rays, int n_samples, float grad_scale,
                      void* stream);

/* The two phases of nerf_mlp_backward, separately launchable (profiling):
 * dgrad walks the chain backwards per tile and fills `workspace` with the per-layer output gradients;
 * wgrad reduces activations x gradients over all samples into `grads` (layer-major, HBM-bound). */
int nerf_mlp_backward_dgrad(const float* d_rgbsigma, const float* rgbsigma, const void* stash, void* workspace,
                            const void* packed, const float* params, int n_rays, int n_samples, void* stream);
int nerf_mlp_backward_wgrad(float* grads, const void* stash, const void* workspace, int n_rays, int n_samples,
                            float grad_scale, void* stream);

/* ---- K7: Adam on a flat parameter buffer (torch.optim.Adam semantics: no weight decay, no amsgrad) ----------
 * reference: src/Methods/NeRF/Trainer.py:32-37,61-63.  `state` = 4 device floats {step, 1-beta1^step,
 * sqrt(1-beta2^step), unused}; nerf_adam_tick advances it once per optimiser step (graph-replay safe), then
 * nerf_adam_update is called once per flat buffer.  `lr` is a DEVICE scalar (the schedule writes it asynchronously). */
int nerf_adam_tick(float* state, float beta1, float beta2, void* stream);
int nerf_adam_update(float* params, float* exp_avg, float* exp_avg_sq, const float* grads, const float* lr, const float* state,
                     float beta1, float beta2, float eps, int64_t n, void* stream);
/* Same update with the gradient multiplied by `grad_mult` on the fly (1/world_size of the data-parallel mean: the NCCL
 * all-reduce stays a plain SUM) and, when zero_grads != 0, the gradient buffer cleared behind the read
 * (optimizer.zero_grad(), src/Methods/NeRF/Trainer.py:62). */
int nerf_adam_update_ex(float* params, float* exp_avg, float* exp_avg_sq, float* grads, const float* lr, const float* state,
                        float beta1, float beta2, float eps, float grad_mult, int zero_grads, int64_t n, void* stream);

/* K8 -- NeRFLoss.forward and its gradient in one launch (reference src/Methods/NeRF/Loss.py:26-43,
 * src/Datasets/utils.py:185-189, src/Optim/Losses/utils.py:54-57):
 *   gt = clamp(lerp(background, rgb_gt, alpha_gt), 0, 1)            (alpha_gt NULL = 1, background NULL = 0)
 *   *loss = lambda_color * [mse(rgb, gt) + mse(rgb_coarse, gt)] + lambda_alpha * [mse(alpha, alpha_gt) + mse(alpha_coarse, alpha_gt)]
 *   g_rgb[n][3] = dloss/drgb, g_rgb_coarse, g_alpha[n], g_alpha_coarse likewise (the coarse / alpha pointers may be NULL;
 *   the alpha gradients are only written when lambda_alpha > 0).  One block: the reduction order is fixed. */
int nerf_loss_mse(float* loss, float* g_rgb, float* g_rgb_coarse, float* g_alpha, float* g_alpha_coarse, const float* rgb,
                  const float* rgb_coarse, const float* alpha, const float* alpha_coarse, const float* rgb_gt,
                  const float* alpha_gt, const float* background, int n_rays, float lambda_color, float lambda_alpha, void* stream);

/* ---- stall accounting (development aid, tools/kernel_timing.py) ---------------------------
 * Registers a device buffer of 32 uint64 counters (or NULL to switch it off, the default): the MLP kernels
 * then add the cycles selected threads spent waiting on each barrier (slot meaning: DESIGN.md "Stall accounting"). */
int nerf_debug_set_timing(void* device_buffer);

/* K0 -- device-side ray generation (SURVEY.md 8(f) rank 1).  View.get_rays (reference src/Datasets/utils.py:1053-1074) with
 * PerspectiveCamera.compute_local_ray_directions (src/Cameras/Perspective.py:64-94, no distortion) and View.cam_to_world
 * (utils.py:1033-1038): origin = camera position, direction = (x, y, 1) @ R^T (NOT normalised), view_direction =
 * normalize(direction), for the pixels `pixel_ids` (row-major ids, DEVICE int64) or, when NULL, for all width*height pixels.
 * c2w_host: HOST pointer to a row-major 3x4 / 4x4 float64 camera-to-world matrix (row stride 4), as View stores it. */
int nerf_generate_rays(float* origin, float* direction, float* view_direction, const int64_t* pixel_ids, int64_t n_rays,
                       const double* c2w_host, int width, int height, double focal_x, double focal_y, double center_x,
                       double center_y, void* stream);
/* RayBatch.__getitem__(index tensor) (reference src/Datasets/utils.py:598-613): gathers origin / direction / view_direction /
 * rgb ([n][3]) and alpha ([n]) of the rays `ids` (DEVICE int64) in one launch; any src/dst pair may be NULL. */
int nerf_gather_rays(float* origin_dst, float* direction_dst, float* view_direction_dst, float* rgb_dst, float* alpha_dst,
                     const float* origin_src, const float* direction_src, const float* view_direction_src, const float* rgb_src,
                     const float* alpha_src, const int64_t* ids, int64_t n_rays, void* stream);

/* ---- self test of the tcgen05 building blocks (used by tests/ only) --------------------
 * D[128][n] = A[128][k] * B[n][k]^T with operand images built on device; mode selects the
 * descriptor flavour (0: K-major fp16, 1: MN-major operands as in wgrad, 2: K-major bf16). */
int nerf_selftest_umma(float* d_out, const float* a, const float* b, int n, int k, int mode, void* stream);
/* CTA-pair flavour (cta_group::2, one 2-CTA cluster): D[256][n] = A[256][k] * B[n][k]^T, K-major fp16. */
int nerf_selftest_umma2(float* d_out, const float* a, const float* b, int n, int k, void* stream);
/* ... with both operands stored reduction-major and read as MN-major (the pair flavour of the weight-gradient MMAs); n % 128 == 0. */
int nerf_selftest_umma2_mn(float* d_out, const float* a, const float* b, int n, int k, void* stream);
/* TMEM read-bandwidth probe (development aid): n_warps warps of one CTA issue `iters` accumulator loads each
 * (mode 0: 32x32b.x32, 1: two x32 in flight, 2: x16); out[0] = cycles, out[1] = bytes read from TMEM. */
int nerf_selftest_tmem_read(unsigned long long* out, int n_warps, int mode, int iters, void* stream);

/* Tensor-pipe rate probe (development aid): `iters` back-to-back cta_group::2 M256 N256 K16 MMAs, K-major or MN-major operands;
 * out[0] = cycles. */
int nerf_selftest_umma2_rate(unsigned long long* out, int mn_major, int iters, void* stream);

/* L2 -> SM streaming probe (development aid): n_ctas CTAs each move `iters` 16 KB chunks between an L2-resident window and
 * shared memory with 1-D bulk copies (mode bit 0: loads, bit 1: stores); out[0] = cycles of the slowest CTA, out[1] = bytes per CTA. */
int nerf_selftest_l2_stream(unsigned long long* out, void* window, uint32_t window_bytes, int mode, int iters, int n_ctas, void* stream);
/* LSU flavour: n_warps warps per CTA copy the chunks with 16-byte ld/st (mode bit 2: shared -> global stores, bit 3: global loads),
 * optionally next to a TMA load ring (bit 0). */
int nerf_selftest_l2_stream_lsu(unsigned long long* out, void* window, uint32_t window_bytes, int mode, int iters, int n_ctas, int n_warps,
                                void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NERF_B200_H */
