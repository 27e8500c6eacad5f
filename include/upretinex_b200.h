/*
 * upretinex_b200.h -- C ABI of libupretinex_b200.so, the B200 (sm_100a) implementation of the
 * classical image-processing hot path of UP-Retinex (xh92117/Retinex-image-Enhancement).
 *
 * The reference has no FFI of its own: its hot path is Python that calls OpenCV / torch on
 * the host.  Each entry point below replaces the arithmetic of one reference function
 * (cited as file:line relative to the reference tree); INTEGRATION.md shows the ctypes stub
 * a maintainer of the reference would add at each call site.
 *
 * Conventions
 *   - All image pointers are DEVICE pointers owned by the caller unless the name ends in
 *     `_host`.  Images are planar NCHW, f32 in [0,1] (values outside are handled exactly
 *     like the reference handles them).
 *   - Every call is asynchronous on the supplied stream (a cudaStream_t passed as void*),
 *     never synchronises, never allocates device memory (workspaces are caller-owned; their
 *     size comes from the matching *_workspace_bytes()).  The `_host` entry points are the
 *     exception: they own a pinned/device staging pool and return after the result is in
 *     the host buffer.
 *   - Return value: 0 = OK, < 0 = invalid argument (UPR_E_*), > 0 = cudaError_t.
 *   - Thread-safe and re-entrant across streams; a workspace must not be shared by calls
 *     that may run concurrently.
 *   - There is no CPU fallback: without an sm_100 device every call fails.
 */
#ifndef UPRETINEX_B200_H
#define UPRETINEX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define UPR_API
#else
#define UPR_API __attribute__((visibility("default")))
#endif

typedef void* upr_stream_t; /* cudaStream_t */

enum {
    UPR_OK = 0,
    UPR_E_NULL = -1,      /* null pointer argument */
    UPR_E_SHAPE = -2,     /* non-positive or unsupported shape */
    UPR_E_WORKSPACE = -3, /* workspace too small or misaligned */
    UPR_E_PARAM = -4,     /* bad scalar parameter */
    UPR_E_DEVICE = -5     /* current device is not sm_100 */
};

UPR_API const char* upr_version(void);
UPR_API const char* upr_status_string(int status);
/* 0 if the current CUDA device is a compute-capability 10.x part, UPR_E_DEVICE otherwise. */
UPR_API int upr_device_check(void);

/* ---- a1: CLAHE in Lab ---------------------------------------------------------------
 * Replaces AdaptiveParameterAdjuster.apply_clahe_enhancement
 * (enhancers/adaptive_params.py:121-169): unclipped trunc-quantise -> sRGB u8 -> OpenCV
 * 8-bit Lab -> CLAHE(clip_limit, tiles) on L -> Lab -> sRGB u8 -> /255.
 * Bit-exact with the reference for every frame of the batch (the reference is batch 1). */
UPR_API size_t upr_clahe_workspace_bytes(int n, int h, int w, int tiles_x, int tiles_y);
UPR_API int upr_clahe_lab_f32(const float* in_nchw, float* out_nchw, int n, int h, int w,
                              double clip_limit, int tiles_x, int tiles_y,
                              void* workspace, size_t workspace_bytes, upr_stream_t stream);
/* The same op at the PACKED u8 boundary (SURVEY 8b/8d): the frames are what an image file decodes to and what is written
 * back -- u8 RGB, HWC -- i.e. exactly the OpenCV part of the reference (adaptive_params.py:145-161) without the float casts
 * around it.  Equivalent to the f32 entry on x = u8 / 255.f followed by (y * 255.f) truncated to u8: both casts are exact
 * (trunc(k / 255.f * 255.f) == k for k = 0..255, pinned in tests/test_oracle_pin.py).  6 instead of 24 bytes per pixel cross
 * the boundary.  upr_clahe_lab_f32_u8 takes the reference's f32 NCHW tensor and writes the packed u8 frame that
 * save_image (enhancers/simple_enhance.py:65-100) would store.  Same workspace as upr_clahe_lab_f32; in place is allowed
 * for the u8 -> u8 entry. */
UPR_API int upr_clahe_lab_u8(const unsigned char* in_nhwc_rgb, unsigned char* out_nhwc_rgb, int n, int h, int w,
                             double clip_limit, int tiles_x, int tiles_y,
                             void* workspace, size_t workspace_bytes, upr_stream_t stream);
UPR_API int upr_clahe_lab_f32_u8(const float* in_nchw, unsigned char* out_nhwc_rgb, int n, int h, int w,
                                 double clip_limit, int tiles_x, int tiles_y,
                                 void* workspace, size_t workspace_bytes, upr_stream_t stream);
/* The enhance path after the CNN in one call: enhanced = R*e + (1-R)*e^2 with R = x/(illu+eps)
 * (models/model.py:405-413, :442) followed by apply_clahe_enhancement(enhanced) (adaptive_params.py:195,
 * :121-169).  x, e: [n][3][h][w]; illu: [n][1][h][w]; out: [n][3][h][w].  The recombined frame is formed in the
 * registers of the histogram kernel and never stored: 40 B/px (x 12 + illu 4 + e 12 read, out 12 written) instead
 * of 64 B/px for upr_retinex_recombine_f32 + upr_clahe_lab_f32.  Bit-identical to those two calls.  Same
 * workspace as upr_clahe_lab_f32. */
UPR_API int upr_retinex_clahe_f32(const float* x_nchw, const float* illu_n1hw, const float* e_nchw, float* out_nchw,
                                  int n, int h, int w, float eps, double clip_limit, int tiles_x, int tiles_y,
                                  void* workspace, size_t workspace_bytes, upr_stream_t stream);
/* Same, writing the packed u8 RGB (HWC) frame that save_image (enhancers/simple_enhance.py:65-100) would store: what the
 * batch driver sends back over PCIe (3 instead of 12 bytes per pixel).  Bit-identical to upr_retinex_clahe_f32 followed by
 * the truncating cast.  Ragged shapes (no vector path) need `enhanced_scratch`, an f32 [n][3][h][w] frame for the
 * recombination; with a NULL scratch they return UPR_E_WORKSPACE. */
UPR_API int upr_retinex_clahe_f32_u8(const float* x_nchw, const float* illu_n1hw, const float* e_nchw,
                                     unsigned char* out_nhwc_rgb, float* enhanced_scratch, int n, int h, int w, float eps,
                                     double clip_limit, int tiles_x, int tiles_y, void* workspace, size_t workspace_bytes,
                                     upr_stream_t stream);
/* Profiling hook: runs only the selected stages of upr_clahe_lab_f32 on a workspace that a full call has
 * already populated.  stage_mask bit 0 = K1 (quantise + Lab + tile histograms + clip/LUT), bit 1 = K3
 * (bilinear LUT map + Lab->RGB); bench.py uses it to time each kernel with CUDA events. */
UPR_API int upr_clahe_lab_stages_f32(const float* in_nchw, float* out_nchw, int n, int h, int w, double clip_limit,
                                     int tiles_x, int tiles_y, void* workspace, size_t workspace_bytes, int stage_mask,
                                     upr_stream_t stream);
/* Copies the per-tile raw histograms ([n][tiles_y*tiles_x][256] int32), LUTs
 * ([n][tiles_y*tiles_x][256] u8) and/or the u8 Lab intermediate ([n][3][h][w]) of the LAST
 * upr_clahe_lab_f32 call that used `workspace` into caller device buffers (any may be NULL). */
UPR_API int upr_clahe_debug_dump(const void* workspace, int n, int h, int w, int tiles_x, int tiles_y,
                                 int32_t* hist_out, uint8_t* lut_out, uint8_t* lab_out,
                                 upr_stream_t stream);
/* The mirror of upr_clahe_debug_dump: copies caller device LUTs ([n][tiles_y*tiles_x][256] u8) and/or Lab planes
 * ([n][3][h][w] u8) into `workspace` (either may be NULL).  With upr_clahe_lab_stages_f32(stage_mask = 2) this runs the
 * map kernel alone on chosen inputs. */
UPR_API int upr_clahe_debug_load(void* workspace, int n, int h, int w, int tiles_x, int tiles_y, const uint8_t* lut_in,
                                 const uint8_t* lab_in, upr_stream_t stream);
/* Host copies of the constant tables the kernels use (for tests/audits). Any may be NULL.
 * gamma[256] u16, cbrt[2048] u16, labyf[256] u32 (ify | y<<16), invgamma[4096] u8. */
UPR_API int upr_get_tables(uint16_t* gamma, uint16_t* cbrt, uint32_t* labyf, uint8_t* invgamma);


/* Same op with HOST buffers (the reference returns a host tensor, adaptive_params.py:164-167): f32 NCHW in
 * host memory in, f32 NCHW in host memory out.  The batch is pipelined through a per-device ring of three
 * streams with library-owned device staging (H2D, kernels and D2H of neighbouring chunks overlap); returns
 * when out_host is complete.  Pinned host memory gives full PCIe speed; pageable memory works.
 * frames_per_chunk <= 0 selects ~96 MB chunks.  upr_host_pool_release() frees the staging pool. */
UPR_API int upr_clahe_lab_f32_host(const float* in_host, float* out_host, int n, int h, int w, double clip_limit,
                                   int tiles_x, int tiles_y, int frames_per_chunk);
/* The packed u8 boundary with HOST buffers: u8 RGB (HWC) in host memory in and out, 3 + 3 instead of 12 + 12 bytes per pixel over
 * PCIe.  Same pipeline, same chunking rule (frames per chunk as for the f32 entry). */
UPR_API int upr_clahe_lab_u8_host(const unsigned char* in_host, unsigned char* out_host, int n, int h, int w, double clip_limit,
                                  int tiles_x, int tiles_y, int frames_per_chunk);
UPR_API int upr_host_pool_release(void);

/* ---- a3: brightness histogram ---------------------------------------------------------
 * Replaces the pixel passes of AdaptiveParameterAdjuster.calculate_brightness_features
 * (enhancers/adaptive_params.py:24-68): trunc-quantise, OpenCV BGR2GRAY fixed point, 256-bin histogram per
 * image ([n][256] u32, zeroed by the call).  mean/std/dark/mid/bright ratios are exact functions of it. */
UPR_API int upr_brightness_hist_f32(const float* in_nchw, int n, int h, int w, uint32_t* hist256_per_image,
                                    upr_stream_t stream);

/* ---- a4/a5: multi-scale statistics and gain ---------------------------------------------
 * Replaces MultiScaleEnhancer.extract_multi_scale_features (enhancers/multi_scale.py:17-60) and the gain of
 * apply_multi_scale_enhancement (:87-94).  means_n_by_3[i] = mean of the 7 feature channels at scales
 * {1, 1/2, 1/4}; gain_per_image[i] = float(1 + 0.1 * (0.5 m1 + 0.3 m2 + 0.2 m3)).
 * flags bit 0: force the generic (non-fused) path.  n <= 65535. */
UPR_API size_t upr_multiscale_workspace_bytes(int n, int h, int w);
UPR_API int upr_multiscale_stats_f32(const float* x_nchw, int n, int h, int w, float* means_n_by_3,
                                     float* gain_per_image, void* workspace, size_t workspace_bytes, int flags,
                                     upr_stream_t stream);
/* Also materialises the three feature tensors [n][7][h_s][w_s] (h_s = int(h*s), w_s = int(w*s)) that
 * extract_multi_scale_features returns; means/gain may be NULL. */
UPR_API int upr_multiscale_features_f32(const float* x_nchw, int n, int h, int w, float* feat_full, float* feat_half,
                                        float* feat_quarter, float* means_n_by_3, float* gain_per_image,
                                        void* workspace, size_t workspace_bytes, upr_stream_t stream);
/* out = clamp(enh * gain_per_image[image], 0, 1)   (enhancers/multi_scale.py:97-98); enh is [n][c][h][w]. */
UPR_API int upr_scale_clamp_f32(const float* enh, const float* gain_per_image, float* out, int n, int c, int h, int w,
                                upr_stream_t stream);
/* a4 + a5 in one call (enhancers/multi_scale.py:62-100 after the CNN): statistics of x, then out = clamp(enh * gain[frame], 0, 1).
 * Batches of two or more ~25 Mpx chunks run chunk by chunk on two library-owned side streams that fork from and join `stream`
 * (graph-capturable): the statistics kernel of one chunk overlaps the gain pass of the previous one.  Same results as
 * upr_multiscale_stats_f32 followed by upr_scale_clamp_f32; means [n][3] and gain [n] are written as by the former;
 * `workspace` = upr_multiscale_workspace_bytes(n, h, w), zero-filled once.  out may alias enh. */
UPR_API int upr_multiscale_enhance_f32(const float* x_nchw, const float* enh_nchw, float* out_nchw, float* means_n_by_3,
                                       float* gain_per_image, int n, int h, int w, void* workspace, size_t workspace_bytes,
                                       upr_stream_t stream);

/* ---- a6/a7: content-aware saliency / attention ------------------------------------------
 * upr_saliency_f32 replaces ContentAwareEnhancer.compute_saliency_map (enhancers/content_aware.py:19-59):
 * u8 gray -> |4-neighbour Laplacian| -> 15x15 Gaussian (sigma 2.6, fp64) -> per-image min-max normalise -> f32
 * [n][1][h][w].  upr_attention_f32 replaces compute_attention_map (:61-91): sal * (1/(luma+0.1)), min-max
 * normalised.  upr_attention_apply_f32 is :119-120: out = clamp(enh * (1 + 0.2*att), 0, 1).  n <= 65535. */
UPR_API size_t upr_saliency_workspace_bytes(int n, int h, int w);
UPR_API int upr_saliency_f32(const float* x_nchw, int n, int h, int w, float* sal_n1hw, void* workspace,
                             size_t workspace_bytes, upr_stream_t stream);
UPR_API int upr_attention_f32(const float* x_nchw, int n, int h, int w, float* att_n1hw, void* workspace,
                              size_t workspace_bytes, upr_stream_t stream);
UPR_API int upr_attention_apply_f32(const float* enh, const float* att_n1hw, float* out, int n, int c, int h, int w,
                                    upr_stream_t stream);
/* The whole of apply_content_aware_enhancement's arithmetic after the CNN (content_aware.py:105-120) in three passes:
 * saliency blur -> raw attention + its min/max -> out = clamp(enh * (1 + 0.2*att), 0, 1).  att_n1hw may be NULL (the
 * reference discards the map); enh/out are [n][3][h][w].  Same workspace as upr_saliency_f32.  Results are identical to
 * upr_attention_f32 followed by upr_attention_apply_f32. */
UPR_API int upr_content_aware_apply_f32(const float* x_nchw, const float* enh_nchw, float* out_nchw, float* att_n1hw, int n,
                                        int h, int w, void* workspace, size_t workspace_bytes, upr_stream_t stream);
/* BASELINE config 5, "content-aware + multi-scale": both gains of the reference's two enhancers applied to the CNN output in
 * ONE epilogue -- out = clamp(clamp(enh * (1 + 0.2 att(x)), 0, 1) * gain[image], 0, 1), i.e. content_aware.py:119-120 followed
 * by multi_scale.py:97-98 -- with gain_per_image from upr_multiscale_stats_f32 on the same input (device memory, no host
 * visit).  Same workspace and attention output as upr_content_aware_apply_f32. */
UPR_API int upr_content_multiscale_apply_f32(const float* x_nchw, const float* enh_nchw, const float* ms_gain_per_image,
                                             float* out_nchw, float* att_n1hw, int n, int h, int w, void* workspace,
                                             size_t workspace_bytes, upr_stream_t stream);
/* The whole chain in one call: the multi-scale statistics of x (means [n][3] and gain [n], as upr_multiscale_stats_f32 writes
 * them; `ms_workspace` = upr_multiscale_workspace_bytes(n, h, w), zero-filled once) are computed INSIDE the chunk schedule of the
 * content-aware passes -- the statistics kernel of a chunk runs on the chunk's stream, overlapping the memory-bound passes of the
 * neighbouring chunk -- and applied in the shared epilogue.  Same results as upr_multiscale_stats_f32 followed by
 * upr_content_multiscale_apply_f32. */
UPR_API int upr_content_multiscale_f32(const float* x_nchw, const float* enh_nchw, float* out_nchw, float* att_n1hw,
                                       float* means_n_by_3, float* gain_per_image, int n, int h, int w, void* workspace,
                                       size_t workspace_bytes, void* ms_workspace, size_t ms_workspace_bytes, upr_stream_t stream);

/* The quantiser of save_image (enhancers/simple_enhance.py:65-100), on the device: [n][c][h][w] f32 -> [n][h][w][c] u8 with
 * (clip(x, 0, 1) * 255).astype(uint8) -- fp32 product, truncation; c = 1 (illumination maps) or 3 (frames).  What the batch
 * driver sends back over PCIe instead of f32 planes (1 resp. 3 instead of 4 resp. 12 bytes per pixel). */
UPR_API int upr_quantize_u8_f32(const float* x_nchw, unsigned char* out_nhwc, int n, int c, int h, int w, upr_stream_t stream);

/* ---- a8: Retinex decomposition / recombination ------------------------------------------
 * models/model.py:405-413 (R = x / (illu + eps), illu broadcast over the 3 channels) and :442
 * (enhanced = R*e + (1-R)*e^2).  refl may be NULL.  Bit-exact with torch eager (no FMA contraction). */
UPR_API int upr_retinex_recombine_f32(const float* x, const float* illu, const float* e, float* refl, float* enh,
                                      int n, int h, int w, float eps, upr_stream_t stream);
UPR_API int upr_retinex_decompose_f32(const float* x, const float* illu, float* refl, int n, int h, int w, float eps,
                                      upr_stream_t stream);

/* ---- a9/a10: texture complexity and the dynamic smoothness weight ------------------------
 * losses/loss.py:523-583: per_image[i] = mean|dx| + mean|dy| ('tv') or the fraction of pixels whose Sobel
 * magnitude exceeds 1.5x its mean ('edge_density').  batch_stats2 (nullable) receives
 * [sum_i per_image[i], n] -- the two numbers a data-parallel all-reduce(SUM) carries so that every rank
 * derives the batch mean of loss.py:710.  The workspace must be zero-filled once before its first use
 * (upr_texture_workspace_init); the kernels leave it clean.  n <= 65535.
 * upr_dynamic_smooth_weight_f32 is loss.py:716-717 on the (all-reduced) pair:
 * weight_out[0] = clamp(weight_smooth * (1 - 0.8 * stats[0]/stats[1]), 0.1, 5.0). */
UPR_API size_t upr_texture_workspace_bytes(int n);
UPR_API int upr_texture_workspace_init(void* workspace, size_t workspace_bytes, int n, upr_stream_t stream);
UPR_API int upr_texture_tv_f32(const float* x, int n, int c, int h, int w, float* per_image, float* batch_stats2,
                               void* workspace, size_t workspace_bytes, upr_stream_t stream);
UPR_API int upr_texture_edge_density_f32(const float* x, int n, int c, int h, int w, float* per_image,
                                         float* batch_stats2, void* workspace, size_t workspace_bytes,
                                         upr_stream_t stream);
UPR_API int upr_dynamic_smooth_weight_f32(const float* batch_stats2, float weight_smooth, float* weight_out,
                                          upr_stream_t stream);
/* ---- N3 (SURVEY 8f): the smoothness term the dynamic weight multiplies ---------------------------------------
 * EdgeAwareSmoothnessLoss.forward(illu_map, img_low) (losses/loss.py:136-176; scaled by the a10 weight at :724):
 *   loss = mean(wh * fh * |dx I|) + mean(wv * fv * |dy I|),  wh/wv = exp(-lambda * mean_c |dx/dy S|),
 *   fh/fv = 1 + alpha * (row / column means of the Sobel edge map of mean_c S; that is what the reference's avg_pool2d
 *   windows (1, W-1) and (H-1, 1) followed by [..., :-1] select).
 * illu: [n][ci][h][w], img_low: [n][cs][h][w] f32.  loss3[0..2] = {loss, horizontal term, vertical term} (device).
 * grad_illu (nullable): d loss / d illu, same shape as illu (sign(0) = 0 like torch.abs).  img_low gets no gradient.
 * Everything derived from img_low is a no-grad image statistic.  Deterministic (ordered fp64 sums).  h, w >= 2. */
/* The three statistics losses of the enhanced image from ONE read of (enhanced, img_low), both [n][3][h][w] f32:
 *   losses3[0] = AdaptiveExposureLoss(enhanced, img_low)   (losses/loss.py:29-58; patch = 16, base_target = 0.6 there)
 *   losses3[1] = ColorLoss(enhanced)                        (:351-368)
 *   losses3[2] = SpatialConsistencyLoss(enhanced, img_low)  (:404-427)
 * `saved` (upr_enh_losses_saved_floats floats, device) keeps the channel means, the adaptive target, the scales and the
 * patch means for the backward entry, which writes  upstream3[0] d exp + upstream3[1] d col + upstream3[2] d spa  w.r.t.
 * `enhanced` in one pass (upstream3: three device floats).  img_low gets no gradient.  h, w >= patch. */
UPR_API size_t upr_enh_losses_workspace_bytes(int n);
UPR_API size_t upr_enh_losses_saved_floats(int n, int h, int w, int patch);
UPR_API int upr_enh_losses_f32(const float* enhanced, const float* img_low, int n, int h, int w, double base_target, int patch,
                               float* losses3, float* saved, void* workspace, size_t workspace_bytes, upr_stream_t stream);
UPR_API int upr_enh_losses_grad_f32(const float* enhanced, const float* img_low, int n, int h, int w, int patch,
                                    const float* saved, const float* upstream3, float* grad_enhanced, upr_stream_t stream);
UPR_API size_t upr_smooth_loss_workspace_bytes(int n, int h, int w);
UPR_API int upr_edge_smooth_loss_f32(const float* illu, const float* img_low, int n, int ci, int cs, int h, int w,
                                     float lambda_val, float alpha, float* loss3, float* grad_illu,
                                     void* workspace, size_t workspace_bytes, upr_stream_t stream);

/* a9 + the data-parallel batch mean + a10 in ONE kernel per rank: the texture statistics kernel exchanges its
 * [sum c, B] pair with every peer through NVLink-mapped symmetric memory (P2P stores + system-scope flags) and writes
 * the all-rank statistics and the dynamic smoothness weight itself -- no NCCL call, no second launch.
 * peer_buffers_dev: device array of `world` addresses, entry r = rank r's buffer of upr_peer_stats_buffer_bytes()
 * bytes (zero-filled once before the first call; allocated with torch.distributed._symmetric_memory or any CUDA IPC /
 * VMM mapping); NULL = single process (then this is upr_texture_*_f32 + upr_dynamic_smooth_weight_f32).  seq: call
 * counter >= 1, the same on every rank, strictly increasing.  method: 0 = 'tv', 1 = 'edge_density'.  All ranks must
 * call it (collective); a peer that never arrives traps the kernel after ~1 s instead of hanging. */
UPR_API size_t upr_peer_stats_buffer_bytes(void);
/* Wall-clock bound on the wait for a peer inside upr_texture_weight_peer_f32 (default 600 000 ms).  A rank whose peer does not
 * arrive in time returns NaN statistics / weight and records {sequence number of the failed call, rank it waited for} in its
 * own buffer; upr_peer_status copies those two words to the host (synchronises `stream`; {0, 0} = no failure so far). */
UPR_API int upr_peer_set_timeout_ms(double ms);
UPR_API int upr_peer_status(const void* own_buffer_dev, unsigned* status2_host, upr_stream_t stream);
UPR_API int upr_texture_weight_peer_f32(const float* x, int n, int c, int h, int w, int method, float* per_image,
                                        float* batch_stats2, void* workspace, size_t workspace_bytes,
                                        const unsigned long long* peer_buffers_dev, int rank, int world, unsigned seq,
                                        float weight_smooth, float* weight_out, upr_stream_t stream);

/* ---- letterbox pre-processing of the enhance drivers (SURVEY 8f N2) ---------------------------------------------
 * utils/letterbox.py:9-102 as called by enhancers/simple_enhance.py:43-58: quantise to u8, cv2.resize INTER_LINEAR
 * (8-bit fixed point) to (rh, rw) when that differs from (h, w), constant border (default 114) to (oh, ow) with the
 * image at (top, left), then /255.  The geometry (ratio, mod-32 padding, rounding) is computed by the caller exactly
 * as the reference does.  Down-scaling only (rh <= h, rw <= w; bit-exact against cv2); up-scaling returns
 * UPR_E_PARAM.  pad_value: c bytes or NULL (114).  The _u8 variant takes the decoded file (u8 HWC) directly. */
UPR_API int upr_letterbox_f32(const float* in_nchw, float* out_nchw, int n, int c, int h, int w, int rh, int rw, int top,
                              int left, int oh, int ow, const unsigned char* pad_value, upr_stream_t stream);
UPR_API int upr_letterbox_u8_f32(const unsigned char* in_nhwc, float* out_nchw, int n, int c, int h, int w, int rh, int rw,
                                 int top, int left, int oh, int ow, const unsigned char* pad_value, upr_stream_t stream);

/* ---- EXTENSION ops (SURVEY 8f N4): not present in the reference, no reference parity target ------------------
 * The north-star names a Gaussian pyramid, log-domain SSR/MSR and gamma; the reference contains none of them
 * (SURVEY 8a "ABSENT").  These entry points implement them against OpenCV / NumPy semantics and are NOT called by
 * any reference-facing entry point.  planes = n*c; all tensors are [planes][h][w] f32.
 *   upr_ext_gaussian_blur_f32 : cv2.GaussianBlur(src, (ksize,ksize), sigma, borderType=BORDER_REFLECT_101), odd
 *                               ksize <= 31 (sigma <= 0: OpenCV's rule, incl. its fixed tables for ksize <= 7).
 *                               The input tile is staged by TMA (cp.async.bulk.tensor) when rows are 16-byte aligned.
 *   upr_ext_msr_f32           : sum_s weights[s] * (log(x + eps) - log(GaussianBlur_s(x) + eps)), 1 <= nscales <= 4
 *                               (nscales == 1: single-scale Retinex); one staged tile serves all scales.
 *   upr_ext_pyr_down_f32      : cv2.pyrDown(src) -> [planes][(h+1)/2][(w+1)/2].
 *   upr_ext_gamma_f32         : pow(clamp(x, 0, 1), gamma).
 * out must not alias x for the two filters. */
UPR_API int upr_ext_gaussian_blur_f32(const float* x, float* out, int planes, int h, int w, int ksize, double sigma,
                                      upr_stream_t stream);
UPR_API int upr_ext_msr_f32(const float* x, float* out, int planes, int h, int w, int nscales, const int* ksizes,
                            const double* sigmas, const float* weights, float eps, upr_stream_t stream);
UPR_API int upr_ext_pyr_down_f32(const float* x, float* out, int planes, int h, int w, upr_stream_t stream);
UPR_API int upr_ext_gamma_f32(const float* x, float* out, long long count, float gamma, upr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* UPRETINEX_B200_H */
