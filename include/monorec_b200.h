/*
 * monorec_b200.h -- C ABI of libmonorec_b200.so (sm_100a kernels for MonoRec's hot path).
 *
 * The reference (Brummi/MonoRec) is pure Python/PyTorch and has no FFI of its own; these entry points are
 * what a binding for the hot path replaces (SURVEY.md §8b).  Every entry point cites the reference code it
 * stands in for.  Conventions:
 *   - plain C types only; device pointers are owned by the caller (PyTorch allocates inputs and outputs);
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *   - return 0 on success, a negative MR_E* code or a positive cudaError_t otherwise;
 *     mr_last_error() returns a thread-local message for the last failure;
 *   - no global mutable state: callable concurrently from several host threads on different devices.
 * All tensors are contiguous fp32 unless stated; image-like tensors are NCHW like the reference's.
 */
#ifndef MONOREC_B200_H
#define MONOREC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MR_OK 0
#define MR_EINVAL -1      /* bad argument (shape, null pointer, unsupported option) */
#define MR_ENOSUPPORT -2  /* valid reference option that this library does not implement */
#define MR_ENOMEM -3      /* workspace too small */

#define MR_MAX_FRAMES 8   /* source frames per keyframe (reference configs use 2..4, BASELINE config 5 uses 6) */

/* Library / build identification: (major<<16 | minor<<8 | patch). */
int mr_version(void);
/* Thread-local description of the last error returned on this thread ("" if none). */
const char* mr_last_error(void);
/* Number of kernels this library has launched from the calling thread since the last reset (for bench.py's
 * `gpu_launches`); mr_launch_count(1) resets after reading. */
long long mr_launch_count(int reset);

/* ---------------------------------------------------------------------------------------------------------
 * Projection tables.  Replaces torch.inverse / matmul at model/monorec/monorec_model.py:171,198,207 and
 * model/layers.py:65 (point_projection): for every (batch b, source frame f)
 *     P = (K_f . inv(pose_f) . pose_kf)[0:3, 0:4],   Kinv = inv(K_kf)[0:3, 0:3]
 *     proj[b,f] = [ P[:, :3] . Kinv | P[:, 3] ]      (3x4 row-major, fp32, evaluated in fp64 on device)
 * with row 0 scaled by W/(W-1), row 1 by H/(H-1) (the reference's normalise-with-(W-1) / sample-with-W quirk,
 * layers.py:67-68 + F.grid_sample default align_corners=False) and 1e-7 added to P[2,3] (layers.py:66), so that
 * for a keyframe pixel (u,v) and plane depth z:   c = proj[:, :3] . [u, v, 1] * z + proj[:, 3]
 *     source pixel  sx = c.x / c.z - 0.5,   sy = c.y / c.z - 0.5 .
 * keyframe_pose, keyframe_K: [B,4,4]; poses[f], intrinsics[f]: host arrays of F device pointers, each [B,4,4].
 * depths (optional, may be NULL): writes 1/linspace(inv_depth_lo, inv_depth_hi, D) to depths[D]
 * (monorec_model.py:184-185; lo = data_dict["inv_depth_max"] = 0.0025, hi = data_dict["inv_depth_min"] = 0.33).
 * No host synchronisation.
 */
int mr_projection_tables(const float* keyframe_pose, const float* keyframe_K,
                         const float* const* poses, const float* const* intrinsics,
                         int B, int F, int H, int W,
                         float* proj /* [B,F,3,4] */,
                         float* depths /* [D] or NULL */, int D, float inv_depth_lo, float inv_depth_hi,
                         void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused plane-sweep cost volume.  Replaces CostVolumeModule.forward, model/monorec/monorec_model.py:150-280
 * (use_ssim=True, sfcv_mult_mask=True, not_center_cv=False, patch_size=3; SSIM = model/layers.py:119-137):
 * per-plane homography warp with bilinear zero-padded sampling, 3x3 SSIM, channel-weighted 3x3 patch cost,
 * validity mask, per-frame view weighting and multi-frame fusion, in one kernel without intermediate tensors.
 *   keyframe      [B,3,H,W]
 *   frames        host array of F device pointers, each [B,3,H,W]
 *   proj          [B,F,3,4] from mr_projection_tables
 *   depths        [D] plane depths (index 0 = farthest)
 *   out_cv        [B,D,H,W]      data_dict["cost_volume"]
 *   out_sfcv      [F,B,D,H,W]    data_dict["single_frame_cvs"][f] = out_sfcv[f]
 *   alpha         view-weight sharpness (reference: 10), chan_w[3] channel weights (reference: 5/32,16/32,11/32)
 * Constraints: 1 <= F <= MR_MAX_FRAMES, 2 <= D <= 128, H >= 5, W >= 5.
 * The source frames are read through TMA (cp.async.bulk.tensor boxes of the NCHW frames into shared-memory windows shared by
 * runs of consecutive depth planes); the frames must stay unmodified until the kernel has finished (stream order).
 */
int mr_cost_volume_fwd(const float* keyframe, const float* const* frames, const float* proj, const float* depths,
                       float* out_cv, float* out_sfcv,
                       int B, int F, int D, int H, int W,
                       float alpha, const float* chan_w /* host, 3 floats, NULL = reference default */,
                       void* stream);

/* The same kernel with the TMA window staging switched off: every bilinear tap is a global-memory load (what
 * mr_cost_volume_fwd itself does for frames TMA cannot address: W % 4 != 0 or a base that is not 16-byte aligned, and for
 * the few (frame, plane) units whose source footprint does not fit a shared-memory window).  Same results up to the
 * last-bit differences of the two interpolation code paths; kept callable for tests and A/B timing. */
int mr_cost_volume_fwd_gather(const float* keyframe, const float* const* frames, const float* proj, const float* depths,
                              float* out_cv, float* out_sfcv,
                              int B, int F, int D, int H, int W,
                              float alpha, const float* chan_w, void* stream);

/* mr_cost_volume_fwd that additionally writes the single-frame volumes in the convolution engine's input layout,
 * out_sfcv_nhwc [F,B,H,W,D] as fp32 (MR_DT_F32) or IEEE half (MR_DT_F16), from the registers of the kernel's per-pixel phase
 * (replaces F layout-change launches in front of the MaskModule, monorec_model.py:357-365).  Needs D <= 32 and D % 8 == 0. */
int mr_cost_volume_fwd_nhwc(const float* keyframe, const float* const* frames, const float* proj, const float* depths,
                            float* out_cv, float* out_sfcv, void* out_sfcv_nhwc, int nhwc_dtype,
                            int B, int F, int D, int H, int W,
                            float alpha, const float* chan_w, void* stream);

/* Same path with HOST buffers (pinned or pageable): uploads the images and matrices, runs
 * mr_projection_tables + mr_cost_volume_fwd and downloads both volumes; batch elements are pipelined on
 * internal streams so copies overlap the kernel.  This is the end-to-end entry bench.py times as `e2e`.
 *   h_keyframe [B,3,H,W]; h_frames [F,B,3,H,W]; h_keyframe_pose,h_keyframe_K [B,4,4]; h_poses,h_intrinsics [F,B,4,4]
 *   h_out_cv [B,D,H,W]; h_out_sfcv [F,B,D,H,W] or NULL: the single-frame volumes then stay in the workspace on the device
 *   (no consumer of the reference reads them on the host: they feed the MaskModule on the device, monorec_model.py:693-699);
 *   their device address is workspace + mr_cost_volume_host_sfcv_offset(B,F,D,H,W).
 * workspace: device buffer of at least mr_cost_volume_host_workspace(B,F,D,H,W) bytes (caller-owned).  It must be idle: the
 * call runs on internal non-blocking streams (created once per host thread and device, reused by later calls) that are not
 * ordered against work the caller has queued on other streams; the call returns after all of its copies have completed.
 */
long long mr_cost_volume_host_workspace(int B, int F, int D, int H, int W);
long long mr_cost_volume_host_sfcv_offset(int B, int F, int D, int H, int W);
int mr_cost_volume_host(const float* h_keyframe, const float* h_frames,
                        const float* h_keyframe_pose, const float* h_keyframe_K,
                        const float* h_poses, const float* h_intrinsics,
                        float* h_out_cv, float* h_out_sfcv,
                        int B, int F, int D, int H, int W,
                        float inv_depth_lo, float inv_depth_hi, float alpha,
                        void* workspace, long long workspace_bytes);

/* ---------------------------------------------------------------------------------------------------------
 * Convolution engine for the MaskModule / DepthModule stacks (model/monorec/monorec_model.py:287-385, :476-557).
 * Activations are NHWC fp32 inside the engine ([B, H, W, C], C contiguous); weights are packed by the host side as
 * [kh][kw][Cin_total][Cout].  One descriptor covers what the reference spreads over several modules:
 *   PadSameConv2d  (model/layers.py:220-252)  -> pad_t / pad_l (asymmetric TF-"SAME" zero padding, out-of-range taps = 0)
 *   torch.cat      (monorec_model.py:372-380, :541-545) -> up to MR_CONV_MAX_SRC channel-concatenated sources
 *   Upsample(x2)   (layers.py:349)            -> upsample2: nearest-neighbour x2 applied while reading
 *   Conv2d + bias + LeakyReLU / Sigmoid / |tanh| (layers.py:301-335, monorec_model.py:340-343, :554-557) -> act
 *   ConvTranspose2d(k4,s2)+crop (layers.py:380-400) -> four sub-pixel 2x2 convolutions written with oy_step = ox_step = 2
 */
#define MR_CONV_MAX_SRC 3
#define MR_DT_F32 0
#define MR_DT_F16 1           /* IEEE half storage: tensor-core path (kind::f16, fp32 accumulate) and the helper kernels */
#define MR_ACT_NONE 0
#define MR_ACT_LEAKY 1     /* x >= 0 ? x : act_a * x  (any slope, on every path) */
#define MR_ACT_SIGMOID 2
#define MR_ACT_ABSTANH 3   /* act_a + act_b * |tanh(x)|  (depth heads + inverse-depth affine, monorec_model.py:717) */

typedef struct mr_conv_desc {
    int n_src;                               /* 1..MR_CONV_MAX_SRC */
    const float* src[MR_CONV_MAX_SRC];       /* each [B, Hs, Ws, src_c[i]] */
    int src_c[MR_CONV_MAX_SRC];
    int B, Hs, Ws;                           /* stored size of every source */
    int upsample2;                           /* 1: virtual input is the nearest-neighbour x2 upsampling of the sources */
    int kh, kw, sy, sx, pad_t, pad_l;
    int Ho, Wo, Cout;                        /* output grid computed by this call */
    const float* weight;                     /* [kh][kw][sum src_c][Cout] */
    const float* bias;                       /* [Cout] or NULL */
    float* dst;                              /* [B, dst_H, dst_W, dst_c] */
    int dst_H, dst_W, dst_c, dst_coff;       /* channel slice [dst_coff, dst_coff + Cout) of the destination */
    int oy_step, ox_step, oy_off, ox_off;    /* output (oy, ox) is stored at (oy*oy_step + oy_off, ox*ox_step + ox_off) */
    int act;
    float act_a, act_b;
    int src_dtype, dst_dtype;                /* MR_DT_F32 / MR_DT_F16 storage of the sources (and packed tensor-core weights) /
                                                of the destination; pointers are typed float* for historical reasons */
} mr_conv_desc;

int mr_conv2d_nhwc(const mr_conv_desc* desc, void* stream);
/* Same descriptor on the tensor cores (tcgen05, kind::tf32: TF32 products, fp32 accumulation in TMEM, fp32 storage).
 * `weight` is packed as [kh*kw][n_pad][k_pad] (K contiguous): Cout padded to n_pad (multiple of 16, <= 256), every source
 * padded to a multiple of 32 channels (k_pad = sum).  Needs src_c[i] % 4 == 0 and upsample2 == 0 (nearest-x2 upsampling is
 * expressed as sub-pixel convolutions on this path).  round_out: round stored activations to TF32 (nearest).
 * With src_dtype = MR_DT_F16 the sources and the packed weights are half, a K chunk is 64 channels (every source padded to
 * a multiple of 64) or, if the caller packed every source to a multiple of 32 instead and that gives a different k_pad,
 * 32 channels (64-byte swizzle rows); the MMA is kind::f16; dst_dtype selects half or float output.
 * Stride-1 layers whose packed weights fit in shared memory twice per SM run on the "halo" variant of the kernel (same
 * results).  Tuning switches (environment, read once): MONOREC_B200_TC_HALO=0|1|2, MONOREC_B200_TC_HALO_F16=0|1,
 * MONOREC_B200_TC_CTAS=n. */
int mr_conv2d_nhwc_tc(const mr_conv_desc* desc, int n_pad, int k_pad, int round_out, void* stream);
/* The sub-pixel convolutions of one layer -- Refine's ConvTranspose2d(k4,s2)+crop = four 2x2 filters (model/layers.py:380-400),
 * Upconv's nearest-x2 + pad + 2x2 conv = 1x1 / 1x2 / 2x1 / 2x2 filters (:338-356) -- in ONE launch: descs[0..n_phases) share the
 * sources, the destination, Cout, bias, activation and strides and differ in kh, kw, pad_t, pad_l, weight, oy_off, ox_off
 * (anything else: MR_EINVAL).  Tiles are ordered (spatial tile, phase), so the phases of a tile run side by side and the input is
 * read from HBM once instead of once per phase.  n_phases = 1 is mr_conv2d_nhwc_tc. */
int mr_conv2d_nhwc_tc_phases(const mr_conv_desc* descs, int n_phases, int n_pad, int k_pad, int round_out, void* stream);
/* Launch plan of mr_conv2d_nhwc_tc_phases(descs, n_phases, n_pad, k_pad, round_out, ...) on a device with `sms` SMs (pure host
 * code, callable without a GPU; the launch itself uses this function with the device's SM count).  Runs every argument check
 * that needs no driver (MR_EINVAL and mr_last_error() like the launch) and reports which kernel, ring and epilogue the call
 * takes.  The MONOREC_B200_TC_* switches above apply.
 *   kernel       MR_TC_REFETCH: one input box and one weight slice per (tap, K chunk); strided layers, sub-pixel phases;
 *                MR_TC_HALO: stride 1, one input box per (tile, K chunk), weights resident in shared memory;
 *                MR_TC_HALO_STREAM: the same with the weights streamed through a ring of b_stream stages
 *   ctas_per_sm  resident CTAs per SM the grid is sized for; stages: input ring stages (MR_TC_REFETCH: input + weight)
 *   row_bytes    bytes of one K-chunk row in shared memory (128 or 64), kc: channels per K chunk
 *   total_tiles  output tiles (8x16 pixels for MR_TC_REFETCH, 16x8 for the halo kernels) over batch and phases;
 *                grid = min(sms * ctas_per_sm, total_tiles) persistent CTAs
 *   epilogue     MR_TC_EPI_STAGED (LeakyReLU / no activation, 16-byte aligned channel slices), MR_TC_EPI_ONE_COLUMN (Cout == 1),
 *                MR_TC_EPI_GENERIC (everything else) */
#define MR_TC_REFETCH 0
#define MR_TC_HALO 1
#define MR_TC_HALO_STREAM 2
#define MR_TC_EPI_STAGED 0
#define MR_TC_EPI_ONE_COLUMN 1
#define MR_TC_EPI_GENERIC 2
typedef struct mr_conv_tc_plan {
    int kernel, ctas_per_sm, stages, b_stream, row_bytes, kc;
    int tmem_cols;                           /* tensor-memory columns per CTA (two accumulators) */
    int smem_bytes;                          /* dynamic shared memory per CTA */
    int total_tiles, grid, epilogue;
} mr_conv_tc_plan;
int mr_conv2d_nhwc_tc_plan(const mr_conv_desc* descs, int n_phases, int n_pad, int k_pad, int round_out, int sms,
                           mr_conv_tc_plan* out);
/* Host-side weight packing for mr_conv2d_nhwc_tc (pure host code, callable without a GPU).
 *   mr_pack_conv_weights_bytes: size of the packed tensor and its n_pad / k_pad for a correlation kernel (Cout, sum src_c, kh, kw)
 *     whose input channels are the concatenation of n_src sources; dtype MR_DT_F32 (TF32-rounded fp32) or MR_DT_F16.
 *   mr_pack_conv_weights: w = host [Cout][Cin][kh][kw] (nn.Conv2d.weight), out = host buffer of that size; upload it and pass
 *     the device copy as mr_conv_desc.weight together with n_pad / k_pad.
 *   mr_subpixel_convt_k4s2: phase (py, px) of Refine's ConvTranspose2d(k4, s2) + crop (model/layers.py:380-400) as a 2x2
 *     correlation: w = host [Cin][Cout][4][4] (nn.ConvTranspose2d.weight), out = host [Cout][Cin][2][2]; run it with
 *     pad_t / pad_l as returned, oy_step = ox_step = 2, oy_off = py, ox_off = px.
 *   mr_subpixel_upconv2: phase (py, px) of Upconv's nearest-x2 + pad(0,1,0,1) + Conv2d(k2) (model/layers.py:338-356):
 *     w = host [Cout][Cin][2][2], out = host [Cout][Cin][kh_out][kw_out] (kh_out = 1 + py, kw_out = 1 + px), pad 0.
 *   mr_conv_workspace_bytes: device scratch a convolution call needs (0: everything is staged in shared / tensor memory). */
long long mr_pack_conv_weights_bytes(int Cout, int n_src, const int* src_c, int kh, int kw, int dtype, int* n_pad, int* k_pad);
int mr_pack_conv_weights(const float* w, int Cout, int n_src, const int* src_c, int kh, int kw, int dtype, void* out);
int mr_subpixel_convt_k4s2(const float* w, int Cin, int Cout, int py, int px, float* out, int* pad_t, int* pad_l);
int mr_subpixel_upconv2(const float* w, int Cout, int Cin, int py, int px, float* out, int* kh_out, int* kw_out);
long long mr_conv_workspace_bytes(const mr_conv_desc* desc);
/* sizeof(mr_conv_desc) as compiled into the library (bindings check their mirror of the struct against it). */
int mr_sizeof_conv_desc(void);

/* NCHW [B,C,H,W] -> channel slice of an NHWC tensor [B,H,W,dst_c]; optional per-pixel multiplier
 * scale[b,h,w] applied as (1 - scale) (monorec_model.py:713: cost_volume * (1 - cv_mask)). */
int mr_nchw_to_nhwc(const float* src, float* dst, int B, int C, int H, int W, int dst_c, int dst_coff,
                    const float* one_minus_scale, void* stream);
/* The same with a half destination; the layout kernels below have _f16 twins for half NHWC tensors. */
int mr_nchw_to_nhwc_f16(const float* src, void* dst, int B, int C, int H, int W, int dst_c, int dst_coff,
                        const float* one_minus_scale, void* stream);
int mr_maxpool2_nhwc_f16(const void* src, void* dst, int B, int H, int W, int C, void* stream);
int mr_max_over_frames_f16(const void* src, void* dst, int F, long long n_per_frame, void* stream);
/* One pass over an encoder level's output x [F*B,H,W,C] (MR_DT_F16: C % 8 == 0, MR_DT_F32: C % 4 == 0; H, W even) that writes both
 * consumers: pooled [F*B,H/2,W/2,C] = nn.MaxPool2d(2) (monorec_model.py:304-316) and frame_max [B,H,W,C] = the element-wise
 * max over the F frames (:362-365). */
int mr_pool_and_frame_max(const void* src, void* pooled, void* frame_max, int dtype, int F, int B, int H, int W, int C,
                          void* stream);
/* torchvision resnet18.maxpool = MaxPool2d(3, stride 2, padding 1) (the trunk's stem pool, monorec_model.py:122) on an NHWC /
 * channels-last tensor: src [B,H,W,C] -> dst [B,(H-1)/2+1,(W-1)/2+1,C]; MR_DT_F16: C % 8 == 0, MR_DT_F32: C % 4 == 0. */
int mr_maxpool3s2_nhwc(const void* src, void* dst, int dtype, int B, int H, int W, int C, void* stream);
/* dst[i] = (half) src[i] for n contiguous fp32 values (used for channels-last feature maps). */
int mr_cast_f32_to_f16(const float* src, void* dst, long long n, void* stream);
/* nn.MaxPool2d(2) on NHWC (monorec_model.py:304-316). H and W must be even. */
int mr_maxpool2_nhwc(const float* src, float* dst, int B, int H, int W, int C, void* stream);
/* Element-wise max over the leading axis: dst[n] = max_f src[f*n_per_frame + n]  (monorec_model.py:362-365). */
int mr_max_over_frames(const float* src, float* dst, int F, long long n_per_frame, void* stream);
/* out[b,d,p] = volume[b,d,p] * (1 - mask[b,p])   (monorec_model.py:713, NCHW volume [B,D,HW], mask [B,HW]). */
int mr_mask_volume(const float* volume, const float* mask, float* out, int B, int D, int HW, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Evaluation-side helpers (SURVEY.md section 8f row 2).
 *
 * mr_sparse_metrics: the seven sparse depth metrics of model/metric_functions/sparse_metrics.py:81-251 (a1, a2, a3, rmse,
 * rmse_log, abs_rel, sq_rel with utils/util.py:36-65, :101-118) in one pass; evaluater/evaluater.py:78-112 calls the seven
 * reference functions (~12 elementwise torch kernels each) one after the other.
 *   result, target   [B,1,H,W] predicted / ground-truth INVERSE depth (target 0 = no measurement)
 *   mvobj_mask       [B,1,H,W] or NULL: with it, pixels whose mask is <= 0.5 are excluded (the *_onlydynamic variants)
 *   roi              host int[4] {r0, r1, c0, c1} (python slice semantics) or NULL; max_distance <= 0: no clamp
 *   pred_all_valid   0: pixels with result == 0 are excluded (the *_onlyvalid variants)
 *   out_metrics      device float[7]: a1, a2, a3, rmse, rmse_log, abs_rel, sq_rel; no host synchronisation
 *   workspace        device buffer of mr_sparse_metrics_workspace(B) bytes, 8-byte aligned
 * mr_images_u8_to_f32: uint8 HWC images [B,Hs,Ws,3] -> float CHW [B,3,H,W] = u / 255 - 0.5 of the crop starting at
 * (crop_top, crop_left) (data_loader/kitti_odometry_dataset.py:121-132 without the PIL resize). */
long long mr_sparse_metrics_workspace(int B);
int mr_sparse_metrics(const float* result, const float* target, const float* mvobj_mask, int B, int H, int W,
                      const int* roi, float max_distance, int pred_all_valid, float* out_metrics,
                      void* workspace, long long workspace_bytes, void* stream);
int mr_images_u8_to_f32(const unsigned char* src, float* dst, int B, int Hs, int Ws, int crop_top, int crop_left,
                        int H, int W, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Point-cloud side (SURVEY.md section 8f row 3): create_pointcloud.py:65-105 + utils/ply_utils.py:34-53 on the device.
 *
 * mr_pointcloud_keep_mask: keep[b,p] = 1 iff no pixel with cv_mask >= thresh lies in the (mask_fill+1)^2 window around p
 *   (create_pointcloud.py:77-78 with mask_fill = 32, thresh = 0.1); cv_mask, keep: [B,1,H,W].
 * mr_pointcloud_add: PLYSaver.add_depthmap with the sliding-window vote folded in.  Appends the vertices (x, y, z, r, g, b)
 *   of a batch to a device buffer, in the reference's order (batch element, then pixel), without host synchronisation.
 *   inv_depth [B,1,H,W] (data_dict["result"]); keyframe [B,3,H,W]; K, pose [B,4,4];
 *   keep_masks: host array of n_masks device pointers [B,1,H,W] (the window's keep masks) -- a pixel survives iff more than
 *     n_masks - min_hits of them are 1 (create_pointcloud.py:93-95); n_masks = 0: no vote;
 *   min_d / max_d: distance range; roi: host int[4] {r0, r1, c0, c1} or NULL; dropout_rand: [B,1,H,W] uniform numbers (a
 *     vertex is kept iff rand > dropout; torch.rand_like in the reference) or NULL;
 *   vertices: device float [capacity][6]; n_before: vertices already stored; n_after: DEVICE long long, the new count, or
 *     minus the needed count if the buffer is too small (then nothing is written);
 *   workspace: device buffer of mr_pointcloud_workspace(B,H,W) bytes. */
int mr_pointcloud_keep_mask(const float* cv_mask, float* keep, int B, int H, int W, int mask_fill, float thresh, void* stream);
long long mr_pointcloud_workspace(int B, int H, int W);
int mr_pointcloud_add(const float* inv_depth, const float* keyframe, const float* K, const float* pose,
                      const float* const* keep_masks, int n_masks, int min_hits, int B, int H, int W,
                      float min_d, float max_d, const int* roi, const float* dropout_rand, float dropout,
                      float* vertices, long long capacity, long long n_before, long long* n_after,
                      void* workspace, long long workspace_bytes, void* stream);

/* ---- photometric reprojection loss, forward and backward (SURVEY.md 8f row 4) -------------------------------------------
 * Replaces reprojection_loss (reference: model/loss_functions/common_losses.py:16-114) with error_function=compute_errors
 * (:10-13), combine_frames="min", mono_auto=False, reduce=False -- the argument sets of model/loss_functions/monorec_loss.py
 * :185-188, :264-265, :355, :361 -- and torch autograd of it w.r.t. the predicted inverse depth (trainer/monorec_trainer.py
 * :143-145).  proj: [B,F,12] rows of mr_projection_tables (depths = NULL) for the F source frames of this call (mono frames
 * and / or the stereo frame); inv_depth: [B,1,H,W] `depth_prediction`.
 *   mr_reprojection_loss_fwd: out_errors [B,H,W] = min over the frames of 0.85 mean_c SSIM + 0.15 mean_c |warped - keyframe|
 *     (Gaussian 3x3 window, zero padding, comp mode: model/layers.py:79-139), +inf where no frame gives a usable sample
 *     (:57 / border > 0: :60-61; automasking != 0: :80-83); out_winner [B,H,W] = index of the frame giving the minimum, -1: none.
 *   mr_reprojection_loss_bwd: out_grad_inv_depth [B,1,H,W] = d (sum_p grad_errors[p] errors[p]) / d inv_depth; grad_errors at
 *     pixels whose winner is -1 is ignored.  Needs nothing from the forward pass but out_winner. */
int mr_reprojection_loss_fwd(const float* keyframe, const float* const* frames, const float* proj, const float* inv_depth,
                             int B, int F, int H, int W, int automasking, int border, float* out_errors, int* out_winner,
                             void* stream);
int mr_reprojection_loss_bwd(const float* keyframe, const float* const* frames, const float* proj, const float* inv_depth,
                             const float* grad_errors, const int* winner, int B, int F, int H, int W,
                             float* out_grad_inv_depth, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MONOREC_B200_H */
