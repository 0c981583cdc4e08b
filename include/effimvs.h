/*
 * effimvs.h -- C-ABI of libeffimvs.so: the B200 (sm_100a) cost-volume hot path of Effi-MVS+.
 *
 * The upstream project (bdwsq1996/Effi-MVS-plus) has no FFI; its boundary is a set of
 * Python call sites.  Each entry point below names the upstream call site it replaces
 * (paths relative to the upstream tree).  INTEGRATION.md shows the ctypes binding and the
 * monkey-patch a maintainer adds on the upstream side.
 *
 * Conventions
 *   - every function returns 0 on success or a negative EFFIMVS_E* code;
 *     effimvs_last_error() returns a thread-local description of the last failure.
 *   - all tensor pointers are DEVICE pointers owned by the caller, fp32, dense, in the
 *     layouts written next to each argument (upstream's NCHW / NCDHW order).  Arrays
 *     documented as "host array" are small host-side arrays of device pointers.
 *   - the library never allocates persistent memory and never synchronises; work is
 *     enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - re-entrant; no mutable global state besides the thread-local error string.
 */
#ifndef EFFIMVS_H
#define EFFIMVS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EFFIMVS_OK 0
#define EFFIMVS_EINVAL (-1)       /* bad argument (null pointer, non-positive size, ...) */
#define EFFIMVS_EUNSUPPORTED (-2) /* shape outside what the kernels are built for */
#define EFFIMVS_ECUDA (-3)        /* CUDA runtime / launch error */
#define EFFIMVS_EWORKSPACE (-4)   /* caller-provided workspace too small */

#define EFFIMVS_MAX_SRC_VIEWS 16

/* hypothesis source for the warp kernels */
#define EFFIMVS_HYP_TENSOR 0 /* hyp = (B,D,H,W) depth per pixel and plane                */
#define EFFIMVS_HYP_PLANES 1 /* hyp = (B,D) one depth per plane (stage-1 plane sweep)    */
#define EFFIMVS_HYP_LOCAL 2  /* hyp = cur_depth (B,1,H,W); D inverse-depth samples around
                                it are generated in-kernel (models/module.py:554-570)    */

/* memory layout of the feature maps handed to the warp kernels */
#define EFFIMVS_FEA_NCHW 0 /* (B,C,H,W) planar, upstream's default                               */
#define EFFIMVS_FEA_NHWC 1 /* (B,H,W,C) channels-last, what a channels_last cuDNN FPN emits      */

/* per-batch scalar (B) or per-pixel (B,H,W) depth range of a volume */
#define EFFIMVS_RANGE_SCALAR 0
#define EFFIMVS_RANGE_PIXEL 1

/* precision of the 3-D regularization nets */
#define EFFIMVS_PREC_F32 0  /* CUDA-core fp32 direct convolution (exact-parity path)     */
#define EFFIMVS_PREC_BF16 1 /* bf16 operands, fp32 accumulate in TMEM (tcgen05 implicit GEMM) */
#define EFFIMVS_PREC_BF16X3 2 /* operands split into hi + lo bf16, three tcgen05 MMAs per product
                                 (hi*hi + hi*lo + lo*hi): fp32-grade results on the tensor cores */

const char* effimvs_last_error(void);
int effimvs_version(void);

/* a1 + models/module.py:314.  cams (B,V,2,4,4): [b,v,0]=extrinsic, [b,v,1,:3,:3]=intrinsic.
 * proj_out (B,V-1,12): rows of rot (9) then trans (3) of  P_src @ inverse(P_ref),
 * P = E with P[:3,:4] = K @ E[:3,:4]  (models/Effi_MVS_plus.py:34-37).  Computed in fp64,
 * rounded once to fp32.  (The torch binding may instead pass upstream's own fp32
 * torch.inverse result to the warp kernels; this entry point serves non-torch callers and
 * CUDA-graph capture.) */
int effimvs_relative_projection_f32(const float* cams, int B, int V, float* proj_out, void* stream);

/* a2 alone: homo_warping_new (models/module.py:303-344), materialising the warped volume.
 *   src_fea (B,C,H,W) planar, proj (B,12) for this source view, hyp TENSOR (B,D,H,W) or PLANES (B,D)
 *   -> warped_out (B,C,D,H,W).  Provided for call-site parity; the fused entry points below never
 *   write this volume. */
int effimvs_homo_warp_f32(const float* src_fea, const float* proj, const float* hyp, int hyp_mode,
                          int B, int C, int H, int W, int D, float* warped_out, void* stream);

/* The scalars the cascade derives from depth_values (B,Dv) alone (models/Effi_MVS_plus.py:409-424, models/module.py:577-585), bit-identical to the
 * torch expressions: out (8 B + B D1 floats) = 8 rows of B scalars [1/min, 1/max, 1/(1/min), 1/(1/max), interval_1..3 =
 * ((max - min) / Dv) * ratios3[s], 0] followed by the (B, D1) plane-sweep hypotheses 1 / (min + k (max - min) / (D1 - 1));
 * min / max = depth_values[:, 0] / [:, -1] (inverse depths).
 * ratios3 is a HOST array of three floats (upstream's depth_interals_ratio 4, 2, 1). */
int effimvs_depth_ranges_f32(const float* depth_values, int B, int Dv, int D1, const float* ratios3, float* out, void* stream);

/* get_cur_depth_range_samples (models/module.py:554-570): ndepth samples around cur (B,H,W) in the
 * caller's space (upstream: inverse depth), half-width (ndepth/2)*interval[b], clamped like upstream.
 *   -> samples_out (B,ndepth,H,W) */
int effimvs_depth_range_samples_f32(const float* cur, const float* interval, int B, int ndepth, int H, int W,
                                    float* samples_out, void* stream);

/* a2 + a3 + a5 + weighted aggregation in one pass; the warped (B,C,D,H,W) volume is never
 * materialised.  Replaces, per source view, homo_warping_new (models/module.py:303-344) +
 * the group-wise correlation (models/Effi_MVS_plus.py:39-40, :222-224) and the aggregation
 * over views (:52-53/:67, :233-234/:244).
 *   ref_fea   (B,C,H,W), or (B,H,W,C) with fea_layout = EFFIMVS_FEA_NHWC
 *   src_fea   host array of n_src device pointers, each laid out like ref_fea
 *   proj      (B,n_src,12) from effimvs_relative_projection_f32 (or torch)
 *   hyp       see EFFIMVS_HYP_*;  interval (B) inverse-depth step, only for HYP_LOCAL
 *   weights   (B,n_src,H,W) view weights or NULL (plain mean over views)
 *   sim_out   (B,G,D,H,W);  hyp_out (B,D,H,W) depth hypotheses actually used, or NULL
 * Alignment: feature pointers need 16 bytes (NCHW: 4).  EFFIMVS_FEA_NHWC maps whose pointers are all 32-byte
 * aligned take the TMA-staged tile kernels (256-bit loads); 16-byte aligned ones run the gather kernels --
 * same results, slower. */
int effimvs_warp_corr_agg_f32(const float* ref_fea, const float* const* src_fea, int n_src,
                              const float* proj, const float* hyp, int hyp_mode, const float* interval,
                              const float* weights, int B, int C, int H, int W, int D, int G, int fea_layout,
                              float* sim_out, float* hyp_out, void* stream);

/* Stage-1 form (models/Effi_MVS_plus.py:32-46): per-view similarity (G must be 1) and the
 * entropy of its softmax over D, which upstream feeds to PixelwiseNet.
 *   sims_out (B,n_src,D,H,W), entropy_out (B,n_src,H,W) */
int effimvs_warp_corr_views_f32(const float* ref_fea, const float* const* src_fea, int n_src,
                                const float* proj, const float* hyp, int hyp_mode,
                                int B, int C, int H, int W, int D, int fea_layout,
                                float* sims_out, float* entropy_out, void* stream);

/* sum_v w_v * sim_v / (sum_v w_v + 1e-6)  (models/Effi_MVS_plus.py:52-53, :67).
 *   sims (B,n_src,D,H,W), weights (B,n_src,H,W) -> out (B,D,H,W) */
int effimvs_weighted_agg_f32(const float* sims, const float* weights, int B, int n_src, int D, int H, int W,
                             float* out, void* stream);

/* a6: pro_bilinear_sampler (models/Effi_MVS_plus.py:102-134) on the un-permuted volume.
 *   volume (B,D,H,W); depth_sample (B,d,H,W); depth_min/depth_max per EFFIMVS_RANGE_*
 *   out (B,d,H,W).  sample_stride: 1, or 2 to read depth_sample from a (B,d,2H,2W) tensor at
 *   even pixels (the nearest x1/2 of Effi_MVS_plus.py:514 fused in; a8). */
int effimvs_volume_lookup_f32(const float* volume, const float* depth_sample, const float* depth_min,
                              const float* depth_max, int range_mode, int sample_stride,
                              int B, int D, int d, int H, int W, float* out, void* stream);

/* a7: GetCost.forward (models/Effi_MVS_plus.py:257-303): ndepth hypotheses around
 * cur_depth (B,1,H,W), looked up in raw (pro[-1]) and reg (pro[0]) volumes (B,D,H,W).
 *   out (B,2*ndepth,H,W): raw samples first, then reg samples. */
int effimvs_dynamic_cost_f32(const float* cur_depth, const float* raw_volume, const float* reg_volume,
                             const float* interval, const float* depth_min, const float* depth_max,
                             int range_mode, int ndepth, int B, int D, int H, int W, float* out, void* stream);

/* a11 + a12: softmax over D, depth expectation, 4-bin confidence
 * (models/Effi_MVS_plus.py:78-88, models/module.py:518-524).
 *   prob_pre (B,D,H,W); hyp per hyp_mode (TENSOR or PLANES) -> depth (B,H,W), conf (B,H,W) */
int effimvs_softmax_regress_conf_f32(const float* prob_pre, const float* hyp, int hyp_mode,
                                     int B, int D, int H, int W, float* depth_out, float* conf_out, void* stream);

/* One 3x3x3 (de)convolution layer with eval-BatchNorm folded in, fp32 CUDA cores
 * (models/module.py:124-209).  x (B,Cin,D,H,W) -> y (B,Cout,Do,Ho,Wo) written at channel
 * offset y_coff of a tensor with y_ctot channels (fuses the torch.cat of module.py:513).
 *   weight: conv (Cout,Cin,3,3,3), deconv (Cin,Cout,3,3,3), BN scale already multiplied in
 *   bias (Cout) or NULL; relu 0/1; residual (B,Cout,Do,Ho,Wo) added after the ReLU, or NULL
 *   stride s* in {1,2}; padding 1; for deconv output_padding = s-1 (so Do = s*D). */
int effimvs_conv3d_f32(const float* x, const float* weight, const float* bias, const float* residual,
                       int B, int Cin, int Cout, int D, int H, int W, int sd, int sh, int sw,
                       int transposed, int relu, float* y, int y_coff, int y_ctot, void* stream);

/* The same layer on the tensor cores: bf16 operands, fp32 accumulation in TMEM (tcgen05 implicit
 * GEMM, operands staged by bulk TMA copies).  Supported: convolution stride 1 or (2,2,2);
 * transposed convolution stride (sd,2,2) with sd in {1,2}.  Cin in {8,16,32}, Cout <= 32.
 * x, residual and y are fp32 NCDHW (converted to / from the kernel's channel-planar bf16 layout
 * inside the call; the net-level entry points below keep activations in that layout between
 * layers).  workspace: effimvs_conv3d_bf16_workspace_bytes() bytes. */
size_t effimvs_conv3d_bf16_workspace_bytes(int B, int Cin, int Cout, int D, int H, int W, int sd, int transposed,
                                           int precision);
int effimvs_conv3d_bf16(const float* x, const float* weight, const float* bias, const float* residual, int B, int Cin,
                        int Cout, int D, int H, int W, int sd, int transposed, int relu, int precision /* BF16 | BF16X3 */,
                        void* workspace, size_t workspace_bytes, float* y, void* stream);

/* a9: CostRegNet_2_sample_FPN3D_Fast.forward (models/module.py:453-463).
 *   x (B,1,D,H,W), D,H,W multiples of 4.  weights: host array of 9 device pointers
 *   (conv0..conv7 BN-folded, prob), biases: host array of 8 device pointers (conv0..conv7).
 *   workspace: effimvs_costreg_workspace_bytes() bytes of device memory.
 *   prob_out (B,1,D,H,W).  precision: EFFIMVS_PREC_*. */
size_t effimvs_costreg_workspace_bytes(int B, int D, int H, int W, int precision);
int effimvs_costreg_fpn3d(const float* x, const float* const* weights, const float* const* biases,
                          int B, int D, int H, int W, int precision, void* workspace, size_t workspace_bytes,
                          float* prob_out, void* stream);

/* a10: cost_up_small.forward (models/module.py:509-516).
 *   x (B,1,D,H,W) full-res local volume, prev (B,1,D,H/2,W/2) resampled previous volume.
 *   weights/biases: host arrays of 4 device pointers (conv0, conv_cost, conv1, conv2).
 *   out (B,1,D,H,W). */
size_t effimvs_cost_up_workspace_bytes(int B, int D, int H, int W, int precision);
int effimvs_cost_up_small(const float* x, const float* prev, const float* const* weights,
                          const float* const* biases, int B, int D, int H, int W, int precision,
                          void* workspace, size_t workspace_bytes, float* out, void* stream);

/* The two net-level calls above, split into phases for callers that keep one workspace per network
 * instance and shape (the tensor-core precisions; EFFIMVS_PREC_F32 has no preparation and ignores phases):
 *   EFFIMVS_WS_PREPARE  clear the halos / guards of the padded activation volumes and pack the weights
 *                       (hi / lo bf16 blocks) into the workspace -- depends on the weights and the shape only;
 *   EFFIMVS_WS_RUN      the layers.  The workspace must have been prepared by this entry point with the same
 *                       weights, shape and precision, and not written by anything else since (the layers never
 *                       store to halo positions, so a prepared workspace stays prepared across runs).
 * phases = PREPARE | RUN is the plain call.  x / prev / outputs may be NULL for a PREPARE-only call. */
#define EFFIMVS_WS_PREPARE 1
#define EFFIMVS_WS_RUN 2
int effimvs_costreg_fpn3d_ex(const float* x, const float* const* weights, const float* const* biases,
                             int B, int D, int H, int W, int precision, int phases, void* workspace,
                             size_t workspace_bytes, float* prob_out, void* stream);
int effimvs_cost_up_small_ex(const float* x, const float* prev, const float* const* weights,
                             const float* const* biases, int B, int D, int H, int W, int precision, int phases,
                             void* workspace, size_t workspace_bytes, float* out, void* stream);

/* Input format next to the path (SURVEY section 8(f) row 4): 8-bit images as they sit in the image files -> fp32 in [0,1],
 * out[i] = (float)images[i] / 255.0f with an IEEE division -- bit for bit what upstream's loaders compute on the host
 * (datasets/general_eval.py:83-87, np.float32 / 255.).  Lets a caller ship a quarter of the bytes over PCIe.
 *   images (n) uint8, any layout;  out (n) fp32, same layout */
int effimvs_images_u8_to_f32(const unsigned char* images, long long n, float* out, void* stream);

/* a13: get_reproj_dynamic (misc/fusion.py:117-154).
 *   ref_depth (n,1,h,w), srcs_depth (n,v,1,h,w), ref_cam (n,2,4,4), srcs_cam (n,v,2,4,4)
 *   -> reproj_xyd (n,v,3,h,w).  Camera inverses are taken in-kernel (fp32 adjugate/LU as
 *   documented in DESIGN.md) unless inv_cams is given: (n,1+v,2,4,4) holding inverse(E) and
 *   inverse(K) (padded to 4x4) for ref then sources, e.g. torch.inverse results. */
int effimvs_fusion_reproject_f32(const float* ref_depth, const float* srcs_depth, const float* ref_cam,
                                 const float* srcs_cam, const float* inv_cams, int n, int v, int h, int w,
                                 float* reproj_xyd, void* stream);

/* inverse(E) and inverse(K) of the reference and the v source cameras of every batch item, fp64 Gauss-Jordan rounded once
 * to fp32 (upstream calls torch's .inverse(), misc/fusion.py:24,32): inv_out (n,1+v,2,4,4) in the layout the inv_cams
 * argument of the two entry points around it takes ([:,:,0] = inverse extrinsic, [:,:,1,:3,:3] = inverse intrinsic).  For
 * callers that want no host synchronisation and no torch LU (CUDA-graph capture). */
int effimvs_fusion_invert_cameras_f32(const float* ref_cam, const float* srcs_cam, int n, int v, float* inv_out, void* stream);

/* a14 alone: vis_filter_dynamic (misc/fusion.py:157-181) on an existing reproj_xyd (n,v,3,h,w).
 *   -> masks_out (n,v,K,h,w) uint8, K = v-thres_view+1 (the last ladder step is upstream's `mask`). */
int effimvs_fusion_masks_f32(const float* ref_depth, const float* reproj_xyd, int n, int v, int h, int w,
                             float dist_base, float rel_diff_base, int thres_view, int relative,
                             uint8_t* masks_out, void* stream);

/* a13 + a14 + a15 fused: reprojection, threshold ladder, votes, masked average and
 * back-projection for one reference view (misc/fusion.py:117-181, test_tank.py:473-515).
 *   conf (n,hc,wc) nearest-resized to (h,w); thresholds k/dist_base px and k/rel_diff_base
 *   for k = thres_view..v; final = (conf > prob_threshold) & OR_k(votes_k >= k).
 *   -> final_mask (n,h,w) uint8, depth_avg (n,h,w), points (n,3,h,w);
 *      optional masks_out (n,v,K,h,w) uint8 (K = v-thres_view+1) or NULL. */
int effimvs_fusion_filter_f32(const float* ref_depth, const float* srcs_depth, const float* conf,
                              const float* ref_cam, const float* srcs_cam, const float* inv_cams,
                              int n, int v, int h, int w, int hc, int wc,
                              float dist_base, float rel_diff_base, int thres_view, float prob_threshold,
                              int relative, uint8_t* final_mask, float* depth_avg, float* points,
                              uint8_t* masks_out, void* stream);

/* The same filter for n reference views of one scene in one launch, reading every depth map in place from one stack.
 *   depths (n_depths,h,w) fp32: the scene's depth maps (e.g. the all-gathered tensor of the scene runner)
 *   ref_idx (n) int32: row of view y's reference depth map in `depths`
 *   src_idx (n,vmax) int32: rows of view y's source depth maps, the first src_count[y] entries used
 *   src_count (n) int32: view y's source count, in [thres_view, vmax]; vmax in [1,16] (EFFIMVS_MAX_SRC_VIEWS)
 *   cams (n_depths,2,4,4) fp32: the camera of every row of `depths`, as ref_cam / srcs_cam of effimvs_fusion_filter_f32
 *   inv_cams (n_depths,2,4,4) fp32: their inverses in the layout of effimvs_fusion_invert_cameras_f32 (for instance its
 *         output for ref_cam = cams, v = 1, column 0)
 *   conf (n,hc,wc) fp32, nearest-resized to (h,w); thresholds, thres_view, prob_threshold and relative as
 *         effimvs_fusion_filter_f32 (the ladder of view y has K = src_count[y] - thres_view + 1 rungs)
 *   -> final_mask (n,h,w) u8, depth_avg (n,h,w), points (n,3,h,w)
 * View y's results are bit-identical to effimvs_fusion_filter_f32 on that view alone with the same cameras and inverses.
 * The host rejects null pointers, vmax outside [1,16], n outside [1,65535], non-positive sizes, non-positive bases and
 * thres_view outside [1,vmax].  All index arrays are device arrays and are NOT validated on the device: every entry of
 * ref_idx and of the used part of src_idx must be in [0, n_depths), and thres_view <= src_count[y] <= vmax for every y
 * (the caller checks its host lists before uploading).  There is no masks_out / reproj_xyd here: the per-rung debugging
 * outputs are single-view only. */
int effimvs_fusion_filter_views_f32(const float* depths, int n_depths, const int* ref_idx, const int* src_idx,
                                    const int* src_count, int vmax, const float* cams, const float* inv_cams,
                                    const float* conf, int hc, int wc, float dist_base, float rel_diff_base,
                                    int thres_view, float prob_threshold, int relative, int n, int h, int w,
                                    uint8_t* final_mask, float* depth_avg, float* points, void* stream);

/* ---- SURVEY section 8(f) row 3: per-pixel glue of the ConvGRU update block and convex upsampling --------
 * The 2-D convolutions stay cuDNN on the upstream side; these entry points replace the elementwise
 * chains between them.  Multi-channel maps are channels-last (B,H,W,C). */

/* ConvGRU.forward, reset half (models/update.py:41-45).  zr_pre (n_pix, 2h) = [convz ; convr] outputs
 * WITHOUT bias, hx (n_pix, h + cx) = cat[h, x]  ->  rhx (n_pix, h + cx) = cat[sigmoid(r_pre + bias_r) * h, x]. */
int effimvs_gru_reset_f32(const float* zr_pre, const float* bias_r, const float* hx, long long n_pix, int h, int cx,
                          float* rhx, void* stream);

/* ConvGRU.forward, update half (models/update.py:43, 45-48).  q_pre (n_pix, h) = convq output without bias.
 * h' = (1 - z) * h + z * tanh(q_pre + bias_q), z = sigmoid(z_pre + bias_z); written in place into hx[:, :h]
 * and densely to net_out (n_pix, h). */
int effimvs_gru_update_f32(const float* zr_pre, const float* bias_z, const float* q_pre, const float* bias_q, float* hx,
                           long long n_pix, int h, int cx, float* net_out, void* stream);

/* Start of a stage's refinement: inv = (1 / cur_depth - lo) / ((hi - lo) + 1e-10) (depth_to_disp, models/Effi_MVS_plus.py:151-164)
 * and depth = 1 / clamp(lo + (hi - lo) * inv, 1e-4) (disp_to_depth, :138-148), both (B,HW); lo_disp / hi_disp (B) as below.
 * Bit-identical to the torch chain (IEEE reciprocal, subtraction, division). */
int effimvs_inv_init_f32(const float* cur_depth, const float* lo_disp, const float* hi_disp, int B, int HW, float* inv_out,
                         float* depth_out, void* stream);

/* DepthHead tail + BasicUpdateBlock step + disp_to_depth (models/update.py:27, 121-125;
 * models/Effi_MVS_plus.py:138-148).  pre (B,HW) = depth_head.conv2 output without bias (NULL: no step),
 * bias (1), inv (B,HW), lo_disp / hi_disp (B)  ->  inv_out = inv + tanh(pre + bias) (optional),
 * depth_out = 1 / clamp(lo + (hi - lo) * inv_out, 1e-4). */
int effimvs_gru_delta_f32(const float* pre, const float* bias, const float* inv, const float* lo_disp, const float* hi_disp,
                          int B, int HW, float* inv_out, float* depth_out, void* stream);

/* DepthHead.conv2 + the step above in one pass (models/update.py:19-27, 121-125; models/Effi_MVS_plus.py:138-148):
 * t (B,H,W,h) channels-last = relu(depth_head.conv1(net)), weight (1,h,3,3), bias (1), inv (B,H,W), lo_disp / hi_disp (B)
 *   -> inv_out = inv + tanh(conv3x3(t, weight; zero padding 1) + bias), depth_out = disp_to_depth(inv_out).
 * h in {16,32,48,64,96,128}. */
int effimvs_delta_head_f32(const float* t, const float* weight, const float* bias, const float* inv, const float* lo_disp,
                           const float* hi_disp, int B, int h, int H, int W, float* inv_out, float* depth_out, void* stream);

/* upsample_depth (models/Effi_MVS_plus.py:167-178) on mask = mask_scale * (mask_pre + mask_bias) (models/update.py:128),
 * mask_pre (B,H,W,9*ratio^2) channels-last conv output without bias, inv (B,H,W)
 *   -> up_out (B,ratio*H,ratio*W) (optional) and depth_out = disp_to_depth(up) (optional).  ratio = 2. */
int effimvs_convex_upsample_f32(const float* mask_pre, const float* mask_bias, float mask_scale, const float* inv,
                                const float* lo_disp, const float* hi_disp, int B, int H, int W, int ratio, float* up_out,
                                float* depth_out, void* stream);

/* The same with the mask head's last layer folded in (models/update.py:109-112, 128): t (B,H,W,K) channels-last =
 * relu(mask[0](net)), mask_w (9*ratio^2, K) = mask[2].weight (1x1), mask = mask_scale * (mask_w t + mask_bias) is formed per
 * pixel in the kernel and never stored.  K a multiple of 4 up to 256. */
int effimvs_convex_upsample_conv_f32(const float* t, int K, const float* mask_w, const float* mask_bias, float mask_scale,
                                     const float* inv, const float* lo_disp, const float* hi_disp, int B, int H, int W, int ratio,
                                     float* up_out, float* depth_out, void* stream);

/* ProjectionInput head (models/update.py:88-91): relu(convc1(cost)) (1x1) and relu(convd1(inv)) (7x7, pad 3).
 * cost (B,CD,H,W) planar (what effimvs_dynamic_cost_f32 writes), inv (B,1,H,W), wc1 (h,CD,1,1), wd1 (h,1,7,7)
 *   -> out (B,H,W,2h) channels-last = cat[relu(convc1), relu(convd1)]: the input of the second encoder layer. */
int effimvs_encoder_head_f32(const float* cost, const float* inv, const float* wc1, const float* bc1, const float* wd1,
                             const float* bd1, int B, int CD, int h, int H, int W, float* out, void* stream);

/* The same head with the weights passed as KERNEL PARAMETERS (constant bank operands of the FMAs: no per-block weight staging, no
 * shared-memory weight reads).  host_tables points to HOST memory holding h / 16 tables of 944 floats each, one per chunk of 16
 * output channels: [49][16] convd1 taps, [8][16] convc1 rows (rows >= CD zero), [16] convc1 bias, [16] convd1 bias.  They are
 * copied into the launch parameters during the call (the array may be reused afterwards; a CUDA graph keeps the values of the
 * capture).  h / 16 launches.  effimvs_encoder_head_pack_host builds the tables from HOST copies of upstream's weight tensors
 * (wc1 (h,CD,1,1), bc1 (h), wd1 (h,1,7,7), bd1 (h)); effimvs_encoder_head_table_floats(h) = (h / 16) * 944 is their size. */
int effimvs_encoder_head_hostw_f32(const float* cost, const float* inv, const float* host_tables, int B, int CD, int h, int H, int W,
                                   float* out, void* stream);
int effimvs_encoder_head_pack_host(const float* wc1, const float* bc1, const float* wd1, const float* bd1, int CD, int h,
                                   float* tables_out);
int effimvs_encoder_head_table_floats(int h);

/* ProjectionInput tail (models/update.py:93-95): x = relu(Wc[:, :hm] m + ctx_term), ctx_term (n_pix, h) = the context half of
 * convc plus both biases (constant over the GRU iterations), m (n_pix, hm) channels-last, w (h, hm) = convc.weight[:, :hm].
 * The result is written into the x half of hx (n_pix, 2h) = cat[h, x] in place. */
int effimvs_encoder_tail_f32(const float* m, const float* w, const float* ctx_term, long long n_pix, int hm, int h,
                             float* hx, void* stream);

/* The same tail with the context half formed in the kernel: x = relu(w_m m + w_ctx act(ctx) + bias), w_ctx (h, cx) =
 * convc.weight[:, hm:], bias (h) = convc.bias + convc.weight[:, :hm] convd.bias.  ctx points at the first context channel
 * of a channels-last map and is read at a pixel stride of ctx_stride floats (cx in {4,8,12}); ctx_relu != 0 applies the
 * relu of models/Effi_MVS_plus.py:466 on the fly. */
int effimvs_encoder_tail_ctx_f32(const float* m, const float* w_m, const float* ctx, int ctx_stride, int cx, int ctx_relu,
                                 const float* w_ctx, const float* bias, long long n_pix, int hm, int h, float* hx, void* stream);

/* GRU start state (models/Effi_MVS_plus.py:464-465): hx[:, :h] = tanh(ctx_map[:, :h]) for ctx_map (n_pix, h + cx) channels-last,
 * hx (n_pix, 2h) = cat[h, x]. */
int effimvs_gru_init_f32(const float* ctx_map, long long n_pix, int h, int cx, float* hx, void* stream);

/* The same start state together with the context half of ProjectionInput.convc (models/update.py:93-95 with the context of
 * models/Effi_MVS_plus.py:466), which does not change over the GRU iterations: ctx_term (n_pix, h) channels-last =
 * w_ctx relu(ctx_map[:, h:h+cx]) + bias, w_ctx (h, cx) = convc.weight[:, hm:], bias (h) = convc.bias + convc.weight[:, :hm] convd.bias
 * (fp32 products).  It is the aux map of effimvs_conv2d_tf32's ADD_RELU epilogue.  h <= 128, cx in 4..64, both multiples of 4. */
int effimvs_gru_init_ctx_f32(const float* ctx_map, long long n_pix, int h, int cx, const float* w_ctx, const float* bias,
                             float* hx, float* ctx_term, void* stream);

/* ---- SURVEY section 8(f) row 3, the convolutions: 3x3 / stride 1 / zero padding 1 convolutions of the update block on the
 * tensor cores (tcgen05 kind::tf32: operands rounded to TF32, fp32 accumulation -- the arithmetic class cuDNN uses for these
 * layers under PyTorch's default torch.backends.cudnn.allow_tf32 = True), with the gate arithmetic as epilogues.
 * Replaces ProjectionInput.convc2 / convd2 / convd (+ convc) (models/update.py:69-99), ConvGRU.convz / convr / convq and the
 * gate expressions (models/update.py:33-49), DepthHead.conv1 (models/update.py:10-27), mask[0] (models/update.py:106-110).
 * All maps are channels-last: a map is addressed as (pointer to channel 0 of pixel 0, pixel stride in floats), so channel
 * slices of wider maps are read and written in place.  Input maps: 32-byte aligned, pixel strides and channel segments
 * multiples of 8 floats; output / aux maps: 16-byte aligned, strides multiples of 4 floats. */
#define EFFIMVS_CONV2D_BIAS 0       /* out = acc + bias (bias may be NULL)                                                  */
#define EFFIMVS_CONV2D_BIAS_RELU 1  /* out = relu(acc + bias)                                                               */
#define EFFIMVS_CONV2D_ADD_RELU 2   /* out = relu(acc + aux0[pixel]), aux0 = addend map with cout channels (bias inside)    */
#define EFFIMVS_CONV2D_GRU_GATES 3  /* cout = 2h, weights [convz ; convr]: aux1 = z = sigmoid(acc[:h] + bias[:h]) (h channels),
                                       out = sigmoid(acc[h:] + bias[h:]) * aux0, aux0 = previous hidden state (h channels)  */
#define EFFIMVS_CONV2D_GRU_UPDATE 4 /* cout = h, weights convq: out = (1 - aux0) * out + aux0 * tanh(acc + bias), aux0 = z;
                                       out is the hidden state, updated in place                                            */

/* 1 if the (cin, cout) pair runs on the tensor-core kernel (cin a multiple of 16, cout a multiple of 4, the whole weight
 * tensor resident in shared memory: 36 * cin * roundup(cout, 16) bytes + the input-row ring <= 220 KiB), else 0. */
int effimvs_conv2d_tf32_supported(int cin, int cout);
size_t effimvs_conv2d_tf32_packed_bytes(int cin, int cout);
/* w (cout, cin, 3, 3) fp32 as nn.Conv2d holds it -> the kernel's shared-memory image (TF32-rounded); once per weight tensor. */
int effimvs_conv2d_tf32_pack(const float* w, int cin, int cout, void* packed, void* stream);
/* The input is the channel concatenation of up to two maps (c0 + c1 channels; in1 = NULL, c1 = 0 for one map) of B images
 * of H x W pixels; packed from effimvs_conv2d_tf32_pack for cin = c0 + c1; bias (cout) or NULL; mode and aux maps as above. */
int effimvs_conv2d_tf32(const float* in0, long long in0_pixstride, int c0, const float* in1, long long in1_pixstride, int c1,
                        const void* packed, const float* bias, int cout, int B, int H, int W, int mode,
                        float* out, long long out_pixstride, const float* aux0, long long aux0_pixstride,
                        float* aux1, long long aux1_pixstride, void* stream);

/* The same convolutions with fp32-grade arithmetic (bf16x3), the class of the 3-D nets' default mode: every operand, input
 * and weight, is carried as hi = bf16(x) and lo = bf16(x - hi) (together ~2^-16 relative), and each product is formed as
 * hi*hi + hi*lo + lo*hi with fp32 accumulation.  Range: fp32's -- nothing saturates.  The packed image is the hi weights
 * followed by the lo weights: 36 * cin * roundup(cout, 16) bytes.  Arguments, modes, layouts and error codes as the
 * _tf32 family above.  Both weight images and a two-copy input ring live in shared memory, so fewer shapes are supported:
 * up to 64 x 64 channels (the update block at hidden sizes 16 and 32), not 96 x 96. */
int effimvs_conv2d_bf16x3_supported(int cin, int cout);
size_t effimvs_conv2d_bf16x3_packed_bytes(int cin, int cout);
int effimvs_conv2d_bf16x3_pack(const float* w, int cin, int cout, void* packed, void* stream);
int effimvs_conv2d_bf16x3(const float* in0, long long in0_pixstride, int c0, const float* in1, long long in1_pixstride, int c1,
                          const void* packed, const float* bias, int cout, int B, int H, int W, int mode,
                          float* out, long long out_pixstride, const float* aux0, long long aux0_pixstride,
                          float* aux1, long long aux1_pixstride, void* stream);

/* ---- SURVEY section 8(f) row 2: the DTU pipeline's NumPy / cv2.remap geometric filter ------------------------
 * reproject_with_depth + check_geometric_consistency + the aggregation of filter_depth
 * (test_dtu_dypcd.py:164-233, 261-309, 320-337) for one reference view in one kernel.
 *   ref_depth (h,w), srcs_depth (v,h,w), conf (h,w) (already resized to the depth map, :258), fp32
 *   mats: device array of 34 + 50*v floats, the float32 matrices exactly as upstream forms them:
 *         [inv(K_ref) 3x3][K_ref 3x3][inv(E_ref) 4x4] then per source view
 *         [E_src @ inv(E_ref) 4x4][K_src 3x3][inv(K_src) 3x3][E_ref @ inv(E_src) 4x4]
 *   thr_dist_host / thr_diff_host: HOST arrays of n_rungs thresholds, i * dist_base (float64) and
 *         log10(max(i, 1.05)) * diff_base (float32), i = first_rung .. first_rung + n_rungs - 1 (:226-228)
 *   full_count: upstream's dy_range of :303 (a pixel also passes if that many views pass the last rung)
 *   conf_thres: args.conf (:261);  conf_keep: 0.75, above which the reference depth is kept (:300)
 *   -> final_mask (h,w) u8, geo_mask (h,w) u8 (optional), depth_avg (h,w), points (3,h,w) world coordinates,
 *      masks_out (v,n_rungs,h,w) u8 (optional), reproj_depth_out (v,h,w) zeroed outside the last rung (optional) */
int effimvs_dtu_filter_f32(const float* ref_depth, const float* srcs_depth, const float* conf, const float* mats,
                           const double* thr_dist_host, const float* thr_diff_host, int n_rungs, int first_rung,
                           int full_count, float conf_thres, float conf_keep, int v, int h, int w,
                           uint8_t* final_mask, uint8_t* geo_mask, float* depth_avg, float* points, uint8_t* masks_out,
                           float* reproj_depth_out, void* stream);

/* The same filter for n reference views of one scene in one launch, reading every depth map in place from one stack.
 *   depths (n_depths,h,w) fp32: the scene's depth maps (e.g. the all-gathered tensor of the scene runner)
 *   ref_idx (n) int32: row of view y's reference depth map in `depths`
 *   src_idx (n,vmax) int32: rows of view y's source depth maps, the first src_count[y] entries used
 *   src_count (n) int32: view y's source count, in [1, vmax]; vmax in [1,31] (the kernel's histogram limit)
 *   mats (n, 34 + 50*vmax) fp32: view y's camera pack in the layout of effimvs_dtu_filter_f32 for its src_count[y]
 *         sources, padded to vmax sources
 *   conf (n,h,w) fp32 at the depth maps' size
 *   thresholds, ladder and conf_thres / conf_keep as effimvs_dtu_filter_f32
 *   -> final_mask (n,h,w) u8, geo_mask (n,h,w) u8 (optional), depth_avg (n,h,w), points (n,3,h,w)
 * View y's results are bit-identical to effimvs_dtu_filter_f32 on that view alone with the same camera pack.
 * All index arrays are device arrays and are NOT validated on the device: every entry of ref_idx and of the used part of
 * src_idx must be in [0, n_depths) and every src_count in [1, vmax] (the caller checks its host lists before uploading).
 * There is no masks_out / reproj_depth_out here: the per-rung debugging outputs are single-view only. */
int effimvs_dtu_filter_views_f32(const float* depths, int n_depths, const int* ref_idx, const int* src_idx,
                                 const int* src_count, int vmax, const float* mats, const float* conf,
                                 const double* thr_dist_host, const float* thr_diff_host, int n_rungs, int first_rung,
                                 int full_count, float conf_thres, float conf_keep, int n, int h, int w,
                                 uint8_t* final_mask, uint8_t* geo_mask, float* depth_avg, float* points, void* stream);

/* ---- the scene's coloured point cloud (upstream's vertex / colour collection, test_tank.py:517-570,
 * test_dtu_dypcd.py:339-350): stream compaction of the filters' dense outputs for n reference views ----------------
 * Views come in the order given; within a view, points come in raster order (row-major over (h,w)).  Offsets come from a
 * scan, never from atomics: two runs give the same bits.  Points are copied, never computed.  Two calls, three launches:
 *
 * Bytes of the tile workspace both calls share (8 per 4096-pixel tile of every view); 0 for bad sizes. */
size_t effimvs_point_offsets_workspace_bytes(int n, int h, int w);

/*   final_mask (n,h,w) uint8: the filters' final masks (nonzero = kept), as effimvs_fusion_filter_views_f32 and
 *         effimvs_dtu_filter_views_f32 write them
 *   workspace: effimvs_point_offsets_workspace_bytes(n, h, w) bytes of device memory, 16-byte aligned; receives the
 *         offset of every tile's first point, which effimvs_gather_points_f32 reads
 *   -> view_offsets (n+1) int64 device array: view y's points are rows view_offsets[y] .. view_offsets[y+1] - 1 of the
 *         output, view_offsets[n] is the total.  Two launches (count, scan). */
int effimvs_point_offsets(const uint8_t* final_mask, int n, int h, int w, void* workspace, size_t workspace_bytes,
                          int64_t* view_offsets, void* stream);

/*   final_mask (n,h,w) uint8 and workspace as effimvs_point_offsets left them
 *   points (n,3,h,w) fp32: the filters' world points
 *   images (n_images,3,h,w) fp32 reference images, or NULL for points only (then image_rows and colors_out are ignored)
 *   image_rows (n) int32 device array: the row of `images` holding view y's image (e.g. its scene view number).  NOT
 *         validated on the device: every entry must be in [0, n_images) (the caller checks its host list before uploading)
 *   -> points_out (total,3) fp32, colors_out (total,3) uint8, both 16-byte aligned, total = view_offsets[n].
 *      Colour channel c is image channel c: trunc(clamp(image * 255, 0, 255)) with an IEEE fp32 multiply, NaN giving 0.
 *      On [0,1] that is NumPy's (image * 255).astype(np.uint8), and it returns the byte of every u8 / 255 image; outside
 *      [0,1] (where NumPy's cast is undefined) the clamp is this library's definition.  One launch. */
int effimvs_gather_points_f32(const uint8_t* final_mask, const float* points, const float* images, int n_images,
                              const int* image_rows, int n, int h, int w, const void* workspace, size_t workspace_bytes,
                              float* points_out, uint8_t* colors_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EFFIMVS_H */
