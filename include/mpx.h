/*
 * mpx.h -- C ABI of libmpx.so, the B200 (sm_100a) render-and-compare engine behind the MegaPose
 * inference API.  This is the drop-in boundary: plain pointers and sizes, no torch types.
 *
 * Conventions (all entry points):
 *   - return 0 on success, negative on error; the message is available from mpx_last_error()
 *     (thread-local, valid until the next failing call on the same thread);
 *   - pointers named d_* are DEVICE pointers (e.g. torch.Tensor.data_ptr()), h_* are HOST pointers;
 *   - the library never allocates or frees caller tensors; outputs are caller-allocated;
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *     no entry point synchronises the device;
 *   - poses are row-major 4x4 float32 (TCO: object -> camera, OpenCV camera axes), intrinsics are
 *     row-major 3x3 float32, boxes are (x1, y1, x2, y2) float32 pixels;
 *   - handles (mpx_meshdb, mpx_net) are opaque and owned by the library.
 *
 * Each group cites the reference interface (under /root/reference/src/megapose) that it replaces.
 */
#ifndef MPX_H_
#define MPX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPX_ABI_VERSION 4

/* ---- library ------------------------------------------------------------------------------ */
int mpx_abi_version(void);
/* 16-bit storage type of weights / activations / the network input tensor ("act16" below): 0 = IEEE fp16 (default: the
 * number format the reference's networks were trained under, training/train_megapose.py:299 torch.cuda.amp.autocast;
 * conversions saturate at +-65504), 1 = bf16 (library built with -DMPX_ACT_BF16).  Accumulation is fp32 in both. */
int mpx_act_dtype(void);
const char* mpx_last_error(void);
/* number of CUDA kernels this library has launched so far in this process (host-side counter) */
long long mpx_launch_count(void);
/* Persistent grids (convolutions, the tiled rasteriser) are sized for mpx_sm_count() SMs: the device's count, or the even
 * limit set here (0 = all).  A limit leaves SMs free for the latency-bound launches of another stream -- the refiner
 * iterations of one frame beside the coarse stage of the next (megapose6d_b200/frame_pipeline.py).  Process-wide; set it
 * before mesh databases are created and before CUDA graphs are captured (both record grid sizes). */
int mpx_set_sm_limit(int n_sms);
int mpx_sm_count(void);
/* measurement aid for bench.py: when enabled every convolution launch is bracketed by CUDA events on
 * its stream; mpx_profile_summary synchronises the device, returns the summed duration (ms), the
 * algorithmic FLOPs (2*M*N*K per launch) and the launch count since enabling, and resets. */
int mpx_profile_enable(int on);
int mpx_profile_summary(double* conv_ms, double* conv_flops, long long* conv_launches);

/* ---- mesh database ---------------------------------------------------------------------------
 * Replaces MeshDataBase / BatchedMeshes (lib3d/rigid_mesh_database.py:57-169) for the point sets
 * and the Panda3D/Assimp model loading (panda3d_renderer/panda3d_scene_renderer.py:195-208) for
 * the triangle meshes.  All meshes of an object dataset are uploaded once.
 *   h_verts   [sum_nv,3] float32, already scaled to metres (RigidObject.scale applied by caller)
 *   h_normals [sum_nv,3] float32 unit vertex normals (object frame)
 *   h_colors  [sum_nv,3] float32 albedo in [0,1]
 *   h_vert_offsets [n_meshes+1] int64 prefix offsets into the vertex arrays
 *   h_faces   [sum_nf,3] int32 vertex indices LOCAL to each mesh
 *   h_face_offsets [n_meshes+1] int64 prefix offsets into h_faces
 */
typedef struct mpx_meshdb mpx_meshdb;
int mpx_meshdb_create(int n_meshes, const float* h_verts, const float* h_normals,
                      const float* h_colors, const int64_t* h_vert_offsets, const int32_t* h_faces,
                      const int64_t* h_face_offsets, mpx_meshdb** out);
int mpx_meshdb_destroy(mpx_meshdb* db);

/* Optional diffuse textures (what Panda3D / Assimp load from the model's material,
 * panda3d_renderer/panda3d_scene_renderer.py:195-208).  Host arrays: h_uv [sum_nv,2] per-vertex texture coordinates
 * (v up), h_tex all RGB8 images back to back (row 0 = top), h_tex_offsets [n+1] byte offsets, h_tex_dims [n,2] =
 * (height, width), (0,0) for an untextured mesh, h_tex_modulate [n] (may be NULL): 1 = multiply the texture with the
 * interpolated vertex colours.  Sampling: repeat wrap, bilinear over texel centres, no mip-mapping.  Call once, after
 * mpx_meshdb_create. */
int mpx_meshdb_set_textures(mpx_meshdb* db, const float* h_uv, const uint8_t* h_tex, const int64_t* h_tex_offsets,
                            const int32_t* h_tex_dims, const int32_t* h_tex_modulate);

/* ---- rasteriser ------------------------------------------------------------------------------
 * Replaces Panda3dBatchRenderer.render (panda3d_renderer/panda3d_batch_renderer.py:217-282) and
 * everything under it (worker_loop :89-150, Panda3dSceneRenderer.render_scene
 * panda3d_scene_renderer.py:298-358, camera model panda3d_renderer/types.py:58-101, depth
 * linearisation and the eye-normal texture panda3d_renderer/utils.py:44-68).
 * One view per (d_label_idx[i], d_TCO[i], d_K[i]); near/far 0.1/10 m; two-sided; black background;
 * non-finite pose or intrinsics => all-zero view (panda3d_batch_renderer.py:109-135).
 */
#define MPX_RASTER_QUANTIZE8 1u      /* round colour/normal channels to k/255 (uint8 read-back)  */
#define MPX_RASTER_NORMALS_GL 2u     /* eye normals in GL Y-up axes instead of Panda Z-up axes  */
#define MPX_RASTER_POINT_LIGHTS 4u   /* rgb lit by make_scene_lights() (ambient 0.1 + six point lights of 0.4 on the object's
                                      * axes at 10 bounding radii, panda3d_scene_renderer.py:104-136) instead of ambient 1.0:
                                      * what models with render_normals=False are fed (models/pose_rigid.py:374-378) */
/* depth normalisation of the fused depth channels (PosePredictor.normalize_depth, models/pose_rigid.py:466-496), applied
 * with d_depth_norm_z[sample] = tCR_z; raster entry points carry it in flags bits 8-9, mpx_roi_align_fused as an argument.
 * NaN follows torch.clamp: a NaN depth / z or depth - z (0 / 0 on the background when z == 0, a NaN z) stays NaN through
 * the clamps, and the network input receives NaN. */
#define MPX_DEPTH_NORM_TCR_SCALE_CLAMP_CENTER 0  /* clamp(depth / z, 0, 2) - 1 (the released RGB-D refiner) */
#define MPX_DEPTH_NORM_TCR_SCALE 1               /* depth / z */
#define MPX_DEPTH_NORM_TCR_CENTER_CLAMP 2        /* clamp(depth - z, -2, 2) */
#define MPX_DEPTH_NORM_NONE 3
#define MPX_RASTER_DEPTH_NORM_SHIFT 8

size_t mpx_raster_workspace_bytes(int h, int w);

/* kernel selection, default 7: bit 0 = batches of at most SMs/8 views (refiner iterations, final scoring) spread
 * the triangles of each view over many CTAs (coverage kernel + resolve kernel) instead of one CTA per
 * (view, row strip); bit 1 = (untiled kernels) visibility through a fire-and-forget 64-bit min reduction instead of
 * read-then-atomic; bit 2 = larger batches use the tiled kernel (triangles binned into screen strips, z-test of a strip in
 * shared memory, candidate fragments dealt out evenly over the threads) instead of one CTA per view with a global
 * visibility buffer.  All combinations produce identical pixels. */
int mpx_raster_set_mode(int mode);

/* contract output: float32 NCHW planes; any of d_rgb [N,3,h,w], d_normals [N,3,h,w],
 * d_depth [N,1,h,w] may be NULL. */
int mpx_raster_render(const mpx_meshdb* db, const int32_t* d_label_idx, const float* d_TCO,
                      const float* d_K, int n_views, int h, int w, uint32_t flags, float* d_rgb,
                      float* d_normals, float* d_depth, void* d_workspace, size_t workspace_bytes,
                      void* stream);

/* fused output: writes act16 channels straight into the network input tensor (see mpx_net):
 * view i belongs to sample i / views_per_sample, view slot v = i % views_per_sample and its
 * channels land at ch_offset + v * ch_per_view: ch_per_view = 3 (rgb), 4 (rgb, depth), 6 (rgb, normals) or
 * 7 (rgb, normals, depth), i.e. what render_normals / render_depth select (models/pose_rigid.py:394-404).
 * d_depth_norm_z [n_samples] (may be NULL = none) applies the depth normalisation selected by flags bits 8-9
 * to the depth channel. */
int mpx_raster_render_fused(const mpx_meshdb* db, const int32_t* d_label_idx, const float* d_TCO,
                            const float* d_K, int n_views, int views_per_sample, int h, int w,
                            uint32_t flags, void* d_x, int c_pad, int ch_offset, int ch_per_view,
                            const float* d_depth_norm_z, void* d_workspace, size_t workspace_bytes,
                            void* stream);

/* single-view samples (coarse / scoring model, models/pose_rigid.py:634-708): crop + render in one pass.
 * Sample i renders (d_label_idx[i], d_TCO[i], d_K[i] = its crop intrinsics) and crops the observation
 * d_img_nhwc4[d_im_idx[i]] with d_boxes_crop[i] (roi_align as in mpx_roi_align); each pixel's complete channel
 * vector [crop rgb(d) | render rgb, normals(, depth) | zero pad] is stored once.  c_in = 3|4, ch_per_view = 6|7. */
int mpx_render_crop_fused(const mpx_meshdb* db, const int32_t* d_label_idx, const float* d_TCO,
                          const float* d_K, int n, int h, int w, uint32_t flags, const float* d_img_nhwc4,
                          int b, int im_h, int im_w, const int32_t* d_im_idx, const float* d_boxes_crop,
                          int c_in, void* d_x, int c_pad, int ch_per_view, const float* d_depth_norm_z,
                          void* d_workspace, size_t workspace_bytes, void* stream);

/* ---- hypothesis geometry -----------------------------------------------------------------------
 * mpx_pose_init_autodepth: TCO_init_from_boxes_autodepth_with_R (lib3d/cosypose_ops.py:169-218).
 *   d_points [n_labels, n_pts, 3]; d_label_idx, d_bboxes [n,4], d_K [n,9], d_R [n,9] -> d_TCO [n,16]
 */
int mpx_pose_init_autodepth(const float* d_points, int n_pts, const int32_t* d_label_idx,
                            const float* d_bboxes, const float* d_K, const float* d_R, int n,
                            float* d_TCO, void* stream);

/* mpx_normalize_T: normalize_T (lib3d/transform_ops.py:106-119), in-place allowed. */
int mpx_normalize_T(const float* d_T_in, int n, float* d_T_out, void* stream);

/* mpx_crop_geometry: the box/intrinsics part of PosePredictor.crop_inputs and
 * compute_crops_multiview (models/pose_rigid.py:180-303): project_points_robust +
 * boxes_from_uv (lib3d/camera_geometry.py:40-64), deepim_boxes via deepim_crops_robust
 * (lib3d/cropping.py:30-110), get_K_crop_resize (lib3d/camera_geometry.py:67-115).
 *   d_points [n_labels, n_pts, 3] (the deterministic 2000- or 200-point subsets)
 *   d_tCR [n,3]; outputs d_boxes_rend [n,4], d_boxes_crop [n,4], d_K_crop [n,9] */
int mpx_crop_geometry(const float* d_points, int n_pts, const int32_t* d_label_idx,
                      const float* d_TCO, const float* d_K, const float* d_tCR, int n, float lamb,
                      int im_h, int im_w, int out_h, int out_w, float* d_boxes_rend,
                      float* d_boxes_crop, float* d_K_crop, void* stream);

/* mpx_multiview_cameras: make_TCO_multiview (lib3d/multiview.py:165-246), closed form of the
 * Panda3D scene-graph look-at (multiview.py:31-92); float64 internally.
 *   h_offsets [n_extra,3] camera positions wrt camera 0 in units of |tCR|
 *   d_TCV_O [n, 1 + n_extra, 16]: view 0 is TCO itself */
int mpx_multiview_cameras(const float* d_TCO, const float* d_tCR, int n, const float* h_offsets,
                          int n_extra, float* d_TCV_O, void* stream);

/* mpx_pose_update: PosePredictor.update_pose (models/pose_rigid.py:305-312) =
 * compute_rotation_matrix_from_ortho6d (lib3d/rotations.py:25-40) +
 * pose_update_with_reference_point (lib3d/cosypose_ops.py:33-58). */
int mpx_pose_update(const float* d_TCO, const float* d_K_crop, const float* d_pose9,
                    const float* d_tCR, int n, float* d_TCO_out, void* stream);

/* mpx_topk_per_group: top-K by logit per detection, the device-side equivalent of
 * PoseEstimator.filter_pose_estimates (inference/pose_estimator.py:643-667) for the coarse
 * stage.  d_logits [n_groups, m]; d_idx [n_groups, k] int32 indices into m, descending logit,
 * ties broken by lower index. */
int mpx_topk_per_group(const float* d_logits, int n_groups, int m, int k, int32_t* d_idx,
                       void* stream);

/* ---- crop ---------------------------------------------------------------------------------------
 * torchvision.ops.roi_align as called by crop_images (lib3d/cropping.py:113-144): sampling_ratio
 * 4, aligned=False, spatial_scale 1, plus the depth validity masking of the RGB-D branch.
 * mpx_image_to_nhwc4 packs an observation [B,C,H,W] float32 (C = 3|4) to [B,H,W,4] float32 once
 * per frame (channel 3 = depth or 0). */
int mpx_image_to_nhwc4(const float* d_images_nchw, int b, int c, int h, int w, float* d_out_nhwc4,
                       void* stream);
/* contract output: d_out [n, c, out_h, out_w] float32 */
int mpx_roi_align(const float* d_img_nhwc4, int b, int h, int w, const int32_t* d_im_idx,
                  const float* d_boxes, int n, int c, int out_h, int out_w, float* d_out,
                  void* stream);
/* fused output: act16 channels 0..c-1 of the network input tensor; for c == 4 the depth channel is
 * normalised with d_depth_norm_z as in mpx_raster_render_fused. */
int mpx_roi_align_fused(const float* d_img_nhwc4, int b, int h, int w, const int32_t* d_im_idx,
                        const float* d_boxes, int n, int c, int out_h, int out_w, void* d_x,
                        int c_pad, const float* d_depth_norm_z, int depth_norm_kind, void* stream);

/* ---- network -------------------------------------------------------------------------------------
 * ResNet-34 + fc + head of PosePredictor.net_forward (models/pose_rigid.py:314-334) with the
 * backbone of models/torchvision_resnet.py:181-316.  Weights are passed already BN-folded and
 * repacked (see megapose6d_b200/backbone.py): per conv an act16 [C_out, R*S*C_in] matrix and an
 * fp32 bias.
 *
 * Network input tensor ("x"): act16, space-to-depth NHWC [n, H/2, W/2, 4*c_pad] with channel
 * index (dy*2+dx)*c_pad + c, c_pad = the channel count rounded up to a multiple of 16: 16 (coarse, 9 real channels) or
 * 32 (refiner, 27|32) for the released models, up to 256 for configurations with more rendered views.
 */
size_t mpx_net_input_bytes(int n, int h, int w, int c_pad);

/* single convolution (also the unit the parity tests exercise):
 *   d_x [n,H,W,C_in] act16, d_w [C_out, R*S*C_in] act16, d_bias [C_out] fp32,
 *   d_residual / d_out [n,P,Q,C_out] act16 (residual may be NULL)
 *   relu: bit 0 = ReLU; bit 1 = the weights are the space-to-depth form of the 7x7 stem (4x4 taps over C_in = 64: the 15 of
 *   64 (tap, 16-channel) slices that are zero by construction are not multiplied, megapose6d_b200/backbone.py: _stem_s2d);
 *   bit 2 = fused 3x3/s2/p1 max-pool (models/torchvision_resnet.py:197 `self.maxpool` right after the stem's ReLU): d_out is
 *   then the ZEROED [n, (P-1)/2+1, (Q-1)/2+1, C_out] tensor and is max-reduced into; needs bit 0, no residual, and returns
 *   MPX_ERR_UNSUPPORTED (nothing launched, no error text) for shapes the pair window kernel does not serve
 *   block_n: 0 = auto, else 64|128|256; max_ctas: 0 = one per SM */
int mpx_conv2d(const void* d_x, int n, int h, int w, int c_in, const void* d_w,
                    const float* d_bias, int c_out, int r, int s, int stride, int pad_lo_h,
                    int pad_lo_w, int pad_hi_h, int pad_hi_w, int relu, const void* d_residual,
                    void* d_out, int block_n, int max_ctas, void* stream);

/* the same convolution with its K loop split over the `splits` (0 = heuristic, 1, 2, 4, 8) CTAs of a thread-block
 * cluster per output tile -- the form the network uses for small batches (refiner iterations: a handful of output
 * tiles, up to 72 serial k-blocks).  The partial tiles are reduced through distributed shared memory in rank order
 * (deterministic).  block_n must be explicit. */
int mpx_conv2d_splitk(const void* d_x, int n, int h, int w, int c_in, const void* d_w,
                           const float* d_bias, int c_out, int r, int s, int stride, int pad_lo_h,
                           int pad_lo_w, int pad_hi_h, int pad_hi_w, int relu, const void* d_residual,
                           void* d_out, int block_n, int splits, void* stream);

/* kernel selection bits for block_n == 0 (auto), default 60866571 = 1 + 2 + 8 + 16384 + 32768 + 2097152 + 8388608 + 16777216 + 33554432:
 *   1   window kernels: 64->64 stride-1 convolutions (stem, layer1) and 128->128 3x3 (layer2) load their activations
 *       once per tile as a contiguous window and address the filter taps as row-shifted operand descriptors
 *   2   the CTA-pair (cta_group::2) kernel serves 256-wide tiles;  4  and 128-wide tiles
 *   8   mpx_net_forward splits the K loop of layers 2-4 over a thread-block cluster for batches <= 64
 *   16  a single epilogue warp set in the 64->64 window kernel (default two)
 *   32  a single MMA-issuing thread in the 64->64 window kernel (default two);  64  three
 *   128 three epilogue warp sets
 *   256 disable the single-CTA layer2 window kernel (TMA-im2col kernel instead)
 *   512 launch without programmatic dependent launch;  1024 older row-group choice of the window kernel (diagnostic)
 *   16384 the layer2 window kernel on CTA pairs (cta_group::2, two MMA issuers in the leader): layer2 0.167 -> 0.153 ms
 *   32768 the 64 -> 64 window kernel (stem, layer1) on CTA pairs: layer1 0.255 -> 0.227 ms per convolution at batch 576
 *   131072 do not skip the structurally zero K slices of the space-to-depth stem weights (diagnostic)
 *   262144 / 524288 cap the automatic small-batch K split (bit 8) at 2 / 1 CTAs per tile: less SM time per layer at a higher
 *       latency (set before graphs are captured; the trade for two frames in flight, frame_pipeline.py)
 *   1048576 row-per-thread epilogue in the 64 -> 64 pair window kernel (round-1 form; default: staged, coalesced)
 *   2097152 mpx_net_forward lets the stem's pair window kernel max-pool in its epilogue (mpx_conv2d relu bit 2): the
 *       full-resolution stem output is never stored; network forward at batch 576: 6.51 -> 6.14 ms
 *   8388608 the 64 -> 64 pair window kernel slides its activation window: every CTA owns a contiguous run of 128-row blocks,
 *       the activations live in a ring of 16 KB chunks (one new chunk per block instead of a whole window: L2 -> SM reads 4x
 *       lower on the stem) and the residual rows arrive by TMA in the layout of the staging tiles: layer1 conv2 + residual
 *       0.246 -> 0.195 ms, bit-identical outputs; runs shorter than 8 blocks per CTA keep the reloading kernel (bit 15)
 *   16777216 the layer2 pair window kernel stages its epilogue through shared memory: residual rows by TMA into 128B-swizzled
 *       tiles, overwritten in place, stored as whole 128-byte lines (the weight ring gives up 3 of 12 stages for the 64 KB):
 *       layer2 conv2 + residual 0.190 -> 0.163 ms, bit-identical outputs
 *   33554432 the same for the 256-wide CTA-pair im2col kernel (layers 3-4), one 128-channel half of the tile at a time through a
 *       32 KB staging tile, bias read from global memory; only for K >= 768 (the 1x1 downsamples keep the row form):
 *       layer3 conv2 + residual 0.151 -> 0.147 ms, bit-identical outputs
 * (r02 A/B, profiles/r02_layer_table_mode_bits.json; the other round-1 candidates -- pair-window kernels for layer3/4 and
 * 128-wide layer2 tiles, residual preload -- measured no gain and were removed.)
 * 0 = single-CTA TMA-im2col kernel only */
int mpx_conv_set_mode(int mode);

/* bring-up probe (tools/gpu_probe_rowshift.py): D[128,64] = A[r0:r0+128, :64] * B[64,64]^T with the UMMA
 * A descriptor started r0 rows into a TMA-written 128B-swizzled tile; d_a [144,64] act16, d_b [64,64] act16 */
int mpx_debug_umma_rowshift(const void* d_a, const void* d_b, int r0, int base_offset, float* d_out,
                            void* stream);

/* measurement probe (tools/gpu_mma_probe.py): mean cycles per tcgen05.mma of shape (128 * cta_group) x n x 16, operands in
 * shared memory, with `chains` (1|2|4) independent accumulators interleaved by each of `issuers` (1..4) issuing threads (one
 * per warp); *h_cycles_per_mma = SM time per MMA, *h_issue_cycles_per_mma (may be NULL) = one thread's time per instruction
 * issued, before the commit; synchronous */
int mpx_debug_mma_probe(int cta_group, int n, int chains, int issuers, int n_mma, double* h_cycles_per_mma,
                        double* h_issue_cycles_per_mma);

/* 3x3/s2/p1 max pool, act16 NHWC (torchvision_resnet.py:302) */
int mpx_maxpool3x3s2(const void* d_x, int n, int h, int w, int c, void* d_out, void* stream);

/* global average pool + folded (fc o head) linear: d_x [n, hw, c] act16, d_w [out_dim, c] fp32,
 * d_b [out_dim] fp32 -> d_out [n, out_dim] fp32 */
int mpx_avgpool_linear(const void* d_x, int n, int hw, int c, const float* d_w, const float* d_b,
                       int out_dim, float* d_out, void* stream);

typedef struct mpx_net mpx_net;
/* h_conv_w / h_conv_b: arrays of 36 DEVICE pointers in execution order (stem, then per BasicBlock
 * conv1, conv2, [downsample]); c_pad as above; d_head_w [out_dim,512] fp32, d_head_b [out_dim]. */
int mpx_net_create(int c_pad, int out_dim, const void* const* h_conv_w, const float* const* h_conv_b,
                   int n_convs, const float* d_head_w, const float* d_head_b, mpx_net** out);
/* Pre-activation backbones (WideResNet34 / WideResNet18 of models/wide_resnet.py:29-126, backbone_str "resnet34" /
 * "resnet18", width 1): h_layer_blocks [4] blocks per layer; h_conv_w / h_conv_b: 1 + 2 * blocks + 3 DEVICE pointers in
 * execution order (stem = the 5x5/s2 convolution as 3x3 over the space-to-depth input, bn1 folded; per block conv1 with
 * bn2 folded, conv2 with a zero bias, [bare 1x1 downsample with a zero bias]); h_block_affine: per block a DEVICE pointer
 * to [2, C_in] fp32 (scale, shift of the block's bn1, applied with ReLU to the block input); d_head_w [out_dim, 512] is
 * the head itself (there is no fc). */
int mpx_net_create_preact(int c_pad, int out_dim, const int32_t* h_layer_blocks, const void* const* h_conv_w,
                          const float* const* h_conv_b, int n_convs, const float* const* h_block_affine, int n_blocks,
                          const float* d_head_w, const float* d_head_b, mpx_net** out);
int mpx_net_destroy(mpx_net* net);
/* mpx_net_forward replays a cached CUDA graph per (buffers, shape) after the first call; 0 disables that
 * (every launch is then issued eagerly on the caller's stream). Default: enabled. */
int mpx_net_set_graphs(int on);
size_t mpx_net_workspace_bytes(const mpx_net* net, int n, int h, int w);
/* d_x: network input tensor (see above) for n samples of size h x w; d_out [n, out_dim] fp32 */
int mpx_net_forward(const mpx_net* net, const void* d_x, int n, int h, int w, float* d_out,
                    void* d_workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPX_H_ */
