// Shared device/host helpers for the mpx kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

namespace mpx {

// ---------------------------------------------------------------------------------------------
// error plumbing (thread-local message, negative return codes; see include/mpx.h)
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define MPX_OK 0
#define MPX_ERR_INVALID -1
#define MPX_ERR_CUDA -2
#define MPX_ERR_UNSUPPORTED -3

#define MPX_CHECK_CUDA(expr)                                                          \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      mpx::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,            \
                     cudaGetErrorString(_e));                                         \
      return MPX_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)

#define MPX_REQUIRE(cond, ...)                                                        \
  do {                                                                                \
    if (!(cond)) {                                                                    \
      mpx::set_error(__VA_ARGS__);                                                    \
      return MPX_ERR_INVALID;                                                         \
    }                                                                                 \
  } while (0)

// Number of SMs the throughput kernels size their persistent grids for: the device's SM count, or the (even) limit set with
// mpx_set_sm_limit -- the SMs left over stay free for latency-bound launches of another stream (two frames in flight:
// the refiner iterations of one frame run beside the coarse stage of the next, see megapose6d_b200/frame_pipeline.py).
extern int g_sm_limit;
inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return (g_sm_limit > 0 && g_sm_limit < n) ? g_sm_limit : n;
}

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------
// 16-bit storage type of weights and activations ("act").  fp16 by default: the tensor core runs fp16 and bf16 operands
// at the same rate (tcgen05 kind::f16, fp32 accumulation either way), fp16 carries three more mantissa bits, and fp16 is
// what the reference's networks were trained under (torch.cuda.amp.autocast, training/train_megapose.py:299).  The
// narrower range is handled by a saturating conversion (values beyond +-65504 clamp instead of becoming inf).
// -DMPX_ACT_BF16 selects bf16 (same kernels; diagnostic A/B of the two number formats).
// ---------------------------------------------------------------------------------------------
#ifdef MPX_ACT_BF16
typedef __nv_bfloat16 act_t;
typedef __nv_bfloat162 act_t2;
constexpr int kActIsFp16 = 0;
constexpr uint32_t kIdescAB = (1u << 7) | (1u << 10);  // InstrDescriptor a_format / b_format = BF16
__device__ __forceinline__ uint32_t pack_act2(float lo, float hi) {
  act_t2 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_act2(uint32_t u) {
  act_t2 v = *reinterpret_cast<act_t2*>(&u);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ act_t to_act(float v) { return __float2bfloat16_rn(v); }
#else
typedef __half act_t;
typedef __half2 act_t2;
constexpr int kActIsFp16 = 1;
constexpr uint32_t kIdescAB = 0u;                      // InstrDescriptor a_format / b_format = F16
__device__ __forceinline__ uint32_t pack_act2(float lo, float hi) {
  uint32_t r;  // cvt packs its first source into the upper half
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float2 unpack_act2(uint32_t u) {
  act_t2 v = *reinterpret_cast<act_t2*>(&u);
  return __half22float2(v);
}
__device__ __forceinline__ act_t to_act(float v) {
  unsigned short r;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(v));
  return __ushort_as_half(r);
}
#endif

// depth normalisation of PosePredictor.normalize_depth (models/pose_rigid.py:466-496); kind as in include/mpx.h
// (MPX_DEPTH_NORM_*): 0 tCR_scale_clamp_center, 1 tCR_scale, 2 tCR_center_clamp, 3 none.  A NaN quotient / difference
// (0 / 0 on the background when z == 0, or a NaN z) passes through as torch.clamp lets it; fminf / fmaxf alone would
// return the bound instead.
__device__ __forceinline__ float depth_norm(float d, float z, int kind) {
  if (kind == 0) {
    const float q = __fdiv_rn(d, z);
    return q != q ? q : fminf(fmaxf(q, 0.f), 2.f) - 1.f;
  }
  if (kind == 1) return __fdiv_rn(d, z);
  if (kind == 2) {
    const float q = d - z;
    return q != q ? q : fminf(fmaxf(q, -2.f), 2.f);
  }
  return d;
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL): a kernel launched through launch_pdl may start while its stream predecessor is
// still running, as soon as every CTA of the predecessor has executed pdl_trigger() (or exited).  It must call pdl_wait()
// before it touches memory the predecessor writes (or writes memory the predecessor reads); everything before that --
// barrier / TMEM set-up, descriptor prefetch, constant loads -- overlaps with the predecessor's tail.  The chains of
// small-batch kernels (36 convolutions of ~6-10 us each per network forward) are bound by exactly that fixed cost.
// Without a PDL-aware predecessor both calls are no-ops.  mpx_conv_set_mode bit 9 (512) launches without the attribute.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
int conv_get_mode();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if ((conv_get_mode() & 512) == 0) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------------------------
// cross-file declarations (conv_tc.cu, net.cu)
// ---------------------------------------------------------------------------------------------
extern long long g_launches;  // kernels launched by this library (host-side counter)
void conv_profile_enable(int on);
bool conv_profile_enabled();
void net_set_graphs(int on);
void conv_set_mode(int mode);
int conv_get_mode();
int conv_profile_summary(double* total_ms, double* total_flops, long long* launches);

struct ConvDesc {
  int n_img, H, W, C_in;  // input NHWC
  int C_out, R, S, stride;
  int pad_lo_h, pad_lo_w, pad_hi_h, pad_hi_w;
  int relu;
  int s2d_stem;  // 1: the weights are the space-to-depth form of the 7x7 stem (zero slices are skipped), see conv_tc.cu
  int pool;      // 1: `out` is the ZERO-INITIALISED [n, (H-1)/2+1, (W-1)/2+1, C_out] tensor and receives the 3x3/s2/p1 max-pool of
                 //    the (ReLU'd) result through vector max-reductions; conv_forward returns MPX_ERR_UNSUPPORTED (no error set)
                 //    when no kernel with that epilogue serves the shape
};
// splitk: 0 = never, -1 = heuristic (few output tiles, long K loop), 1|2|4|8 = that many k-splits (cluster size)
int conv_forward(const ConvDesc& d, const void* x, const void* w, const float* bias,
                 const void* residual, void* out, int block_n_override, int max_ctas,
                 cudaStream_t stream, int splitk = 0);
int conv_out_dim(int in, int pad_lo, int pad_hi, int k, int stride);
int mma_probe(int cta_group, int n, int chains, int issuers, int n_mma, double* cycles_per_mma, double* issue_cycles_per_mma);
int umma_rowshift_probe(const void* a, const void* b, int r0, int base_off, float* out, cudaStream_t stream);
int maxpool3x3s2(const void* x, int n, int h, int w, int c, void* out, cudaStream_t stream);
int avgpool_linear(const void* x, int n, int hw, int c, const float* w, const float* b, int out_dim,
                   float* out, cudaStream_t stream);
struct Net;
int net_create(int c_pad, int out_dim, const void* const* conv_w, const float* const* conv_b,
               int n_convs, const float* head_w, const float* head_b, Net** out);
int net_create_preact(int c_pad, int out_dim, const int* layer_blocks, const void* const* conv_w, const float* const* conv_b,
                      int n_convs, const float* const* block_affine, int n_blocks, const float* head_w, const float* head_b,
                      Net** out);
size_t net_workspace_bytes(const Net* net, int n, int h, int w);
int net_forward(const Net* net, const void* x, int n, int h, int w, float* out, void* workspace,
                size_t workspace_bytes, cudaStream_t stream);
void net_destroy(Net* net);

// raster.cu
struct MeshDb {
  int n_meshes;
  int nv_max;
  float* verts;             // [sum_nv,3]
  float* normals;           // [sum_nv,3]
  float* colors;            // [sum_nv,3]
  int* faces;               // [sum_nf,3] local indices
  long long* vert_offsets;  // [n+1]
  long long* face_offsets;  // [n+1]
  int4* vtx_cache;          // [slots, nv_max] {X, Y, 1/z bits, behind}
  int slots;
  int nf_max;
  // packed copies for the kernels (same values as the arrays above): faces padded to 16 B, and two float4 per vertex
  // {r, g, b, nx}, {ny, nz, u, v} so that a resolved pixel gathers its triangle with 1 + 6 16-byte loads
  int4* faces4;             // [sum_nf] {ia, ib, ic, 0}
  float4* vattr;            // [sum_nv, 2]
  float* radius;            // [n_meshes] max |vertex| (point lights sit at 10 radii, panda3d_scene_renderer.py:104-136)
  // per-CTA scratch of the tiled kernel: row-range word per triangle, per-strip triangle lists, large-triangle list
  unsigned* tile_scratch;   // [slots, tile_words]
  long long tile_words;
  // optional textures (meshdb_set_textures): per-vertex uv, RGB8 images back to back, per mesh {byte offset, th, tw,
  // modulate-with-vertex-colours}; tex_info == nullptr: no mesh is textured
  float* uv;                // [sum_nv,2]
  unsigned char* tex;
  long long* tex_offsets;   // [n]
  int4* tex_info;           // [n] {th, tw, modulate, 0}; th == 0: untextured
};
struct RasterOut {
  float* rgb;      // contract planes (fp32 NCHW), any may be null
  float* normals;
  float* depth;
  act_t* x;  // fused network input (16-bit s2d NHWC), may be null
  int c_pad, ch_offset, ch_per_view, views_per_sample;  // ch_per_view: 3 rgb | 4 rgb+depth | 6 rgb+normals | 7 all
  const float* depth_norm_z;
  int depth_norm_kind;  // MPX_DEPTH_NORM_*
  // optional: observation crop computed in the resolve pass (views_per_sample == 1), so that each
  // pixel's whole channel vector (crop | render | zero pad) is written with 16-byte stores
  const float4* crop_images;  // [crop_b, crop_h, crop_w] NHWC4, nullptr = no fused crop
  int crop_b, crop_h, crop_w, crop_c;
  const int* crop_im_idx;     // [n_samples] or nullptr
  const float* crop_boxes;    // [n_samples, 4]
};
int meshdb_create(int n_meshes, const float* verts, const float* normals, const float* colors,
                  const int64_t* vert_offsets, const int32_t* faces, const int64_t* face_offsets,
                  MeshDb** out);
void meshdb_destroy(MeshDb* db);
int meshdb_set_textures(MeshDb* db, const float* uv, const unsigned char* tex, const int64_t* tex_offsets,
                        const int32_t* tex_dims, const int32_t* tex_modulate);
size_t raster_workspace_bytes(int h, int w);
void raster_set_scatter(int on);
void raster_set_tiled(int on);
int raster_set_red_only(int on);
int raster_launch(const MeshDb* db, const int32_t* label_idx, const float* TCO, const float* K, int n_views,
                  int h, int w, unsigned flags, const RasterOut& out, void* workspace, size_t workspace_bytes,
                  cudaStream_t stream);

// geom.cu
int pose_init_autodepth(const float* points, int n_pts, const int* label_idx, const float* bboxes,
                        const float* K, const float* R, int n, float* TCO, cudaStream_t stream);
int normalize_T(const float* Tin, int n, float* Tout, cudaStream_t stream);
int crop_geometry(const float* points, int n_pts, const int* label_idx, const float* TCO, const float* K,
                  const float* tCR, int n, float lamb, int im_h, int im_w, int out_h, int out_w,
                  float* boxes_rend, float* boxes_crop, float* K_crop, cudaStream_t stream);
int multiview_cameras(const float* TCO, const float* tCR, int n, const float* h_offsets, int n_extra,
                      float* TCV_O, cudaStream_t stream);
int pose_update(const float* TCO, const float* K_crop, const float* pose9, const float* tCR, int n,
                float* TCO_out, cudaStream_t stream);
int topk_per_group(const float* logits, int n_groups, int m, int k, int* idx, cudaStream_t stream);

// crop.cu
struct CropOut {
  float* nchw;       // [n, c, oh, ow] or null
  act_t* x;  // fused network input or null
  int c_pad;
  const float* depth_norm_z;
  int depth_norm_kind;
};
int image_to_nhwc4(const float* in, int b, int c, int h, int w, float* out, cudaStream_t stream);
int roi_align_launch(const float* images, int b, int h, int w, const int* im_idx, const float* boxes, int n,
                     int c, int oh, int ow, const CropOut& out, cudaStream_t stream);

}  // namespace mpx
