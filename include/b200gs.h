/* b200gs — C ABI of the B200-native 4D Gaussian-splatting hot path.
 *
 * This is the drop-in boundary: every entry point replaces one pybind11 / torch::Tensor
 * entry point (or one PyTorch-operator chain) of cvsp-lab/ICLR2025_3D-MOM and is what the
 * reference-side Python binding (ctypes, see INTEGRATION.md) loads from libb200gs.so.
 *
 * Conventions
 *  - Plain C: raw DEVICE pointers (unless a parameter says "host"), explicit sizes, and the
 *    CUDA stream to launch on (pass PyTorch's current stream). No torch types.
 *  - Every function returns 0 on success and non-zero on error; b200gs_last_error() returns
 *    the message of the last error raised on the calling thread.
 *  - Ownership: the caller owns every buffer, scratch included. The library never allocates
 *    or frees device memory and keeps no global state besides the per-thread error string and the
 *    process-wide settings of b200gs_set_option / b200gs_profile_enable.
 *  - No implicit device synchronisation except where stated (b200gs_rast_forward_stage1).
 *  - "null" for an optional tensor has the meaning of the reference's empty tensor.
 *  Citations: RAST = submodules/depth-diff-gaussian-rasterization, KNN = submodules/simple-knn.
 */
#ifndef B200GS_H_INCLUDED
#define B200GS_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200gs_stream_t; /* cudaStream_t */

const char* b200gs_last_error(void);
int b200gs_version(void);
/* Process-wide launch settings (the library reads no environment variables):
 *   "mlp_fwd_sms" / "mlp_bwd_sms" (default 0 = all 148): CTAs of the persistent deformation-MLP kernels (mlp_bwd_sms caps the
 *                    feature-dim-64 backward only: the feature-dim-128 backward always launches one CTA per SM).  The view-pipelining trainer
 *                    sets 120 around a step so that the other stream's sorts / emission / preprocess find free SMs next to them
 *                    (377 -> 383 view-iterations/s; 96: slower again); same results up to the order of the weight-gradient flushes
 * set: 0 on success, non-zero for an unknown name; get: the value, or -1 for an unknown name. */
int b200gs_set_option(const char* name, int value);
int b200gs_get_option(const char* name);

/* Opt-in phase timing for the multi-kernel rasterizer entry points (what bench.py's per-kernel roofline rows are measured with):
 * while enabled, every call records CUDA events on the launching stream around each phase -- "preprocess_fwd", "depth_sort",
 * "emit_instances", "tile_sort", "tile_ranges", "composite_fwd", "composite_bwd", "preprocess_bwd".  enable(1) / enable(0) both
 * clear the record; read() synchronises on the recorded events and returns how many calls were recorded and their summed
 * duration in milliseconds.  Process-wide, not thread-safe, off by default (no events are created or recorded then). */
int b200gs_profile_enable(int enable);
int b200gs_profile_read(const char* phase, int* calls, float* total_ms);

/* ---------------------------------------------------------------------------------------
 * Rasterizer — replaces _C.rasterize_gaussians / rasterize_gaussians_backward / mark_visible
 * (RAST/ext.cpp:15-19; RAST/rasterize_points.cu:35-117, :119-202, :204-223) and underneath
 * them CudaRasterizer::Rasterizer::{forward,backward,markVisible}
 * (RAST/cuda_rasterizer/rasterizer.h:24-87).
 * ------------------------------------------------------------------------------------- */

/* Sizes in bytes of the geometry / binning / image scratch buffers for P Gaussians, R
 * (tile, Gaussian) instances and a W x H image. Replaces required<GeometryState>() etc.
 * (RAST/cuda_rasterizer/rasterizer_impl.h:65-72). */
int b200gs_rast_buffer_sizes(int P, long long R, int W, int H, size_t out_bytes[3]);

/* Stage 1 of the forward pass: per-Gaussian projection, covariance, SH colour, tile
 * rectangle (RAST/cuda_rasterizer/forward.cu:155-256). Writes radii[P] (int32) and fills
 * geom_buf. host_counters (HOST memory, 2 x uint64) receives {num_rendered, num_visible};
 * this is the forward pass's single device->host read and synchronises `stream`, like the
 * reference's cudaMemcpy at rasterizer_impl.cu:282. The caller then sizes the binning
 * buffer with b200gs_rast_buffer_sizes(P, num_rendered, ...). */
int b200gs_rast_forward_stage1(int P, int D, int M, int W, int H,
                               const float* means3D, const float* shs, const float* colors_precomp,
                               const float* opacities, const float* scales, float scale_modifier,
                               const float* rotations, const float* cov3D_precomp,
                               const float* viewmatrix, const float* projmatrix, const float* campos,
                               float tan_fovx, float tan_fovy, int prefiltered,
                               int* radii, void* geom_buf, size_t geom_bytes,
                               unsigned long long* host_counters, b200gs_stream_t stream);

/* Stage 2: depth sort, instance emission, tile sort, tile ranges, compositing
 * (rasterizer_impl.cu:284-336; forward.cu:261-379). Writes out_color[3,H,W] and
 * out_depth[1,H,W]; keeps final transmittance / contributor counts in img_buf. */
int b200gs_rast_forward_stage2(int P, long long num_rendered, long long num_visible, int W, int H,
                               const float* background, void* geom_buf, void* bin_buf, size_t bin_bytes,
                               void* img_buf, size_t img_bytes, float* out_color, float* out_depth,
                               b200gs_stream_t stream);

/* Backward pass (rasterizer_impl.cu:343-444; backward.cu). grad_arena is scratch of
 * 12*P floats. All eight outputs are fully written (zeros for culled Gaussians), so they
 * may be uninitialised on entry: dL_dmean2D[P,3], dL_dcolor[P,3], dL_dopacity[P],
 * dL_dmean3D[P,3], dL_dcov3D[P,6], dL_dsh[P,M,3] (may be null), dL_dscale[P,3], dL_drot[P,4]. */
int b200gs_rast_backward(int P, int D, int M, long long num_rendered, int W, int H,
                         const float* background, const float* means3D, const float* shs,
                         const float* colors_precomp, const float* scales, float scale_modifier,
                         const float* rotations, const float* cov3D_precomp,
                         const float* viewmatrix, const float* projmatrix, const float* campos,
                         float tan_fovx, float tan_fovy, const int* radii,
                         void* geom_buf, void* bin_buf, void* img_buf,
                         const float* dL_dpix, const float* dL_dpix_depth, float* grad_arena,
                         float* dL_dmean2D, float* dL_dcolor, float* dL_dopacity, float* dL_dmean3D,
                         float* dL_dcov3D, float* dL_dsh, float* dL_dscale, float* dL_drot,
                         b200gs_stream_t stream);

/* Same, but the SH gradient is ADDED to dL_dsh_accum[P,M,3] instead of written (rows of invisible Gaussians are left
 * untouched): a trainer that renders several views per optimiser step keeps ONE gradient buffer for the step's shared SH
 * tensor and saves the per-view [P,16,3] allocation plus a full accumulation pass over it. */
int b200gs_rast_backward_accumulate_sh(int P, int D, int M, long long num_rendered, int W, int H,
                                       const float* background, const float* means3D, const float* shs,
                                       const float* colors_precomp, const float* scales, float scale_modifier,
                                       const float* rotations, const float* cov3D_precomp,
                                       const float* viewmatrix, const float* projmatrix, const float* campos,
                                       float tan_fovx, float tan_fovy, const int* radii,
                                       void* geom_buf, void* bin_buf, void* img_buf,
                                       const float* dL_dpix, const float* dL_dpix_depth, float* grad_arena,
                                       float* dL_dmean2D, float* dL_dcolor, float* dL_dopacity, float* dL_dmean3D,
                                       float* dL_dcov3D, float* dL_dsh_accum, float* dL_dscale, float* dL_drot,
                                       b200gs_stream_t stream);

/* present[P] (uint8/bool) = view-space z > 0.2 (rasterizer_impl.cu:54-66, :141-153). */
int b200gs_mark_visible(int P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                        unsigned char* present, b200gs_stream_t stream);

/* Parity/debug: re-expresses one field of the internal state of the last forward call in the
 * REFERENCE's layout (rasterizer_impl.h:21-73) into a device buffer `dst` of dst_bytes.
 * Fields: "depths" f32[P], "means2D" f32[P,2], "conic_opacity" f32[P,4], "rgb" f32[P,3],
 * "clamped" u8[P,3], "cov3D" f32[P,6], "tiles_touched" u32[P], "point_list" u32[R],
 * "keys" u64[R] (tile<<32 | depth bits, sorted), "ranges" u32[tiles,2], "n_contrib" u32[H*W],
 * "accum_alpha" f32[H*W]. Returns the number of bytes written, or -1. */
long long b200gs_rast_export(const char* field, int P, long long num_rendered, int W, int H,
                             void* geom_buf, void* bin_buf, void* img_buf, void* dst, long long dst_bytes,
                             b200gs_stream_t stream);

/* Stand-alone stable radix sort of (u32 key, u32 value) pairs on key bits [begin_bit, end_bit);
 * replaces cub::DeviceRadixSort::SortPairs (rasterizer_impl.cu:304-309; KNN/simple_knn.cu:208-213).
 * keys_a/vals_a hold the input, *_b are ping-pong buffers; returns 0 or 1 = which side holds the
 * result, or -1. temp_bytes from b200gs_sort_temp_bytes. */
size_t b200gs_sort_temp_bytes(size_t n, int begin_bit, int end_bit);
int b200gs_sort_pairs_u32(uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b,
                          size_t n, int begin_bit, int end_bit, void* temp, size_t temp_bytes,
                          b200gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * simple-knn — replaces simple_knn._C.distCUDA2 (KNN/spatial.cu:15-26, KNN/ext.cpp) and
 * SimpleKNN::knn (KNN/simple_knn.cu:185-220): mean_dists[i] = mean of the three smallest
 * squared distances from point i to the other points. points[P,3] float32.
 * ------------------------------------------------------------------------------------- */
size_t b200gs_dist2_scratch_bytes(size_t P);
int b200gs_dist2(int P, const float* points, float* mean_dists, void* scratch, size_t scratch_bytes,
                 b200gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Optimiser — replaces the ~8 foreach launches of torch.optim.Adam.step() that the reference
 * runs every iteration (scene/gaussian_model.py:197-209; train_4DGS.py:295-297) with one
 * launch over all parameter tensors. Arithmetic = torch/optim/adam.py::_multi_tensor_adam
 * (no weight decay, no amsgrad, not capturable): the caller computes, per tensor and in
 * double precision like torch does, neg_step_size = -(lr / (1 - beta1^step)) and
 * bias_correction2_sqrt = sqrt(1 - beta2^step) after incrementing that tensor's step.
 * The table is HOST memory (copied into kernel arguments). Tensors whose grad is None are
 * simply not listed, which is how torch skips them.
 * ------------------------------------------------------------------------------------- */
#define B200GS_ADAM_MAX_TENSORS 56
typedef struct {
    float* param; const float* grad; float* exp_avg; float* exp_avg_sq;
    long long numel;
    float neg_step_size;
    float bias_correction2_sqrt;
} b200gs_adam_tensor;
int b200gs_adam_multi(int n_tensors, const b200gs_adam_tensor* tensors /* host */, double beta1, double beta2,
                      double eps, b200gs_stream_t stream);

/* The same step for the two SH tensors of scene/gaussian_model.py:136-140 (_features_dc [P,1,3], _features_rest [P,M-1,3]) with
 * their gradient read from ONE [P,M,3] buffer -- the layout the rasterizer backward writes (RAST/cuda_rasterizer/backward.cu:20-139)
 * -- so the per-step split of that gradient into two tensors never happens.  `grad` of the two descriptors is ignored. */
int b200gs_adam_sh(long long P, int M, const b200gs_adam_tensor* dc, const b200gs_adam_tensor* rest, const float* grad_pm3,
                   double beta1, double beta2, double eps, b200gs_stream_t stream);

/* Densify / prune bookkeeping — replaces the per-tensor boolean-mask indexing and torch.cat
 * chains of scene/gaussian_model.py:424-482 (_prune_optimizer, cat_tensors_to_optimizer):
 * for every listed tensor, dst[i, :] = src[index[i], :], i < n_out, rows of row_floats floats.
 * index = int64 row ids on the device (null = identity, i.e. a plain multi-tensor copy). */
#define B200GS_GATHER_MAX_TENSORS 64
typedef struct { const float* src; float* dst; int row_floats; int zero_tail_rows; /* the last zero_tail_rows of the n_out rows are set to 0
                 instead of gathered: the fresh rows of exp_avg / exp_avg_sq (gaussian_model.py:470-471) */ } b200gs_gather_tensor;
int b200gs_gather_rows_multi(int n_tensors, const b200gs_gather_tensor* tensors /* host */,
                             const long long* index, long long n_out, b200gs_stream_t stream);

/* The DECISIONS of a densification / pruning event, one pass over the Gaussians each (the moves are b200gs_gather_rows_multi):
 *   densify_select  GaussianModel.densify -> densify_and_clone / densify_and_split (scene/gaussian_model.py:693-698, :541-565, :511-523):
 *                   g = grad_accum / denom (NaN -> 0); clone_flag = |g| >= thr and max(exp(scaling)) <= dense_extent;
 *                   split_flag = g >= thr and max(exp(scaling)) > dense_extent   (dense_extent = percent_dense * scene_extent)
 *   prune_select    GaussianModel.prune (:681-690): sigmoid(opacity) < min_opacity, or -- when max_screen_size > 0 -- max_radii2D >
 *                   max_screen_size or max(exp(scaling)) > max_world_extent (= 0.1 * extent)
 *   densification_stats  add_densification_stats (:713-715): for update_filter[i] != 0: grad_accum[i] += |viewspace_grad[i, :2]|, denom[i] += 1
 *   reset_opacity   (:362-365): out = inverse_sigmoid(min(sigmoid(opacity), 0.01))
 * flags are bytes (0 / 1; a torch.bool tensor's storage).  Same float operations as the torch expressions they replace. */
int b200gs_densify_select(long long N, const float* grad_accum, const float* denom, const float* scaling_raw, float grad_threshold,
                          float dense_extent, unsigned char* clone_flag, unsigned char* split_flag, b200gs_stream_t stream);
int b200gs_prune_select(long long N, const float* opacity_raw, const float* scaling_raw, const float* max_radii2D, float min_opacity,
                        float max_screen_size, float max_world_extent, unsigned char* prune_flag, b200gs_stream_t stream);
int b200gs_densification_stats(long long N, const float* viewspace_grad /* [N,3] */, const unsigned char* update_filter, float* grad_accum,
                               float* denom, b200gs_stream_t stream);
int b200gs_reset_opacity(long long N, const float* opacity_raw, float* out, b200gs_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Deformation field — replaces the PyTorch operator chains behind
 * scene/hexplane.py::HexPlaneField.forward (:177, interpolate_ms_features :73-106: 6*levels
 * F.grid_sample + products + cat) and scene/deformation.py::Deformation.forward_dynamic
 * (:97-153: feature_out Linear + three ReLU-Linear-ReLU-Linear heads on cuBLAS), forward and
 * backward. Planes are CHANNELS-LAST: plane[l][k] points at [res_b][res_a][32] floats for the
 * coordinate pair k = (a,b) in (0,1)(0,2)(0,3)(1,2)(1,3)(2,3); res[l] = resolution of x,y,z,t.
 * ------------------------------------------------------------------------------------- */
#define B200GS_HEXPLANE_MAX_LEVELS 4
typedef struct {
    int levels;
    int channels;                                   /* 32 */
    int res[B200GS_HEXPLANE_MAX_LEVELS][4];
    const float* plane[B200GS_HEXPLANE_MAX_LEVELS][6];
    float* grad_plane[B200GS_HEXPLANE_MAX_LEVELS][6]; /* backward: accumulated into (caller zero-fills); null = skip */
    const float* aabb;                              /* device, 6 floats: max xyz, then min xyz (hexplane.py:116-120) */
} b200gs_hexplane_desc;

/* Optional visiting order: order[P] = permutation of the points sorted by the cell they fall in, so
 * neighbouring warps touch the same texels (L1 hits instead of L2 gathers). Purely a performance hint:
 * results do not depend on it; pass null to visit points in index order. */
size_t b200gs_hexplane_order_scratch_bytes(long long P);
int b200gs_hexplane_order(long long P, const float* pts, const float* aabb, unsigned int* order, void* scratch,
                          size_t scratch_bytes, b200gs_stream_t stream);
/* features[P, 32*levels] = HexPlaneField(pts[P,3], t). times[P] may be null -> time_scalar for all. */
int b200gs_hexplane_forward(const b200gs_hexplane_desc* desc /* host */, long long P, const float* pts,
                            const unsigned int* order, const float* times, float time_scalar, float* features,
                            b200gs_stream_t stream);
/* plane gradients are ACCUMULATED into desc->grad_plane; d_pts[P,3] (may be null) is written. */
int b200gs_hexplane_backward(const b200gs_hexplane_desc* desc /* host */, long long P, const float* pts,
                             const unsigned int* order, const float* times, float time_scalar,
                             const float* d_features, float* d_pts, b200gs_stream_t stream);

typedef struct {
    int feat_dim;                 /* 32 * levels (64 or 128) */
    int width;                    /* net_width, 64 */
    const float* w1; const float* b1;           /* feature_out.0  [64, feat_dim], [64] */
    const float* w2[3]; const float* b2[3];     /* {pos,scales,rotations}_deform.1  [64,64],[64]; null = head off (no_dx/no_ds/no_dr) */
    const float* w3[3]; const float* b3[3];     /* {pos,scales,rotations}_deform.3  [k,64],[k], k = 3,3,4 */
    int feat_tiled;               /* 0: features / d_features are row-major [P, feat_dim]; 1 (feat_dim 64 only): both use the
                                     4-point-group tile layout of the activation stash ([tile of 128][32 groups][16 chunks][4 points][4]),
                                     which is what b200gs_hexplane_time_forward / _backward produce / consume with tiled = 1 */
} b200gs_mlp_weights;
/* gradients of b200gs_mlp_weights' arrays.  With feat_dim 64, w1 and the w2[h] of every enabled head must be 16-byte aligned
 * (they are accumulated with 128-bit vector reductions); b200gs_deform_mlp_backward refuses other pointers. */
typedef struct { float* w1; float* b1; float* w2[3]; float* b2[3]; float* w3[3]; float* b3[3]; } b200gs_mlp_grads;

/* floats of the buffer the forward leaves for the backward (opaque to the caller, who only allocates it and hands the same
 * pointer to both calls of one view): four planes of ReLU'd activations in 4-point-group tiles, followed by the transposed
 * TF32 hi / lo weight images the tcgen05 backward streams into shared memory */
size_t b200gs_deform_mlp_saved_floats(long long P);
/* pts_out = xyz + pos_head + delta_scale*(frame_num*scene_flow); scales_out = scales + scale_head;
 * rot_out = rot + rot_head (deformation.py:113-135). frame_num_dev (device float, may be null)
 * overrides frame_num: the reference hands frame_num over as a 0-d CUDA tensor (scene/dataset.py:39)
 * and reading it on the host would cost a device sync per view.
 * saved: the activation stash the backward reads (b200gs_deform_mlp_saved_floats(P) floats), or NULL for INFERENCE
 * (render_4DGS.py, torch.no_grad()): nothing is stashed, 1 KB per point less HBM traffic (needs all three heads enabled). */
int b200gs_deform_mlp_forward(const b200gs_mlp_weights* w /* host */, long long P, const float* features,
                              const float* xyz, const float* scales, const float* rot, const float* scene_flow,
                              float frame_num, const float* frame_num_dev, float delta_scale, float* pts_out, float* scales_out, float* rot_out,
                              float* saved, b200gs_stream_t stream);
/* weight gradients are ACCUMULATED into gw (caller zero-fills); d_features[P, feat_dim] is written.
 * d_pts / d_scales / d_rot: upstream gradients of the three outputs (null = zero). `w` and `saved` must be the ones the
 * matching b200gs_deform_mlp_forward call was given. */
int b200gs_deform_mlp_backward(const b200gs_mlp_weights* w /* host */, const b200gs_mlp_grads* gw /* host */,
                               long long P, const float* features, const float* saved, const float* d_pts,
                               const float* d_scales, const float* d_rot, float* d_features, b200gs_stream_t stream);

/* Opacity and SH deformation heads (no_do = False / no_dshs = False; deformation.py:97-153 with mask = ones):
 *     opacity_out[P,1] = opacity * 1 + opacity_deform(hidden)      opacity_deform: ReLU, Linear(64,64), ReLU, Linear(64,1)
 *     shs_out[P,16,3]  = shs * 1 + shs_deform(hidden)              shs_deform:     ReLU, Linear(64,64), ReLU, Linear(64,48)
 * They run beside the three geometry heads and read relu(hidden) from the stash b200gs_deform_mlp_forward left (which must
 * therefore have been given one).  w2[0] / w2[1] null = that head off; at least one must be on. */
typedef struct {
    int feat_dim;                 /* 64 or 128, as in b200gs_mlp_weights */
    int width;                    /* net_width, 64 */
    const float* w1;              /* feature_out.0 [64, feat_dim] (backward only: d_features += d_h W1) */
    const float* w2[2]; const float* b2[2];     /* {opacity,shs}_deform.1  [64,64], [64] */
    const float* w3[2]; const float* b3[2];     /* {opacity,shs}_deform.3  [k,64], [k], k = 1, 48 */
    int feat_tiled;               /* layout of features / d_features, as in b200gs_mlp_weights */
} b200gs_heads_weights;
/* gradients of b200gs_heads_weights' arrays (w1 / b1: feature_out.0).  w1, the w2[h] of every enabled head and the SH head's
 * w3 must be 16-byte aligned (128-bit vector reductions). */
typedef struct { float* w1; float* b1; float* w2[2]; float* b2[2]; float* w3[2]; float* b3[2]; } b200gs_heads_grads;
/* floats of the heads' own activation stash: relu(z_opacity), relu(z_sh) in the layout of the three-head stash */
size_t b200gs_deform_heads_saved_floats(long long P);
/* mlp_saved: the stash of the matching b200gs_deform_mlp_forward call.  opacity [P,1], shs [P,sh_coeffs,3] (sh_coeffs must
 * be 16 when the SH head is on).  heads_saved: b200gs_deform_heads_saved_floats(P) floats for the backward, or NULL. */
int b200gs_deform_heads_forward(const b200gs_heads_weights* w /* host */, long long P, int sh_coeffs, const float* mlp_saved,
                                const float* opacity, const float* shs, float* opacity_out, float* shs_out, float* heads_saved,
                                b200gs_stream_t stream);
/* Run AFTER b200gs_deform_mlp_backward of the same view: ADDS the heads' share into d_features (same layout), gw->w1 and
 * gw->b1, and accumulates the heads' own weight gradients.  d_opacity [P,1] / d_shs [P,16,3]: upstream gradients of the
 * outputs (null = zero).  sh_grad (may be null): a [P,16,3] buffer that receives d_shs as well (the gradient of the `shs`
 * input: an identity path), written instead of added to when sh_grad_overwrite != 0. */
int b200gs_deform_heads_backward(const b200gs_heads_weights* w /* host */, const b200gs_heads_grads* gw /* host */, long long P,
                                 int sh_coeffs, const float* features, const float* mlp_saved, const float* heads_saved,
                                 const float* d_opacity, const float* d_shs, float* d_features, float* sh_grad,
                                 int sh_grad_overwrite, b200gs_stream_t stream);

/* Plane-subset variants: features = factor * prod_{k in plane_mask} plane_k (bit k of plane_mask = plane k; factor may be
 * null = 1).  With the spatial planes (0,1,3: mask 0x0B) evaluated once per optimiser step and handed back as `factor`,
 * each view of a multi-view batch only samples the time planes (2,4,5: mask 0x34): the Gaussians' xyz do not change
 * within a step, so the spatial product is shared by all its views.  The backward additionally ACCUMULATES
 * d_factor_accum[P,F] += d_features * prod_{k in plane_mask} plane_k (null = skip), which is the upstream gradient of the
 * deferred spatial pass.  mask 0x3F with null factor is exactly b200gs_hexplane_forward / _backward. */
int b200gs_hexplane_forward_masked(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                   const float* times, float time_scalar, int plane_mask, const float* factor, float* features,
                                   b200gs_stream_t stream);
int b200gs_hexplane_backward_masked(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                    const float* times, float time_scalar, int plane_mask, const float* factor, float* d_factor_accum,
                                    const float* d_features, float* d_pts, void* time_row_scratch, size_t time_row_scratch_bytes,
                                    b200gs_stream_t stream);
/* Optional scratch for the backward above when the whole launch shares ONE timestamp (times == null): the time planes'
 * gradient is then reduced along x into up to 64 replicas of a 1-D row per plane (so the few hundred hot 128-byte lines of
 * the two touched time rows do not serialise in L2) and added to the planes by a small follow-up kernel. null = classic path. */
size_t b200gs_hexplane_time_row_scratch_bytes(const b200gs_hexplane_desc* desc, int replicas);

/* Time planes only (mask 0x34), ONE timestamp for the whole launch, served from shared memory: every CTA pre-blends the two
 * touched time rows of each (x,t) / (y,t) / (z,t) plane into a 1-D row, samples become 1-D lerps without global texel traffic,
 * and the backward reduces the row gradients into replicated 1-D rows (time_row_scratch, as for the _masked variant; required). Same contract as the
 * _masked variants with plane_mask = 0x34 and times = null (results differ from them by FP32 re-association only).
 * b200gs_hexplane_time_supported: 1 when the rows of this descriptor fit one CTA's shared memory (2 levels at 64 / 128).
 * d_features_tiled of the backward is a flag word: bit 0 = d_features in the MLP kernels' tiled layout, bit 1 = d_factor_accum is
 * WRITTEN instead of accumulated (a fresh per-view buffer under autograd: saves its zero fill and the read). */
int b200gs_hexplane_time_supported(const b200gs_hexplane_desc* desc);
int b200gs_hexplane_time_forward(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                 float time_scalar, const float* factor, float* features, int features_tiled, b200gs_stream_t stream);
int b200gs_hexplane_time_backward(const b200gs_hexplane_desc* desc, long long P, const float* pts, const unsigned int* order,
                                  float time_scalar, const float* factor, float* d_factor_accum, const float* d_features,
                                  float* d_pts, void* time_row_scratch, size_t time_row_scratch_bytes, int d_features_tiled,
                                  b200gs_stream_t stream);

/* HexPlane regulariser, value and gradient in one pass (scene/gaussian_model.py:730-769 compute_regulation;
 * scene/regulation.py:22-28 compute_plane_smoothness): per level
 *   plane_tv_weight * sum_{k in 0,1,3} S(G_k) + time_smoothness_weight * sum_{k in 2,4,5} S(G_k)
 *   + l1_time_planes_weight * sum_{k in 2,4,5} mean |1 - G_k|,   S = mean squared second difference along a plane's height.
 * The value is ADDED to loss_accum[0] (device float, may be null); the gradient is ADDED into desc->grad_plane
 * (entries may be null). desc->aabb is not used. */
int b200gs_hexplane_regulation(const b200gs_hexplane_desc* desc, float plane_tv_weight, float time_smoothness_weight,
                               float l1_time_planes_weight, float* loss_accum, b200gs_stream_t stream);

/* ---- fused elementwise pieces of the training loop ------------------------------------------------
 * activations: scales = exp(s), rotations = F.normalize(r) (x / max(||x||, 1e-12)), opacity = sigmoid(o)
 * (gaussian_renderer/__init__.py:130-132; scene/gaussian_model.py:37-47). [P,3] / [P,4] / [P,1] FP32.
 * The backward takes the forward's OUTPUTS for exp / sigmoid and the raw quaternion; null upstream gradients
 * count as zero, null outputs are skipped. */
int b200gs_activations_forward(long long P, const float* scales_raw, const float* rot_raw, const float* opacity_raw,
                               float* scales_out, float* rot_out, float* opacity_out, b200gs_stream_t stream);
int b200gs_activations_backward(long long P, const float* scales_out, const float* rot_raw, const float* opacity_out,
                                const float* d_scales_out, const float* d_rot_out, const float* d_opacity_out,
                                float* d_scales_raw, float* d_rot_raw, float* d_opacity_raw, b200gs_stream_t stream);
/* L1 loss of utils/loss_utils.py:23-24 with its gradient in one pass: loss_accum[0] += scale * sum |render - target|,
 * d_render[i] = scale * sign(render[i] - target[i]) (d_render may be null). scale = 1 / (n * batch) gives the
 * per-view share of train_4DGS.py:205-210's batch-mean L1. loss_accum is a device float the caller zeroes.
 * sse_accum (may be null): sse_accum[0] += sum (render - target)^2, the numerator of utils/image_utils.py:17-38 `psnr`, which
 * train_4DGS.py:212 evaluates on the same two images every iteration: psnr = 20 log10(1 / sqrt(sse / n)). */
int b200gs_l1_loss_fwd_bwd(long long n, const float* render, const float* target, float scale, float* loss_accum, float* sse_accum,
                           float* d_render, b200gs_stream_t stream);
/* The same against the ground truth as the dataset holds it -- uint8 [H,W,3] (scene/dataset_readers.py:1041), converted on the
 * device the way utils/general_utils.py:PILtoTorch does on the host (float(u8) / 255.0f): 3 B/pixel cross PCIe instead of 12.
 * render / d_render are [3,H,W]. */
int b200gs_l1_loss_fwd_bwd_u8(int H, int W, const float* render_chw, const unsigned char* target_hwc, float scale, float* loss_accum,
                              float* sse_accum, float* d_render_chw, b200gs_stream_t stream);

/* SSIM of utils/loss_utils.py:ssim (the 3DGS formulation: 11x11 Gaussian window, sigma 1.5, zero padding, C1 = 0.01^2,
 * C2 = 0.03^2) with its gradient, for the D-SSIM term lambda_dssim * (1 - ssim) of train_4DGS.py.  x, y are [N,C,H,W] FP32
 * (any N, C, H, W >= 1, N * C <= 65535); map(n,c,p) is the SSIM map of that pixel.
 *   ssim_sum (may be null): ssim_sum[n] += value_offset + value_scale * sum_{c,p} map(n,c,p) for every image n, one FP32 add
 *     of a value formed in FP64 (the map sums are accumulated in FP64 in the scratch).  value_offset 0, value_scale
 *     1 / (C*H*W) on a zeroed ssim_sum gives each image's SSIM; offset w, scale -w / (C*H*W) adds w * (1 - SSIM) to a loss.
 *   d_x (may be null = value only): d_x += weight * d(sum_{n,c,p} map)/dx, ADDED to what the buffer holds (so it can share
 *     the buffer the L1 kernel wrote).  Forward, then backward launch; the map's partial derivatives pass between them
 *     through the scratch.
 *   scratch: b200gs_ssim_scratch_bytes(N, C, H, W, with_grad = d_x != null) bytes of device memory, no initial contents
 *     (8 bytes per image, plus 12 bytes per element with the gradient).
 * Returns 0 without launching when both ssim_sum and d_x are null. */
size_t b200gs_ssim_scratch_bytes(int N, int C, int H, int W, int with_grad);
int b200gs_ssim_fwd_bwd(int N, int C, int H, int W, const float* x, const float* y, float value_offset, float value_scale,
                        float* ssim_sum, float weight, float* d_x, void* scratch, size_t scratch_bytes, b200gs_stream_t stream);
/* The same for one [3,H,W] image against the uint8 [H,W,3] ground truth (N = 1, C = 3), converted on the device as
 * float(u8) / 255.0f like b200gs_l1_loss_fwd_bwd_u8: identical results to the FP32 entry on the converted target. */
int b200gs_ssim_fwd_bwd_u8(int H, int W, const float* x_chw, const unsigned char* y_hwc, float value_offset, float value_scale,
                           float* ssim_sum, float weight, float* d_x_chw, void* scratch, size_t scratch_bytes, b200gs_stream_t stream);

/* Is the [n] float tensor x one value repeated?  gaussian_renderer/__init__.py:56 hands the field the camera's single timestamp as
 * a materialised [P,1] tensor; when it is uniform the field takes its one-timestamp fast path (time planes from shared memory).
 * scratch_dev2: 8 bytes of device memory; host_pinned2: 8 bytes of PINNED host memory, on return [0] = 1 if uniform else 0,
 * [1] = the bits of x[0].  HOST SYNC: waits for the stream (the second documented one next to b200gs_rast_forward_stage1). */
int b200gs_uniform_value(long long n, const float* x, unsigned int* scratch_dev2, unsigned int* host_pinned2, b200gs_stream_t stream);

/* to8b of render_4DGS.py:49 / train_4DGS.py:335 on the device: out_hwc[y][x][c] = (uint8)(255 * clip(image_chw[c][y][x], 0, 1)),
 * truncating like numpy's astype; [3,H,W] FP32 -> [H,W,3] bytes (SURVEY.md 8f rank 3: the frame leaves the GPU as 3 B/pixel). */
int b200gs_to8b_hwc(int H, int W, const float* image_chw, unsigned char* out_hwc, b200gs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200GS_H_INCLUDED */
