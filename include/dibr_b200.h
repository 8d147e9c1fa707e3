/*
 * dibr_b200.h — C ABI of libdibr_b200.so: B200 (sm_100a) kernels for Kaolin's
 * DIB-R hot path (rasterize + dibr_soft_mask, forward and backward).
 *
 * Plain pointers and sizes only; no torch / ATen types.  All pointers are DEVICE
 * pointers on the current CUDA device unless stated otherwise; all tensors are
 * dense row-major ("contiguous") fp32 / int64 / uint8 exactly as the reference
 * operators take them.  Nothing is allocated by the library: the caller passes
 * the outputs and a scratch `workspace` of at least dibr_b200_workspace_bytes().
 * Every output is fully written (no pre-zeroing needed).  Calls are asynchronous
 * on `stream` and never synchronise; they are re-entrant (no global state).
 *
 * Alignment: every device tensor pointer (inputs and outputs) must be a multiple of
 * DIBR_B200_ALIGNMENT (16) bytes; NULL is allowed where documented.  The kernels access caller
 * tensors with 16-byte vector loads / stores and 16- or 8-byte cp.async copies, so a tensor
 * view at a storage offset (e.g. buf[1:] of a float buffer, 4 bytes in) is rejected with
 * DIBR_B200_EINVAL before anything is launched; copy it first.  The workspace is exempt (it
 * is aligned internally) and so are host pointers (camera_proj_host, peer-push arrays).
 *
 * Return value: 0 on success; DIBR_B200_E* (<0) for argument errors detected on
 * the host; a positive cudaError_t if a launch failed (cudaGetLastError()).
 *
 * The four "operator" entry points replace, one for one, the functions the
 * reference registers in kaolin/csrc/bindings.cpp:111-115; the two "fused"
 * entry points implement the same mathematics directly on the public-API
 * tensors (kaolin/render/mesh/dibr.py:119-209) without the packed temporaries.
 */
#ifndef DIBR_B200_H_
#define DIBR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIBR_B200_OK 0
#define DIBR_B200_EINVAL (-1)      /* null or misaligned pointer / non-positive size / bad flag */
#define DIBR_B200_EWORKSPACE (-3)  /* workspace_bytes too small */
#define DIBR_B200_ESIZE (-4)       /* image larger than 16384 px or index overflow */

#define DIBR_B200_MAX_IMAGE_DIM 16384
#define DIBR_B200_ALIGNMENT 16     /* bytes, every device tensor pointer (see above) */

/* forward `mode` bits */
#define DIBR_B200_RASTER 1     /* compute face_idx / weights / features */
#define DIBR_B200_SOFT_MASK 2  /* compute soft_mask */

/* backward `flags` bits */
#define DIBR_B200_BINS_VALID 1  /* workspace still holds forward's bins / hit cache for the same inputs */
#define DIBR_B200_ACCUMULATE 2  /* add into grad_face_vertices_image instead of overwriting it */

typedef struct CUstream_st* dibr_b200_stream_t; /* == cudaStream_t */

int dibr_b200_version(void);

/* Diagnostics: per-kernel device time of every launch made by the CALLING THREAD between
 * _begin and _end (thread-local: concurrent callers do not interact; no global state).
 * _end synchronises the recorded events, writes up to `capacity` durations (ms, launch
 * order) and the '\n'-separated kernel names, and returns the number of launches. */
int dibr_b200_trace_begin(void);
int dibr_b200_trace_end(char* names, size_t names_bytes, float* ms, int capacity);

/* Scratch needed by any entry point for `batch` views with `total_faces` faces
 * in all views together on a height x width image. */
size_t dibr_b200_workspace_bytes(int batch, int64_t total_faces, int height, int width);

/* Minimum scratch + a soft-mask hit cache for `cache_tiles` 16x16 screen tiles
 * (3072*knum + 16 bytes each, + 17 412 bytes when knum <= 32).  Any workspace larger than the minimum is used by
 * dibr_b200_forward (mode & SOFT_MASK) to record, per tile that has any, the
 * (pixel, face, probability, distance type) hits — what the reference stores as
 * 13*knum bytes for EVERY pixel (dibr.py:49-54) — so that dibr_b200_backward with
 * bins_valid = 1 streams over them instead of recomputing the neighbour walk.
 * Tiles that do not fit are recomputed in backward; results are identical. */
size_t dibr_b200_workspace_bytes_cached(int batch, int64_t total_faces, int height, int width,
                                        int knum, int64_t cache_tiles);

/*
 * Fused forward on the public-API tensors.
 * Replaces: kaolin/render/mesh/rasterization.py:273-352 (RasterizeCuda.forward:
 * valid-face packing, x multiplier, bboxes, op call, index remap) and
 * kaolin/render/mesh/dibr.py:29-55 (DibrSoftMaskCuda.forward) in one pass.
 *
 *  face_vertices_z      (B,F,3)   f32
 *  face_vertices_image  (B,F,3,2) f32, NOT multiplied
 *  face_features        (B,F,3,D) f32 (may be NULL when D == 0)
 *  face_normals_z       (B,F) f32 or NULL: faces with value >= 0 are rasterized
 *  valid_faces          (B,F) u8  or NULL: faces with non-zero are rasterized
 *  boxlen_m             = (float)(boxlen * multiplier)   (dibr.py:36-37)
 *  mode                 DIBR_B200_RASTER | DIBR_B200_SOFT_MASK
 *  face_idx             (B,H,W) i64: output if RASTER, else INPUT (dibr_soft_mask alone)
 *  interpolated_features(B,H,W,D) f32, output_weights (B,H,W,3) f32: outputs if RASTER
 *  soft_mask            (B,H,W) f32: output if SOFT_MASK
 * The workspace keeps the face bins; pass it unchanged to dibr_b200_backward
 * with bins_valid = 1 to skip rebuilding them.
 */
int dibr_b200_forward(
    int batch, int num_faces, int height, int width, int feat_dim,
    const float* face_vertices_z, const float* face_vertices_image,
    const float* face_features, const float* face_normals_z, const uint8_t* valid_faces,
    float multiplier, float eps, int mode, float sigmainv, float boxlen_m, int knum,
    float* interpolated_features, int64_t* face_idx, float* output_weights, float* soft_mask,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

/*
 * Fused backward: grad wrt face_vertices_image (sum of the rasterize and the
 * soft-mask branches, as autograd would add them) and wrt face_features.
 * Replaces rasterization.py:355-371 + dibr.py:58-73 and the kernels behind them.
 *  grad_features  (B,H,W,D) f32 or NULL (skips the rasterize branch; grad_face_features is zeroed)
 *  grad_soft_mask (B,H,W)   f32 or NULL (skips the soft-mask branch)
 *  soft_mask      forward's output (needed only with grad_soft_mask)
 *  flags          DIBR_B200_BINS_VALID: workspace still holds forward's bins for the same
 *                 inputs.  DIBR_B200_ACCUMULATE: grad_face_vertices_image is added to, not
 *                 zeroed first - lets a caller run the two branches as two calls (e.g. to
 *                 start sending grad_face_features while the soft-mask branch still runs);
 *                 grad_face_features is only touched when grad_features is given.
 *  workspace      may be NULL when grad_soft_mask is NULL.  When it is at least
 *                 dibr_b200_workspace_bytes() the rasterize branch (fp32 features, D <= 4,
 *                 width a multiple of 4) runs the row-walk kernel, which scatters into padded
 *                 per-face records in the workspace with 16-byte vector reductions; otherwise
 *                 the warp-reduction kernel scatters straight into the outputs.
 */
int dibr_b200_backward(
    int batch, int num_faces, int height, int width, int feat_dim,
    const float* grad_features, const float* grad_soft_mask,
    const int64_t* face_idx, const float* output_weights, const float* soft_mask,
    const float* face_vertices_image, const float* face_features,
    float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
    float* grad_face_vertices_image, float* grad_face_features,
    void* workspace, size_t workspace_bytes, int flags, dibr_b200_stream_t stream);

/*
 * dibr_b200_backward restricted to the views [view_begin, view_end) of the batch.  ALL pointers are
 * the full-batch tensors and the forward's workspace (exactly what dibr_b200_backward takes;
 * grad_features / face_features hold bfloat16 bit patterns when features_bf16 != 0); only the rows
 * of grad_face_vertices_image / grad_face_features that belong to those views are written.  Lets a
 * caller pipeline the backward of one view chunk with the exchange (all-gather) of the previous
 * chunk's gradients: kaolin_b200.multi_gpu.pipelined_backward_all_gather.
 */
int dibr_b200_backward_views(
    int batch, int num_faces, int height, int width, int feat_dim,
    const void* grad_features, const float* grad_soft_mask,
    const int64_t* face_idx, const float* output_weights, const float* soft_mask,
    const float* face_vertices_image, const void* face_features, int features_bf16,
    float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
    float* grad_face_vertices_image, float* grad_face_features,
    void* workspace, size_t workspace_bytes, int flags, int view_begin, int view_end,
    dibr_b200_stream_t stream);

/*
 * float64 instantiation of the fused entry points (the reference dispatches float and double:
 * rasterization_cuda.cu:218/427, dibr_soft_mask_cuda.cu:205/376; its tests parametrise the dtype).
 * Same contract as dibr_b200_forward / dibr_b200_backward with double tensors (face_idx stays i64;
 * multiplier / eps / sigmainv are C floats exactly as in the reference kernels' signatures, the
 * enlarged-bbox margin boxlen * multiplier is a double as in dibr.py:33-39).  Every per-pixel decision
 * is taken with the reference's <double> arithmetic (pixel centres computed in float and widened);
 * built for exactness, not speed (one thread per pixel walks its tile's bins; double atomics in the
 * backward).  workspace >= dibr_b200_workspace_bytes_f64(); pass it unchanged to the backward with
 * DIBR_B200_BINS_VALID to reuse the forward's bins.
 */
size_t dibr_b200_workspace_bytes_f64(int batch, int64_t total_faces, int height, int width);
int dibr_b200_forward_f64(
    int batch, int num_faces, int height, int width, int feat_dim,
    const double* face_vertices_z, const double* face_vertices_image,
    const double* face_features, const double* face_normals_z, const uint8_t* valid_faces,
    float multiplier, float eps, int mode, float sigmainv, double boxlen_m, int knum,
    double* interpolated_features, int64_t* face_idx, double* output_weights, double* soft_mask,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);
int dibr_b200_backward_f64(
    int batch, int num_faces, int height, int width, int feat_dim,
    const double* grad_features, const double* grad_soft_mask,
    const int64_t* face_idx, const double* output_weights, const double* soft_mask,
    const double* face_vertices_image, const double* face_features,
    float multiplier, float eps, float sigmainv, double boxlen_m, int knum,
    double* grad_face_vertices_image, double* grad_face_features,
    void* workspace, size_t workspace_bytes, int flags, dibr_b200_stream_t stream);

/*
 * bf16 feature storage (BASELINE.json configs[3], "bf16 features"; an extension - the
 * reference dispatches float/double only, rasterization_cuda.cu:218): same as
 * dibr_b200_forward / dibr_b200_backward except that face_features (B,F,3,D),
 * interpolated_features (B,H,W,D) and grad_features (B,H,W,D) hold bfloat16 bit patterns.
 * Arithmetic is the fp32 arithmetic of the fp32 entry points on the upcast values; the
 * interpolated feature is rounded to nearest-even once, on store, so it equals the fp32
 * entry point's output converted to bf16.  Geometry, weights, soft mask and BOTH output
 * gradients (fp32 accumulation) stay fp32.
 */
int dibr_b200_forward_bf16(
    int batch, int num_faces, int height, int width, int feat_dim,
    const float* face_vertices_z, const float* face_vertices_image,
    const uint16_t* face_features, const float* face_normals_z, const uint8_t* valid_faces,
    float multiplier, float eps, int mode, float sigmainv, float boxlen_m, int knum,
    uint16_t* interpolated_features, int64_t* face_idx, float* output_weights, float* soft_mask,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

int dibr_b200_backward_bf16(
    int batch, int num_faces, int height, int width, int feat_dim,
    const uint16_t* grad_features, const float* grad_soft_mask,
    const int64_t* face_idx, const float* output_weights, const float* soft_mask,
    const float* face_vertices_image, const uint16_t* face_features,
    float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
    float* grad_face_vertices_image, float* grad_face_features,
    void* workspace, size_t workspace_bytes, int flags, dibr_b200_stream_t stream);

/*
 * Operator: kaolin::packed_rasterize_forward_cuda
 * (kaolin/csrc/render/mesh/rasterization.h:23-32, rasterization.cpp:49-104).
 * Packed valid faces of all meshes; coordinates already multiplied; tight bboxes
 * [xmin,ymin,xmax,ymax]; first_idx_face_per_mesh is a DEVICE int64 array (B+1).
 * selected_face_idx is relative to the mesh's first face, -1 = background.
 */
int dibr_b200_packed_rasterize_forward(
    int batch, int64_t total_faces, int height, int width, int feat_dim,
    const float* face_vertices_z, const float* face_vertices_image,
    const float* face_bboxes, const float* face_features,
    const int64_t* first_idx_face_per_mesh, float multiplier, float eps,
    float* interpolated_features, int64_t* selected_face_idx, float* output_weights,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

/*
 * Operator: kaolin::rasterize_backward_cuda
 * (rasterization.h:34-41, rasterization.cpp:106-168).  face_vertices_image is the
 * UNSCALED (B,F,3,2) tensor; selected_face_idx holds original face ids.
 * (The reference's `interpolated_features` argument is never read by its kernel
 * and is therefore not part of this ABI.)
 */
int dibr_b200_rasterize_backward(
    int batch, int num_faces, int height, int width, int feat_dim,
    const float* grad_interpolated_features, const int64_t* selected_face_idx,
    const float* output_weights, const float* face_vertices_image,
    const float* face_features, float eps,
    float* grad_face_vertices_image, float* grad_face_features,
    dibr_b200_stream_t stream);

/*
 * Operator: kaolin::dibr_soft_mask_forward_cuda
 * (kaolin/csrc/render/mesh/dibr_soft_mask.h:23-30, dibr_soft_mask.cpp:48-108).
 * face_vertices_image already multiplied; face_large_bboxes (B,F,4).
 * close_face_prob (B,H,W,K) f32, close_face_idx (B,H,W,K) i64 (-1 padded),
 * close_face_dist_type (B,H,W,K) u8 (0 padded; 1-3 edge, 4-6 vertex).
 */
int dibr_b200_soft_mask_forward(
    int batch, int num_faces, int height, int width, int knum,
    const float* face_vertices_image, const float* face_large_bboxes,
    const int64_t* selected_face_idx, float sigmainv, float multiplier,
    float* soft_mask, float* close_face_prob, int64_t* close_face_idx,
    uint8_t* close_face_dist_type,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

/*
 * Operator: kaolin::dibr_soft_mask_backward_cuda
 * (dibr_soft_mask.h:32-42, dibr_soft_mask.cpp:110-183).
 */
int dibr_b200_soft_mask_backward(
    int batch, int num_faces, int height, int width, int knum,
    const float* grad_soft_mask, const float* soft_mask, const int64_t* selected_face_idx,
    const float* close_face_prob, const int64_t* close_face_idx,
    const uint8_t* close_face_dist_type, const float* face_vertices_image,
    float sigmainv, float multiplier, float* grad_face_vertices_image,
    dibr_b200_stream_t stream);

/*
 * float64 instantiation of the four operators (the reference dispatches float and double:
 * rasterization_cuda.cu:218/427, dibr_soft_mask_cuda.cu:205/376).  Each takes the arguments of its
 * float sibling above, with double tensors where the reference uses scalar_t; indices, K-list ids and
 * dist types keep their types, multiplier / eps / sigmainv stay C floats as in the reference kernels.
 * Every decision is the reference's <double> arithmetic on the caller's tensors as given: the half-open
 * bbox tests read face_bboxes / face_large_bboxes, the coordinates are not multiplied again, pixel
 * centres are computed in float and widened.  Built for exactness, not speed.  The two forwards take a
 * workspace of at least dibr_b200_workspace_bytes_f64(); the two backwards zero their outputs inside.
 */

/* Operator: kaolin::packed_rasterize_forward_cuda<double> (rasterization.h:23-32). */
int dibr_b200_packed_rasterize_forward_f64(
    int batch, int64_t total_faces, int height, int width, int feat_dim,
    const double* face_vertices_z, const double* face_vertices_image,
    const double* face_bboxes, const double* face_features,
    const int64_t* first_idx_face_per_mesh, float multiplier, float eps,
    double* interpolated_features, int64_t* selected_face_idx, double* output_weights,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

/* Operator: kaolin::rasterize_backward_cuda<double> (rasterization.h:34-41); no workspace. */
int dibr_b200_rasterize_backward_f64(
    int batch, int num_faces, int height, int width, int feat_dim,
    const double* grad_interpolated_features, const int64_t* selected_face_idx,
    const double* output_weights, const double* face_vertices_image,
    const double* face_features, float eps,
    double* grad_face_vertices_image, double* grad_face_features,
    dibr_b200_stream_t stream);

/* Operator: kaolin::dibr_soft_mask_forward_cuda<double> (dibr_soft_mask.h:23-30).  close_face_prob
 * (B,H,W,K) f64; the three K-lists are all given or all NULL. */
int dibr_b200_soft_mask_forward_f64(
    int batch, int num_faces, int height, int width, int knum,
    const double* face_vertices_image, const double* face_large_bboxes,
    const int64_t* selected_face_idx, float sigmainv, float multiplier,
    double* soft_mask, double* close_face_prob, int64_t* close_face_idx,
    uint8_t* close_face_dist_type,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

/* Operator: kaolin::dibr_soft_mask_backward_cuda<double> (dibr_soft_mask.h:32-42). */
int dibr_b200_soft_mask_backward_f64(
    int batch, int num_faces, int height, int width, int knum,
    const double* grad_soft_mask, const double* soft_mask, const int64_t* selected_face_idx,
    const double* close_face_prob, const int64_t* close_face_idx,
    const uint8_t* close_face_dist_type, const double* face_vertices_image,
    float sigmainv, float multiplier, double* grad_face_vertices_image,
    dibr_b200_stream_t stream);

/* =========================================================================
 * The steps either side of the rasterizer in every DIB-R caller (SURVEY.md 8f rank 1, 2);
 * kaolin_b200/csrc/mesh_pipeline.cu.  The reference has no native interface for them: they
 * are chains of PyTorch ops (cited per entry point); the signatures below are what a
 * binding for a fused version would take.  No workspace; asynchronous on `stream`.
 * ========================================================================= */

/*
 * prepare_vertices (kaolin/render/mesh/utils.py:129-175): camera transform
 * (camera/legacy.py:22-37 with camera_rot (B,3,3) + camera_trans (B,3), or
 * [p,1] @ camera_transform (B,4,3); pass exactly one of the two), perspective divide
 * (camera/legacy.py:120-138; camera_proj_host = 3 floats on the HOST), gather by `faces`
 * (F,3) i64 (ops/mesh/mesh.py:54-76) and unit face normals (ops/mesh/trianglemesh.py:314-338).
 * Outputs: face_vertices_camera (B,F,3,3), face_vertices_image (B,F,3,2), face_normals (B,F,3).
 */
int dibr_b200_prepare_vertices_forward(
    int batch, int num_vertices, int num_faces, const float* vertices, const int64_t* faces,
    const float* camera_transform, const float* camera_rot, const float* camera_trans,
    const float* camera_proj_host, float* face_vertices_camera, float* face_vertices_image,
    float* face_normals, dibr_b200_stream_t stream);

/* Gradient wrt the CAMERA-SPACE vertices (B,V,3) (zeroed inside, scattered with float
 * atomics); any of the three upstream gradients may be NULL.  The linear map back to
 * world-space vertices / camera parameters is a (B,V,3)x(3,3) product left to the caller. */
int dibr_b200_prepare_vertices_backward(
    int batch, int num_vertices, int num_faces, const float* vertices, const int64_t* faces,
    const float* camera_transform, const float* camera_rot, const float* camera_trans,
    const float* camera_proj_host, const float* grad_face_vertices_camera,
    const float* grad_face_vertices_image, const float* grad_face_normals,
    float* grad_vertices_camera, dibr_b200_stream_t stream);

/*
 * texture_mapping (kaolin/render/mesh/utils.py:22-79): texture_coordinates (B,N,2) in [0,1]
 * (OpenGL convention), texture_maps (B,C,Ht,Wt); clamp, y flip,
 * grid_sample(align_corners=False, padding_mode='border'), mode nearest (1) or bilinear (0).
 * out (B,N,C).  Backward: grad_texture_maps (B,C,Ht,Wt) (zeroed inside) and/or
 * grad_texture_coordinates (B,N,2); either may be NULL.
 */
int dibr_b200_texture_mapping_forward(
    int batch, int64_t num_points, int channels, int tex_height, int tex_width,
    const float* texture_coordinates, const float* texture_maps, int nearest, float* out,
    dibr_b200_stream_t stream);
int dibr_b200_texture_mapping_backward(
    int batch, int64_t num_points, int channels, int tex_height, int tex_width,
    const float* texture_coordinates, const float* texture_maps, int nearest,
    const float* grad_out, float* grad_texture_maps, float* grad_texture_coordinates,
    dibr_b200_stream_t stream);

/*
 * mask_iou (kaolin/metrics/render.py:18-41): loss = 1 - mean_b(sum(l*r) / (sum(l+r-l*r) + 1e-10)).
 * sums (B,2) f32 scratch/output {sum(l*r), sum(l+r-l*r)} kept for the backward; loss: 1 f32.
 */
int dibr_b200_mask_iou_forward(
    int batch, int64_t pixels_per_view, const float* lhs_mask, const float* rhs_mask,
    float* sums, float* loss, dibr_b200_stream_t stream);
int dibr_b200_mask_iou_backward(
    int batch, int64_t pixels_per_view, const float* lhs_mask, const float* rhs_mask,
    const float* sums, const float* grad_loss, float* grad_lhs, float* grad_rhs,
    dibr_b200_stream_t stream);

/*
 * DefTet volumetric renderer operators (SURVEY.md 8f rank 3; kaolin_b200/csrc/deftet.cu).
 * Operator: kaolin::deftet_sparse_render_forward_cuda (kaolin/csrc/render/mesh/deftet.h,
 * deftet.cpp:48-113, kernel deftet_cuda.cu:31-194; registered at bindings.cpp next to the four
 * DIB-R operators).  For every query point the first `knum` faces IN INDEX ORDER whose half-open
 * bbox holds the point, whose eps-normalised barycentric weights are all >= 0 and whose
 * interpolated depth lies in [render_ranges[...,0], render_ranges[...,1]).
 *  face_vertices_z (B,F,3), face_vertices_image (B,F,3,2), face_bboxes (B,F,4) [xmin,ymin,xmax,ymax],
 *  pixel_coords (B,P,2), render_ranges (B,P,2)  f32
 *  outputs (B,P,K): face_idx i64 (-1 padded), pixel_depth f32 (-inf padded), w0, w1 f32 (0 padded),
 *  fully written.  workspace >= dibr_b200_deftet_workspace_bytes(batch, num_faces).
 */
size_t dibr_b200_deftet_workspace_bytes(int batch, int num_faces);
int dibr_b200_deftet_sparse_render_forward(
    int batch, int num_faces, int num_pixels, int knum,
    const float* face_vertices_z, const float* face_vertices_image, const float* face_bboxes,
    const float* pixel_coords, const float* render_ranges, float eps,
    int64_t* face_idx, float* pixel_depth, float* w0, float* w1,
    void* workspace, size_t workspace_bytes, dibr_b200_stream_t stream);

/*
 * Operator: kaolin::deftet_sparse_render_backward_cuda (deftet.cpp:115-170, kernel
 * deftet_cuda.cu:238-430).  grad_interpolated_features (B,P,K,D), face_idx (B,P,K) i64,
 * weights (B,P,K,3), face_vertices_image (B,F,3,2), face_features (B,F,3,D);
 * outputs grad_face_vertices_image (B,F,3,2), grad_face_features (B,F,3,D), zeroed inside.
 */
int dibr_b200_deftet_sparse_render_backward(
    int batch, int num_faces, int num_pixels, int knum, int feat_dim,
    const float* grad_interpolated_features, const int64_t* face_idx, const float* weights,
    const float* face_vertices_image, const float* face_features, float eps,
    float* grad_face_vertices_image, float* grad_face_features, dibr_b200_stream_t stream);

/*
 * Exchange step of the view-sharded path (SURVEY.md 8e; kaolin_b200/csrc/peer_push.cu): the
 * reference has no multi-GPU code - its callers all-gather the per-view gradients with
 * torch.distributed.  All-gather by STORES over NVLink: copies `bytes` (multiple of 16) from the
 * local device buffer `src` to dst[i] + dst_offset_bytes for i < n_dst (<= 16), where dst[i] are
 * device pointers valid in this process (local memory or peer memory mapped through CUDA
 * symmetric / IPC memory; host array of pointers).  `ctas` bounds the grid (<= 0: 32) so that the
 * kernel can run underneath compute.  Asynchronous on `stream`; a cross-rank barrier after it is
 * the caller's (kaolin_b200/multi_gpu.py:PeerGradAllGather).
 */
int dibr_b200_peer_push(const void* src, size_t bytes, void* const* dst, int n_dst, size_t dst_offset_bytes,
                        int ctas, dibr_b200_stream_t stream);
/*
 * The same through an NVSwitch MULTICAST address (multimem.st): `multicast_dst` is the multicast
 * mapping of the symmetric landing buffer; one store per 16 bytes lands at multicast_dst +
 * dst_offset_bytes in EVERY GPU bound to the multicast object, this one included - a rank's
 * egress is its shard once, not once per peer.
 */
int dibr_b200_peer_push_multicast(const void* src, size_t bytes, void* multicast_dst, size_t dst_offset_bytes,
                                  int ctas, dibr_b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DIBR_B200_H_ */
