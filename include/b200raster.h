/*
 * b200raster.h -- C ABI of libb200raster.so, the B200 (sm_100a) differentiable
 * mesh rasterizer that drops in behind Jittor/jrender's rasterizer Functions.
 *
 * Every entry point replaces one `jt.code(...)` op of the reference (paths are
 * relative to the reference checkout):
 *
 *   b200r_softras_forward   <- jrender/renderer/dr/softras/cuda/soft_rasterize.py:3-521
 *                              (forward_soft_rasterize: memsets + K1 + K2), called from
 *                              jrender/renderer/dr/softras/soft_rasterize.py:75-82; also
 *                              serves the bin_size>0 call site (:91-99,
 *                              soft_rasterize_coarse_to_fine.py:7-879) -- binning is
 *                              internal here and exact, so one entry point covers both.
 *   b200r_softras_backward  <- jrender/renderer/dr/softras/cuda/soft_rasterize.py:966-1416
 *                              (backward_soft_rasterize, top-K), called from
 *                              jrender/renderer/dr/softras/soft_rasterize.py:125-132.
 *   b200r_nmr_forward       <- jrender/renderer/dr/n3mr/cuda/rasterize.py:5-217 and :219-339
 *                              (forward_face_index_map + forward_texture_sampling),
 *                              called from jrender/renderer/dr/n3mr/n3mr.py:125-133.
 *   b200r_nmr_backward      <- jrender/renderer/dr/n3mr/cuda/rasterize.py:342-648, :650-727,
 *                              :729-822 (backward_pixel_map, backward_textures,
 *                              backward_depth_map), called from n3mr.py:29-67.
 *   b200r_sss_blur_chain    <- jrender/renderer/utils/ToStretchMap.py and the 36 _blur_for_SSS ops
 *                              (renderer/utils/gaussian_blur.py:34-165) of SSS(), called from
 *                              jrender/renderer/lighting/lighting.py:86-156 (Mesh.with_SSS).
 *
 * Conventions
 *   - All tensor pointers are DEVICE pointers owned by the caller (contiguous, fp32 /
 *     int32).  No allocation and no host synchronisation happens inside; all work is
 *     enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - Scalar parameters are runtime arguments (the reference bakes them into JIT source).
 *   - Return 0 on success; a negative B200R_E* code for argument errors; a positive
 *     cudaError_t for CUDA failures.  b200r_last_error() returns a thread-local message.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef B200RASTER_H
#define B200RASTER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B200R_API __attribute__((visibility("default")))
#else
#define B200R_API
#endif

#define B200R_EINVAL (-1)      /* bad argument (NULL pointer, size, enum out of range) */
#define B200R_EWORKSPACE (-2)  /* workspace too small */
#define B200R_EUNSUPPORTED (-3)

/* enum values = the reference's maps, jrender/renderer/dr/softras/soft_rasterize.py:39-42 */
enum { B200R_DIST_HARD = 0, B200R_DIST_BARYCENTRIC = 1, B200R_DIST_EUCLIDEAN = 2 };
enum { B200R_RGB_HARD = 0, B200R_RGB_SOFTMAX = 1, B200R_RGB_NONE = 2 };
enum { B200R_ALPHA_HARD = 0, B200R_ALPHA_SUM = 1, B200R_ALPHA_PROD = 2 };
enum { B200R_TEX_SURFACE = 0, B200R_TEX_VERTEX = 1 };

#define B200R_MAX_FACES_PER_PIXEL 64 /* kMaxPointsPerPixel, cuda/soft_rasterize.py:16 */

B200R_API const char* b200r_version(void);
B200R_API const char* b200r_last_error(void);

/* Device memory of one forward / backward pair, in two caller-allocated blocks:
 *   state      b200r_softras_state_bytes(batch, num_faces): written by the forward, handed to the backward -- the per-face
 *              records (what the reference keeps in `faces_info`, soft_rasterize.py:62,101) and the backward's gradient
 *              accumulator.  208 bytes per (batch, face).
 *   workspace  b200r_softras_workspace_bytes(batch, num_faces, image_size): transient scratch of the forward only (binning
 *              lists in a pool of 512-id chunks budgeted at 8 list entries per face -- bins that find the pool exhausted
 *              are flagged and their blocks filter the whole face list, so nothing is ever dropped -- and the block
 *              queue); free to be released or reused once the forward has been enqueued.  ~12 MB for 4 x 1024^2 images of
 *              39 200 faces. */
B200R_API size_t b200r_softras_workspace_bytes(int batch_size, int num_faces, int image_size);
B200R_API size_t b200r_softras_state_bytes(int batch_size, int num_faces);

/* SoftRas forward.
 *   face_vertices  [B, nf, 3, 3]  NDC x,y (+y up) and camera-space z per vertex
 *   textures       [B, nf, T, 3]  T = R*R texels (surface) or 3 (vertex)
 *   soft_colors    [B, 4, H, W]   out, planar RGBA, row 0 = top (y = +1)
 *   aggrs_info     [B, 2, H, W]   out: softmax -> (sum, max); hard rgb -> (depth_min, face_index_min)
 *   faces_id_buffer[B, K, H, W]   out, int32, the <=K nearest-z face ids per pixel in the
 *                                 reference's slot order, -1 TERMINATED: slots [0, n) hold ids, slot n (if n < K) is
 *                                 -1, and the slots behind it are left untouched (the reference memsets all of them
 *                                 to -1, soft_rasterize.py:470; the backward only ever reads up to the first -1,
 *                                 :1236-1237, and so does b200r_softras_backward).  Nothing to initialise on the caller's
 *                                 side.
 *   faces_info     [B, nf, 27]    out, optional (may be NULL): the reference's K1 output
 *   dist_eps_logit = ln(1/dist_eps - 1) computed by the host as soft_rasterize.py:25
 * Background colour is always 0, as in the reference (the op memsets soft_colors). */
B200R_API int b200r_softras_forward(const float* face_vertices, const float* textures,
                          float* soft_colors, float* aggrs_info, int32_t* faces_id_buffer,
                          float* faces_info, void* state, size_t state_bytes,
                          void* workspace, size_t workspace_bytes,
                          int batch_size, int num_faces, int texture_size, int image_size,
                          int max_faces_per_pixel, float near, float far, float eps,
                          float sigma_val, float gamma_val, float dist_eps_logit,
                          int dist_func, int rgb_func, int alpha_func, int texture_type,
                          int double_side, void* stream);

/* SoftRas top-K backward.  grad_face_vertices [B,nf,3,3] and grad_textures [B,nf,T,3]
 * are overwritten (zeroed inside, then accumulated). */
B200R_API int b200r_softras_backward(const float* face_vertices, const float* textures,
                           const float* soft_colors, const float* aggrs_info,
                           const int32_t* faces_id_buffer, void* state,
                           size_t state_bytes, const float* grad_soft_colors,
                           float* grad_face_vertices, float* grad_textures,
                           int batch_size, int num_faces, int texture_size, int image_size,
                           int max_faces_per_pixel, float near, float far, float eps,
                           float sigma_val, float gamma_val, float dist_eps_logit,
                           int dist_func, int rgb_func, int alpha_func, int texture_type,
                           int double_side, void* stream);

/* Anti-aliased flavours (SURVEY.md section 8f rank 2): replace SoftRasterizer.execute's "render at 2 x image_size, then
 * 2x2 mean-pool" (jrender/renderer/dr/softras/rasterizer.py:45,54-55) without the extra passes.  image_size is the
 * SUPERSAMPLED size (even).  forward_aa additionally writes pooled_colors [B,4,image_size/2,image_size/2], the 2x2 means of
 * soft_colors, from the forward kernel's output staging (soft_colors is still written: the backward reads it);
 * backward_aa takes grad_pooled_colors [B,4,image_size/2,image_size/2] and forms avg_pool2d's backward (grad / 4 at each
 * of the four source pixels) while loading, instead of materialising a 4x larger gradient tensor. */
B200R_API int b200r_softras_forward_aa(const float* face_vertices, const float* textures, float* soft_colors,
                           float* pooled_colors, float* aggrs_info, int32_t* faces_id_buffer, float* faces_info,
                           void* state, size_t state_bytes, void* workspace, size_t workspace_bytes,
                           int batch_size, int num_faces, int texture_size, int image_size,
                           int max_faces_per_pixel, float near, float far, float eps,
                           float sigma_val, float gamma_val, float dist_eps_logit,
                           int dist_func, int rgb_func, int alpha_func, int texture_type,
                           int double_side, void* stream);
B200R_API int b200r_softras_backward_aa(const float* face_vertices, const float* textures,
                           const float* soft_colors, const float* aggrs_info,
                           const int32_t* faces_id_buffer, void* state,
                           size_t state_bytes, const float* grad_pooled_colors,
                           float* grad_face_vertices, float* grad_textures,
                           int batch_size, int num_faces, int texture_size, int image_size,
                           int max_faces_per_pixel, float near, float far, float eps,
                           float sigma_val, float gamma_val, float dist_eps_logit,
                           int dist_func, int rgb_func, int alpha_func, int texture_type,
                           int double_side, void* stream);

/* ---- NMR (dr_type='n3mr') hard rasterizer -------------------------------------------------
 * Maps keep the reference kernels' orientation [B, yi, xi] with yi UP (row 0 = bottom); the
 * vertical flip to image orientation belongs to the caller (n3mr.py:239-247).
 *   faces               [B, nf, 3, 3]
 *   textures            [B, nf, ts, ts, ts, 3]           (return_rgb)
 *   face_index_map      [B, H, W] int32, -1 = background
 *   weight_map          [B, H, W, 3]      depth_map [B, H, W] (far where uncovered)
 *   rgb_map             [B, H, W, 3]      already mixed with background_rgb (host float[3], may be NULL = black)
 *   alpha_map           [B, H, W]         (face_index >= 0)
 *   sampling_index_map  [B, H, W, 8] int32, sampling_weight_map [B, H, W, 8]
 *   face_inv_map        [B, H, W, 9]      (return_depth)
 * Equal-depth ties are won by the lowest face id (the reference's winner is race-dependent). */
B200R_API size_t b200r_nmr_workspace_bytes(int batch_size, int num_faces, int image_size);
B200R_API int b200r_nmr_forward(const float* faces, const float* textures, int32_t* face_index_map,
                                float* weight_map, float* depth_map, float* rgb_map, float* alpha_map,
                                int32_t* sampling_index_map, float* sampling_weight_map, float* face_inv_map,
                                void* workspace, size_t workspace_bytes, int batch_size, int num_faces,
                                int texture_size, int image_size, float near, float far, float eps,
                                const float* background_rgb, int return_rgb, int return_alpha,
                                int return_depth, void* stream);
/* grad_faces [B,nf,3,3] and grad_textures [B,nf,ts,ts,ts,3] are overwritten.  Sub-ops follow
 * n3mr.py:29-67: pixel-map gradient (x,y) -> texture gradient -> depth gradient accumulated in place.
 * `scratch` (b200r_nmr_backward_scratch_bytes) holds the packed row-/column-major pixel records the
 * pixel-map gradient scans; it is only needed when return_rgb or return_alpha. */
B200R_API size_t b200r_nmr_backward_scratch_bytes(int batch_size, int image_size);
B200R_API int b200r_nmr_backward(const float* faces, const int32_t* face_index_map, const float* weight_map,
                                 const float* depth_map, const float* rgb_map, const float* alpha_map,
                                 const int32_t* sampling_index_map, const float* sampling_weight_map,
                                 const float* face_inv_map, const float* grad_rgb_map,
                                 const float* grad_alpha_map, const float* grad_depth_map, float* grad_faces,
                                 float* grad_textures, void* scratch, size_t scratch_bytes,
                                 int batch_size, int num_faces, int texture_size,
                                 int image_size, float eps, int return_rgb, int return_alpha,
                                 int return_depth, void* stream);

/* ---- fused pre-raster geometry stage (SURVEY.md section 8f rank 1) ------------------------------
 * World-space vertices -> camera space -> projection -> per-face gather in ONE launch.  Replaces
 * the tensor-op chain of jrender/renderer/transform/look_at.py:24-38 (or look.py:23-53),
 * transform/perspective.py:11-16 / orthogonal.py:12-15 and structures/utils/faces_vertices.py:14-19,
 * called from transform/transform.py:52-58 and structures/mesh.py (face_vertices property).
 *   vertices       [vertices_batch, nv, 3]   world space; vertices_batch = B, or 1 = shared mesh
 *   faces          [faces_batch, nf, 3] int32; faces_batch = B or 1; an index outside [0, nv) makes
 *                  that corner NaN (the reference reads out of bounds)
 *   eye            [eye_batch, 3] device; eye_batch = B or 1
 *   face_vertices  [B, nf, 3, 3]   out: x, y projected (perspective: X/Z/width; orthogonal: X*scale), z = camera Z
 *   at_or_direction, up: HOST float[3] (look_at: the `at` point; look: the viewing direction)
 *   width_or_scale: tan(viewing_angle) (perspective.py:11-12) or viewing_scale (orthogonal)
 * The backward overwrites grad_vertices [vertices_batch, nv, 3] with the sum over every (batch, face,
 * corner) that references the vertex (float atomics).  No gradient for eye / at / up. */
enum { B200R_CAM_LOOK_AT = 0, B200R_CAM_LOOK_RIGHT = 1, B200R_CAM_LOOK_LEFT = 2 };
enum { B200R_PROJ_PERSPECTIVE = 0, B200R_PROJ_ORTHOGONAL = 1 };
B200R_API int b200r_project_faces_forward(const float* vertices, const int32_t* faces, const float* eye,
                                          float* face_vertices,
                                          const float* at_or_direction, const float* up, float width_or_scale,
                                          int camera_mode, int projection, int batch_size, int num_vertices,
                                          int num_faces, int vertices_batch, int faces_batch, int eye_batch, void* stream);
B200R_API int b200r_project_faces_backward(const float* vertices, const int32_t* faces, const float* eye,
                                           const float* grad_face_vertices, float* grad_vertices,
                                           const float* at_or_direction, const float* up, float width_or_scale,
                                           int camera_mode, int projection, int batch_size, int num_vertices,
                                           int num_faces, int vertices_batch, int faces_batch, int eye_batch, void* stream);

/* ---- fused mesh regularisers of the fitting loop (SURVEY.md section 8f rank 4) ---------------------
 * Each call writes loss [B] AND d(loss_b)/d(vertices) [B, nv, 3] (both overwritten) in one launch.
 *   b200r_flatten_loss   <- jrender/loss/flatten_loss.py:38-79; v0s..v3s [E] int32 = the edge table the
 *                           reference builds at :14-36 (edge v0-v1 shared by the faces with apexes v2, v3)
 *   b200r_laplacian_loss <- jrender/loss/laplacian_loss.py:29-36 with the row-normalised Laplacian of :11-27
 *                           stored as a padded neighbour table: (L x)_i = diag[i] x_i + sum_k w[i,k] x[nbr[i,k]],
 *                           neighbours / neighbour_weights [nv, max_degree] (weight 0 = padding), diag [nv] */
B200R_API int b200r_flatten_loss(const float* vertices, const int32_t* v0s, const int32_t* v1s, const int32_t* v2s,
                                 const int32_t* v3s, float* loss, float* grad_vertices, int batch_size,
                                 int num_vertices, int num_edges, float eps, void* stream);
B200R_API int b200r_laplacian_loss(const float* vertices, const int32_t* neighbours, const float* neighbour_weights,
                                   const float* diag, float* loss, float* grad_vertices, int batch_size,
                                   int num_vertices, int max_degree, void* stream);

/* Launch counter: number of kernels this library has launched in this process
 * (bench.py reports the delta over the timed region as "gpu_launches"). */
/* ---- texture baking (SURVEY.md section 8f rank 3) -------------------------------------------------------------
 * Replaces _load_textures_for_softras / load_textures_cuda_kernel (jrender/io/utils/load_textures.py:3-101):
 * image [H, W, 3] f32 (already flipped vertically by the caller, _load_obj_for_softras.py:136), faces_uv [nf, 3, 2],
 * is_update [nf] int32, textures [nf, R*R, 3] updated in place where is_update != 0.  Device pointers. */
B200R_API int b200r_bake_textures_softras(const float* image, const float* faces_uv, const int32_t* is_update, float* textures,
                                          int nf, int texture_res, int image_height, int image_width, void* stream);
/* Replaces _load_textures_for_n3mr / load_textures_cuda_kernel (jrender/io/utils/load_textures.py:103-246), the bake of
 * the NMR rasterizer's [nf, ts, ts, ts, 3] textures: texel (a, b, c) samples the image at the barycentric point
 * (a, b, c) / (ts - 1) normalised to sum 1, through the face's wrapped UVs.  texture_wrapping: 0 REPEAT, 1 MIRRORED_REPEAT,
 * 2 CLAMP_TO_EDGE, 3 CLAMP_TO_BORDER (writes zeros, like the reference); use_bilinear: bilinear (1) or nearest (0) fetch.
 * texture_size >= 2 (the reference divides by texture_size - 1).  faces_uv is read-only here (the reference wraps it in
 * place from every thread of the face, a race).  textures updated in place where is_update != 0. */
B200R_API int b200r_bake_textures_n3mr(const float* image, const float* faces_uv, const int32_t* is_update, float* textures,
                                       int nf, int texture_size, int image_height, int image_width, int texture_wrapping,
                                       int use_bilinear, void* stream);

/* ---- fused surface-mode lighting of the pre-raster stage (SURVEY.md section 8f rank 1) -------------------------
 * Replaces Lighting.execute with light_mode='surface', no normal map, no SSS, one directional light:
 *   jrender/renderer/lighting/lighting.py:186-204, ambient_lighting.py:4-9, directional_lighting.py:54-135
 *   (diffuse branch, and the Cook-Torrance branch when with_specular and eye / metallic / roughness are given),
 *   surface normals of jrender/structures/mesh.py:213-229.
 * vertices [vertices_batch, nv, 3] world space, faces [faces_batch, nf, 3] int32, textures / out_textures
 * [B, nf, T, 3] (T = texture_res^2, or ts^3 for n3mr), metallic / roughness [B, nf, Tm] or NULL, eye [eye_batch, 3]
 * (eye_batch 0: none).  Batches of 1 broadcast.  ambient_color, directional_color, direction: HOST pointers to 3 floats
 * (direction already normalised).  backward overwrites grad_textures [B, nf, T, 3] and grad_vertices
 * [vertices_batch, nv, 3] (NULL: not needed). */
B200R_API int b200r_surface_lighting_forward(const float* vertices, const int32_t* faces, const float* textures, const float* metallic,
                                             const float* roughness, const float* eye, float* out_textures, int B, int vertices_batch,
                                             int faces_batch, int eye_batch, int nv, int nf, int T, int Tm, float ambient_intensity,
                                             const float* ambient_color, float directional_intensity, const float* directional_color,
                                             const float* direction, int with_specular, void* stream);
B200R_API int b200r_surface_lighting_backward(const float* vertices, const int32_t* faces, const float* textures, const float* metallic,
                                              const float* roughness, const float* eye, const float* grad_out, float* grad_textures,
                                              float* grad_vertices, int B, int vertices_batch, int faces_batch, int eye_batch, int nv,
                                              int nf, int T, int Tm, float ambient_intensity, const float* ambient_color,
                                              float directional_intensity, const float* directional_color, const float* direction,
                                              int with_specular, void* stream);

/* ---- texture-space subsurface scattering (Mesh.with_SSS) ------------------------------------------------------
 * b200r_sss_blur_chain replaces the image-space part of SSS() (jrender/renderer/lighting/lighting.py:86-156): the stretch
 * map of renderer/utils/ToStretchMap.py (of worldcoord * 7, clamped to [0, 1]) and the 36 launches of the stretch-modulated
 * 7-tap Gaussian blur _blur_for_SSS (renderer/utils/gaussian_blur.py:34-165) for the variances 25, 75, 300, the weighted
 * sum of the three basis images, `* irradiance + specular` and the vertical flip, in seven launches.
 *   worldcoord_map, irradiance_map, specular_map  [>=3, S, S] planar (soft_colors of a texture-space rasterization)
 *   final_map      [S, S, 3] out, flipped vertically, ready for b200r_bake_textures_softras
 *   workspace      b200r_sss_workspace_bytes(S) bytes of device scratch (13 planes of S x S floats)
 *   taps           HOST float[3][7]: Gauss[i] = sqrt(v) * N(v, -sqrt(v) * (3 - i)) per variance, computed in double and
 *                  rounded to float (gaussian_blur.py:8-10); gauss_widths HOST float[3] = sqrt(v)
 *   weights        HOST float[3][3]: weights[channel][basis] (R 0.7 0.2 0.1, G and B 0.1 0.2 0.7 in the reference)
 * b200r_sss_blur is one _blur_for_SSS launch on a single S x S map: dim 1 blurs along x, dim 0 along y; taps HOST
 * float[7].  Both keep the reference's FFMA contraction of the tap interpolation and accumulation (csrc/sss_api.cu). */
B200R_API size_t b200r_sss_workspace_bytes(int image_size);
B200R_API int b200r_sss_blur_chain(const float* worldcoord_map, const float* irradiance_map, const float* specular_map,
                                   float* final_map, void* workspace, size_t workspace_bytes, int image_size,
                                   const float* taps, const float* gauss_widths, const float* weights, void* stream);
B200R_API int b200r_sss_blur(const float* image, const float* modulate, float* out, int image_size, const float* taps,
                             float gauss_width, int dim, void* stream);

B200R_API unsigned long long b200r_launch_count(void);

/* Tuning knobs (process-wide; results are identical for every setting except softras_exact_tail):
 *   "softras_fwd_persistent" 0 = one CTA per tile, 1 = persistent grid + tile queue (default)
 *   "softras_exact_tail"     1 = the reference's double-precision sigmoid / alpha-product tails bit for bit;
 *                            0 (default) = the same expressions in fp32 for the default euclidean+softmax
 *                            mode (<= 1 ulp on D; all index / depth outputs are identical either way)
 *   "softras_list_pool_chunks" >= 0 caps the binning-list chunk pool (exercises the pool-exhausted path in tests);
 *                            -1 (default) = the size b200r_softras_workspace_bytes accounts for */
B200R_API int b200r_set_option(const char* name, int value);

/* Per-kernel device timing (CUDA events recorded on the launch stream around every kernel
 * this library launches).  Off by default.  bench.py uses it for the roofline of the
 * dominant kernel; b200r_profile_read synchronises the outstanding events. */
enum { B200R_K_FACE_SETUP = 0, B200R_K_COARSE_BIN = 1, B200R_K_SOFTRAS_FWD = 2, B200R_K_SOFTRAS_BWD = 3,
       B200R_K_TILE_ORDER = 4, B200R_K_NMR_SETUP = 5, B200R_K_NMR_FWD = 6, B200R_K_NMR_BWD_PIXEL = 7,
       B200R_K_NMR_BWD_MAPS = 8, B200R_K_SOFTRAS_BWD_FINALIZE = 9, B200R_K_NMR_PACK = 10,
       B200R_K_PROJECT_FWD = 11, B200R_K_PROJECT_BWD = 12, B200R_K_FLATTEN_LOSS = 13, B200R_K_LAPLACIAN_LOSS = 14,
       B200R_K_LIGHTING = 15, B200R_K_BAKE = 16, B200R_K_SSS = 17 };
B200R_API void b200r_profile_enable(int on);
B200R_API void b200r_profile_reset(void);
B200R_API int b200r_profile_read(int kernel, double* total_ms, long long* launches);

/* Test hook: checks the exact-arithmetic helpers (csrc/exact_math.cuh) against the plain
 * IEEE expressions they replace on n (a[i], b[i]) pairs; mismatch7[0..5] count bit
 * differences (must all be 0), mismatch7[6] counts pairs that took the reciprocal fast path. */
B200R_API int b200r_debug_exact_math(const float* a, const float* b, int n, int* mismatch7, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200RASTER_H */
