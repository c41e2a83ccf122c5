/* gsr_b200 — C ABI of the B200-native 3D-Gaussian-splatting rasterizer hot path.
 *
 * This is the drop-in boundary for the reference's native entry points ("DGR/" =
 * sugar/gaussian_splatting/submodules/diff-gaussian-rasterization, "KNN/" = .../simple-knn of
 * haoyuhsu/autovfx):
 *
 *   gsr_forward       replaces  _C.rasterize_gaussians           DGR/rasterize_points.cu:35-119
 *                               (CudaRasterizer::Rasterizer::forward, DGR/cuda_rasterizer/rasterizer_impl.cu:197-339)
 *   gsr_backward      replaces  _C.rasterize_gaussians_backward  DGR/rasterize_points.cu:121-209
 *                               (Rasterizer::backward, rasterizer_impl.cu:343-446)
 *   gsr_mark_visible  replaces  _C.mark_visible                  DGR/rasterize_points.cu:211-230
 *   gsr_dist2         replaces  simple_knn._C.distCUDA2          KNN/spatial.cu:15-26 (SimpleKNN::knn, KNN/simple_knn.cu:185-220)
 *
 * and, for the render() wrapper around the two rasterizer passes ("GR/" = sugar/gaussian_splatting/gaussian_renderer/__init__.py):
 *
 *   gsr_forward_multi replaces  both rasterizer(...) calls of one frame           GR/:134-166 (same geometry, second colour set)
 *   gsr_backward_multi replaces the two rasterizer backward passes of that frame under autograd
 *   gsr_axis_normals  replaces  pc.get_normal(dir_pp_normalized) * 0.5 + 0.5      GR/:131-132,146-147; scene/gaussian_model.py:120-128
 *   gsr_normal_maps   replaces  normal normalisation + depth pseudo normal        GR/:168-191 (depth_pcd2normal GR/:23-38)
 *   gsr_pack_frame    replaces  the per-frame 8-bit conversions before encoding   scene_representation.py:424-438, sugar/render.py:18-22
 *   gsr_activate_gaussians replaces the activations of every render call and the per-frame object edit
 *                               get_scaling/get_rotation/get_opacity/get_features   sugar/gaussian_splatting/scene/gaussian_model.py:95-115
 *                               transform_gaussians + merge_two_gaussians            gaussians_utils.py:71-125, scene_representation.py:357-371
 *
 * Conventions (same as the reference's C++ layer):
 *   - every pointer is a DEVICE pointer to contiguous fp32 / int32 data unless it says "host";
 *   - a NULL pointer means "input absent" (the reference encodes None as an empty tensor whose
 *     data_ptr is null, DGR/diff_gaussian_rasterization/__init__.py:200-210);
 *   - no torch types; the caller owns every buffer, the library never allocates device memory;
 *   - `stream` is a cudaStream_t (the reference uses the legacy default stream; pass 0 for that);
 *   - functions return GSR_OK or a negative error code, gsr_last_error() gives the message;
 *     CUDA errors are only checked synchronously when frame->debug != 0 (reference: CHECK_CUDA,
 *     DGR/cuda_rasterizer/auxiliary.h:166-173).
 */
#ifndef GSR_B200_H_INCLUDED
#define GSR_B200_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSR_ABI_VERSION 4

enum {
    GSR_OK = 0,
    GSR_ERR_INVALID = -1,   /* bad argument combination / sizes                                   */
    GSR_ERR_WORKSPACE = -2, /* a workspace is smaller than the gsr_*_bytes() query                 */
    GSR_ERR_CUDA = -3,      /* CUDA runtime error (launch failure, or any error when debug is set) */
};

/* gsr_forward flags */
enum {
    GSR_FLAG_FOR_BACKWARD = 1, /* also keep cov3D, SH clamp flags and n_contrib for gsr_backward   */
    GSR_FLAG_SORTED_KEYS = 2,  /* also write the sorted 64-bit (tile<<32 | depth bits) keys (parity/debug) */
    GSR_FLAG_TIGHT_TILES = 4,  /* opt-in: emit a (Gaussian, tile) instance only if the splat can reach alpha >= 1/255 at a
                                  pixel of the tile; per-tile lists become a sub-sequence of the reference's, num_rendered and
                                  n_contrib shrink accordingly, color/depth/alpha/radii and all gradients are unchanged */
    GSR_FLAG_REUSE_GEOMETRY = 8, /* second pass of a frame: the workspaces still hold the projection + binning of the previous
                                  gsr_forward on the SAME geometry / camera / image size; only colors_precomp is re-read and the
                                  blend re-run.  `radii` must point to the radii written by that previous call (input). */
    GSR_FLAG_EXACT_IMAGES = 16, /* blend with the reference's own fp32 instruction sequence (expf, separate opacity multiply):
                                  color / depth / alpha are bit-identical to the reference's CUDA.  Default (flag clear): alpha =
                                  ex2.approx(power * log2e + log2(opacity)); every skip / termination decision that falls inside
                                  the approximation's error band is detected and that warp's pixels are re-blended exactly, so
                                  the images differ from the exact ones by ~1e-6 relative (requirement: 1e-4 max abs) and
                                  n_contrib / all integer outputs are unchanged. */
    GSR_FLAG_BINNING_ONLY = 32, /* first half of a frame issued in two calls: projection + tile scan only.  Afterwards the counters
                                  (num_rendered, overflow, max_tile, trapped, num_visible) are final, so a caller that validates the
                                  binning capacity on the host (the reference blocks on the same number, rasterizer_impl.cu:281-282)
                                  can start that copy now and let it overlap the rest of the frame. */
    GSR_FLAG_RESUME = 64,       /* second half: same arguments and workspaces as the GSR_FLAG_BINNING_ONLY call; runs colour +
                                  emission, the tile sort and the blend. */
};

/* One rasterizer invocation = the argument list of Rasterizer::forward (DGR/cuda_rasterizer/rasterizer.h:33-58). */
typedef struct gsr_frame {
    int32_t P;              /* number of Gaussians                                                 */
    int32_t D;              /* active SH degree (0..3; larger values are treated as 3, forward.cu:29-59) */
    int32_t M;              /* SH coefficients per channel in `shs` (stride), 0 if shs == NULL      */
    int32_t W, H;           /* image width / height                                               */
    float scale_modifier;
    float tanfovx, tanfovy;
    int32_t prefiltered;    /* !=0: a near-culled point is an error (reference __trap()s, auxiliary.h:156-160) */
    int32_t debug;          /* !=0: synchronise and check for CUDA errors after the call          */
    const float* bg;            /* [3]                                                            */
    const float* means3D;       /* [P,3]                                                          */
    const float* shs;           /* [P,M,3] coefficient-major, or NULL                             */
    const float* colors_precomp;/* [P,3] or NULL  (exactly one of shs / colors_precomp)            */
    const float* opacities;     /* [P]                                                            */
    const float* scales;        /* [P,3] or NULL                                                  */
    const float* rotations;     /* [P,4] (r,x,y,z), NOT normalised here, or NULL                  */
    const float* cov3D_precomp; /* [P,6] or NULL  (exactly one of scales+rotations / cov3D_precomp) */
    const float* viewmatrix;    /* [16] row-major torch buffer of the transposed W2C              */
    const float* projmatrix;    /* [16] view @ proj                                               */
    const float* campos;        /* [3]                                                            */
} gsr_frame;

/* Opaque workspaces, the analogue of the reference's geomBuffer / binningBuffer / imgBuffer
 * (rasterizer_impl.h:30-63).  They must stay untouched between gsr_forward and the matching
 * gsr_backward.  `binning` is sized by a CAPACITY in splat instances, not by the exact count: the
 * pipeline never reads the instance count back to the host (the reference's blocking cudaMemcpy,
 * rasterizer_impl.cu:281-282).  If the frame produces more instances than the capacity the frame is
 * incomplete, gsr_counters.overflow is set, and the caller re-runs with a larger binning workspace. */
typedef struct gsr_workspace {
    void* geom;    size_t geom_bytes;    /* >= gsr_geom_bytes(P)                                   */
    void* binning; size_t binning_bytes; /* >= gsr_binning_bytes(capacity), capacity >= 1          */
    void* image;   size_t image_bytes;   /* >= gsr_image_bytes(W, H)                               */
} gsr_workspace;

/* First bytes of the image workspace; copy them to the host (async) to learn the frame's statistics. */
typedef struct gsr_counters {
    uint32_t num_rendered; /* R = sum over Gaussians of tiles touched (what the reference returns)  */
    uint32_t overflow;     /* 1 if R > binning capacity: outputs are incomplete                    */
    uint32_t max_tile;     /* longest per-tile list                                               */
    uint32_t trapped;      /* 1 if prefiltered was set and a point was near-culled                 */
    uint32_t num_visible;  /* Gaussians with radii > 0                                             */
    uint32_t foot_total;   /* reserved (0)                                                          */
    uint32_t exact_redos;  /* warps whose pixels were re-blended exactly (default image mode)       */
    uint32_t blend_next;   /* work cursor of the persistent blend (gsr_set_option("blend_persist", K)); 0 otherwise          */
} gsr_counters;

size_t gsr_geom_bytes(int32_t P);
/* 13 bytes per instance of capacity (8-byte sort pair, 4-byte list entry, 1 byte of the footprint ballot matrix) + a fixed 4 MiB of
 * ballot rows (one 32-byte row per 32 list entries and one extra per tile: enough for 131,072 tiles; an image with more tiles needs
 * capacity >= 32 * (tiles - 131072)). */
size_t gsr_binning_bytes(size_t capacity_instances);
size_t gsr_image_bytes(int32_t W, int32_t H);
/* Largest capacity (in instances) a binning workspace of `bytes` bytes provides. */
size_t gsr_binning_capacity(size_t bytes);

/* Forward: projection (+ per-tile histogram) -> tile scan -> colour + key emission (+ footprint masks) -> per-tile depth sort
 * (+ footprint ballot matrix) -> blend (one warp per 8x4-pixel footprint).
 * Outputs: out_color [3,H,W], out_depth [1,H,W], out_alpha [1,H,W], radii [P] (int32).
 * All four are fully written (no pre-zeroing needed).  With P == 0 the images are zero-filled
 * (reference: rasterize_points.cu:68-71,82).  Asynchronous on `stream`. */
int gsr_forward(const gsr_frame* frame, const gsr_workspace* ws, float* out_color, float* out_depth,
                float* out_alpha, int32_t* radii, int flags, void* stream);

/* gsr_forward plus a second colour set blended with the SAME per-pixel weights: out_extra [3,H,W] is what a second
 * gsr_forward with colors_precomp = extra_colors ([P,3]) would write to out_color (bit for bit), at the cost of three
 * more accumulators in the blend instead of a second pass.  extra_colors == NULL && out_extra == NULL is gsr_forward.
 * With GSR_FLAG_REUSE_GEOMETRY, colors_precomp recolours the cached records and extra_colors is blended alongside. */
int gsr_forward_multi(const gsr_frame* frame, const gsr_workspace* ws, float* out_color, float* out_depth, float* out_alpha,
                      int32_t* radii, const float* extra_colors, float* out_extra, int flags, void* stream);

/* Per-Gaussian shading normal of the reference's GaussianModel.get_normal: the rotation-matrix column of the smallest
 * scale (ties: lowest index), flipped so that it faces the camera, normalised; remap01 != 0 stores normal*0.5+0.5.
 * out [P,3]. */
int gsr_axis_normals(int32_t P, const float* means3D, const float* scales, const float* rotations, const float* campos,
                     int remap01, float* out, void* stream);

/* normal_img [3,H,W] (a rendered normal*0.5+0.5 image) -> out_normal [H,W,3] = normalize((img - 0.5) * 2);
 * depth [H,W] -> out_pseudo [H,W,3] = normalised cross product of central differences of the unprojected depth map,
 * zero on the 1-pixel border.  c2w: DEVICE pointer to >= 12 floats, rows 0..2 of the 4x4 the reference calls c2w
 * (world_view_transform.inverse(), row-major); fx, fy, cx, cy as in GR/:180-184.  Either pair may be NULL. */
int gsr_normal_maps(int32_t W, int32_t H, const float* normal_img, const float* depth, const float* c2w, float fx, float fy,
                    float cx, float cy, float* out_normal, float* out_pseudo, void* stream);

/* 8-bit hand-off of a finished frame (any output may be NULL):
 *   rgba8   [H,W,4] = clamp(v*255+0.5, 0, 255) of rgb [3,H,W] and alpha [H,W] (alpha NULL -> 255)
 *   normal8 [H,W,3] = trunc((n+1)/2*255) of normal_hwc [H,W,3]
 *   depth8  [H,W]   = trunc(clip(depth/depth_scale, 0, 1)*255), the colormap index */
int gsr_pack_frame(int32_t W, int32_t H, const float* rgb, const float* alpha, const float* depth, const float* normal_hwc,
                   float depth_scale, uint8_t* rgba8, uint8_t* normal8, uint8_t* depth8, void* stream);

/* Rigid edit of one inserted object for one frame = the arguments of the reference's transform_gaussians(gaussians, center,
 * rotation, scaling, initial_center) (gaussians_utils.py:88-125), plus the two values its host code derives from them. */
typedef struct gsr_object_xform {
    float rotation[9];       /* R, row-major 3x3                                                       */
    float quat[4];           /* matrix_to_quaternion(R), (w,x,y,z) (rotation_utils.py:24-84)           */
    float center[3];         /* target position of the pivot                                          */
    float initial_center[3]; /* the pivot: centre of the object's mesh                                 */
    float scaling;           /* uniform scale                                                          */
    float log_scaling;       /* (float)log(scaling), added to the log-scales                           */
} gsr_object_xform;

/* RAW parameters (the reference's GaussianModel fields: _xyz [N,3], _features_dc [N,1,3], _features_rest [N,M-1,3],
 * _opacity [N], _scaling [N,3], _rotation [N,4]) -> the ACTIVATED tensors the rasterizer takes: means3D [N,3],
 * shs [N,M,3] = cat(dc, rest), opacities [N] = sigmoid, scales [N,3] = exp, rotations [N,4] = normalize.
 * xform (HOST pointer, may be NULL) applies transform_gaussians first: scale about the pivot, rotate, translate,
 * compose the quaternions, shift the log-scales.  The output pointers may address a sub-range of larger arrays
 * (the tail of a resident scene): this replaces merge_two_gaussians' concatenation.  M >= 1. */
int gsr_activate_gaussians(int32_t N, int32_t M, const float* xyz, const float* f_dc, const float* f_rest, const float* opacity_raw,
                           const float* scaling_raw, const float* rotation_raw, const gsr_object_xform* xform, float* means3D,
                           float* shs, float* opacities, float* scales, float* rotations, void* stream);

/* Gradient buffers, all caller-allocated; the library zero-fills what it accumulates into (the
 * reference's torch::zeros, rasterize_points.cu:158-168).  dL_dsh may be NULL when shs is NULL,
 * dL_dscales / dL_drotations may be NULL when scales is NULL. */
typedef struct gsr_grads {
    float* dL_dmeans2D;   /* [P,3]  (x,y in NDC-scaled units, z = 0), returned to Python            */
    float* dL_dconic;     /* [P,4]  scratch (slots 0,1,3)                                          */
    float* dL_dopacity;   /* [P]                                                                   */
    float* dL_dcolors;    /* [P,3]  = grad of colors_precomp, or scratch for the SH backward        */
    float* dL_ddepths;    /* [P]    scratch                                                        */
    float* dL_dmeans3D;   /* [P,3]                                                                 */
    float* dL_dcov3D;     /* [P,6]                                                                 */
    float* dL_dsh;        /* [P,M,3] or NULL                                                       */
    float* dL_dscales;    /* [P,3] or NULL                                                         */
    float* dL_drotations; /* [P,4] or NULL                                                         */
} gsr_grads;

/* Backward of the frame last run through gsr_forward(..., GSR_FLAG_FOR_BACKWARD) on `ws`.
 * out_alpha is the forward's alpha image; dL_dout_* are the three image gradients
 * ([3,H,W], [1,H,W], [1,H,W]); radii is the forward's radii output. */
int gsr_backward(const gsr_frame* frame, const gsr_workspace* ws, const int32_t* radii, const float* out_alpha,
                 const float* dL_dout_color, const float* dL_dout_depth, const float* dL_dout_alpha,
                 const gsr_grads* grads, void* stream);

/* Backward of a gsr_forward_multi(..., extra_colors, out_extra, GSR_FLAG_FOR_BACKWARD) frame on `ws`, called with the same
 * extra_colors [P,3].  dL_dout_extra [3,H,W] is the gradient of out_extra; the blend backward folds it into the same single
 * pass, so every gradient in `grads` is the sum of what two gsr_backward calls would return (one for the colour image, one for
 * a colors_precomp = extra_colors frame with zero depth and alpha gradients), up to summation order.  dL_dextra_colors [P,3]
 * receives the gradient of extra_colors and is zero-filled by the library.  extra_colors == dL_dout_extra ==
 * dL_dextra_colors == NULL is gsr_backward; a partial set returns GSR_ERR_INVALID. */
int gsr_backward_multi(const gsr_frame* frame, const gsr_workspace* ws, const int32_t* radii, const float* out_alpha,
                       const float* dL_dout_color, const float* dL_dout_depth, const float* dL_dout_alpha, const float* extra_colors,
                       const float* dL_dout_extra, const gsr_grads* grads, float* dL_dextra_colors, void* stream);

/* present[i] = (view-space z of means3D[i] > 0.2)  — checkFrustum, rasterizer_impl.cu:54-66. */
int gsr_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix,
                     uint8_t* present, void* stream);

/* Mean squared distance to the 3 nearest neighbours.  `workspace` needs gsr_dist2_bytes(P) bytes. */
size_t gsr_dist2_bytes(int32_t P);
int gsr_dist2(int32_t P, const float* points, float* mean_dists, void* workspace, size_t workspace_bytes,
              void* stream);

/* Device pointers into the workspaces of the last layout (P, capacity, W, H) — for parity tests that
 * compare per-stage buffers with the reference (SURVEY §4).  Pure pointer arithmetic, no CUDA calls. */
typedef struct gsr_views {
    const float* records;        /* [P,12]: x, y, conic_a, conic_b | conic_c, opacity, depth, radius (int bits) | r, g, b, log2 opacity */
    const float* cov3D;          /* [P,6]  (GSR_FLAG_FOR_BACKWARD only)                             */
    const uint8_t* clamped;      /* [P]    bit c set = channel c clamped (GSR_FLAG_FOR_BACKWARD only) */
    const uint32_t* point_list;  /* [capacity] Gaussian ids, per tile front-to-back                 */
    const uint64_t* sorted_keys; /* [capacity] (GSR_FLAG_SORTED_KEYS only)                          */
    const uint32_t* ranges;      /* [tiles,2]                                                       */
    const uint32_t* n_contrib;   /* [H,W]  (GSR_FLAG_FOR_BACKWARD only)                             */
    const uint32_t* tile_count;  /* [tiles] instances of Gaussians touching <= 8 tiles                   */
    const uint32_t* tile_big;    /* [tiles] instances of Gaussians touching > 8 tiles                    */
    const gsr_counters* counters;
} gsr_views;
int gsr_get_views(const gsr_workspace* ws, int32_t P, int32_t W, int32_t H, gsr_views* out);

/* Per-kernel device timing of gsr_forward (CUDA events on the launching stream), for roofline reports.
 * ms_per_kernel[5] = average ms of {preprocess, tile_scan, emit, sort_tiles, blend} over the profiled frames. */
int gsr_profile_begin(int max_frames);
/* Same, timing only every stride-th gsr_forward call (the six event records per timed frame cost about 1.5 % of a 0.9 ms frame). */
int gsr_profile_begin_strided(int max_frames, int stride);
int gsr_profile_end(float* ms_per_kernel, int* frames);

/* Process-wide tuning options (not part of the reference's surface; defaults are what bench.py measures unless it says so):
 *   "blend_persist" = K   0: one CTA per half tile (default).  K in 1..16: the blend runs as a persistent kernel with K CTAs per SM
 *                         drawing work from gsr_counters.blend_next, so that it never holds more than 4 K warps of an SM and the
 *                         geometry kernels of the next frame, issued on another stream, run beside it.
 *   "sort_single_pass" = 0|1   1 (default): the per-tile sort reads a tile of <= 2048 instances from global memory once. */
int gsr_set_option(const char* name, int value);

const char* gsr_last_error(void);
int gsr_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GSR_B200_H_INCLUDED */
