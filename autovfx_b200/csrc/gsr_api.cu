// gsr_b200 — extern "C" surface declared in include/gsr_b200.h.
#include "gsr_common.cuh"
#include <cstring>
#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: the ranges cost nothing unless a profiler is attached

namespace {
struct NvtxRange {  // one named range per C-ABI call (SURVEY §5: the reference has no instrumentation; this build adds NVTX)
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
}  // namespace

namespace gsr {
int forward_impl(const gsr_frame* f, const gsr_workspace* ws, float* out_color, float* out_depth, float* out_alpha,
                 int32_t* radii, const float* extra_colors, float* out_extra, int flags, cudaStream_t st);
int axis_normals_impl(int P, const float* means3D, const float* scales, const float* rotations, const float* campos, int remap01,
                      float* out, cudaStream_t st);
int normal_maps_impl(int W, int H, const float* normal_img, const float* depth, const float* c2w, float fx, float fy, float cx, float cy,
                     float* out_normal, float* out_pseudo, cudaStream_t st);
int pack_frame_impl(int W, int H, const float* rgb, const float* alpha, const float* depth, const float* normal_hwc, float depth_scale,
                    uint8_t* rgba8, uint8_t* normal8, uint8_t* depth8, cudaStream_t st);
int backward_impl(const gsr_frame* f, const gsr_workspace* ws, const int32_t* radii, const float* out_alpha, const float* dL_dc,
                  const float* dL_dd, const float* dL_da, const float* extra, const float* dL_de, float* dL_dextra, const gsr_grads* g,
                  cudaStream_t st);
int compose_impl(int N, int M, const float* xyz, const float* f_dc, const float* f_rest, const float* opacity_raw, const float* scaling_raw,
                 const float* rotation_raw, const gsr_object_xform* xform, float* means3D, float* shs, float* opacities, float* scales,
                 float* rotations, cudaStream_t st);
int dist2_impl(int P, const float* points, float* out, void* ws, size_t ws_bytes, cudaStream_t st);
size_t dist2_bytes(int P);
int profile_begin(int max_frames, int stride);
int set_option(const char* name, int value);
int profile_end(float* ms, int* frames);

// checkFrustum (rasterizer_impl.cu:54-66): in_frustum() only tests view-space z (auxiliary.h:154)
__global__ void k_mark_visible(int P, const float* __restrict__ means3D, const float* __restrict__ view, uint8_t* __restrict__ present) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P) return;
    const float3 p = {means3D[3 * (size_t)idx], means3D[3 * (size_t)idx + 1], means3D[3 * (size_t)idx + 2]};
    const float3 pv = xform4x3(p, view);
    present[idx] = !(pv.z <= 0.2f);
}
}  // namespace gsr

extern "C" {

int gsr_abi_version(void) { return GSR_ABI_VERSION; }
const char* gsr_last_error(void) { return gsr::last_error(); }

size_t gsr_geom_bytes(int32_t P) { return gsr::GeomLayout((size_t)(P < 0 ? 0 : P)).total; }
size_t gsr_binning_bytes(size_t capacity) { return gsr::BinLayout(capacity < 1 ? 1 : capacity).total; }
size_t gsr_binning_capacity(size_t bytes) { return gsr::BinLayout::capacity_of(bytes); }
size_t gsr_image_bytes(int32_t W, int32_t H) { return gsr::ImageLayout(W < 1 ? 1 : W, H < 1 ? 1 : H).total; }

int gsr_forward(const gsr_frame* frame, const gsr_workspace* ws, float* out_color, float* out_depth, float* out_alpha,
                int32_t* radii, int flags, void* stream) {
    NvtxRange nvtx_("gsr_forward");
    return gsr::forward_impl(frame, ws, out_color, out_depth, out_alpha, radii, nullptr, nullptr, flags, (cudaStream_t)stream);
}

int gsr_forward_multi(const gsr_frame* frame, const gsr_workspace* ws, float* out_color, float* out_depth, float* out_alpha,
                      int32_t* radii, const float* extra_colors, float* out_extra, int flags, void* stream) {
    NvtxRange nvtx_("gsr_forward_multi");
    return gsr::forward_impl(frame, ws, out_color, out_depth, out_alpha, radii, extra_colors, out_extra, flags, (cudaStream_t)stream);
}

int gsr_axis_normals(int32_t P, const float* means3D, const float* scales, const float* rotations, const float* campos, int remap01,
                     float* out, void* stream) {
    NvtxRange nvtx_("gsr_axis_normals");
    return gsr::axis_normals_impl(P, means3D, scales, rotations, campos, remap01, out, (cudaStream_t)stream);
}

int gsr_normal_maps(int32_t W, int32_t H, const float* normal_img, const float* depth, const float* c2w, float fx, float fy, float cx,
                    float cy, float* out_normal, float* out_pseudo, void* stream) {
    NvtxRange nvtx_("gsr_normal_maps");
    return gsr::normal_maps_impl(W, H, normal_img, depth, c2w, fx, fy, cx, cy, out_normal, out_pseudo, (cudaStream_t)stream);
}

int gsr_pack_frame(int32_t W, int32_t H, const float* rgb, const float* alpha, const float* depth, const float* normal_hwc,
                   float depth_scale, uint8_t* rgba8, uint8_t* normal8, uint8_t* depth8, void* stream) {
    NvtxRange nvtx_("gsr_pack_frame");
    return gsr::pack_frame_impl(W, H, rgb, alpha, depth, normal_hwc, depth_scale, rgba8, normal8, depth8, (cudaStream_t)stream);
}

int gsr_activate_gaussians(int32_t N, int32_t M, const float* xyz, const float* f_dc, const float* f_rest, const float* opacity_raw,
                           const float* scaling_raw, const float* rotation_raw, const gsr_object_xform* xform, float* means3D, float* shs,
                           float* opacities, float* scales, float* rotations, void* stream) {
    NvtxRange nvtx_("gsr_activate_gaussians");
    return gsr::compose_impl(N, M, xyz, f_dc, f_rest, opacity_raw, scaling_raw, rotation_raw, xform, means3D, shs, opacities, scales, rotations,
                             (cudaStream_t)stream);
}

int gsr_backward(const gsr_frame* frame, const gsr_workspace* ws, const int32_t* radii, const float* out_alpha,
                 const float* dL_dout_color, const float* dL_dout_depth, const float* dL_dout_alpha, const gsr_grads* grads,
                 void* stream) {
    NvtxRange nvtx_("gsr_backward");
    return gsr::backward_impl(frame, ws, radii, out_alpha, dL_dout_color, dL_dout_depth, dL_dout_alpha, nullptr, nullptr, nullptr, grads,
                              (cudaStream_t)stream);
}

int gsr_backward_multi(const gsr_frame* frame, const gsr_workspace* ws, const int32_t* radii, const float* out_alpha,
                       const float* dL_dout_color, const float* dL_dout_depth, const float* dL_dout_alpha, const float* extra_colors,
                       const float* dL_dout_extra, const gsr_grads* grads, float* dL_dextra_colors, void* stream) {
    NvtxRange nvtx_("gsr_backward_multi");
    return gsr::backward_impl(frame, ws, radii, out_alpha, dL_dout_color, dL_dout_depth, dL_dout_alpha, extra_colors, dL_dout_extra,
                              dL_dextra_colors, grads, (cudaStream_t)stream);
}

int gsr_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* projmatrix, uint8_t* present,
                     void* stream) {
    (void)projmatrix;
    if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !present))) { gsr::set_error("gsr_mark_visible: bad arguments"); return GSR_ERR_INVALID; }
    if (P == 0) return GSR_OK;
    gsr::k_mark_visible<<<(P + 255) / 256, 256, 0, (cudaStream_t)stream>>>(P, means3D, viewmatrix, present);
    return gsr::check_launch("gsr_mark_visible", false, (cudaStream_t)stream);
}

size_t gsr_dist2_bytes(int32_t P) { return gsr::dist2_bytes(P); }
int gsr_dist2(int32_t P, const float* points, float* mean_dists, void* workspace, size_t workspace_bytes, void* stream) {
    NvtxRange nvtx_("gsr_dist2");
    return gsr::dist2_impl(P, points, mean_dists, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gsr_profile_begin(int max_frames) { return gsr::profile_begin(max_frames, 1); }
int gsr_profile_begin_strided(int max_frames, int stride) { return gsr::profile_begin(max_frames, stride); }
int gsr_profile_end(float* ms_per_kernel, int* frames) { return gsr::profile_end(ms_per_kernel, frames); }

int gsr_set_option(const char* name, int value) {
    if (!name) { gsr::set_error("gsr_set_option: null name"); return GSR_ERR_INVALID; }
    const int rc = gsr::set_option(name, value);
    if (rc != GSR_OK) gsr::set_error("gsr_set_option: unknown option or bad value (%s = %d)", name, value);
    return rc;
}

int gsr_get_views(const gsr_workspace* ws, int32_t P, int32_t W, int32_t H, gsr_views* out) {
    if (!ws || !out) { gsr::set_error("gsr_get_views: null argument"); return GSR_ERR_INVALID; }
    const gsr::GeomLayout gl((size_t)P);
    const gsr::ImageLayout il(W, H);
    const gsr::BinLayout bl(gsr::BinLayout::capacity_of(ws->binning_bytes));
    const char* geo = (const char*)ws->geom; const char* img = (const char*)ws->image; const char* bin = (const char*)ws->binning;
    out->records = (const float*)(geo + gl.records);
    out->cov3D = (const float*)(geo + gl.cov3D);
    out->clamped = (const uint8_t*)(geo + gl.clamped);
    out->point_list = (const uint32_t*)(bin + bl.point_list);
    out->sorted_keys = (const uint64_t*)(bin + bl.pairs);
    out->ranges = (const uint32_t*)(img + il.ranges);
    out->n_contrib = (const uint32_t*)(img + il.n_contrib);
    out->tile_count = (const uint32_t*)(img + il.tile_count);
    out->tile_big = (const uint32_t*)(img + il.tile_big);
    out->counters = (const gsr_counters*)(img + il.counters);
    return GSR_OK;
}

}  // extern "C"
