"""``render()`` — the per-frame wrapper around the rasterizer, mirror of the reference's
``sugar/gaussian_splatting/gaussian_renderer/__init__.py:83-218`` ("GR/"; the SuGaR variant ``sugar_scene/sugar_model.py:
1956-2228`` has the same two-pass structure).

The reference renders every camera twice with identical geometry (SH colours, then ``colors_precomp`` = per-Gaussian
normals), and surrounds the two passes with ~25 elementwise torch launches over P Gaussians and over H·W pixels
(direction normalisation, ``get_normal``, remaps, ``F.normalize``, meshgrid, ray directions, a 3x3 matmul per pixel, the
central-difference stencil).  Here, under ``torch.no_grad()`` (the frame loop of ``scene_representation.py:355-438``), one
frame is

    gsr_axis_normals -> gsr_forward_multi (ONE projection/binning/sort/blend pass, 6 colour channels) -> gsr_normal_maps

When gradients are required (training) one frame is ONE autograd rasterizer call, ``rasterize_gaussians_multi``: one
projection/binning/sort/blend forward for the SH colours and the normal colours, one blend backward for both images
(gsr_backward_multi) and one per-Gaussian backward on the summed contributions.  The per-Gaussian normals
(``pc.get_normal(dir_pp_normalized) * 0.5 + 0.5``), the normal-image normalisation and the pseudo-normal stencil stay torch ops
of the caller's graph, as in the reference, so the gradient reaches rotations and scales through ``get_normal``.  ``render``,
``depth`` and ``radii`` are bit-identical to the reference's two-pass structure; gradients differ only in summation order.
``set_fused_training(False)`` restores the two-call graph (for A/B comparisons).

Same argument names, return keys and error behaviour as the reference function.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import lib as _L
from . import rasterizer as R
from .rasterizer import GaussianRasterizationSettings, GaussianRasterizer

__all__ = ["render", "axis_normals", "normal_maps", "pack_frame", "fov2focal", "TURBO_LUT_BGR", "set_fused_training",
           "get_fused_training"]

_FUSED_TRAINING = True


def set_fused_training(on: bool) -> None:
    """Default on: under autograd ``render()`` rasterizes the colour and normal images in one ``rasterize_gaussians_multi`` call
    (one forward and one backward pass).  Off: two ``GaussianRasterizer`` calls, the reference's graph."""
    global _FUSED_TRAINING
    _FUSED_TRAINING = bool(on)


def get_fused_training() -> bool:
    return _FUSED_TRAINING


def fov2focal(fov: float, pixels: float) -> float:
    """utils/graphics_utils.py:74-75."""
    return pixels / (2 * math.tan(fov / 2))


def _stream(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _f32c(t: torch.Tensor, device) -> torch.Tensor:
    if t.device != device:
        t = t.to(device, non_blocking=True)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ------------------------------------------------------------------------------------------ the three post kernels
def axis_normals(means3D: torch.Tensor, scales: torch.Tensor, rotations: torch.Tensor, campos: torch.Tensor, remap01: bool = False,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``GaussianModel.get_normal(dir_pp_normalized)`` (scene/gaussian_model.py:120-128) for every Gaussian: the axis of
    the smallest scale, flipped towards ``campos``, unit length; ``remap01`` additionally applies ``*0.5+0.5`` (GR/:147).
    [P,3] float32 on the device of ``means3D``.  Forward only."""
    if not means3D.is_cuda:
        raise RuntimeError("autovfx_b200.renderer: CUDA tensors required (there is no CPU path)")
    device = means3D.device
    with torch.cuda.device(device):
        m, s, r, c = _f32c(means3D.detach(), device), _f32c(scales.detach(), device), _f32c(rotations.detach(), device), _f32c(campos.detach(), device)
        P = m.shape[0]
        if s.shape != (P, 3) or r.shape != (P, 4) or c.numel() != 3:
            raise ValueError("axis_normals: expected scales [P,3], rotations [P,4], campos [3]")
        if out is None:
            out = torch.empty((P, 3), dtype=torch.float32, device=device)
        rc = _L.gsr_axis_normals(P, m.data_ptr() if P else None, s.data_ptr() if P else None, r.data_ptr() if P else None, c.data_ptr(),
                                 int(bool(remap01)), out.data_ptr() if P else None, _stream(device))
        _lib.check(rc, "gsr_axis_normals")
    return out


def normal_maps(normal_img: Optional[torch.Tensor], depth: Optional[torch.Tensor], c2w: Optional[torch.Tensor], fx: float, fy: float,
                cx: float, cy: float, out: Optional[Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]] = None
                ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(normal [H,W,3], pseudo_normal [H,W,3]) from the rendered ``normal*0.5+0.5`` image [3,H,W] and the depth map [H,W]
    (GR/:168-191).  ``c2w`` is the 4x4 the reference calls c2w (``world_view_transform.inverse()``)."""
    src = normal_img if normal_img is not None else depth
    if src is None:
        return None, None
    device = src.device
    with torch.cuda.device(device):
        out_n = out_p = None
        H, W = src.shape[-2], src.shape[-1]
        if normal_img is not None:
            normal_img = _f32c(normal_img, device)
            out_n = out[0] if out is not None and out[0] is not None else torch.empty((H, W, 3), dtype=torch.float32, device=device)
        if depth is not None:
            depth = _f32c(depth, device)
            c2w = _f32c(c2w, device)
            if c2w.numel() < 12:
                raise ValueError("normal_maps: c2w must hold at least 3x4 floats")
            out_p = out[1] if out is not None and out[1] is not None else torch.empty((H, W, 3), dtype=torch.float32, device=device)
        rc = _L.gsr_normal_maps(W, H, R._ptr(normal_img), R._ptr(depth), R._ptr(c2w) if depth is not None else None, fx, fy, cx, cy,
                                R._ptr(out_n), R._ptr(out_p), _stream(device))
        _lib.check(rc, "gsr_normal_maps")
    return out_n, out_p


def pack_frame(rgb: Optional[torch.Tensor] = None, alpha: Optional[torch.Tensor] = None, depth: Optional[torch.Tensor] = None,
               normal_hwc: Optional[torch.Tensor] = None, depth_scale: float = 3.0, out: Optional[Dict[str, torch.Tensor]] = None
               ) -> Dict[str, torch.Tensor]:
    """8-bit images of a finished frame, exactly the bytes the reference's frame loop hands to its encoders
    (scene_representation.py:424-438): ``rgba8`` [H,W,4] (torchvision ``save_image`` rounding of cat(rgb, alpha)),
    ``normal8`` [H,W,3] (RGB order; the reference swaps to BGR only for cv2.imwrite) and ``depth8`` [H,W], the index of
    ``depth2img``'s TURBO colormap (``TURBO_LUT_BGR[depth8]`` is the image cv2.applyColorMap returns)."""
    src = rgb if rgb is not None else (depth if depth is not None else normal_hwc)
    if src is None:
        return {}
    device = src.device
    res: Dict[str, torch.Tensor] = {}
    with torch.cuda.device(device):
        if rgb is not None:
            H, W = rgb.shape[-2], rgb.shape[-1]
        elif depth is not None:
            H, W = depth.shape[-2], depth.shape[-1]
        else:
            H, W = normal_hwc.shape[0], normal_hwc.shape[1]
        rgb = _f32c(rgb, device) if rgb is not None else None
        alpha = _f32c(alpha, device) if alpha is not None else None
        depth = _f32c(depth, device) if depth is not None else None
        normal_hwc = _f32c(normal_hwc, device) if normal_hwc is not None else None

        def buf(name, shape):
            if out is not None and name in out:
                return out[name]
            return torch.empty(shape, dtype=torch.uint8, device=device)
        if rgb is not None:
            res["rgba8"] = buf("rgba8", (H, W, 4))
        if normal_hwc is not None:
            res["normal8"] = buf("normal8", (H, W, 3))
        if depth is not None:
            res["depth8"] = buf("depth8", (H, W))
        rc = _L.gsr_pack_frame(W, H, R._ptr(rgb), R._ptr(alpha), R._ptr(depth), R._ptr(normal_hwc), float(depth_scale),
                               R._ptr(res.get("rgba8")), R._ptr(res.get("normal8")), R._ptr(res.get("depth8")), _stream(device))
        _lib.check(rc, "gsr_pack_frame")
    return res


# 256x3 uint8 (B,G,R): the table cv2.applyColorMap(..., cv2.COLORMAP_TURBO) applies (depth2img, sugar/render.py:18-22),
# generated by tools/make_turbo_lut.py from OpenCV 4.13 so that the hand-off does not need cv2 on the render box.
_TURBO_HEX = (
    "3b12304315324a1833511b34581e355f21366624376d2738732a39792d3a802f3b86323c8b353d91383e973b3f9c3e3fa24040a74341ac4641b14942"
    "b54b42ba4e43bf5144c35444c75644cb5945cf5c45d35e45d66146da6446dd6646e06946e36b46e66e47e97147eb7347ee7647f07847f27b47f47d46"
    "f68046f88246fa8546fb8746fc8a45fd8c45fe8f44fe9143ff9442ff9641ff9940fe9b3efe9e3dfda03bfca33afba538faa837f8ab35f7ad33f5af31"
    "f4b22ff2b42ef0b72ceeb92aebbc28e9be27e7c025e4c323e2c522dfc720ddc91fdacb1ed8cd1cd5d01bd2d21ad0d41acdd519cad718c8d918c5db18"
    "c2dd18c0de18bde018bbe219b9e319b6e41ab4e61cb2e71dafe91facea20aaeb22a7ec25a4ee27a1ef2a9ef02c9bf12f98f23294f33591f4388ef53c"
    "8af63f87f74384f84680f84a7df94e7afa5276fa5573fb596ffc5d6cfc6169fd6566fd6962fe6d5ffe715cfe7559fe7956ff7d53ff8051ff844eff88"
    "4bff8b49ff8f47ff9244fe9642fe9940fe9c3ffd9f3dfda13cfca43afca739fba938fbac37faaf36f9b136f8b435f7b735f6b934f5bc34f4be34f3c1"
    "34f1c334f0c634efc834edcb34eccd34ead035e9d235e7d435e5d736e4d936e2db37e0dd37dfdf37dde138dbe338d9e539d7e739d5e939d3eb3ad1ec"
    "3acfee3acdef3acbf13ac9f23ac7f43ac5f53ac3f63ac1f739bef839bcf939bafa38b8fb37b6fb36b3fc36b1fc35aefd34acfd33a9fe32a7fe31a4fe"
    "30a1fe2f9efe2d9bfe2c99fe2b96fe2a93fe2990fe278dfd268afd2587fc2384fc2281fb217efb1f7bfa1e78f91d75f91c72f81a6ff7196cf61869f5"
    "1766f41563f31460f2135df1125bf01158ef1055ed0f53ec0e50eb0d4eea0c4be80c49e70b47e50a45e40a43e20941e1083fdf083ddd073bdc0739da"
    "0637d80635d60533d40531d2052fd0042dce042bcc042aca0328c80326c50325c30223c10221be0220bc021eb9021db7011bb4011ab20118af0117ac"
    "0116a90114a70113a40112a101109e010f9b010e98010d95010b92010a8e02098b02088802078502068102057e03047a"
)
TURBO_LUT_BGR = torch.frombuffer(bytearray(bytes.fromhex(_TURBO_HEX)), dtype=torch.uint8).reshape(256, 3).clone()


# ------------------------------------------------------------------------------------------ SH -> RGB in Python (pipe.convert_SHs_python)
def _eval_sh_torch(deg: int, sh: torch.Tensor, dirs: torch.Tensor) -> torch.Tensor:
    """Real spherical harmonics up to degree 3, sh [...,3,(max_deg+1)^2], dirs [...,3] unit -> [...,3]
    (same basis and sign convention as utils/sh_utils.py:57-112 and DGR/cuda_rasterizer/forward.cu:20-71)."""
    x, y, z = dirs[..., 0:1], dirs[..., 1:2], dirs[..., 2:3]
    basis = [torch.full_like(x, 0.28209479177387814)]
    if deg > 0:
        c1 = 0.4886025119029199
        basis += [-c1 * y, c1 * z, -c1 * x]
    if deg > 1:
        xx, yy, zz, xy, yz, xz = x * x, y * y, z * z, x * y, y * z, x * z
        basis += [1.0925484305920792 * xy, -1.0925484305920792 * yz, 0.31539156525252005 * (2.0 * zz - xx - yy),
                  -1.0925484305920792 * xz, 0.5462742152960396 * (xx - yy)]
        if deg > 2:
            basis += [-0.5900435899266435 * y * (3 * xx - yy), 2.890611442640554 * xy * z, -0.4570457994644658 * y * (4 * zz - xx - yy),
                      0.3731763325901154 * z * (2 * zz - 3 * xx - 3 * yy), -0.4570457994644658 * x * (4 * zz - xx - yy),
                      1.445305721320277 * z * (xx - yy), -0.5900435899266435 * x * (xx - 3 * yy)]
    B = torch.cat(basis, dim=-1)  # [..., n]
    return (sh[..., : B.shape[-1]] * B.unsqueeze(-2)).sum(-1)


# ------------------------------------------------------------------------------------------ render()
def _depth_pcd2normal(xyz: torch.Tensor) -> torch.Tensor:
    """Differentiable torch form of GR/:23-38 (used only when gradients are required)."""
    hd, wd, _ = xyz.shape
    l2r = xyz[1:hd - 1, 2:wd, :] - xyz[1:hd - 1, 0:wd - 2, :]
    b2t = xyz[0:hd - 2, 1:wd - 1, :] - xyz[2:hd, 1:wd - 1, :]
    n = torch.nn.functional.normalize(torch.cross(l2r, b2t, dim=-1), p=2, dim=-1)
    return torch.nn.functional.pad(n.permute(2, 0, 1), (1, 1, 1, 1), mode="constant").permute(1, 2, 0)


def render(viewpoint_camera, pc, pipe, bg_color: torch.Tensor, scaling_modifier: float = 1.0, override_color=None):
    """Render the scene.  Background tensor (bg_color) must be on GPU!  (GR/:83-218)

    viewpoint_camera: FoVx, FoVy, image_height, image_width, world_view_transform, full_proj_transform, camera_center.
    pc: get_xyz, get_opacity, get_scaling, get_rotation, get_features, active_sh_degree, max_sh_degree,
        get_covariance(scaling_modifier), get_normal(dir_pp_normalized=...).
    pipe: debug, compute_cov3D_python, convert_SHs_python.
    Returns {"render" [4,H,W] (rgb|alpha), "depth" [H,W], "normal" [H,W,3], "pseudo_normal" [H,W,3], "viewspace_points",
    "visibility_filter", "radii"}."""
    xyz = pc.get_xyz
    device = xyz.device
    grad_mode = torch.is_grad_enabled() and any(
        isinstance(t, torch.Tensor) and t.requires_grad
        for t in (xyz, pc.get_opacity, pc.get_scaling, pc.get_rotation, pc.get_features, override_color))

    # zero tensor whose gradient is the screen-space positional gradient (densification statistics, GR/:90-95)
    screenspace_points = torch.zeros_like(xyz, dtype=xyz.dtype, requires_grad=True, device=device) + 0
    try:
        screenspace_points.retain_grad()
    except Exception:  # noqa: BLE001
        pass

    tanfovx = math.tan(viewpoint_camera.FoVx * 0.5)
    tanfovy = math.tan(viewpoint_camera.FoVy * 0.5)
    H, W = int(viewpoint_camera.image_height), int(viewpoint_camera.image_width)
    raster_settings = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=tanfovx, tanfovy=tanfovy, bg=bg_color, scale_modifier=scaling_modifier,
        viewmatrix=viewpoint_camera.world_view_transform, projmatrix=viewpoint_camera.full_proj_transform,
        sh_degree=pc.active_sh_degree, campos=viewpoint_camera.camera_center, prefiltered=False, debug=pipe.debug)

    means3D, means2D, opacity = xyz, screenspace_points, pc.get_opacity
    scales = rotations = cov3D_precomp = None
    if pipe.compute_cov3D_python:
        cov3D_precomp = pc.get_covariance(scaling_modifier)
    else:
        scales, rotations = pc.get_scaling, pc.get_rotation

    shs = colors_precomp = None
    dir_pp_normalized = None
    if override_color is None:
        if pipe.convert_SHs_python:
            dir_pp = xyz - viewpoint_camera.camera_center.repeat(pc.get_features.shape[0], 1)
            dir_pp_normalized = dir_pp / dir_pp.norm(dim=1, keepdim=True)
            shs_view = pc.get_features.transpose(1, 2).view(-1, 3, (pc.max_sh_degree + 1) ** 2)
            colors_precomp = torch.clamp_min(_eval_sh_torch(pc.active_sh_degree, shs_view, dir_pp_normalized) + 0.5, 0.0)
        else:
            shs = pc.get_features
    else:
        colors_precomp = override_color

    fx, fy = fov2focal(viewpoint_camera.FoVx, W), fov2focal(viewpoint_camera.FoVy, H)
    cx, cy = W / 2, H / 2

    if not grad_mode:
        # ---- one pass: normals kernel -> 6-channel forward -> normal maps
        with torch.no_grad(), torch.cuda.device(device):
            normal_normed = axis_normals(xyz, pc.get_scaling, pc.get_rotation, viewpoint_camera.camera_center, remap01=True)
            frame = torch.empty((5, H, W), dtype=torch.float32, device=device)  # rgb | alpha | depth: "render" = frame[0:4] without a cat
            radii = torch.empty((xyz.shape[0],), dtype=torch.int32, device=device)
            _c, _d, _a, normal_img, radii, _ticket = R.forward_multi(
                means3D, shs, colors_precomp, normal_normed, opacity, scales, rotations, cov3D_precomp, raster_settings,
                out=(frame[0:3], frame[4:5], frame[3:4], radii))
            c2w = torch.linalg.inv_ex(viewpoint_camera.world_view_transform.float())[0]  # no error-check sync; GR/:185
            normal_image, pseudo_normal = normal_maps(normal_img, frame[4], c2w, fx, fy, cx, cy)
        return {"render": frame[0:4], "depth": frame[4], "normal": normal_image, "pseudo_normal": pseudo_normal,
                "viewspace_points": screenspace_points, "visibility_filter": radii > 0, "radii": radii}

    # ---- gradients required: the reference's graph with its two rasterizer calls merged into one (set_fused_training)
    if dir_pp_normalized is None:
        dir_pp = xyz - viewpoint_camera.camera_center.repeat(pc.get_features.shape[0], 1)
        dir_pp_normalized = dir_pp / dir_pp.norm(dim=1, keepdim=True)
    if _FUSED_TRAINING:
        normal_normed = pc.get_normal(dir_pp_normalized=dir_pp_normalized) * 0.5 + 0.5
        rendered_image, depth_image, alpha_image, normal_image, radii = R.rasterize_gaussians_multi(
            means3D, means2D, shs, colors_precomp, normal_normed, opacity, scales, rotations, cov3D_precomp, raster_settings)
        rendered_image = torch.cat((rendered_image, alpha_image), dim=0)
        depth_image = depth_image.squeeze(0)
    else:
        rasterizer = GaussianRasterizer(raster_settings=raster_settings)
        rendered_image, depth_image, alpha_image, radii = rasterizer(
            means3D=means3D, means2D=means2D, shs=shs, colors_precomp=colors_precomp, opacities=opacity, scales=scales, rotations=rotations,
            cov3D_precomp=cov3D_precomp)
        rendered_image = torch.cat((rendered_image, alpha_image), dim=0)
        depth_image = depth_image.squeeze(0)
        normal_normed = pc.get_normal(dir_pp_normalized=dir_pp_normalized) * 0.5 + 0.5
        normal_image = rasterizer(means3D=means3D, means2D=means2D, shs=None, colors_precomp=normal_normed, opacities=opacity, scales=scales,
                                  rotations=rotations, cov3D_precomp=cov3D_precomp)[0]
    normal_image = (normal_image - 0.5) * 2.
    normal_image = torch.nn.functional.normalize(normal_image.permute(1, 2, 0), p=2, dim=-1)
    c2w = viewpoint_camera.world_view_transform.inverse()
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32, device=device), torch.arange(W, dtype=torch.float32, device=device), indexing="ij")
    K = torch.tensor([fx, fy, cx, cy], dtype=torch.float32)
    directions = torch.stack([(xs - K[2] + 0.5) / K[0], (ys - K[3] + 0.5) / K[1], torch.ones_like(xs)], -1)
    rays_d = directions @ c2w[:3, :3].T
    rays_o = c2w[:3, 3].expand_as(rays_d)
    points3D = rays_o + rays_d * depth_image.unsqueeze(-1)
    pseudo_normal = _depth_pcd2normal(points3D)
    return {"render": rendered_image, "depth": depth_image, "normal": normal_image, "pseudo_normal": pseudo_normal,
            "viewspace_points": screenspace_points, "visibility_filter": radii > 0, "radii": radii}
