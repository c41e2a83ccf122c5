"""Differentiable fp64 PyTorch restatement of the rasterizer at small sizes (test infrastructure).

Purpose: pin the CPU oracle's and the CUDA kernels' forward AND backward independently of their fp32 arithmetic: the
continuous part of the forward (reference forward.cu:74-256 preprocess math, forward.cu:330-366 blend recurrence) is restated
in torch fp64 and differentiated by autograd, while the discrete decisions are constants handed in by the caller, taken from
the forward under test (the C oracle's buffers or the kernel's workspaces): the visible set (radii > 0), the tile lists
(ranges, point_list) and each pixel's last contributor (n_contrib).  That is exactly what the reference's hand-written
backward does (backward.cu:415-599 replays the forward's decisions).  The only decision evaluated here, in fp64, is the
per-(pixel, splat) skip test (power > 0 or alpha < 1/255); the pairs and Gaussians where an fp32 evaluation could decide a
threshold differently are reported, so that callers can leave them out (``Fp64Render.ambiguous_pixels`` / ``ambiguous_gaussians``).

The reference's deliberate departures from the true derivative are restated as straight-through terms, so that a kernel can
be held to a tight tolerance:
  * alpha = min(0.99, o G) in value, but its derivative is that of o G (backward.cu:528, :580 use dL/dG = o dL/dalpha);
  * where tx / tz or ty / tz is clamped to +-1.3 tan(fov), the clamped image-plane coordinate is a constant of the Jacobian
    (backward.cu:168-175, :262-264 zero its t.x derivative and keep the clamped value in the t.z derivative);
  * ``kernel_grads`` reports dL/dscale for the effective scale (scale_modifier * scale, backward.cu:322-325 omit the factor)
    and dL/dmean2D in NDC-scaled units (pixel gradient * (W/2, H/2), backward.cu:488-489).
The 1 / (det^2 + 1e-7) regularisation of the conic backward (backward.cu:203) is not restated: det >= 0.09 for every
projected covariance (the 0.3 px^2 dilation), so it changes a gradient by less than 1.3e-5 of its value.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, Optional

import numpy as np
import torch

SH_C0 = 0.28209479177387814
SH_C1 = 0.4886025119029199
SH_C2 = [1.0925484305920792, -1.0925484305920792, 0.31539156525252005, -1.0925484305920792, 0.5462742152960396]
SH_C3 = [-0.5900435899266435, 2.890611442640554, -0.4570457994644658, 0.3731763325901154, -0.4570457994644658, 1.445305721320277,
         -0.5900435899266435]

# Thresholds of the "could an fp32 evaluation decide this differently" tests (relative to the decision's scale)
NEAR_ALPHA = 1e-5   # |o G 255 - 1|: the alpha >= 1/255 skip test
NEAR_POWER = 1e-6   # |power|: the power > 0 skip test
NEAR_CLAMP = 1e-6   # |rgb| (colour clamp at 0) and | |t.x / t.z| / (1.3 tan fov) - 1 | (frustum clamp)


def eval_sh(deg, sh, dirs):
    """sh [P,M,3], dirs [P,3] unit.  Same polynomials as forward.cu:20-71 / utils/sh_utils.py:57-112."""
    x, y, z = dirs[:, 0:1], dirs[:, 1:2], dirs[:, 2:3]
    res = SH_C0 * sh[:, 0]
    if deg > 0:
        res = res - SH_C1 * y * sh[:, 1] + SH_C1 * z * sh[:, 2] - SH_C1 * x * sh[:, 3]
        if deg > 1:
            xx, yy, zz, xy, yz, xz = x * x, y * y, z * z, x * y, y * z, x * z
            res = res + SH_C2[0] * xy * sh[:, 4] + SH_C2[1] * yz * sh[:, 5] + SH_C2[2] * (2 * zz - xx - yy) * sh[:, 6] + \
                SH_C2[3] * xz * sh[:, 7] + SH_C2[4] * (xx - yy) * sh[:, 8]
            if deg > 2:
                res = res + SH_C3[0] * y * (3 * xx - yy) * sh[:, 9] + SH_C3[1] * xy * z * sh[:, 10] + SH_C3[2] * y * (4 * zz - xx - yy) * sh[:, 11] + \
                    SH_C3[3] * z * (2 * zz - 3 * xx - 3 * yy) * sh[:, 12] + SH_C3[4] * x * (4 * zz - xx - yy) * sh[:, 13] + \
                    SH_C3[5] * z * (xx - yy) * sh[:, 14] + SH_C3[6] * x * (xx - 3 * yy) * sh[:, 15]
    return res


def _clamped_coord(t, tz, lim):
    """t / tz clamped to +-lim, times tz.  Inside the clamp the coordinate is t itself; outside it is a constant (the
    reference's derivative, see the module docstring).  Also returns |t / tz| / lim for the near-clamp test."""
    r = t / tz
    inside = (r >= -lim) & (r <= lim)
    clamped = (torch.clamp(r, -lim, lim) * tz).detach()
    return torch.where(inside, t, clamped), (r.abs() / lim).detach()


def preprocess(means3D, scales, rotations, opacities, shs, view, proj, campos, W, H, tanfovx, tanfovy, sh_degree, scale_modifier,
               cov3D=None, colors=None):
    """Continuous per-Gaussian quantities in fp64: means2D [P,2] (pixels), conic [P,3], rgb [P,3] (SH clamped at 0, or
    ``colors``), depth [P], and [P] bool tensors {"near": within rounding of the colour or frustum clamp, "frustum": tx / tz or
    ty / tz clamped, "rgb_clamped": a colour channel clamped at 0}.
    ``cov3D`` [P,6] (upper triangle, row-major) replaces scales / rotations, ``colors`` [P,3] replaces the SH colours."""
    P = means3D.shape[0]
    hom = torch.cat([means3D, torch.ones(P, 1, dtype=means3D.dtype)], dim=1)
    p_hom = hom @ proj  # row-vector convention on the row-major buffer (auxiliary.h:58-77)
    p_w = 1.0 / (p_hom[:, 3] + 0.0000001)
    p_proj = p_hom[:, :3] * p_w[:, None]
    t = (hom @ view)[:, :3]
    depth = t[:, 2]
    fx, fy = W / (2.0 * tanfovx), H / (2.0 * tanfovy)
    if cov3D is None:
        r, x, y, z = rotations.unbind(-1)
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y), 2 * (x * y + r * z), 1 - 2 * (x * x + z * z),
                         2 * (y * z - r * x), 2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], dim=-1).view(P, 3, 3)
        L = R * (scales * scale_modifier).unsqueeze(1)
        Sigma = L @ L.transpose(1, 2)
    else:
        c = cov3D.unbind(-1)
        Sigma = torch.stack([c[0], c[1], c[2], c[1], c[3], c[4], c[2], c[4], c[5]], dim=-1).view(P, 3, 3)
    tz = t[:, 2]
    tx, nx = _clamped_coord(t[:, 0], tz, 1.3 * tanfovx)
    ty, ny = _clamped_coord(t[:, 1], tz, 1.3 * tanfovy)
    near = ((nx - 1).abs() < NEAR_CLAMP) | ((ny - 1).abs() < NEAR_CLAMP)
    info = {"frustum": (nx > 1) | (ny > 1), "rgb_clamped": torch.zeros(P, dtype=torch.bool)}
    zero = torch.zeros_like(tz)
    J = torch.stack([fx / tz, zero, -(fx * tx) / (tz * tz), zero, fy / tz, -(fy * ty) / (tz * tz)], dim=-1).view(P, 2, 3)
    Wr = view[:3, :3].T  # world -> camera rotation (the buffer holds the transpose)
    T = J @ Wr
    cov = T @ Sigma @ T.transpose(1, 2)
    a = cov[:, 0, 0] + 0.3
    b = cov[:, 0, 1]
    c = cov[:, 1, 1] + 0.3
    det = a * c - b * b
    conic = torch.stack([c / det, -b / det, a / det], dim=-1)
    px = ((p_proj[:, 0] + 1.0) * W - 1.0) * 0.5
    py = ((p_proj[:, 1] + 1.0) * H - 1.0) * 0.5
    if colors is None:
        d = means3D - campos[None]
        d = d / d.norm(dim=1, keepdim=True)
        raw = eval_sh(sh_degree, shs, d) + 0.5
        near = near | (raw.detach().abs() < NEAR_CLAMP).any(dim=1)
        info["rgb_clamped"] = (raw.detach() < 0).any(dim=1)
        rgb = torch.clamp_min(raw, 0.0)
    else:
        rgb = colors
    info["near"] = near
    return torch.stack([px, py], dim=-1), conic, rgb, depth, info


def blend(means2D, conic, opac, rgb, depth, ranges, point_list, n_contrib, W, H, bg, extra=None):
    """The blend recurrence with the given tile lists: pixel p blends the entries of its tile's list up to its last
    contributor (1-based list position n_contrib[p]) that pass the skip test.  Per tile, the [pixels x entries] alphas are
    masked and the transmittance in front of every entry is an exclusive cumulative product of (1 - alpha).
    Returns color [3,H,W], depth [1,H,W], alpha [1,H,W], the extra image [3,H,W] (``extra`` [P,3] blended with the same
    weights over the same background) or None, a [H,W] bool map of the pixels with a pair inside a skip test's rounding band, and
    counts {"clamped_pairs": blended pairs with o G > 0.99}."""
    dt = means2D.dtype
    bgv = bg.to(dt)
    color = bgv.view(3, 1, 1).repeat(1, H, W)
    eimg = None if extra is None else bgv.view(3, 1, 1).repeat(1, H, W)
    dimg = torch.zeros(1, H, W, dtype=dt)
    aimg = torch.zeros(1, H, W, dtype=dt)
    amb = torch.zeros(H, W, dtype=torch.bool)
    stats = {"clamped_pairs": 0}
    gx = (W + 15) // 16
    for tile in range(ranges.shape[0]):
        lo, hi = int(ranges[tile, 0]), int(ranges[tile, 1])
        ty, tx = divmod(tile, gx)
        y0, x0 = ty * 16, tx * 16
        hh, ww = min(16, H - y0), min(16, W - x0)
        if hi <= lo or hh <= 0 or ww <= 0:
            continue
        nc = n_contrib[y0:y0 + hh, x0:x0 + ww].reshape(-1)
        L = int(nc.max())
        if L == 0:
            continue
        g = point_list[lo:lo + L]
        yy, xx = torch.meshgrid(torch.arange(y0, y0 + hh, dtype=dt), torch.arange(x0, x0 + ww, dtype=dt), indexing="ij")
        dx = means2D[g, 0][None, :] - xx.reshape(-1, 1)
        dy = means2D[g, 1][None, :] - yy.reshape(-1, 1)
        cg = conic[g]
        power = -0.5 * (cg[:, 0][None] * dx * dx + cg[:, 2][None] * dy * dy) - cg[:, 1][None] * dx * dy
        oG = opac[g][None, :] * torch.exp(power)
        alpha = oG - (oG - torch.clamp_max(oG, 0.99)).detach()  # min(0.99, oG) in value, d(oG) in derivative
        with torch.no_grad():
            listed = torch.arange(L)[None, :] < nc[:, None]
            hit = listed & (power <= 0) & (oG * 255.0 >= 1.0)
            near = listed & (((oG * 255.0 - 1.0).abs() < NEAR_ALPHA) | (power.abs() < NEAR_POWER))
        amb[y0:y0 + hh, x0:x0 + ww] = near.any(dim=1).reshape(hh, ww)
        stats["clamped_pairs"] += int((hit & (oG > 0.99)).sum())
        a_eff = torch.where(hit, alpha, torch.zeros_like(alpha))
        T_after = torch.cumprod(1.0 - a_eff, dim=1)
        T_before = torch.cat([torch.ones(a_eff.shape[0], 1, dtype=dt), T_after[:, :-1]], dim=1)
        w = a_eff * T_before
        T_fin = T_after[:, -1]
        color[:, y0:y0 + hh, x0:x0 + ww] = (w @ rgb[g] + T_fin[:, None] * bgv[None]).T.reshape(3, hh, ww)
        dimg[0, y0:y0 + hh, x0:x0 + ww] = (w @ depth[g]).reshape(hh, ww)
        aimg[0, y0:y0 + hh, x0:x0 + ww] = (1.0 - T_fin).reshape(hh, ww)
        if extra is not None:
            eimg[:, y0:y0 + hh, x0:x0 + ww] = (w @ extra[g] + T_fin[:, None] * bgv[None]).T.reshape(3, hh, ww)
    return color, dimg, aimg, eimg, amb, stats


def _i64(x) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x.detach().cpu().to(torch.int64)
    return torch.from_numpy(np.asarray(x).astype(np.int64))


LEAVES = ("means3D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D_precomp")


@dataclass
class Fp64Render:
    color: torch.Tensor
    depth: torch.Tensor
    alpha: torch.Tensor
    extra_image: Optional[torch.Tensor]
    leaves: Dict[str, torch.Tensor]       # fp64 leaves [P, ...]; "means2D" is a zero offset whose gradient is dL/d(pixel position)
    ambiguous_pixels: torch.Tensor        # [H,W] bool
    ambiguous_gaussians: torch.Tensor     # [P] bool (visible Gaussians only)
    visible: torch.Tensor                 # [P] bool
    meta: Dict = field(default_factory=dict)

    def loss(self, dc, dd, da, de=None, stored_alpha=None):
        """sum(image * dL/dimage) over the images; the gradient tensors may be float32 or on any device.

        ``stored_alpha``: the fp32 alpha image of the forward under test.  The reference's backward does not keep a pixel's
        final transmittance; it recovers it as 1 - alpha from that image (backward.cu:462-463) and every transmittance in front
        of it by dividing (1 - alpha_k) back out, so each of the pixel's gradient terms is scaled by
        rho = (1 - stored alpha) / T_final.  rho - 1 reaches 6e-4 where T_final nears the 1e-4 termination threshold (half an
        ulp of an fp32 alpha near 1, relative to T_final).  Given the image, the loss weights pixel p by rho_p, so that the
        fp64 gradient carries the same factor."""
        f = lambda t: torch.as_tensor(t).detach().double().cpu()  # noqa: E731
        dc, dd, da = f(dc), f(dd), f(da)
        de = None if de is None else f(de)
        if stored_alpha is not None:
            T = 1.0 - self.alpha.detach()
            rho = (1.0 - f(stored_alpha).reshape(T.shape)) / T
            dc, dd, da = dc * rho, dd * rho, da * rho
            de = None if de is None else de * rho
        out = (self.color * dc).sum() + (self.depth * dd).sum() + (self.alpha * da).sum()
        if de is not None:
            out = out + (self.extra_image * de).sum()
        return out

    def kernel_grads(self) -> Dict[str, torch.Tensor]:
        """Leaf gradients after ``loss().backward()``, under the names and in the conventions of the rasterizer's gradient
        buffers (dL/dscale for the effective scale, dL/dmean2D [P,2] in NDC-scaled units)."""
        L, m = self.leaves, self.meta
        names = {"means3D": "dL_dmeans3D", "opacities": "dL_dopacity", "shs": "dL_dsh", "colors_precomp": "dL_dcolors", "scales": "dL_dscales",
                 "rotations": "dL_drotations", "cov3D_precomp": "dL_dcov3D", "extra": "dL_dextra"}
        out = {names[k]: L[k].grad.detach().clone() for k in names if k in L}
        if "dL_dscales" in out:
            out["dL_dscales"] = out["dL_dscales"] / m["scale_modifier"]
        out["dL_dmeans2D"] = L["means2D"].grad.detach() * torch.tensor([0.5 * m["W"], 0.5 * m["H"]], dtype=torch.float64)
        return out


def render_fp64(a, dec, extra=None) -> Fp64Render:
    """a: resolved case (tests/helpers.resolve), on any device.  dec: the forward's decisions, {radii [P], ranges [tiles,2],
    point_list, n_contrib [H,W]} as numpy arrays or tensors.  ``extra`` [P,3]: a second colour set blended with the same weights.
    Only the visible Gaussians are preprocessed, so that a culled point's unused branch (e.g. behind the camera) cannot put
    inf / NaN into the graph."""
    f64 = lambda t: t.detach().double().cpu().clone().requires_grad_(True)  # noqa: E731
    leaves = {k: f64(a[k]) for k in LEAVES if a[k] is not None}
    if extra is not None:
        leaves["extra"] = f64(extra)
    P = leaves["means3D"].shape[0]
    leaves["means2D"] = torch.zeros(P, 2, dtype=torch.float64, requires_grad=True)
    W, H = a["W"], a["H"]
    visible = _i64(dec["radii"]) > 0
    vis = torch.nonzero(visible).squeeze(1)
    sub = lambda k: leaves[k][vis] if k in leaves else None  # noqa: E731
    cpu64 = lambda t: t.detach().double().cpu()  # noqa: E731
    m2d, conic, rgb, depth, info = preprocess(sub("means3D"), sub("scales"), sub("rotations"), sub("opacities"), sub("shs"), cpu64(a["view"]),
                                              cpu64(a["proj"]), cpu64(a["campos"]), W, H, a["tanfovx"], a["tanfovy"], a["sh_degree"],
                                              a["scale_modifier"], cov3D=sub("cov3D_precomp"), colors=sub("colors_precomp"))
    m2d = m2d + leaves["means2D"][vis]
    compact = torch.full((P,), -1, dtype=torch.int64)
    compact[vis] = torch.arange(vis.numel())
    ranges = _i64(dec["ranges"]).reshape(-1, 2)
    plist = compact[_i64(dec["point_list"])[:int(ranges.max()) if ranges.numel() else 0]]  # a workspace's list may run on past the last range
    color, dimg, aimg, eimg, amb, stats = blend(m2d, conic, sub("opacities").reshape(-1), rgb, depth, ranges, plist, _i64(dec["n_contrib"]).reshape(H, W),
                                         W, H, cpu64(a["bg"]), extra=sub("extra"))
    amb_g = torch.zeros(P, dtype=torch.bool)
    amb_g[vis] = info["near"]
    meta = dict(W=W, H=H, scale_modifier=a["scale_modifier"], means2D=m2d.detach(), conic=conic.detach(), frustum_clamped=int(info["frustum"].sum()),
                rgb_clamped=int(info["rgb_clamped"].sum()), visible_index=vis, **stats)
    return Fp64Render(color, dimg, aimg, eimg, leaves, amb, amb_g, visible, meta)


def render(a, oracle_fw):
    """a: resolved case with scales/rotations/shs, decisions from the C oracle's forward; returns images + the fp64 leaf
    tensors + the pixel-position leaf (whose gradient is dL/d(pixel position))."""
    r = render_fp64(a, oracle_fw)
    return r.color, r.depth, r.alpha, r.leaves, r.leaves["means2D"]
