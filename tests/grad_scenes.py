"""Seeded scenes aimed at the branches of the blend and preprocess backward, and the per-element gradient criterion that
tests/test_grad_fp64_cpu.py (C oracle) and tests/test_gpu_grad_fp64.py (CUDA kernels) check them with against the fp64
restatement (tests/torch_ref.py).  Each builder returns the argument set of one rasterizer call (tests/helpers.resolve form)
on the CPU."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from autovfx_b200 import scene
from tests import helpers as Hh

RAGGED_SIZES = ((1, 1), (7, 3), (9, 5), (17, 1), (8, 4), (37, 29))
MODES_SH = ((0, 1), (1, 4), (2, 9), (3, 16), (1, 25), (3, 25), None)  # (sh_degree, M); None: colors_precomp


def _points(cam, u, v, z):
    """World points that project to pixel (u, v) at view depth z."""
    W, H = cam.image_width, cam.image_height
    u, v, z = u.double(), v.double(), z.double()
    x = ((2 * u + 1) / W - 1) * cam.tanfovx * z
    y = ((2 * v + 1) / H - 1) * cam.tanfovy * z
    c2w = torch.linalg.inv(cam.world_view_transform.double().T)
    pc = torch.stack([x, y, z, torch.ones_like(z)], dim=1)
    return (pc @ c2w.T)[:, :3].float().contiguous()


def _gaussians(cam, gen, u, v, z, sigma_px, opacity, sh_degree=3, M=None):
    """Gaussians at pixel (u, v), depth z, with a world scale that spans about sigma_px pixels."""
    P = u.shape[0]
    M = (sh_degree + 1) ** 2 if M is None else M
    fx = cam.image_width / (2 * cam.tanfovx)
    scales = (sigma_px * z / fx)[:, None] * torch.exp(torch.randn(P, 3, generator=gen) * 0.3)
    q = torch.randn(P, 4, generator=gen)
    shs = torch.randn(P, M, 3, generator=gen) * 0.1
    shs[:, 0] = torch.randn(P, 3, generator=gen) * 0.5
    return {"means3D": _points(cam, u, v, z), "scales": scales.float().contiguous(), "rotations": (q / q.norm(dim=1, keepdim=True)).contiguous(),
            "opacities": opacity.reshape(P, 1).float().contiguous(), "shs": shs.contiguous()}


def _cat(*gs):
    return {k: torch.cat([g[k] for g in gs]).contiguous() for k in gs[0]}


def _case(g, cam, sh_degree=3, bg=(0.3, 0.1, 0.6), scale_modifier=1.0):
    return Hh.resolve(dict(g=g, cam=cam, sh_degree=sh_degree, bg=bg, scale_modifier=scale_modifier))


def ragged(W: int, H: int) -> Dict:
    """Splats straddling the right and bottom edges of a W x H image (and a few anywhere)."""
    gen = torch.Generator().manual_seed(1000 + 37 * W + H)
    cam = scene.lookat_camera((0.0, -3.0, 0.3), (0, 0, 0), W, H, 60.0)
    n = 40
    U = lambda lo, hi, k=n: lo + (hi - lo) * torch.rand(k, generator=gen)  # noqa: E731
    # small splats centred just past the right / bottom edge reach only the last column / row; larger ones anywhere
    u = torch.cat([U(W, W + 1.5), U(-0.5, W - 0.5), U(-2.0, W + 2.0)])
    v = torch.cat([U(-0.5, H - 0.5), U(H, H + 1.5), U(-2.0, H + 2.0)])
    P = u.shape[0]
    z = U(2.0, 4.0, P)
    sigma = torch.cat([U(0.2, 0.6, 2 * n), torch.exp(torch.randn(n, generator=gen) * 0.5) * 1.5])
    op = torch.sigmoid(torch.randn(P, generator=gen) * 1.5)
    return _case(_gaussians(cam, gen, u, v, z, sigma, op), cam)


def opaque() -> Dict:
    """Opacity near 1 and large splats a few layers deep: alpha reaches the 0.99 clamp and pixels terminate early."""
    gen = torch.Generator().manual_seed(2001)
    W, H = 48, 40
    cam = scene.lookat_camera((0.2, -3.0, 0.4), (0, 0, 0), W, H, 55.0)
    P = 160
    u, v = torch.rand(P, generator=gen) * (W + 8) - 4, torch.rand(P, generator=gen) * (H + 8) - 4
    z = 2.0 + 2.0 * torch.rand(P, generator=gen)
    sigma = torch.exp(torch.randn(P, generator=gen) * 0.4) * 5.0
    op = torch.sigmoid(torch.randn(P, generator=gen) * 1.5 + 6.0)
    return _case(_gaussians(cam, gen, u, v, z, sigma, op), cam, bg=(0.9, 0.5, 0.1))


def deep(P: int = 2600) -> Dict:
    """Hundreds of faint, overlapping splats on a 32 x 32 image: long contributor lists (many 16-survivor batches, more than
    the 128-entry survivor ring) and tiles with more than 2048 instances."""
    gen = torch.Generator().manual_seed(3001)
    W = H = 32
    cam = scene.lookat_camera((0.0, -3.0, 0.0), (0, 0, 0), W, H, 50.0)
    u, v = 4 + 24 * torch.rand(P, generator=gen), 4 + 24 * torch.rand(P, generator=gen)
    z = 2.0 + 2.0 * torch.rand(P, generator=gen)
    sigma = 8.0 + 6.0 * torch.rand(P, generator=gen)
    op = 0.01 + 0.02 * torch.rand(P, generator=gen)
    return _case(_gaussians(cam, gen, u, v, z, sigma, op), cam, bg=(0.2, 0.6, 0.3))


def frustum() -> Dict:
    """Splats beyond +-1.3 tan(fov) that reach into the image, points just past the near plane, points behind the camera
    (the camera inside the cloud) and strongly negative SH DC terms (colour channels clamped at 0)."""
    gen = torch.Generator().manual_seed(4001)
    W, H = 48, 36
    cam = scene.lookat_camera((0.0, -2.0, 0.2), (0, 0, 0), W, H, 60.0)
    U = lambda lo, hi, k: lo + (hi - lo) * torch.rand(k, generator=gen)  # noqa: E731
    ndc_px = lambda ndc, n: ((ndc + 1) * n - 1) / 2  # noqa: E731
    k = 40
    side = torch.where(torch.rand(k, generator=gen) < 0.5, -1.0, 1.0)
    out_ndc = side * 1.3 * U(1.03, 1.5, k)
    horiz = torch.rand(k, generator=gen) < 0.5  # beyond the left / right or the top / bottom limit
    u_out = torch.where(horiz, ndc_px(out_ndc, W), U(0, W - 1, k))
    v_out = torch.where(horiz, U(0, H - 1, k), ndc_px(out_ndc, H))
    g_out = _gaussians(cam, gen, u_out, v_out, U(1.5, 3.0, k), U(14.0, 24.0, k), U(0.3, 0.95, k))
    g_near = _gaussians(cam, gen, U(0, W - 1, 20), U(0, H - 1, 20), U(0.205, 0.3, 20), U(2.0, 6.0, 20), U(0.2, 0.9, 20))
    g_behind = _gaussians(cam, gen, U(0, W - 1, 30), U(0, H - 1, 30), U(-1.0, 0.19, 30), U(2.0, 6.0, 30), U(0.2, 0.9, 30))
    g_in = _gaussians(cam, gen, U(-2, W + 1, 60), U(-2, H + 1, 60), U(1.5, 4.0, 60), U(1.5, 5.0, 60), U(0.2, 0.95, 60))
    g = _cat(g_out, g_near, g_behind, g_in)
    P = g["means3D"].shape[0]
    dark = torch.rand(P, generator=gen) < 0.5
    g["shs"][dark, 0] = torch.randn(int(dark.sum()), 3, generator=gen) * 0.5 - 1.6
    return _case(g, cam, bg=(0.1, 0.2, 0.3))


def modes(sh: Optional[tuple], cov3d: bool) -> Dict:
    """One scene in every parametrisation: SH at (degree, M) or colors_precomp, scales + rotations or cov3D_precomp; a scale
    modifier of 0.7, quaternions of norm 0.5 to 2 (the rasterizer does not normalise them) and a coloured background."""
    gen = torch.Generator().manual_seed(5001)
    W, H = 40, 30
    cam = scene.lookat_camera((0.5, -3.0, 0.6), (0, 0, 0), W, H, 60.0)
    P = 300
    D, M = sh if sh is not None else (3, 16)
    g = _gaussians(cam, gen, torch.rand(P, generator=gen) * (W + 4) - 2, torch.rand(P, generator=gen) * (H + 4) - 2,
                   2.0 + 2.0 * torch.rand(P, generator=gen), torch.exp(torch.randn(P, generator=gen) * 0.5) * 2.0,
                   torch.sigmoid(torch.randn(P, generator=gen) * 1.5), M=M)
    g["rotations"] = (g["rotations"] * (0.5 + 1.5 * torch.rand(P, 1, generator=gen))).contiguous()
    g["scales"] = (g["scales"] / 0.7).contiguous()
    a = _case(g, cam, sh_degree=D, bg=(0.2, 0.4, 0.7), scale_modifier=0.7)
    if sh is None:
        a["shs"], a["colors_precomp"] = None, torch.rand(P, 3, generator=gen)
    if cov3d:
        a["cov3D_precomp"] = Hh.cov3d_from(a["scales"], a["rotations"], 0.7)
        a["scales"] = a["rotations"] = None
    return a


def extra_colours(a: Dict, seed: int = 6) -> torch.Tensor:
    """A second colour set [P,3] for the fused (gsr_forward_multi) image."""
    return torch.rand(a["means3D"].shape[0], 3, generator=torch.Generator().manual_seed(seed))


# --------------------------------------------------------------------------------------------------------- loss gradients
LOSSES = ("randn", "color", "depth", "alpha", "onehot_footprint", "onehot_tile", "onehot_last")


def loss_grads(a: Dict, kind: str, seed: int = 7, extra: bool = False):
    """(dL/dcolor [3,H,W], dL/ddepth [1,H,W], dL/dalpha [1,H,W], dL/dextra [3,H,W] or None) on the CPU.
    randn: all N(0,1); color / depth / alpha: N(0,1) on that image alone; onehot_*: 1 at a single pixel of every image —
    a footprint corner (pixel (7, 3) clipped to the image), a tile corner ((15, 15) clipped) or the image's last pixel."""
    H, W = a["H"], a["W"]
    g = torch.Generator().manual_seed(seed)
    dc, dd, da, de = torch.randn(3, H, W, generator=g), torch.randn(1, H, W, generator=g), torch.randn(1, H, W, generator=g), \
        torch.randn(3, H, W, generator=g)
    if kind in ("color", "depth", "alpha"):
        dc, dd, da, de = [t if kind == k else torch.zeros_like(t) for t, k in ((dc, "color"), (dd, "depth"), (da, "alpha"), (de, "color"))]
    elif kind.startswith("onehot"):
        x, y = {"onehot_footprint": (7, 3), "onehot_tile": (15, 15), "onehot_last": (W - 1, H - 1)}[kind]
        x, y = min(x, W - 1), min(y, H - 1)
        dc, dd, da, de = [torch.zeros_like(t) for t in (dc, dd, da, de)]
        for t, val in ((dc, (1.0, -0.5, 0.25)), (dd, (0.3,)), (da, (-0.7,)), (de, (0.5, 0.2, -1.0))):
            t[:, y, x] = torch.tensor(val)
    elif kind != "randn":
        raise KeyError(kind)
    return dc, dd, da, (de if extra else None)


def mask_pixels(grads, amb):
    """Zero the rows of dL/dimage at the pixels ``amb`` [H,W] (returns new tensors, None stays None)."""
    keep = (~amb).to(torch.float32)
    return tuple(None if t is None else t * keep.to(t.device) for t in grads)


# ----------------------------------------------------------------------------------------------------- per-element criterion
def worst_ratio(got, want, keep, rtol: float, atol: float) -> float:
    """max over the kept rows of |g - r| / (rtol |r| + atol rms(r)): the criterion holds when it is <= 1.  ``want`` is the fp64
    value; ``keep`` [P] bool selects the compared Gaussians."""
    g = torch.as_tensor(got).detach().double().cpu()
    r = torch.as_tensor(want).detach().double().cpu()
    P = keep.shape[0]
    g, r = g.reshape(P, -1)[keep], r.reshape(P, -1)[keep]
    g = g[:, :r.shape[1]]
    if r.numel() == 0:
        return 0.0
    rms = float(r.pow(2).mean().sqrt())
    bound = rtol * r.abs() + atol * rms + 1e-30
    return float(((g - r).abs() / bound).max())


def atol_for(kind: str, atol: float) -> float:
    """The alpha-only loss gets atol 1e-3.  Its gradient to splat k of a pixel is T_final / (1 - alpha_k), which the
    reference's recursion forms as T_k (1 - R) with R, the alpha accumulated behind the splat, near 1 in an opaque pixel
    (backward.cu:561-562, the kernel's scalar recursion likewise): an fp32 difference with an absolute error of ~6e-8 per pixel,
    against gradients that are all of the order of T_final >= 1e-4, so no rms-relative floor far below 1e-3 can hold."""
    return max(atol, 1e-3) if kind == "alpha" else atol


def compare_grads(got: Dict, want: Dict, keep, rtol: float, atol: float, names=None) -> Dict[str, float]:
    """worst_ratio for every gradient both dicts hold (``names`` restricts them)."""
    names = [k for k in want if k in got] if names is None else names
    return {k: worst_ratio(got[k], want[k], keep, rtol, atol) for k in names}


def check_masked(amb_pixels, amb_gauss, visible):
    """Masking must stay a rounding-band exception: fewer than 1% of the pixels and of the visible Gaussians."""
    npx = int(amb_pixels.sum())
    ng = int(amb_gauss.sum())
    nvis = max(1, int(visible.sum()))
    assert npx < 0.01 * amb_pixels.numel() or npx == 0, "masked pixels: %d of %d" % (npx, amb_pixels.numel())
    assert ng < 0.01 * nvis or ng == 0, "masked Gaussians: %d of %d visible" % (ng, nvis)
    return npx, ng


def partial_footprint_only(r) -> int:
    """Number of visible Gaussians of the fp64 render ``r`` whose reach (the pixels where o G >= 1/255 is possible: distance
    <= sqrt(2 ln(255 o) / lambda_min(conic))) inside the image lies entirely in 8x4 footprints that the image border cuts
    (footprints whose columns reach past W or rows past H)."""
    W, H = r.meta["W"], r.meta["H"]
    px0 = W - W % 8 if W % 8 else W  # first column of a cut footprint (W: none)
    py0 = H - H % 4 if H % 4 else H
    m, k = r.meta["means2D"], r.meta["conic"]
    o = r.leaves["opacities"].detach().reshape(-1)[r.meta["visible_index"]]
    lam = 0.5 * (k[:, 0] + k[:, 2]) - torch.sqrt(0.25 * (k[:, 0] - k[:, 2]) ** 2 + k[:, 1] ** 2)
    reach = torch.sqrt(torch.clamp_min(2 * torch.log(255 * o), 0) / lam)
    x0, x1 = torch.clamp(torch.ceil(m[:, 0] - reach), min=0), torch.clamp(torch.floor(m[:, 0] + reach), max=W - 1)
    y0, y1 = torch.clamp(torch.ceil(m[:, 1] - reach), min=0), torch.clamp(torch.floor(m[:, 1] + reach), max=H - 1)
    inside = (x0 <= x1) & (y0 <= y1)
    return int((inside & ((x0 >= px0) | (y0 >= py0))).sum())
