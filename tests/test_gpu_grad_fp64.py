"""The CUDA backward (gsr_backward / gsr_backward_multi: k_blend_backward + k_gaussian_backward), element by element, against
fp64 autograd (tests/torch_ref.py), on scenes built to reach the branches the kernels special-case (tests/grad_scenes.py):
partial 8x4 footprints at ragged image borders, the 0.99 alpha clamp and early termination, contributor lists far longer than
the 128-entry survivor ring and tiles of more than 2048 instances, the +-1.3 tan(fov) and colour clamps, every SH layout and
parametrisation, and the fused extra-colour image.  Every scene asserts, from the kernel's own outputs, that it reaches its regime.

Plumbing: forward_raw(for_backward=True), then the C-ABI backward on the same workspaces; the fp64 restatement takes that
forward's decisions (radii, ranges, point_list, n_contrib through gsr_get_views) as constants.  Pixels with a (pixel, splat) pair
inside the rounding band of a skip test get a zero loss gradient in both; Gaussians within rounding of the colour or frustum
clamp are not compared; both stay under 1% (asserted).

Criterion, per gradient tensor over the compared Gaussians, r the fp64 value and g the kernel's:
    |g - r| <= rtol |r| + atol rms(r),   rtol = 1e-3, atol = 1e-4
(atol 1e-3 for the alpha-only loss, see grad_scenes.atol_for).  The fp64 loss weights each pixel by the kernel's recovered
final transmittance over the exact one (torch_ref.Fp64Render.loss, stored_alpha).  Forward images agree with the fp64 forward
to 1e-4.  The deep scene does not run the alpha-only loss: there the reference's own arithmetic is the limit.  A splat's gradient from
the alpha image is T_final / (1 - alpha_k), and both the reference's backward and this kernel form it as T_k (1 - R) with R,
the alpha accumulated behind the splat, summed over some 500 faint splats to within 1e-4 of 1.  The fp32 rounding of that sum
and of the transmittance recovery (T_k: T_final divided by (1 - alpha_j) splat by splat) leaves front splats' alpha gradients
percent-level errors.  At rtol = atol = 1e-3 the worst ratio there is 3.9 for the C oracle (tests/test_grad_fp64_cpu.py's
scene and decisions) and 8.9 for the kernel, whose recovery multiplies by an approximate reciprocal (rcp.approx, 1 ulp) where
the oracle divides.  The colour and depth terms carry no such cancellation and are checked at full strictness.
Worst ratios |g - r| / bound observed on an NVIDIA B200 at a 1000 W power limit (the largest over image modes, tile modes and
losses; <= 1 passes): ragged 0.18, opaque 0.13, deep 0.46, frustum 0.04, modes 0.18, fused 0.21.  The whole file runs in
about 10 s.
"""
import pytest
import torch

from tests import grad_scenes as S
from tests import helpers as Hh
from tests import torch_ref
from tests.test_gpu_fused_training import _backward

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
RTOL, ATOL = 1e-3, 1e-4


def _dev(a):
    return {k: (v.to(DEV) if isinstance(v, torch.Tensor) else v) for k, v in a.items()}


def _check(a, exact, tight=False, kinds=("randn",), extra=None):
    """Kernel forward + backward on ``a`` against fp64 autograd for each loss in ``kinds``; returns (fp64 render, kernel
    views, worst ratio)."""
    from autovfx_b200 import rasterizer as R
    ad = _dev(a)
    P, W, H = a["means3D"].shape[0], a["W"], a["H"]
    ex = None if extra is None else extra.to(DEV)
    eo = None if extra is None else torch.empty((3, H, W), device=DEV)
    res = R.forward_raw(ad["means3D"], ad["shs"], ad["colors_precomp"], ad["opacities"], ad["scales"], ad["rotations"], ad["cov3D_precomp"],
                        Hh.settings_from(ad), for_backward=True, sync=True, exact=exact, tight=tight, extra=ex, extra_out=eo)
    views = {k: v.cpu() for k, v in R.debug_views(res[4], P, W, H).items()}
    radii = res[3].cpu()
    r = torch_ref.render_fp64(a, dict(radii=radii, ranges=views["ranges"], point_list=views["point_list"], n_contrib=views["n_contrib"]),
                              extra=extra)
    for name, got, want in (("color", res[0], r.color), ("depth", res[1], r.depth), ("alpha", res[2], r.alpha),
                            ("extra", eo, r.extra_image)):
        if got is not None:
            assert Hh.maxabs(got, want.detach()) <= 1e-4, name
    S.check_masked(r.ambiguous_pixels, r.ambiguous_gaussians, r.visible)
    keep = ~r.ambiguous_gaussians
    worst = 0.0
    for kind in kinds:
        dc, dd, da, de = S.mask_pixels(S.loss_grads(a, kind, extra=extra is not None), r.ambiguous_pixels)
        dextra = None if extra is None else torch.full((P, 3), float("nan"), device=DEV)
        rc, g = _backward(ad, res, dc.to(DEV), dd.to(DEV), da.to(DEV), extra=ex, de=None if de is None else de.to(DEV), dextra=dextra,
                          multi=extra is not None)
        assert rc == 0
        if extra is not None:
            g["dL_dextra"] = dextra
        for t in r.leaves.values():
            t.grad = None
        r.loss(dc, dd, da, de, stored_alpha=res[2]).backward(retain_graph=True)
        want = r.kernel_grads()
        for k in want:
            assert torch.isfinite(g[k]).all(), (kind, k)
        ratios = S.compare_grads(g, want, keep, RTOL, S.atol_for(kind, ATOL))
        bad = {k: v for k, v in ratios.items() if v > 1.0}
        assert not bad, (kind, bad)
        worst = max([worst] + list(ratios.values()))
    print("worst ratio %.3g" % worst)
    return r, views, radii


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
@pytest.mark.parametrize("W,H", S.RAGGED_SIZES)
def test_ragged(W, H, exact):
    r, _, _ = _check(S.ragged(W, H), exact, kinds=S.LOSSES)
    assert r.visible.any()
    if W % 8 or H % 4:
        assert S.partial_footprint_only(r) > 0


def _terminated_pixels(views, W, H):
    rg = views["ranges"].to(torch.int64)
    lens = rg[:, 1] - rg[:, 0]
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    return int((views["n_contrib"].to(torch.int64) < lens[(ys // 16) * ((W + 15) // 16) + xs // 16]).sum())


@pytest.mark.parametrize("tight", [False, True], ids=["tiles", "tight"])
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
def test_opaque(exact, tight):
    a = S.opaque()
    r, views, _ = _check(a, exact, tight, kinds=S.LOSSES)
    assert r.meta["clamped_pairs"] > 0
    assert _terminated_pixels(views, a["W"], a["H"]) > 0.1 * a["W"] * a["H"]


@pytest.mark.parametrize("tight", [False, True], ids=["tiles", "tight"])
@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
def test_deep(exact, tight):
    a = S.deep()
    # no alpha-only loss here: see the module docstring
    r, views, _ = _check(a, exact, tight, kinds=("randn", "color", "depth", "onehot_tile", "onehot_last"))
    assert int(views["n_contrib"].max()) > 300
    rg = views["ranges"].to(torch.int64)
    assert int((rg[:, 1] - rg[:, 0]).max()) > 2048


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
def test_frustum(exact):
    r, views, radii = _check(S.frustum(), exact, kinds=("randn", "color", "depth", "onehot_footprint"))
    assert r.meta["frustum_clamped"] > 0
    assert int(((views["clamped"] != 0) & (radii > 0)).sum()) > 0
    assert not r.visible.all()  # points behind the camera are culled


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
@pytest.mark.parametrize("cov3d", [False, True], ids=["scalerot", "cov3D"])
@pytest.mark.parametrize("sh", S.MODES_SH, ids=lambda s: "precomp" if s is None else "D%dM%d" % s)
def test_modes(sh, cov3d, exact):
    _check(S.modes(sh, cov3d), exact)


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact"])
@pytest.mark.parametrize("scene", ["modes", "opaque", "deep"])
def test_fused_extra_colours(scene, exact):
    a = S.modes((3, 16), False) if scene == "modes" else getattr(S, scene)()
    _check(a, exact, kinds=("randn", "color", "onehot_footprint"), extra=S.extra_colours(a))
