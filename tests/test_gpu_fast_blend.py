"""Default blend (alpha = ex2.approx(power*log2e + log2 opacity), guarded decisions + exact repair, gsr_blend.cu) against the
bit-exact blend (GSR_FLAG_EXACT_IMAGES) and the reference's CUDA (tests/golden/): images within BASELINE's 1e-4 (measured: ~1e-6 of the
value), every integer output identical — radii, per-tile lists and n_contrib (the last blended splat of every pixel, i.e. every
skip / termination decision of the default mode equals the reference's)."""
import math

import pytest
import torch

from tests import helpers as Hh
from autovfx_b200 import scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CASES = ["config1", "small_sh", "small_deg1_m25", "deg3_m25", "deg2_m25", "small_precomp", "big_splats", "dense_tile", "coplanar"]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("for_backward", [False, True])
def test_fast_equals_exact_decisions_and_is_close(name, for_backward):
    a = Hh.resolve(Hh.case_inputs(name), DEV)
    fast = Hh.run_ours(a, for_backward=for_backward)
    f_img = {k: fast[k].clone() for k in ("color", "depth", "alpha")}
    nc_fast = fast["views"]["n_contrib"].clone()
    exact = Hh.run_ours(a, for_backward=for_backward, exact=True)
    Hh.assert_images_close(f_img, exact)
    assert torch.equal(fast["radii"], exact["radii"])
    if for_backward:
        assert torch.equal(nc_fast, exact["views"]["n_contrib"])
    Hh.assert_images_close(f_img, Hh.golden_case(name), tol=1e-4)  # the reference's images on the same case


def test_fast_product_frame_six_channels():
    """k_blend_lists<3>: the second colour set rides on the same weights in the default mode too."""
    from autovfx_b200 import rasterizer as R
    a = Hh.resolve(Hh.case_inputs("config1"), DEV)
    extra = torch.rand(a["means3D"].shape[0], 3, generator=torch.Generator().manual_seed(21)).to(DEV)
    s = Hh.settings_from(a)
    f = R.forward_multi(a["means3D"], a["shs"], None, extra, a["opacities"], a["scales"], a["rotations"], None, s, sync=True)
    f = [t.clone() for t in f[:5]]
    e = R.forward_multi(a["means3D"], a["shs"], None, extra, a["opacities"], a["scales"], a["rotations"], None, s, sync=True, exact=True)
    for i, tol in enumerate((1e-5, 5e-5, 1e-5, 1e-5)):
        assert Hh.maxabs(f[i], e[i]) <= tol, i
    assert torch.equal(f[4], e[4])
    one = Hh.run_ours(a)
    assert torch.equal(f[0], one["color"]) and torch.equal(f[1], one["depth"])  # same weights with or without the extra channels


def test_ill_conditioned_and_degenerate_splats_take_the_exact_drain():
    """Needle-like splats (conic determinant below 1e-5 a c), zero opacity and opacity 1: batches holding such splats are
    drained with the reference's arithmetic, so the default mode equals the exact mode bit for bit on them."""
    g = scene.synthetic_gaussians(400, seed=41, extent=(1, 1, 1), log_scale_mean=math.log(0.05), log_scale_std=0.3)
    g["scales"][:, 0] = 40.0     # sigma_max / sigma_min ~ 1e3 in screen space
    g["scales"][:, 1:] = 2e-4
    g["opacities"][:50] = 0.0
    g["opacities"][50:100] = 1.0
    cam = scene.lookat_camera((0.0, -3.0, 0.5), (0, 0, 0), 160, 96, 60.0)
    a = Hh.resolve(dict(g=g, cam=cam, sh_degree=3, bg=(0.1, 0.1, 0.1), scale_modifier=1.0), DEV)
    fast = Hh.run_ours(a, for_backward=True)
    f_img = {k: fast[k].clone() for k in ("color", "depth", "alpha")}
    nc = fast["views"]["n_contrib"].clone()
    exact = Hh.run_ours(a, for_backward=True, exact=True)
    for k in ("color", "depth", "alpha"):
        assert torch.equal(f_img[k], exact[k]), k
    assert torch.equal(nc, exact["views"]["n_contrib"])
    ref = Hh.ref_forward("fast_blend", "ill_conditioned", a, names=("color", "depth", "alpha"))
    for k in ("color", "depth", "alpha"):
        assert Hh.same(exact[k], ref[k]), k


def test_fast_blend_full_size_three_cameras():
    """3M Gaussians, 1920x1080, three trajectory cameras: max abs error of the default images against the exact ones, and
    identical n_contrib (every decision), with the repair path touching well under 10 % of the warps."""
    g = scene.config3_scene()
    cams = scene.cameras_from_trajectory(scene.trajectory_dict(num_views=300))
    worst = {"color": 0.0, "depth": 0.0, "alpha": 0.0}
    for ci in (7, 150, 271):
        a = Hh.resolve(dict(g=g, cam=cams[ci], sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0), DEV)
        fast = Hh.run_ours(a, for_backward=True, debug=False)
        f_img = {k: fast[k].clone() for k in ("color", "depth", "alpha")}
        nc = fast["views"]["n_contrib"].clone()
        redos = fast["stats"]["exact_redos"]
        exact = Hh.run_ours(a, for_backward=True, debug=False, exact=True)
        for k in worst:
            worst[k] = max(worst[k], Hh.maxabs(f_img[k], exact[k]))
        assert torch.equal(nc, exact["views"]["n_contrib"]), ci
        assert 0 < redos < 6000, redos
    print("fast vs exact, 3M/1080p, max abs:", worst)
    assert worst["color"] <= 1e-5 and worst["alpha"] <= 1e-5 and worst["depth"] <= 5e-5
