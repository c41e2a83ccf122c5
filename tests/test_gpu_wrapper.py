"""GPU parity of the render() wrapper row (SURVEY §8 a19 / f1 / f2): the 6-channel forward, the per-Gaussian normals, the
normal maps and the 8-bit hand-off, through the C ABI, against (a) the reference rasterizer called twice the way the
reference's render() does (its outputs stored under tests/golden/) and (b) the torch restatement of the wrapper's helper functions run with torch's CUDA kernels."""
import math
import types

import numpy as np
import pytest
import torch

from tests import wrapper_ref as WR
from tests.helpers import case_inputs, maxabs, ref_forward, resolve, run_ours, same

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(autouse=True, params=["exact"])
def _image_mode(request):
    """These tests compare images bit for bit with the compiled reference: run them with GSR_FLAG_EXACT_IMAGES.  The default
    (fast-alpha) blend is compared with the exact one in tests/test_gpu_fast_blend.py."""
    from autovfx_b200 import rasterizer as R
    R.set_exact_images(True)
    yield
    R.set_exact_images(False)


def _extra(P, seed=21):
    return torch.rand(P, 3, generator=torch.Generator().manual_seed(seed)).to(DEV)


@pytest.mark.parametrize("name", ["config1", "small_sh", "small_deg1_m25", "small_precomp", "big_splats", "dense_tile", "coplanar"])
@pytest.mark.parametrize("tight", [False, True])
def test_forward_multi_is_two_passes(name, tight):
    from autovfx_b200 import rasterizer as R
    from tests.helpers import settings_from
    a = resolve(case_inputs(name), DEV)
    P = a["means3D"].shape[0]
    extra = _extra(P)
    s = settings_from(a, debug=True)
    color, depth, alpha, eimg, radii, ticket = R.forward_multi(a["means3D"], a["shs"], a["colors_precomp"], extra, a["opacities"], a["scales"],
                                                              a["rotations"], a["cov3D_precomp"], s, sync=True, tight=tight)
    one = run_ours(a, tight=tight)
    assert torch.equal(color, one["color"]) and torch.equal(depth, one["depth"]) and torch.equal(alpha, one["alpha"]) and torch.equal(radii, one["radii"])
    b = dict(a)
    b["shs"], b["colors_precomp"] = None, extra
    second = run_ours(b, tight=tight)
    assert torch.equal(eimg, second["color"])  # bit for bit what a second pass returns
    ref2 = ref_forward("wrapper", "second_pass_" + name, b, names=("color",))
    assert same(eimg, ref2["color"])  # ... and what the reference's second pass returns


def test_forward_multi_empty_and_errors():
    from autovfx_b200 import rasterizer as R
    from tests.helpers import settings_from
    a = resolve(case_inputs("small_sh"), DEV)
    s = settings_from(a)
    z = lambda *sh: torch.zeros(*sh, device=DEV)  # noqa: E731
    color, depth, alpha, eimg, radii, _ = R.forward_multi(z(0, 3), z(0, 16, 3), None, z(0, 3), z(0, 1), z(0, 3), z(0, 4), None, s, sync=True)
    assert float(eimg.abs().max()) == 0.0 and float(color.abs().max()) == 0.0 and radii.numel() == 0
    with pytest.raises(ValueError):
        R.forward_raw(a["means3D"], a["shs"], None, a["opacities"], a["scales"], a["rotations"], None, s, extra=_extra(a["means3D"].shape[0]))
    with pytest.raises(ValueError):
        R.forward_multi(a["means3D"], a["shs"], None, _extra(5), a["opacities"], a["scales"], a["rotations"], None, s)


def test_axis_normals_vs_torch():
    from autovfx_b200 import renderer
    g = torch.Generator().manual_seed(0)
    P = 200_000
    xyz = (torch.rand(P, 3, generator=g) * 8 - 4).to(DEV)
    scales = torch.exp(torch.randn(P, 3, generator=g) * 0.6 - 4).to(DEV)
    rot = torch.randn(P, 4, generator=g).to(DEV)
    campos = torch.tensor([0.3, -3.5, 0.7], device=DEV)
    ref = WR.get_normal(xyz, scales, rot, campos)
    got = renderer.axis_normals(xyz, scales, rot, campos)
    assert maxabs(got, ref) <= 5e-7
    frac_exact = float((got == ref).all(dim=1).float().mean())
    assert frac_exact > 0.8, frac_exact  # the rest differ in the last bit (torch's reductions sum in another order)
    got01 = renderer.axis_normals(xyz, scales, rot, campos, remap01=True)
    assert maxabs(got01, ref * 0.5 + 0.5) <= 5e-7
    assert renderer.axis_normals(xyz[:0], scales[:0], rot[:0], campos).shape == (0, 3)


@pytest.mark.parametrize("H,W", [(75, 100), (1080, 1920), (3, 3), (2, 7)])
def test_normal_maps_vs_torch(H, W):
    from autovfx_b200 import renderer
    g = torch.Generator().manual_seed(H + W)
    nimg = torch.rand(3, H, W, generator=g).to(DEV)
    nimg[:, 0, 0] = 0.5
    depth = (torch.rand(H, W, generator=g) * 3 + 0.5).to(DEV)
    depth[H // 2:, : W // 3] = 0.0
    cam = case_inputs("small_sh")["cam"]
    view = cam.world_view_transform.to(DEV)
    FoVx, FoVy = 2 * math.atan(cam.tanfovx), 2 * math.atan(cam.tanfovy)
    ref_n = WR.normal_image(nimg)
    ref_p = WR.pseudo_normal(depth, view, FoVx, FoVy)
    c2w = view.inverse()
    got_n, got_p = renderer.normal_maps(nimg, depth, c2w, WR.fov2focal(FoVx, W), WR.fov2focal(FoVy, H), W / 2, H / 2)
    assert got_n.shape == (H, W, 3) and got_p.shape == (H, W, 3)
    assert maxabs(got_n, ref_n) <= 5e-7
    # pseudo normal: a cancelling stencil over a GEMM whose summation order torch does not fix -> compare as directions
    assert maxabs(got_p, ref_p) < 5e-3
    only_n, none_p = renderer.normal_maps(nimg, None, None, 1.0, 1.0, 0.0, 0.0)
    assert none_p is None and torch.equal(only_n, got_n)


def test_pack_frame_bytes():
    from autovfx_b200 import renderer
    from oracle import render_oracle as RO
    g = torch.Generator().manual_seed(9)
    H, W = 270, 480
    rgb = (torch.rand(3, H, W, generator=g) * 1.4 - 0.2).to(DEV)
    alpha = torch.rand(H, W, generator=g).to(DEV)
    depth = (torch.rand(H, W, generator=g) * 5 - 0.5).to(DEV)
    nrm = torch.nn.functional.normalize(torch.randn(H, W, 3, generator=g), dim=-1).to(DEV)
    out = renderer.pack_frame(rgb, alpha, depth, nrm, depth_scale=3.0)
    ref_rgba = WR.save_image_bytes(torch.cat([rgb, alpha[None]], 0))
    assert torch.equal(out["rgba8"], ref_rgba)
    assert (out["normal8"].cpu().numpy() == RO.normal8(nrm.cpu().numpy())).all()
    assert (out["depth8"].cpu().numpy() == RO.depth8(depth.cpu().numpy(), 3.0)).all()
    assert (out["rgba8"].cpu().numpy() == RO.rgba8(rgb.cpu().numpy(), alpha.cpu().numpy())).all()
    lut = renderer.TURBO_LUT_BGR
    assert lut.shape == (256, 3) and lut.dtype == torch.uint8
    only = renderer.pack_frame(rgb=rgb)
    assert set(only) == {"rgba8"} and int(only["rgba8"][..., 3].min()) == 255


def test_pack_frame_bytes_against_torchvision_and_cv2(tmp_path):
    """The per-frame conversions of the reference's loop (scene_representation.py:424-438) executed with the REAL libraries it calls —
    torchvision.utils.save_image -> PNG, cv2.applyColorMap(COLORMAP_TURBO) (sugar/render.py:18-22), numpy astype(uint8) + cv2.cvtColor —
    against gsr_pack_frame's bytes and the exported TURBO table."""
    import cv2
    import torchvision
    from autovfx_b200 import renderer
    g = torch.Generator().manual_seed(19)
    H, W = 135, 240
    rgb = (torch.rand(3, H, W, generator=g) * 1.3 - 0.15).to(DEV)
    alpha = torch.rand(H, W, generator=g).to(DEV)
    depth = (torch.rand(H, W, generator=g) * 4.5 - 0.4).to(DEV)
    nrm = torch.nn.functional.normalize(torch.randn(H, W, 3, generator=g), dim=-1).to(DEV)
    out = renderer.pack_frame(rgb, alpha, depth, nrm, depth_scale=3.0)
    # rgb image: torchvision.utils.save_image(result["render"], png)
    png = str(tmp_path / "f.png")
    torchvision.utils.save_image(torch.cat([rgb, alpha[None]], 0), png)
    bgra = cv2.imread(png, cv2.IMREAD_UNCHANGED)
    assert bgra.shape == (H, W, 4)
    assert np.array_equal(out["rgba8"].cpu().numpy(), bgra[..., [2, 1, 0, 3]])
    # depth map: depth2img(depth_raw, scale=3.0) = cv2.applyColorMap((clip(depth / scale, 0, 1) * 255).astype(uint8), COLORMAP_TURBO)
    d = depth.cpu().numpy()
    idx = (np.clip(d / 3.0, a_min=0., a_max=1.) * 255).astype(np.uint8)
    assert np.array_equal(out["depth8"].cpu().numpy(), idx)
    assert np.array_equal(renderer.TURBO_LUT_BGR.numpy()[out["depth8"].cpu().numpy()], cv2.applyColorMap(idx, cv2.COLORMAP_TURBO))
    # normal map: ((normal + 1) / 2 * 255).astype(uint8), written through cv2.cvtColor(RGB2BGR)
    n8 = (((nrm.cpu().numpy() + 1) / 2) * 255).astype(np.uint8)
    assert np.array_equal(out["normal8"].cpu().numpy(), n8)
    assert np.array_equal(out["normal8"].cpu().numpy()[..., ::-1], cv2.cvtColor(n8, cv2.COLOR_RGB2BGR))


class _PC:
    """Duck-typed stand-in for the reference's GaussianModel (scene/gaussian_model.py): activated parameters."""

    def __init__(self, g, sh_degree, max_sh_degree=3, requires_grad=False):
        self._xyz = g["means3D"].clone().requires_grad_(requires_grad)
        self._scales, self._rot, self._op, self._shs = g["scales"], g["rotations"], g["opacities"], g["shs"]
        self.active_sh_degree, self.max_sh_degree = sh_degree, max_sh_degree

    get_xyz = property(lambda s: s._xyz)
    get_scaling = property(lambda s: s._scales)
    get_rotation = property(lambda s: s._rot)
    get_opacity = property(lambda s: s._op)
    get_features = property(lambda s: s._shs)

    def get_normal(self, dir_pp_normalized=None):
        n, _ = WR.flip_align_view(WR.get_minimum_axis(self._scales, self._rot), dir_pp_normalized)
        return n / n.norm(dim=1, keepdim=True)


def _cam_obj(cam):
    return types.SimpleNamespace(FoVx=2 * math.atan(cam.tanfovx), FoVy=2 * math.atan(cam.tanfovy), image_height=cam.image_height,
                                 image_width=cam.image_width, world_view_transform=cam.world_view_transform.to(DEV),
                                 full_proj_transform=cam.full_proj_transform.to(DEV), camera_center=cam.camera_center.to(DEV))


@pytest.mark.parametrize("name", ["config1", "small_sh", "big_splats"])
def test_render_matches_reference_structure(name):
    from autovfx_b200 import renderer
    case = case_inputs(name)
    a = resolve(case, DEV)
    g = {k: v.to(DEV) for k, v in case["g"].items()}
    pc = _PC(g, case["sh_degree"])
    cam = _cam_obj(case["cam"])
    pipe = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    with torch.no_grad():
        out = renderer.render(cam, pc, pipe, a["bg"], scaling_modifier=case["scale_modifier"])

    def rasterize(shs=None, colors_precomp=None):
        """The reference rasterizer's pass: this repository's exact-image pass, checked bit for bit against the reference's."""
        b = dict(a)
        b["shs"], b["colors_precomp"] = shs, colors_precomp
        fw = run_ours(b, exact=True)
        ref = ref_forward("wrapper", "render_%s_%s" % (name, "sh" if shs is not None else "precomp"), b, names=("color", "depth", "alpha", "radii"))
        for k in ("color", "depth", "alpha", "radii"):
            assert same(fw[k], ref[k]), k
        return fw["color"].clone(), fw["depth"].clone(), fw["alpha"].clone(), fw["radii"].clone()
    ref = WR.render_two_pass(rasterize, a["means3D"], a["shs"], a["opacities"], a["scales"], a["rotations"], case["sh_degree"],
                             dict(campos=a["campos"], viewmatrix=a["view"], FoVx=cam.FoVx, FoVy=cam.FoVy), a["bg"])
    assert set(out) == {"render", "depth", "normal", "pseudo_normal", "viewspace_points", "visibility_filter", "radii"}
    assert out["render"].shape == ref["render"].shape and torch.equal(out["render"], ref["render"])
    assert out["depth"].shape == ref["depth"].shape and torch.equal(out["depth"], ref["depth"])
    assert torch.equal(out["radii"], ref["radii"]) and torch.equal(out["visibility_filter"], ref["radii"] > 0)
    assert maxabs(out["normal"], ref["normal"]) < 1e-4
    assert maxabs(out["pseudo_normal"], ref["pseudo_normal"]) < 5e-3
    assert out["viewspace_points"].shape == a["means3D"].shape and float(out["viewspace_points"].abs().max()) == 0.0


def test_render_with_gradients_keeps_the_graph():
    from autovfx_b200 import renderer
    case = case_inputs("small_sh")
    a = resolve(case, DEV)
    g = {k: v.to(DEV) for k, v in case["g"].items()}
    cam = _cam_obj(case["cam"])
    pipe = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    with torch.no_grad():
        fused = renderer.render(cam, _PC(g, case["sh_degree"]), pipe, a["bg"])
    pc = _PC(g, case["sh_degree"], requires_grad=True)
    out = renderer.render(cam, pc, pipe, a["bg"])
    assert maxabs(out["render"], fused["render"]) < 1e-6 and maxabs(out["depth"], fused["depth"]) < 1e-6
    assert maxabs(out["normal"], fused["normal"]) < 1e-4
    loss = out["render"].sum() + out["depth"].sum() + out["normal"].sum() + out["pseudo_normal"].sum()
    loss.backward()
    assert pc._xyz.grad is not None and torch.isfinite(pc._xyz.grad).all() and float(pc._xyz.grad.abs().max()) > 0
    assert out["viewspace_points"].grad is not None


def test_render_python_sh_and_cov_paths():
    """pipe.convert_SHs_python / pipe.compute_cov3D_python (GR/:116-141): same image within fp32 round-off of the in-kernel paths."""
    from autovfx_b200 import renderer
    from tests.helpers import cov3d_from
    case = case_inputs("small_sh")
    a = resolve(case, DEV)
    g = {k: v.to(DEV) for k, v in case["g"].items()}
    cam = _cam_obj(case["cam"])
    pc = _PC(g, case["sh_degree"])
    pc.get_covariance = lambda mod: cov3d_from(g["scales"], g["rotations"], mod)
    base = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    py = types.SimpleNamespace(debug=False, compute_cov3D_python=True, convert_SHs_python=True)
    with torch.no_grad():
        o0 = renderer.render(cam, pc, base, a["bg"])
        o1 = renderer.render(cam, pc, py, a["bg"])
    assert maxabs(o0["render"], o1["render"]) < 2e-3  # colours/covariances computed by torch ops differ in the last bits; rare skip flips
    assert float((o0["render"] - o1["render"]).abs().mean()) < 1e-5


@pytest.mark.parametrize("pack8", [False, True])
def test_frame_loop_product_mode(pack8):
    """FrameLoop(product=True): every frame equals render() called per camera; pack8 hands off the 8-bit bytes."""
    from autovfx_b200 import renderer, scene
    from autovfx_b200.render_loop import FrameLoop, pack_cameras
    case = case_inputs("config1")
    g = {k: v.to(DEV) for k, v in case["g"].items()}
    traj = scene.trajectory_dict(radius=3.5, num_views=5, theta=30.0, w=160, h=120)
    cams = scene.cameras_from_trajectory(traj)
    loop = FrameLoop(g, 3, 160, 120, device=DEV, ring=2, to_host=True, product=True, pack8=pack8)
    got = {}

    def consume(i, frame, stats):
        got[i] = {k: v.clone() for k, v in frame.items()}
    stats = loop.render(pack_cameras(cams), consume)
    assert len(stats) == 5 and all(s["overflow"] == 0 for s in stats)
    pipe = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    pc = _PC(g, 3)
    for i, cam in enumerate(cams):
        with torch.no_grad():
            ref = renderer.render(_cam_obj(cam), pc, pipe, torch.zeros(3, device=DEV))
        if not pack8:
            fr = got[i]["frame"].to(DEV)
            assert torch.equal(fr[0:3], ref["render"][0:3]) and torch.equal(fr[4], ref["render"][3]) and torch.equal(fr[3], ref["depth"])
            assert maxabs(got[i]["normal"], ref["normal"]) < 1e-6
            assert maxabs(got[i]["pseudo_normal"], ref["pseudo_normal"]) < 5e-3
        else:
            packed = renderer.pack_frame(ref["render"][0:3], ref["render"][3], ref["depth"], ref["normal"], 3.0)
            assert torch.equal(got[i]["rgba8"].to(DEV), packed["rgba8"])
            assert torch.equal(got[i]["depth8"].to(DEV), packed["depth8"])
            assert int((got[i]["normal8"].to(DEV).int() - packed["normal8"].int()).abs().max()) <= 1  # inverse computed per call: last-bit normal differences
            assert torch.equal(got[i]["depth"].to(DEV), ref["depth"])
    assert loop.d2h_bytes_per_frame == (120 * 160 * (4 + 4 + 1 + 3) if pack8 else 120 * 160 * 4 * (5 + 3 + 3))
