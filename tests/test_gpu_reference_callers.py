"""The reference's OWN Python callers of the hot path, executed on the GPU box against the drop-in (SURVEY §8 rows a17, a19, b, f-1..f-4).

What the reference's ``render()`` (gaussian_renderer/__init__.py:83-218), ``GaussianModel`` (scene/gaussian_model.py: activations,
get_normal, create_from_pcd -> distCUDA2, save_ply / load_ply), ``Camera`` (scene/cameras.py) and ``transform_gaussians`` /
``merge_two_gaussians`` (gaussians_utils.py:71-125) computed on their own rasterizer and kNN is stored under
tests/golden/ref_callers*.npz; ``rp`` runs that code (``oracle/ref_py.py``, staged by ``make -C oracle refpy``) only when
those values are recorded.  This repository's side is the drop-in package (``diff_gaussian_rasterization``, ``simple_knn._C``)
driven by the torch restatement of the callers (tests/wrapper_ref.py) or the product's own API.
"""
import math
import os

import numpy as np
import pytest
import torch

from tests import helpers as Hh
from tests import wrapper_ref as WR
from tests.test_wrapper_cpu import _raw, _rot
from autovfx_b200 import scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def rp():
    """oracle.ref_py when recording the reference's values, else None (the stored values are used)."""
    if not Hh.RECORD_DIR:
        return None
    from oracle import ref_py
    assert ref_py.available(), "recording needs oracle/_ref and oracle/_ref_py (make -C oracle ref refpy)"
    return ref_py


def _camera(Rm, T, fovx, fovy, W, H, c2w, fx):
    """The matrices of the reference's Camera: the view and projection of scene.camera_from_c2w (equal to the reference's,
    test_reference_camera_class_matches_scene_helpers) and the centre inverted on the GPU as Camera does."""
    cam = scene.camera_from_c2w(c2w, fx, fx, W, H)
    wv = cam.world_view_transform.to(DEV)
    return dict(world_view_transform=wv, full_proj_transform=cam.full_proj_transform.to(DEV), camera_center=wv.inverse()[3, :3],
                FoVx=fovx, FoVy=fovy, image_width=W, image_height=H)


def _dropin_render(cam, g, sh_degree, bg, means2D=None):
    """render() (tests/wrapper_ref.py restatement) on the drop-in diff_gaussian_rasterization.GaussianRasterizer."""
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    st = GaussianRasterizationSettings(image_height=cam["image_height"], image_width=cam["image_width"], tanfovx=math.tan(cam["FoVx"] * 0.5),
                                       tanfovy=math.tan(cam["FoVy"] * 0.5), bg=bg, scale_modifier=1.0, viewmatrix=cam["world_view_transform"],
                                       projmatrix=cam["full_proj_transform"], sh_degree=sh_degree, campos=cam["camera_center"], prefiltered=False,
                                       debug=False)
    rast = GaussianRasterizer(st)
    m2 = torch.zeros_like(g["means3D"]) if means2D is None else means2D

    def rasterize(shs=None, colors_precomp=None):
        return rast(means3D=g["means3D"], means2D=m2, shs=shs, colors_precomp=colors_precomp, opacities=g["opacities"], scales=g["scales"],
                    rotations=g["rotations"], cov3D_precomp=None)
    out = WR.render_two_pass(rasterize, g["means3D"], g["shs"], g["opacities"], g["scales"], g["rotations"], sh_degree,
                             dict(campos=cam["camera_center"], viewmatrix=cam["world_view_transform"], FoVx=cam["FoVx"], FoVy=cam["FoVy"]), bg)
    out["visibility_filter"] = out["radii"] > 0
    return out


def _scene_raw(N, M, seed, spread=1.0, log_scale=-3.3):
    r = _raw(N, M, seed)
    r["xyz"] = r["xyz"] * spread
    r["scaling"] = r["scaling"] * 0.6 + (log_scale + 3.0)
    r["f_dc"] = r["f_dc"] * 0.5
    return r


def _cam_args(eye=(0.4, -3.2, 0.6), target=(0, 0, 0), W=160, H=112, fovx_deg=58.0):
    """R, T, FoVx, FoVy exactly as scene_representation.py:144-156 derives them from a c2w."""
    eye, target = np.asarray(eye, np.float64), np.asarray(target, np.float64)
    Rc = scene.rotm_from_lookat(target - eye, np.asarray((0.0, 0.0, 1.0)))
    c2w = np.vstack((np.hstack((Rc, eye.reshape(3, 1))), np.array([0, 0, 0, 1])))
    w2c = np.linalg.inv(c2w)
    fx = W / (2 * math.tan(math.radians(fovx_deg) / 2))
    return np.transpose(w2c[:3, :3]), w2c[:3, 3], scene.focal2fov(fx, W), scene.focal2fov(fx, H), W, H, c2w, fx


def test_reference_camera_class_matches_scene_helpers(rp):
    """scene/cameras.py Camera (the reference's own class) vs autovfx_b200.scene.camera_from_c2w: identical matrices."""
    R, T, fovx, fovy, W, H, c2w, fx = _cam_args()

    def compute():
        cam = rp.make_camera(rp.load("ref"), R, T, fovx, fovy, W, H)
        return {"world_view_transform": cam.world_view_transform, "full_proj_transform": cam.full_proj_transform,
                "camera_center": cam.camera_center, "size": np.array([cam.image_width, cam.image_height]), "fov": np.array([cam.FoVx, cam.FoVy])}
    cam = Hh.reference("callers", "camera", compute)
    mine = scene.camera_from_c2w(c2w, fx, fx, W, H)
    assert Hh.same(mine.world_view_transform, cam["world_view_transform"])
    assert Hh.same(mine.full_proj_transform, cam["full_proj_transform"])
    # the reference inverts the view matrix on the GPU (cuSOLVER), scene.py on the CPU (LAPACK): last-bit differences only
    assert torch.allclose(torch.from_numpy(cam["camera_center"]), mine.camera_center, rtol=0, atol=1e-6)
    assert cam["size"].tolist() == [W, H] and cam["fov"].tolist() == [mine.FoVx, mine.FoVy]


def _ref_render(rp, group, key, raw, M, deg, cam_args, bg, full=()):
    """The reference's render() on its own rasterizer, for the stored values."""
    def compute():
        ns = rp.load("ref")
        Rm, T, fovx, fovy, W, H, _, _ = cam_args
        pc = rp.make_model(ns, raw, int(math.isqrt(M)) - 1, deg)
        cam = rp.make_camera(ns, Rm, T, fovx, fovy, W, H)
        with torch.no_grad():
            o = ns.renderer.render(cam, pc, rp.Pipe(), bg)
        return {k: o[k] for k in ("render", "depth", "normal", "pseudo_normal", "radii", "visibility_filter")}
    return Hh.reference(group, key, compute, full=full)


@pytest.mark.parametrize("M,deg", [(16, 3), (25, 1), (25, 3)])
def test_reference_render_on_dropin_equals_reference_render_on_reference(rp, M, deg):
    """render() with `diff_gaussian_rasterization` = this repo's drop-in, against the reference's render() on the reference's
    Python + CUDA rasterizer.  Exact image mode: every output bit-identical (the torch post-processing is the same computation
    fed identical rasterizer outputs).  Default mode: within the 1e-4 image tolerance."""
    from autovfx_b200 import rasterizer as R
    raw = _scene_raw(5000, M, 11)
    cam_args = _cam_args()
    bg = torch.tensor([0.1, 0.3, 0.2], device=DEV)
    want = _ref_render(rp, "callers_render", "dropin_%d_%d" % (M, deg), raw, M, deg, cam_args, bg)
    cam = _camera(*cam_args)
    g = WR.activate({k: v.to(DEV) for k, v in raw.items()})
    outs = {}
    for exact in (True, False):
        R.set_exact_images(exact)
        try:
            with torch.no_grad():
                outs[exact] = {k: v.detach().clone() for k, v in _dropin_render(cam, g, deg, bg).items()}
        finally:
            R.set_exact_images(False)
    ex = outs[True]
    for k in ("render", "depth", "normal", "pseudo_normal", "radii", "visibility_filter"):
        assert Hh.same(ex[k], want[k]), k
    fast = outs[False]
    assert Hh.same(fast["radii"], want["radii"])
    assert Hh.maxabs(fast["render"], ex["render"]) <= 1e-5 and Hh.maxabs(fast["depth"], ex["depth"]) <= 5e-5
    assert Hh.maxabs(fast["normal"], ex["normal"]) <= 1e-4


@pytest.mark.parametrize("M,deg", [(16, 3), (25, 2)])
def test_fused_render_matches_reference_render(rp, M, deg):
    """autovfx_b200.renderer.render (axis normals + ONE 6-channel pass + normal-map kernel) fed the activations and camera of the
    reference's GaussianModel and Camera, against the reference's render() on the reference rasterizer."""
    import types
    from autovfx_b200 import rasterizer as R, renderer as RD
    raw = _scene_raw(6000, M, 5)
    cam_args = _cam_args(eye=(-2.0, -2.4, 1.1), W=176, H=96)
    bg = torch.tensor([0.0, 0.0, 0.0], device=DEV)
    want = _ref_render(rp, "callers_fused", "fused_%d_%d" % (M, deg), raw, M, deg, cam_args, bg, full=("normal", "pseudo_normal"))
    g = WR.activate({k: v.to(DEV) for k, v in raw.items()})
    pc = types.SimpleNamespace(get_xyz=g["means3D"], get_features=g["shs"], get_opacity=g["opacities"], get_scaling=g["scales"],
                               get_rotation=g["rotations"], active_sh_degree=deg, max_sh_degree=int(math.isqrt(M)) - 1)
    cam = types.SimpleNamespace(**_camera(*cam_args))
    with torch.no_grad():
        R.set_exact_images(True)
        try:
            got = RD.render(cam, pc, rp_pipe(), bg)
        finally:
            R.set_exact_images(False)
        fast = RD.render(cam, pc, rp_pipe(), bg)
    assert Hh.same(got["render"], want["render"]) and Hh.same(got["depth"], want["depth"]) and Hh.same(got["radii"], want["radii"])
    assert Hh.same(got["visibility_filter"], want["visibility_filter"])
    # blended normal image: the per-Gaussian normals differ in the last bit (torch norm reduction order)
    assert Hh.maxabs(got["normal"], want["normal"]) <= 1e-4
    # pseudo normal: normalised cross product of depth differences (cancellation): compare directions where the normal is defined
    a, b = got["pseudo_normal"].cpu(), torch.from_numpy(want["pseudo_normal"])
    defined = (b.norm(dim=-1) > 0.5) & (a.norm(dim=-1) > 0.5)
    cos = (a * b).sum(-1)[defined]
    assert defined.float().mean() > 0.5 and float((cos > 1 - 5e-3).float().mean()) > 0.999
    assert Hh.maxabs(fast["render"], got["render"]) <= 1e-5 and Hh.maxabs(fast["depth"], got["depth"]) <= 5e-5


def rp_pipe():
    """pipeline parameters render() reads (arguments/__init__.py PipelineParams)."""
    import types
    return types.SimpleNamespace(convert_SHs_python=False, compute_cov3D_python=False, debug=False)


def test_training_step_through_reference_render_gradients(rp):
    """Backward through render() (two rasterizer passes, gradients w.r.t. the raw GaussianModel parameters) on the drop-in vs the
    reference's render() on its autograd front end + CUDA backward."""
    raw = _scene_raw(3000, 16, 23)
    cam_args = _cam_args(W=128, H=96)
    Rm, T, fovx, fovy, W, H, _, _ = cam_args
    bg = torch.tensor([0.2, 0.2, 0.2], device=DEV)
    gen = torch.Generator().manual_seed(3)
    w_img, w_d, w_n = torch.randn(4, H, W, generator=gen).to(DEV), torch.randn(H, W, generator=gen).to(DEV), torch.randn(H, W, 3, generator=gen).to(DEV)
    names = ("xyz", "f_dc", "f_rest", "opacity", "scaling", "rotation", "screen")

    def compute():
        ns = rp.load("ref")
        pc = rp.make_model(ns, raw, 3, 3)
        cam = rp.make_camera(ns, Rm, T, fovx, fovy, W, H)
        o = ns.renderer.render(cam, pc, rp.Pipe(), bg)
        loss = (o["render"] * w_img).sum() + (o["depth"] * w_d).sum() + (o["normal"] * w_n).sum()
        loss.backward()
        return dict(zip(names, (pc._xyz.grad, pc._features_dc.grad, pc._features_rest.grad, pc._opacity.grad, pc._scaling.grad,
                                pc._rotation.grad, o["viewspace_points"].grad)))
    want = Hh.reference("callers_grads", "training_step", compute, full=names)
    leaves = {k: v.to(DEV).float().contiguous().requires_grad_(True) for k, v in raw.items()}
    screen = torch.zeros_like(leaves["xyz"], requires_grad=True)
    o = _dropin_render(_camera(*cam_args), WR.activate(leaves), 3, bg, means2D=screen)
    loss = (o["render"] * w_img).sum() + (o["depth"] * w_d).sum() + (o["normal"] * w_n).sum()
    loss.backward()
    got = dict(zip(names, (leaves["xyz"].grad, leaves["f_dc"].grad, leaves["f_rest"].grad, leaves["opacity"].grad, leaves["scaling"].grad,
                           leaves["rotation"].grad, screen.grad)))
    for k, g in got.items():
        assert g is not None, k
        assert Hh.relerr(g, want[k]) < 3e-4, k


def test_create_from_pcd_uses_distcuda2(rp):
    """GaussianModel.create_from_pcd (gaussian_model.py:134-157), the only real distCUDA2 call site: initial log-scales from the
    drop-in simple_knn._C vs the reference's simple-knn CUDA."""
    from simple_knn._C import distCUDA2
    gen = np.random.default_rng(4)
    pts = (gen.standard_normal((20000, 3)) * np.array([2.0, 1.0, 0.4])).astype(np.float32)
    cols = gen.random((20000, 3)).astype(np.float32)

    def compute():
        ns = rp.load("ref")
        pcd = ns.graphics_utils.BasicPointCloud(points=pts, colors=cols, normals=np.zeros_like(pts))
        m = ns.gaussian_model.GaussianModel(3)
        m.create_from_pcd(pcd, 1.0)
        return {"scaling": m._scaling, "xyz": m._xyz, "f_dc": m._features_dc, "opacity": m._opacity, "rotation": m._rotation}
    b = Hh.reference("callers", "create_from_pcd", compute, full=("scaling",))
    # create_from_pcd's initial parameters: log(sqrt(clamped squared kNN distance)) per axis, the points, RGB2SH colours, opacity 0.1
    dist2 = torch.clamp_min(distCUDA2(torch.from_numpy(pts).float().to(DEV)), 0.0000001)
    scaling = torch.log(torch.sqrt(dist2))[..., None].repeat(1, 3)
    assert torch.allclose(scaling.cpu(), torch.from_numpy(b["scaling"]), rtol=0, atol=2e-6) and Hh.same(torch.from_numpy(pts), b["xyz"])
    C0 = 0.28209479177387814
    assert Hh.same(((torch.from_numpy(cols).float().to(DEV) - 0.5) / C0)[:, None, :], b["f_dc"])
    opacity = torch.log(0.1 * torch.ones((20000, 1), dtype=torch.float, device=DEV) / (1 - 0.1 * torch.ones((20000, 1), dtype=torch.float, device=DEV)))
    rots = torch.zeros((20000, 4), device=DEV)
    rots[:, 0] = 1
    assert Hh.same(opacity, b["opacity"]) and Hh.same(rots, b["rotation"])


@pytest.mark.parametrize("M", [16, 25])
def test_activations_match_reference_gaussian_model(rp, M):
    """edit.activate (gsr_activate_gaussians) vs the reference GaussianModel's get_* properties (gaussian_model.py:95-115); the
    tolerance-compared ones over a seeded sample of 4096 Gaussians."""
    from autovfx_b200 import edit
    raw = _scene_raw(40000, M, 9)
    idx = torch.randperm(40000, generator=torch.Generator().manual_seed(M))[:4096].to(DEV)

    def compute():
        pc = rp.make_model(rp.load("ref"), raw, int(math.isqrt(M)) - 1, 0)
        with torch.no_grad():
            return {"xyz": pc.get_xyz, "features": pc.get_features, "scaling": pc.get_scaling, "opacity": pc.get_opacity[idx],
                    "rotation": pc.get_rotation[idx]}
    want = Hh.reference("callers", "activations_%d" % M, compute, full=("opacity", "rotation"))
    got = edit.activate({k: v.to(DEV) for k, v in raw.items()}, DEV)
    assert Hh.same(got["means3D"], want["xyz"]) and Hh.same(got["shs"], want["features"])
    assert Hh.same(got["scales"], want["scaling"])
    assert Hh.maxabs(got["opacities"][idx], want["opacity"]) <= 1.2e-7
    assert Hh.maxabs(got["rotations"][idx], want["rotation"]) <= 2.4e-7


def test_get_normal_matches_reference(rp):
    """renderer.axis_normals (gsr_axis_normals) vs GaussianModel.get_normal (gaussian_model.py:120-128), over a seeded sample of
    4096 Gaussians."""
    from autovfx_b200 import renderer as RD
    raw = _scene_raw(50000, 16, 13)
    campos = torch.tensor([0.3, -2.0, 0.7], device=DEV)
    idx = torch.randperm(50000, generator=torch.Generator().manual_seed(13))[:4096].to(DEV)

    def compute():
        pc = rp.make_model(rp.load("ref"), raw, 3, 3)
        with torch.no_grad():
            d = pc.get_xyz - campos
            d = d / d.norm(dim=1, keepdim=True)
            return {"normal": pc.get_normal(dir_pp_normalized=d)[idx]}
    want = Hh.reference("callers", "get_normal", compute, full=("normal",))
    g = WR.activate({k: v.to(DEV) for k, v in raw.items()})
    with torch.no_grad():
        got = RD.axis_normals(g["means3D"], g["scales"], g["rotations"], campos, remap01=False)
    assert Hh.maxabs(got[idx], want["normal"]) <= 5e-7


def test_transform_and_merge_match_reference(rp):
    """edit.ResidentScene.compose vs the reference's transform_gaussians + merge_two_gaussians executed from gaussians_utils.py
    (:71-125), then both scenes through the rasterizer."""
    from autovfx_b200 import edit
    M = 25
    scene_raw, obj_raw = _scene_raw(8000, M, 1), _scene_raw(1500, M, 2, spread=0.3)
    Rot = _rot(5)
    center, init_c, scaling = torch.tensor([0.4, -0.2, 0.3]), torch.tensor([0.05, 0.02, -0.01]), 1.7
    Rm, T, fovx, fovy, W, H, c2w, fx = _cam_args(W=144, H=96)
    cam = scene.camera_from_c2w(c2w, fx, fx, W, H).to(DEV)
    a = dict(means3D=None, opacities=None, view=cam.world_view_transform, proj=cam.full_proj_transform, campos=cam.camera_center, W=W, H=H,
             tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, sh_degree=0, scale_modifier=1.0, bg=torch.zeros(3, device=DEV),
             shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None)
    keys = ("means3D", "opacities", "shs", "scales", "rotations")

    def compute():
        ns = rp.load("ref")
        bg_model, obj_model = rp.make_model(ns, scene_raw, 4, 0), rp.make_model(ns, obj_raw, 4, 0)
        with torch.no_grad():
            moved = ns.gaussians_utils.transform_gaussians(obj_model, center.to(DEV), Rot.to(DEV), scaling, init_c.to(DEV))
            merged = ns.gaussians_utils.merge_two_gaussians(bg_model, moved)
            want = {"means3D": merged.get_xyz, "shs": merged.get_features, "opacities": merged.get_opacity, "scales": merged.get_scaling,
                    "rotations": merged.get_rotation}
        b = dict(a)
        b.update({k: want[k].contiguous() for k in keys})
        b["sh_degree"] = merged.active_sh_degree
        out = {"color": Hh.run_ref(b)["color"], "active_sh_degree": merged.active_sh_degree}
        out.update(want)
        return out
    want = Hh.reference("callers_merge", "transform_and_merge", compute, full=("means3D", "opacities", "scales", "rotations", "color"))
    rs = edit.ResidentScene({k: v.to(DEV) for k, v in scene_raw.items()}, {"obj": {k: v.to(DEV) for k, v in obj_raw.items()}}, DEV)
    got = rs.compose({"obj": (center, Rot, scaling, init_c)})
    w = {k: torch.from_numpy(want[k]).to(DEV) for k in keys if k != "shs"}
    assert got["means3D"].shape == w["means3D"].shape
    assert Hh.maxabs(got["means3D"], w["means3D"]) <= 2e-6 and Hh.same(got["shs"], want["shs"])
    assert Hh.maxabs(got["scales"], w["scales"]) <= 1e-6 * float(w["scales"].max()) + 1e-9
    assert Hh.maxabs(got["opacities"], w["opacities"]) <= 1.2e-7 and Hh.maxabs(got["rotations"], w["rotations"]) <= 1e-6
    # the merged model renders at active_sh_degree 0 (gaussians_utils.py:75 builds GaussianModel(4): active degree 0)
    assert int(want["active_sh_degree"]) == 0
    imgs = []
    # the reference-built SH coefficients (transform_gaussians leaves them as they are), checked against the stored digest
    w["shs"] = WR.activate(WR.merge_two_gaussians(*[{k: v.to(DEV) for k, v in r.items()} for r in (scene_raw, obj_raw)]))["shs"]
    assert Hh.same(w["shs"], want["shs"])
    for tag, src in (("got", got), ("want", w)):
        b = dict(a)
        b.update({k: src[k].contiguous() for k in keys})
        imgs.append((Hh.run_ours(b, exact=True)["color"].clone(), Hh.ref_forward("callers_merge", "render_" + tag, b, names=("color", "radii"))))
    for ours_c, ref_o in imgs:  # each parameter set: drop-in == reference rasterizer, bit for bit
        assert Hh.same(ours_c, ref_o["color"])
    assert Hh.maxabs(imgs[0][0], want["color"]) <= 2e-4  # composed on the GPU vs composed by the reference's torch ops


def test_ply_round_trip_with_reference_gaussian_model(rp, tmp_path):
    """save_ply written by the reference GaussianModel is read by scene.load_ply, and scene.save_ply is read by the reference's
    load_ply (gaussian_model.py:201-266): identical raw parameters both ways; both files are byte-identical."""
    M = 16
    raw = _scene_raw(3000, M, 31)
    n = lambda t: t.detach().cpu().numpy()  # noqa: E731
    p_ours = str(tmp_path / "ours.ply")
    scene.save_ply(p_ours, n(raw["xyz"]), n(raw["f_dc"]), n(raw["f_rest"]), n(raw["opacity"]), n(raw["scaling"]), n(raw["rotation"]))

    def compute():
        ns = rp.load("ref")
        pc = rp.make_model(ns, raw, 3, 3)
        p_ref = str(tmp_path / "ref" / "point_cloud.ply")
        pc.save_ply(p_ref)
        back = ns.gaussian_model.GaussianModel(3)
        back.load_ply(p_ours)
        out = {"file": np.frombuffer(open(p_ref, "rb").read(), dtype=np.uint8)}
        out.update({k: getattr(back, "_" + k) for k in ("xyz", "features_dc", "features_rest", "opacity", "scaling", "rotation")})
        return out
    want = Hh.reference("callers", "ply_round_trip", compute)
    data = open(p_ours, "rb").read()
    assert Hh.same(np.frombuffer(data, dtype=np.uint8), want["file"])  # the reference's save_ply wrote these very bytes
    mine = scene.load_ply(p_ours)
    for k, kk in (("xyz", "xyz"), ("f_dc", "f_dc"), ("f_rest", "f_rest"), ("opacity", "opacity"), ("scale", "scaling"), ("rot", "rotation")):
        assert np.array_equal(mine[k], n(raw[kk])), k
    # the reference's load_ply read scene.save_ply's file back to the raw parameters
    for k, kk in (("xyz", "xyz"), ("features_dc", "f_dc"), ("features_rest", "f_rest"), ("opacity", "opacity"), ("scaling", "scaling"),
                  ("rotation", "rotation")):
        assert Hh.same(raw[kk].float().contiguous(), want[k]), k


def test_sugar_style_call_offcentre_projection_and_python_sh(rp):
    """The SuGaR wrapper's call shape (sugar_model.py:2010-2071): M = 25 storage, colours from the reference's Python eval_sh
    (utils/sh_utils.py) passed as colors_precomp, and a projection matrix whose principal point is patched off-centre
    (proj[2,0], proj[2,1] overwritten, sugar_model.py:2029-2030) — drop-in vs compiled reference, bit for bit."""
    g = scene.synthetic_gaussians(20000, seed=77, extent=(1.2, 1.2, 0.6), log_scale_mean=math.log(0.02), log_scale_std=0.5, sh_degree=4)
    cam = scene.lookat_camera((0.5, -3.0, 0.8), (0, 0, 0), 208, 144, 62.0)
    view = cam.world_view_transform.clone()
    proj = scene.projection_matrix(0.01, 100.0, cam.FoVx, cam.FoVy).transpose(0, 1).contiguous()
    proj[2, 0], proj[2, 1] = -0.11, 0.07  # principal point away from the image centre
    full = (view.unsqueeze(0).bmm(proj.unsqueeze(0))).squeeze(0).contiguous()
    a = Hh.resolve(dict(g=g, cam=cam, sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0), DEV)
    a["proj"] = full.to(DEV)

    def compute():
        ns = rp.load("ref")
        with torch.no_grad():
            d = a["means3D"] - a["campos"]
            d = d / d.norm(dim=1, keepdim=True)
            shs_view = a["shs"].transpose(1, 2).reshape(-1, 3, 25)
            return {"rgb": torch.clamp_min(ns.sh_utils.eval_sh(3, shs_view, d) + 0.5, 0.0).contiguous()}
    rgb = torch.from_numpy(Hh.reference("callers_sugar", "python_sh", compute, full=("rgb",))["rgb"]).to(DEV)
    b = dict(a)
    b["shs"], b["colors_precomp"] = None, rgb
    for tag, case in (("sh", a), ("precomp", b)):  # SH evaluated by the rasterizer at an off-centre projection, and the Python-SH colors_precomp call
        ours = Hh.run_ours(case, exact=True, for_backward=True)
        ours = {k: ours[k].clone() for k in ("color", "depth", "alpha", "radii")}
        ref = Hh.ref_forward("callers_sugar", tag, case)
        for k in ("color", "depth", "alpha", "radii"):
            assert Hh.same(ours[k], ref[k]), k
        Hh.assert_images_close(Hh.run_ours(case), ours)  # = against the reference's images
    # the CUDA SH evaluation agrees with the reference's Python eval_sh to float rounding
    assert Hh.maxabs(Hh.run_ours(a)["color"], Hh.run_ours(b)["color"]) <= 2e-5


def test_config2_one_million_through_the_ply_path(rp, tmp_path):
    """BASELINE config 2 stand-in (SURVEY §8d): P = 1,000,000, seed 1, 4-unit scene, written and re-read through the 3DGS .ply vertex
    layout, activated on the GPU, one 1920x1080 camera, forward — drop-in vs compiled reference, bit for bit (exact image mode),
    and the default mode within tolerance."""
    from autovfx_b200 import edit
    raw = scene.config2_raw()
    path = str(tmp_path / "config2.ply")
    n = lambda t: t.numpy()  # noqa: E731
    scene.save_ply(path, n(raw["xyz"]), n(raw["f_dc"]), n(raw["f_rest"]), n(raw["opacity"]), n(raw["scaling"]), n(raw["rotation"]))
    assert os.path.getsize(path) > 1_000_000 * 62 * 4
    loaded = scene.load_ply(path)
    g = edit.activate({"xyz": torch.from_numpy(loaded["xyz"]), "f_dc": torch.from_numpy(loaded["f_dc"]), "f_rest": torch.from_numpy(loaded["f_rest"]),
                       "opacity": torch.from_numpy(loaded["opacity"]), "scaling": torch.from_numpy(loaded["scale"]),
                       "rotation": torch.from_numpy(loaded["rot"])}, DEV)
    cam = scene.config2_camera()
    a = Hh.resolve(dict(g=g, cam=cam, sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0), DEV)
    ours = Hh.run_ours(a, exact=True, debug=False)
    ours = {k: ours[k].clone() for k in ("color", "depth", "alpha", "radii")} | {"num_rendered": ours["stats"]["num_rendered"]}
    ref = Hh.ref_forward("callers", "config2", a)
    assert int(ref["num_rendered"]) == ours["num_rendered"] > 1_000_000
    for k in ("color", "depth", "alpha", "radii"):
        assert Hh.same(ours[k], ref[k]), k
    Hh.assert_images_close(Hh.run_ours(a, debug=False), ours)  # = against the reference's images
    # the reference's own loader reads the same file to the same parameters (subset check: its per-property Python loops are slow)
    small = str(tmp_path / "small.ply")
    sl = slice(0, 20000)
    scene.save_ply(small, loaded["xyz"][sl], loaded["f_dc"][sl], loaded["f_rest"][sl], loaded["opacity"][sl], loaded["scale"][sl], loaded["rot"][sl])

    def compute():
        m = rp.load("ref").gaussian_model.GaussianModel(3)
        m.load_ply(small)
        with torch.no_grad():
            return {"xyz": m.get_xyz, "features": m.get_features, "scaling": m.get_scaling}
    want = Hh.reference("callers", "config2_load_ply", compute)
    assert Hh.same(g["means3D"][sl], want["xyz"]) and Hh.same(g["shs"][sl], want["features"]) and Hh.same(g["scales"][sl], want["scaling"])
