"""GPU parity of the activation / per-frame edit row (SURVEY §8 f-3, f-4): gsr_activate_gaussians through autovfx_b200.edit
against the torch restatement of the reference's transform_gaussians + merge_two_gaussians + GaussianModel activations run
with torch's CUDA kernels, and the rendered result of a composed scene against the reference rasterizer's (tests/golden/)."""
import numpy as np
import pytest
import torch

from tests import wrapper_ref as WR
from tests.helpers import maxabs
from tests.test_wrapper_cpu import _raw, _rot

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


def _to(d, dev=DEV):
    return {k: v.to(dev) for k, v in d.items()}


@pytest.mark.parametrize("M", [16, 25, 1])
def test_activate_matches_torch(M):
    from autovfx_b200 import edit
    raw = _to(_raw(50_000, M, 1)) if M > 1 else _to({**_raw(50_000, 2, 1), "f_rest": torch.zeros(50_000, 0, 3)})
    got = edit.activate(raw, DEV)
    ref = WR.activate(raw)
    assert torch.equal(got["means3D"], ref["means3D"]) and torch.equal(got["shs"], ref["shs"])
    assert torch.equal(got["scales"], ref["scales"])  # expf is the same libdevice routine torch calls
    assert maxabs(got["opacities"], ref["opacities"]) <= 1.2e-7
    assert maxabs(got["rotations"], ref["rotations"]) <= 2.4e-7  # torch's norm reduction sums the four squares in another order
    assert got["shs"].shape == (50_000, M, 3) and got["opacities"].shape == (50_000, 1)


def test_transform_matches_torch():
    from autovfx_b200 import edit
    raw = _to(_raw(40_000, 16, 2))
    R = _rot(7)
    center, pivot, s = torch.tensor([0.4, -1.2, 0.3]), torch.tensor([0.1, 0.2, -0.5]), 1.7
    xf = edit.make_xform(center, R, s, pivot)
    got = edit.activate(raw, DEV, xform=xf)
    quat = torch.tensor(list(xf.quat), device=DEV)
    ref = WR.activate(WR.transform_gaussians(raw, center.to(DEV), R.to(DEV), s, pivot.to(DEV), quat=quat))
    assert maxabs(got["means3D"], ref["means3D"]) < 2e-6
    frac = float((got["means3D"] == ref["means3D"]).float().mean())
    assert frac > 0.9, frac  # the K=3 GEMM's accumulation order is the only unknown
    assert torch.equal(got["scales"], ref["scales"])
    assert maxabs(got["rotations"], ref["rotations"]) <= 3e-7
    assert torch.equal(got["shs"], ref["shs"])
    # the host quaternion agrees with an independent implementation
    qs = WR.matrix_to_quaternion(R)
    q = torch.tensor(list(xf.quat))
    assert float((q - qs).abs().max()) < 1e-6 or float((q + qs).abs().max()) < 1e-6


def test_resident_scene_compose_and_render():
    """Scene + two objects, one of them absent in the second frame: arrays equal the reference's merge, and the rendered
    frame equals the compiled reference rasterizer on the reference-built tensors."""
    from autovfx_b200 import edit, scene
    from autovfx_b200 import rasterizer as R
    from tests.helpers import ref_forward, same, settings_from
    scene_raw, objA, objB = _to(_raw(20_000, 16, 3)), _to(_raw(3_000, 16, 4)), _to(_raw(1_500, 16, 5))
    for r in (scene_raw, objA, objB):
        r["scaling"] = r["scaling"] - 1.0  # small splats
    rs = edit.ResidentScene(scene_raw, {"A": objA, "B": objB}, DEV)
    tfA = (torch.tensor([0.5, 0.0, 0.2]), _rot(1), 0.6, torch.tensor([0.0, 0.1, 0.0]))
    tfB = (torch.tensor([-0.7, 0.3, 0.0]), _rot(2), 1.3, torch.tensor([0.2, 0.0, 0.1]))
    cam = scene.lookat_camera((0.0, -4.5, 0.8), (0, 0, 0), 160, 120, 60.0)

    def reference_merge(tfs):
        merged = scene_raw
        for obj, tf in tfs:
            c, Rm, s, p = tf
            xf = edit.make_xform(c, Rm, s, p)
            t = WR.transform_gaussians(obj, c.to(DEV), Rm.to(DEV), s, p.to(DEV), quat=torch.tensor(list(xf.quat), device=DEV))
            merged = WR.merge_two_gaussians(merged, t)
        return WR.activate(merged)

    for frame, tfs in enumerate([{"A": tfA, "B": tfB}, {"B": tfB}]):
        got = rs.compose(tfs)
        ref = reference_merge([({"A": objA, "B": objB}[k], v) for k, v in tfs.items()])
        n = ref["means3D"].shape[0]
        assert got["means3D"].shape[0] == n == rs.count
        for k in ("means3D", "scales", "rotations", "opacities", "shs"):
            assert got[k].shape == ref[k].shape, k
            assert maxabs(got[k], ref[k]) < 3e-6, k
        a = dict(means3D=got["means3D"], opacities=got["opacities"], shs=got["shs"], scales=got["scales"], rotations=got["rotations"],
                 colors_precomp=None, cov3D_precomp=None, view=cam.world_view_transform.to(DEV), proj=cam.full_proj_transform.to(DEV),
                 campos=cam.camera_center.to(DEV), W=160, H=120, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, sh_degree=0, scale_modifier=1.0,
                 bg=torch.zeros(3, device=DEV))
        color, depth, alpha, radii, _ws, _t, _k = R.forward_raw(a["means3D"], a["shs"], None, a["opacities"], a["scales"], a["rotations"], None,
                                                               settings_from(a), sync=True)
        # same composed tensors through the reference rasterizer: bit-identical images
        fw = ref_forward("edit", "compose_%d" % frame, a, names=("color", "depth", "radii"))
        assert same(color, fw["color"]) and same(depth, fw["depth"]) and same(radii, fw["radii"])
        b = dict(a)
        for k in ("means3D", "scales", "rotations", "opacities", "shs"):
            b[k] = ref[k].contiguous()
        # reference-built tensors (torch ops): agree up to the few last-bit parameter differences
        fw2 = torch.from_numpy(ref_forward("edit", "compose_torch_%d" % frame, b, names=("color",), full=("color",))["color"]).to(DEV)
        assert float((color - fw2).abs().mean()) < 1e-6 and maxabs(color, fw2) < 5e-3


def test_edit_errors():
    from autovfx_b200 import edit
    raw = _to(_raw(100, 16, 6))
    rs = edit.ResidentScene(raw, {"A": _to(_raw(10, 16, 7))}, DEV)
    with pytest.raises(KeyError):
        rs.compose({"nope": (torch.zeros(3), torch.eye(3), 1.0, torch.zeros(3))})
    with pytest.raises(ValueError):
        edit.ResidentScene(raw, {"A": _to(_raw(10, 9, 7))}, DEV)  # SH storage mismatch
    with pytest.raises(RuntimeError):
        edit.activate_into({k: v.cpu() for k, v in raw.items()}, {k: v.cpu() for k, v in rs.arrays.items()})


def test_frame_loop_with_per_frame_edits():
    """FrameLoop.render(before_frame=compose): every frame shows the scene with that frame's object transform; equals rendering
    the composed tensors directly."""
    from autovfx_b200 import edit, scene
    from autovfx_b200 import rasterizer as R
    from autovfx_b200.render_loop import FrameLoop, pack_cameras
    from tests.helpers import settings_from
    scene_raw, obj = _to(_raw(8_000, 16, 11)), _to(_raw(2_000, 16, 12))
    for r in (scene_raw, obj):
        r["scaling"] = r["scaling"] - 1.0
    rs = edit.ResidentScene(scene_raw, {"A": obj}, DEV)
    cams = scene.cameras_from_trajectory(scene.trajectory_dict(radius=4.5, num_views=4, theta=25.0, w=128, h=96))
    tfs = [{"A": (torch.tensor([0.3 * i, 0.0, 0.1]), _rot(i), 1.0 + 0.2 * i, torch.zeros(3))} if i != 2 else {} for i in range(4)]
    loop = FrameLoop(rs.compose({}), 0, 128, 96, device=DEV, ring=2, to_host=True)
    got = {}
    loop.render(pack_cameras(cams), lambda i, fr, st: got.__setitem__(i, fr.clone()), before_frame=lambda i: rs.compose(tfs[i]))
    for i, cam in enumerate(cams):
        g = rs.compose(tfs[i])
        a = dict(view=cam.world_view_transform.to(DEV), proj=cam.full_proj_transform.to(DEV), campos=cam.camera_center.to(DEV), W=128, H=96,
                 tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, sh_degree=0, scale_modifier=1.0, bg=torch.zeros(3, device=DEV))
        color, depth, alpha, radii, _w, _t, _k = R.forward_raw(g["means3D"], g["shs"], None, g["opacities"], g["scales"], g["rotations"], None,
                                                               settings_from(a), sync=True)
        assert g["means3D"].shape[0] == (8_000 if i == 2 else 10_000)
        fr = got[i].to(DEV)
        assert torch.equal(fr[0:3], color) and torch.equal(fr[3:4], depth) and torch.equal(fr[4:5], alpha), i
