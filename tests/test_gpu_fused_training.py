"""Training through render() in one rasterizer pass: gsr_backward_multi (the backward of the 6-channel gsr_forward_multi),
rasterize_gaussians_multi and render()'s fused autograd path, against two single-image passes, the CPU oracle and the stored
gradients of the reference's own training step."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from tests import helpers as Hh
from tests.test_gpu_reference_callers import _cam_args, _camera, _scene_raw, rp_pipe
from tools.time_render_training import TrainableGaussians, training_loss

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")

GRAD_SHAPES = (("dL_dmeans2D", 3), ("dL_dconic", 4), ("dL_dopacity", 1), ("dL_dcolors", 3), ("dL_ddepths", 1), ("dL_dmeans3D", 3),
               ("dL_dcov3D", 6), ("dL_dsh", None), ("dL_dscales", 3), ("dL_drotations", 4))


def _forward(a, exact, extra=None, colors=None):
    """forward_raw(for_backward) of the case; ``colors`` replaces the SH / precomputed colours (the second pass of a frame)."""
    from autovfx_b200 import rasterizer as R
    shs, cp = (None, colors) if colors is not None else (a["shs"], a["colors_precomp"])
    eo = None if extra is None else torch.empty((3, a["H"], a["W"]), device=DEV)
    res = R.forward_raw(a["means3D"], shs, cp, a["opacities"], a["scales"], a["rotations"], a["cov3D_precomp"], Hh.settings_from(a),
                        for_backward=True, sync=True, exact=exact, extra=extra, extra_out=eo)
    return res, eo


def _backward(a, res, dc, dd, da, extra=None, de=None, dextra=None, multi=True):
    """gsr_backward_multi (or gsr_backward) through the C ABI on the workspaces of ``res``.  Returns (status, gradient buffers)."""
    from autovfx_b200 import _lib, rasterizer as R
    color, depth, alpha, radii, (geom, binning, image), _ticket, keep = res
    m3, shs, cp, _op, sc, ro, cov, bg, view, proj, campos, _ex = keep
    P = m3.shape[0]
    M = shs.shape[1] if shs is not None else 0
    fr = _lib.gsr_frame()
    R._fill_frame(fr, P, a["sh_degree"], M, a["W"], a["H"], Hh.settings_from(a), bg, m3, shs, cp, None, sc, ro, cov, view, proj, campos)
    ws = _lib.gsr_workspace(geom.data_ptr(), geom.numel(), binning.data_ptr(), binning.numel(), image.data_ptr(), image.numel())
    g = {k: torch.full((P, n) if n else (P, M, 3), float("nan"), device=DEV) for k, n in GRAD_SHAPES}
    gr = _lib.gsr_grads(*[R._ptr(g[k]) for k, _ in GRAD_SHAPES])
    st = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    p = R._ptr
    if multi:
        rc = _lib.lib.gsr_backward_multi(C.byref(fr), C.byref(ws), p(radii), p(alpha), p(dc), p(dd), p(da), p(extra), p(de), C.byref(gr),
                                         p(dextra), st)
    else:
        rc = _lib.lib.gsr_backward(C.byref(fr), C.byref(ws), p(radii), p(alpha), p(dc), p(dd), p(da), C.byref(gr), st)
    torch.cuda.synchronize()
    return rc, g


def _extra_inputs(a, seed=5):
    gen = torch.Generator().manual_seed(seed)
    P = a["means3D"].shape[0]
    return torch.rand(P, 3, generator=gen).to(DEV), torch.randn(3, a["H"], a["W"], generator=gen).to(DEV)


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("name", ["config1", "small_sh", "big_splats", "dense_tile", "deg3_m25", "small_precomp"])
def test_backward_multi_equals_two_single_passes(name, exact):
    a = Hh.resolve(Hh.case_inputs(name), DEV)
    P = a["means3D"].shape[0]
    dc, dd, da = Hh.image_grads(a, device=DEV)
    extra, de = _extra_inputs(a)
    zeros1 = torch.zeros(1, a["H"], a["W"], device=DEV)
    res, eo = _forward(a, exact, extra=extra)
    dextra = torch.full((P, 3), float("nan"), device=DEV)
    rc, fused = _backward(a, res, dc, dd, da, extra=extra, de=de, dextra=dextra)
    assert rc == 0
    res1, _ = _forward(a, exact)
    rc1, g1 = _backward(a, res1, dc, dd, da, multi=False)
    res2, _ = _forward(a, exact, colors=extra)
    rc2, g2 = _backward(a, res2, de, zeros1, zeros1, multi=False)
    assert rc1 == 0 and rc2 == 0
    assert torch.equal(eo, res2[0]) and torch.equal(res[0], res1[0])  # the forward's two images are the two passes' colour images
    for k, _ in GRAD_SHAPES:
        want = g1[k] if k in ("dL_dcolors", "dL_dsh") else g1[k] + g2[k]  # colour gradients belong to pass 1 alone
        assert torch.isfinite(fused[k]).all(), k
        assert Hh.relerr(fused[k], want) < 1e-4, (k, Hh.relerr(fused[k], want))
    assert Hh.relerr(dextra, g2["dL_dcolors"]) < 1e-4


def test_backward_multi_against_cpu_oracle():
    """config1: gsr_backward_multi against the sum of two CPU oracle backward passes (colour image, then the extra colours as
    colors_precomp with zero depth / alpha gradients).  Tolerance as for the single-pass oracle comparison (fp32 sums in
    different orders, relative to the largest entry)."""
    a = Hh.resolve(Hh.case_inputs("config1"), DEV)
    P = a["means3D"].shape[0]
    dc, dd, da = Hh.image_grads(a, device=DEV)
    extra, de = _extra_inputs(a)
    res, _ = _forward(a, False, extra=extra)
    dextra = torch.empty((P, 3), device=DEV)
    rc, g = _backward(a, res, dc, dd, da, extra=extra, de=de, dextra=dextra)
    assert rc == 0
    og1 = Hh.oracle_backward(a, Hh.run_oracle(a), dc, dd, da)
    b = dict(a, shs=None, colors_precomp=extra)
    z = torch.zeros(1, a["H"], a["W"], device=DEV)
    og2 = Hh.oracle_backward(b, Hh.run_oracle(b), de, z, z)
    tol = 1e-3

    def cmp(mine, want):
        want = np.asarray(want).reshape(P, -1)
        return Hh.relerr(mine.reshape(P, -1)[:, :want.shape[1]], want)
    for mine, k in (("dL_dmeans3D", "dL_dmeans3D"), ("dL_dmeans2D", "dL_dmeans2D"), ("dL_dopacity", "dL_dopacity"),
                    ("dL_dscales", "dL_dscales"), ("dL_drotations", "dL_drotations")):
        assert cmp(g[mine], np.asarray(og1[k]) + np.asarray(og2[k])) < tol, mine
    assert cmp(g["dL_dsh"], og1["dL_dsh"]) < tol
    assert cmp(dextra, og2["dL_dcolors"]) < tol


def test_backward_multi_null_extras_and_validation():
    from autovfx_b200 import _lib
    a = Hh.resolve(Hh.case_inputs("small_sh"), DEV)
    P = a["means3D"].shape[0]
    dc, dd, da = Hh.image_grads(a, device=DEV)
    res, _ = _forward(a, False)
    rc, g_null = _backward(a, res, dc, dd, da)
    assert rc == 0
    rc, g_ref = _backward(a, res, dc, dd, da, multi=False)
    assert rc == 0
    for k, _ in GRAD_SHAPES:
        assert Hh.relerr(g_null[k], g_ref[k]) < 1e-5, k  # same kernels; only the order of the atomic sums may differ
    extra, de = _extra_inputs(a)
    dextra = torch.empty((P, 3), device=DEV)
    for partial in (dict(extra=extra), dict(de=de), dict(dextra=dextra), dict(extra=extra, de=de), dict(de=de, dextra=dextra)):
        rc, _ = _backward(a, res, dc, dd, da, **partial)
        assert rc == -1, partial
        assert b"gsr_backward_multi" in _lib.lib.gsr_last_error()


# ----------------------------------------------------------------------------------------------------------- render()
PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)


def _render_case(name="small_sh", P=None):
    case = Hh.case_inputs(name)
    g = case["g"]
    if P is not None:
        g = {k: v[:P] for k, v in g.items()}
    pc = TrainableGaussians.from_activated(g, 3, DEV)
    cam = case["cam"].to(DEV)
    bg = torch.tensor(case["bg"], dtype=torch.float32, device=DEV)
    gen = torch.Generator().manual_seed(11)
    H, W = cam.image_height, cam.image_width
    targets = (torch.rand(3, H, W, generator=gen).to(DEV), (torch.rand(H, W, generator=gen) * 3 + 1).to(DEV))
    return pc, cam, bg, targets


def _raster_nodes(t):
    """Rasterizer backward nodes in the autograd graph of ``t``."""
    seen, stack, n = set(), [t.grad_fn], 0
    while stack:
        f = stack.pop()
        if f is None or f in seen:
            continue
        seen.add(f)
        n += "RasterizeGaussians" in type(f).__name__
        stack.extend(nf for nf, _ in f.next_functions)
    return n


def test_render_training_forward_equals_inference_and_uses_one_rasterizer_node():
    from autovfx_b200 import renderer as RD
    pc, cam, bg, _ = _render_case("config1")
    with torch.no_grad():
        want = RD.render(cam, pc, PIPE, bg)
    assert RD.get_fused_training()
    got = RD.render(cam, pc, PIPE, bg)
    assert got["render"].requires_grad
    for k in ("render", "depth", "radii"):
        assert torch.equal(got[k].detach(), want[k]), k
    assert Hh.maxabs(got["normal"].detach(), want["normal"]) <= 1e-4
    assert _raster_nodes(got["render"]) == 1
    assert _raster_nodes(got["render"].sum() + got["depth"].sum() + got["normal"].sum()) == 1
    RD.set_fused_training(False)
    try:
        two = RD.render(cam, pc, PIPE, bg)
    finally:
        RD.set_fused_training(True)
    assert _raster_nodes(two["render"].sum() + two["depth"].sum() + two["normal"].sum()) == 2
    for k in ("render", "depth", "radii"):
        assert torch.equal(got[k].detach(), two[k].detach()), k


def _step(fused, pc, cam, bg, targets, pipe=PIPE, override=None, rgb_only=False):
    from autovfx_b200 import renderer as RD
    RD.set_fused_training(fused)
    try:
        pc.zero_grad()
        if override is not None:
            override.grad = None
        out = RD.render(cam, pc, pipe, bg, override_color=override)
        training_loss(out, targets[0], targets[1], rgb_only).backward()
    finally:
        RD.set_fused_training(True)
    grads = {k: None if v.grad is None else v.grad.detach().clone() for k, v in pc.raw.items()}  # override_color: no SH gradient
    grads["viewspace_points"] = out["viewspace_points"].grad.detach().clone()
    if override is not None:
        grads["override_color"] = override.grad.detach().clone()
    return out, grads


@pytest.mark.parametrize("variant", ["full_loss", "rgb_only", "override_color", "python_cov_and_sh", "no_gaussians"])
def test_fused_training_matches_two_pass(variant):
    pc, cam, bg, targets = _render_case("small_sh", P=0 if variant == "no_gaussians" else None)
    kw = {}
    if variant == "rgb_only":
        kw["rgb_only"] = True
    if variant == "override_color":
        gen = torch.Generator().manual_seed(2)
        kw["override"] = torch.rand(pc.get_xyz.shape[0], 3, generator=gen).to(DEV).requires_grad_(True)
    if variant == "python_cov_and_sh":
        kw["pipe"] = types.SimpleNamespace(debug=False, compute_cov3D_python=True, convert_SHs_python=True)
    out_f, g_f = _step(True, pc, cam, bg, targets, **kw)
    out_t, g_t = _step(False, pc, cam, bg, targets, **kw)
    for k in ("render", "depth", "radii"):
        assert torch.equal(out_f[k].detach(), out_t[k].detach()), k
    assert Hh.maxabs(out_f["normal"].detach(), out_t["normal"].detach()) <= 1e-6
    assert g_f.keys() == g_t.keys()
    for k in g_t:
        assert (g_f[k] is None) == (g_t[k] is None), k
        if g_t[k] is None:
            continue
        assert g_f[k].shape == g_t[k].shape, k
        assert torch.isfinite(g_f[k]).all(), k
        assert Hh.relerr(g_f[k], g_t[k]) < 1e-4, (k, Hh.relerr(g_f[k], g_t[k]))


def test_fused_training_step_matches_reference_training_step():
    """The inputs of test_training_step_through_reference_render_gradients through render()'s fused path, against the gradients
    the reference's own render() + autograd rasterizer computed (tests/golden/ref_callers_grads.npz)."""
    raw = _scene_raw(3000, 16, 23)
    cam_args = _cam_args(W=128, H=96)
    _, _, _, _, W, H, _, _ = cam_args
    bg = torch.tensor([0.2, 0.2, 0.2], device=DEV)
    gen = torch.Generator().manual_seed(3)
    w_img, w_d, w_n = torch.randn(4, H, W, generator=gen).to(DEV), torch.randn(H, W, generator=gen).to(DEV), torch.randn(H, W, 3, generator=gen).to(DEV)
    names = ("xyz", "f_dc", "f_rest", "opacity", "scaling", "rotation", "screen")

    def compute():
        raise RuntimeError("recorded by test_gpu_reference_callers.py::test_training_step_through_reference_render_gradients")
    want = Hh.reference("callers_grads", "training_step", compute, full=names)
    from autovfx_b200 import renderer as RD
    assert RD.get_fused_training()
    pc = TrainableGaussians({k: v.to(DEV).float().contiguous().requires_grad_(True) for k, v in raw.items()}, 3)
    o = RD.render(types.SimpleNamespace(**_camera(*cam_args)), pc, rp_pipe(), bg)
    loss = (o["render"] * w_img).sum() + (o["depth"] * w_d).sum() + (o["normal"] * w_n).sum()
    loss.backward()
    got = dict(zip(names, [pc.raw[k].grad for k in names[:-1]] + [o["viewspace_points"].grad]))
    for k, g in got.items():
        assert g is not None, k
        assert Hh.relerr(g, want[k]) < 3e-4, k
