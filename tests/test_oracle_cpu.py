"""CPU tests of the oracle (no GPU): self-consistency, autograd pinning, golden vectors from the reference's own CUDA code."""
import glob
import math
import os

import numpy as np
import pytest
import torch

from tests import helpers as Hh
from tests import torch_ref
from autovfx_b200 import scene
from oracle import gsr_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def tiny_case():
    g = scene.synthetic_gaussians(60, seed=21, extent=(0.8, 0.8, 0.8), log_scale_mean=math.log(0.12), log_scale_std=0.4, opacity_mean=-0.5,
                                  opacity_std=0.8)
    g["opacities"] = g["opacities"].clamp(max=0.9)  # keep alpha below the 0.99 clamp (its derivative differs by design)
    cam = scene.lookat_camera((0.4, -3.0, 0.5), (0, 0, 0), 40, 28, 50.0)
    return dict(g=g, cam=cam, sh_degree=3, bg=(0.3, 0.1, 0.6), scale_modifier=1.1)


def test_oracle_forward_matches_fp64_torch_restatement():
    a = Hh.resolve(tiny_case())
    fw = Hh.run_oracle(a)
    color, depth, alpha, _, _ = torch_ref.render(a, fw)
    assert Hh.maxabs(color.detach(), fw["color"]) < 2e-5
    assert Hh.maxabs(depth.detach(), fw["depth"]) < 2e-5
    assert Hh.maxabs(alpha.detach(), fw["alpha"]) < 2e-5


def test_oracle_backward_matches_autograd():
    a = Hh.resolve(tiny_case())
    fw = Hh.run_oracle(a)
    dc, dd, da = Hh.image_grads(a)
    og = Hh.oracle_backward(a, fw, dc, dd, da)
    color, depth, alpha, leaves, m2d = torch_ref.render(a, fw)
    loss = (color * dc.double()).sum() + (depth * dd.double()).sum() + (alpha * da.double()).sum()
    loss.backward()
    tol = 2e-3  # fp32 oracle vs fp64 autograd, relative to the largest entry
    assert Hh.relerr(og["dL_dmeans3D"], leaves["means3D"].grad) < tol
    # reference quirk: dL/dscale is the gradient w.r.t. (scale_modifier * scale) — backward.cu:318-321 omits the
    # factor scale_modifier — so the true gradient is the reported one times the modifier
    assert Hh.relerr(og["dL_dscales"] * a["scale_modifier"], leaves["scales"].grad) < tol
    assert Hh.relerr(og["dL_drotations"], leaves["rotations"].grad) < tol
    assert Hh.relerr(og["dL_dopacity"], leaves["opacities"].grad) < tol
    assert Hh.relerr(og["dL_dsh"], leaves["shs"].grad) < tol
    # dL/dmean2D is reported in NDC-scaled units: pixel gradient * 0.5*W (backward.cu:488-489)
    scale = torch.tensor([0.5 * a["W"], 0.5 * a["H"]], dtype=torch.float64)
    assert Hh.relerr(og["dL_dmeans2D"][:, :2], m2d.grad * scale) < tol
    assert np.all(og["dL_dmeans2D"][:, 2] == 0)


@pytest.mark.parametrize("name", ["config1", "small_sh", "small_deg1_m25", "deg3_m25", "deg2_m25", "small_precomp", "big_splats", "dense_tile", "coplanar"])
def test_oracle_binning_invariants(name):
    a = Hh.resolve(Hh.case_inputs(name))
    fw = Hh.run_oracle(a, stop_after="binning")
    R = fw["num_rendered"]
    assert R == int(fw["tiles_touched"].sum())
    keys, pl, rg = fw["keys"], fw["point_list"], fw["ranges"].astype(np.int64)
    gx = (a["W"] + 15) // 16
    # keys sorted (tile, depth bits); ties keep ascending Gaussian id (stable sort of id-ordered emission)
    assert np.all(keys[1:] >= keys[:-1])
    same = keys[1:] == keys[:-1]
    assert np.all(pl[1:][same] > pl[:-1][same])
    # ranges partition [0,R) in tile order and agree with the key's tile field
    cnt = rg[:, 1] - rg[:, 0]
    assert cnt.sum() == R
    tiles = (keys >> np.uint64(32)).astype(np.int64)
    assert np.array_equal(np.bincount(tiles, minlength=rg.shape[0]), cnt)
    nz = cnt > 0
    assert np.array_equal(rg[nz, 0], (np.cumsum(cnt) - cnt)[nz])
    # every instance lies inside its Gaussian's tile rectangle, depth bits come from the Gaussian
    dbits = fw["depths"].view(np.uint32)[pl]
    assert np.array_equal((keys & np.uint64(0xFFFFFFFF)).astype(np.uint32), dbits)
    assert np.all(fw["radii"][pl] > 0)
    assert tiles.max(initial=0) < gx * ((a["H"] + 15) // 16)


def test_oracle_render_invariants():
    a = Hh.resolve(Hh.case_inputs("small_sh"))
    fw = Hh.run_oracle(a)
    assert fw["alpha"].min() >= 0 and fw["alpha"].max() <= 1.0
    rg = fw["ranges"].astype(np.int64)
    gx = (a["W"] + 15) // 16
    lens = (rg[:, 1] - rg[:, 0])
    for y in range(0, a["H"], 7):
        for x in range(0, a["W"], 9):
            assert fw["n_contrib"][y, x] <= lens[(y // 16) * gx + x // 16]
    # empty pixels show the background exactly
    empty = fw["alpha"][0] == 0
    if empty.any():
        for c in range(3):
            assert np.all(fw["color"][c][empty] == np.float32(a["bg"][c]))


def test_oracle_prefiltered_traps():
    case = Hh.case_inputs("big_splats")  # the camera sits inside the cloud: some points are near-culled
    a = Hh.resolve(case)
    n = lambda t: None if t is None else t.numpy()  # noqa: E731
    with pytest.raises(RuntimeError):
        O.forward(n(a["means3D"]), n(a["opacities"]), n(a["view"]), n(a["proj"]), n(a["campos"]), a["W"], a["H"], a["tanfovx"], a["tanfovy"],
                  shs=n(a["shs"]), scales=n(a["scales"]), rotations=n(a["rotations"]), sh_degree=a["sh_degree"], prefiltered=True)


def test_oracle_mark_visible_is_near_plane_only():
    a = Hh.resolve(Hh.case_inputs("big_splats"))
    vis = O.mark_visible(a["means3D"].numpy(), a["view"].numpy(), a["proj"].numpy())
    hom = torch.cat([a["means3D"], torch.ones(a["means3D"].shape[0], 1)], dim=1)
    z = (hom @ a["view"])[:, 2].numpy()
    margin = np.abs(z - 0.2) > 1e-5
    assert np.array_equal(vis[margin], (z > 0.2)[margin])
    assert 0 < vis.sum() < vis.size


@pytest.mark.parametrize("P", [1, 5, 1500, 5000])
def test_oracle_dist2_matches_brute_force(P):
    g = torch.Generator().manual_seed(P)
    pts = (torch.randn(P, 3, generator=g) * torch.tensor([2.0, 1.0, 0.3]) + torch.tensor([3.0, -1.0, 0.5])).numpy()
    fast, brute = O.dist2(pts), O.dist2(pts, brute=True)
    if P < 4:
        assert not np.all(np.isfinite(brute)) or True  # fewer than 3 neighbours: FLT_MAX arithmetic, same in both
    np.testing.assert_allclose(fast, brute, rtol=1e-6, atol=0)


def _golden_files():
    return sorted(p for p in glob.glob(os.path.join(GOLDEN, "*.npz")) if not os.path.basename(p).startswith(("wrapper_", "grads_", "ref_")))


@pytest.mark.parametrize("path", _golden_files() or [None])
def test_oracle_against_reference_golden(path):
    """Golden vectors = outputs of the reference's own CUDA rasterizer (oracle/_ref) on a B200 for the named cases
    (tests/golden/make_golden.py).  fp32 images agree to 1e-4 (FMA contraction differs between nvcc and gcc);
    integer outputs may differ only where a float sits within an ulp of a rounding boundary."""
    if path is None:
        pytest.skip("no golden fixtures committed yet")
    gold = Hh.golden_case(os.path.basename(path)[:-4])
    name = str(gold["case"])
    a = Hh.resolve(Hh.case_inputs(name))
    fw = Hh.run_oracle(a)
    P = a["means3D"].shape[0]
    assert int((fw["radii"] != gold["radii"]).sum()) <= max(1, P // 5000)
    for k in ("color", "depth", "alpha"):
        assert Hh.maxabs(fw[k], gold[k]) <= 1e-4, k
    if int((fw["radii"] != gold["radii"]).sum()) == 0 and fw["num_rendered"] == int(gold["num_rendered"]):
        assert np.array_equal(fw["point_list"], gold["point_list"].astype(np.uint32))
        assert np.array_equal(fw["ranges"].reshape(-1), gold["ranges"].reshape(-1).astype(np.uint32))
        assert int((fw["n_contrib"] != gold["n_contrib"].astype(np.uint32)).sum()) <= 2
    if "dL_dmeans3D" in gold:
        dc, dd, da = Hh.image_grads(a)
        og = Hh.oracle_backward(a, fw, dc, dd, da)
        for k in ("dL_dmeans3D", "dL_dmeans2D", "dL_dopacity", "dL_dsh", "dL_dscales", "dL_drotations", "dL_dcolors", "dL_dcov3D"):
            if k in gold and gold[k].size:
                assert Hh.relerr(og[k].reshape(gold[k].shape), gold[k]) < 5e-3, k


def test_torch_cpu_rasterize_loop_matches_the_c_oracle():
    """The pure-CPU PyTorch rasterize loop that bench.py times as `torch_cpu_baseline` (oracle/torch_cpu_raster.py) renders the
    same images as the C oracle (and hence the reference) on BASELINE config 1 and a small ragged-image case."""
    import torch
    from oracle import torch_cpu_raster as TR
    from tests import helpers as Hh
    for name in ("config1", "small_sh"):
        a = Hh.resolve(Hh.case_inputs(name))
        c, d, al, r = TR.rasterize(a["means3D"], a["scales"], a["rotations"], a["opacities"], a["shs"], a["view"], a["proj"], a["campos"], a["W"], a["H"],
                                   a["tanfovx"], a["tanfovy"], a["sh_degree"], a["scale_modifier"], tuple(float(v) for v in a["bg"]))
        o = Hh.run_oracle(a)
        assert Hh.maxabs(c, o["color"]) <= 1e-4 and Hh.maxabs(d, o["depth"]) <= 1e-4 and Hh.maxabs(al, o["alpha"]) <= 1e-4
        assert int((r != torch.from_numpy(o["radii"])).sum()) <= 1
