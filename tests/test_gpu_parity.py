"""GPU parity tests (run with -m gpu on the B200 box).  Every call goes through the public Python API / the C ABI of
include/gsr_b200.h.  Two checkers: the CPU oracle (oracle/gsr_oracle.c) and what the reference's own CUDA code computed on
identical inputs, stored under tests/golden/ (bit-exact integer outputs; images within 1e-4 as BASELINE.json's north_star
states)."""
import glob
import math
import os

import numpy as np
import pytest
import torch

from tests import helpers as Hh
from autovfx_b200 import scene

pytestmark = pytest.mark.gpu

CASES = ["config1", "small_sh", "small_deg1_m25", "deg3_m25", "deg2_m25", "small_precomp", "big_splats", "dense_tile", "coplanar"]
GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz"))
                if not os.path.basename(p).startswith(("wrapper_", "grads_", "ref_")))
IMG_TOL = 1e-4  # BASELINE.json: "within 1e-4 max abs per channel"


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from autovfx_b200 import rasterizer  # noqa: F401  (fails loudly if the CUDA library is missing)
    return torch.device("cuda:0")


@pytest.mark.parametrize("name", CASES)
def test_forward_matches_cpu_oracle(dev, name):
    a = Hh.resolve(Hh.case_inputs(name), dev)
    ours = Hh.run_ours(a, for_backward=True, sorted_keys=True)
    orc = Hh.run_oracle(a)
    P = a["means3D"].shape[0]
    mism = int((ours["radii"].cpu() != torch.from_numpy(orc["radii"])).sum())
    assert mism <= max(1, P // 5000)
    for k in ("color", "depth", "alpha"):
        assert Hh.maxabs(ours[k], orc[k]) <= IMG_TOL, k
    if mism == 0:
        assert ours["stats"]["num_rendered"] == orc["num_rendered"]
        assert ours["stats"]["num_visible"] == int((orc["radii"] > 0).sum())
        R = orc["num_rendered"]
        assert np.array_equal(ours["views"]["point_list"][:R].cpu().numpy().astype(np.uint32), orc["point_list"])
        assert np.array_equal(ours["views"]["ranges"].cpu().numpy().astype(np.uint32), orc["ranges"])


@pytest.mark.parametrize("name", CASES)
def test_forward_bit_exact_vs_compiled_reference(dev, name):
    a = Hh.resolve(Hh.case_inputs(name), dev)
    ours = Hh.run_ours(a, for_backward=True, sorted_keys=True)

    def compute():
        from oracle import ref_cuda
        ref = Hh.run_ref(a)
        rs = ref_cuda.state(dev)
        vis = ref["radii"] > 0
        out = {k: ref[k] for k in ("color", "depth", "alpha", "radii", "num_rendered")}
        out.update({k: rs[k] for k in ("point_list", "ranges", "n_contrib", "point_list_keys")})
        out.update(means2D=rs["means2D"][vis], depths=rs["depths"][vis], conic=rs["conic_opacity"][vis][:, 0:3].contiguous().view(torch.int32))
        torch.cuda.synchronize()
        return out
    ref = Hh.reference("parity", "bit_exact_" + name, compute)
    v = ours["views"]
    R = int(ref["num_rendered"])
    assert Hh.same(ours["radii"], ref["radii"])
    assert ours["stats"]["num_rendered"] == R
    assert Hh.same(v["point_list"][:R], ref["point_list"])
    assert Hh.same(v["ranges"], ref["ranges"])
    assert Hh.same(v["n_contrib"], ref["n_contrib"])
    # (tile << 32 | depth bits) keys of the reference, rebuilt from our (depth bits << 32 | id) pairs and the ranges
    rg = v["ranges"].long()
    tile_of = torch.repeat_interleave(torch.arange(rg.shape[0], device=dev), rg[:, 1] - rg[:, 0])
    key = (tile_of << 32) | ((v["sorted_keys"][:R] >> 32) & 0xFFFFFFFF)
    assert Hh.same(key, ref["point_list_keys"])
    assert torch.equal(v["sorted_keys"][:R] & 0xFFFFFFFF, v["point_list"][:R].long() & 0xFFFFFFFF)
    vis = ours["radii"] > 0
    rec = v["records"]
    assert Hh.same(rec[vis][:, 0:2], ref["means2D"])
    assert Hh.same(rec[vis][:, 6], ref["depths"])
    assert Hh.same(rec[vis][:, 2:5].contiguous().view(torch.int32), ref["conic"])
    fast = {k: ours[k].clone() for k in ("color", "depth", "alpha")}
    nc_fast = v["n_contrib"].clone()
    exact = Hh.run_ours(a, for_backward=True, exact=True)
    for k in ("color", "depth", "alpha"):
        assert Hh.same(exact[k], ref[k]), k  # GSR_FLAG_EXACT_IMAGES: bit-identical images
    Hh.assert_images_close(fast, exact)  # default blend (ex2.approx alpha, guarded decisions) against the reference's images
    assert torch.equal(exact["views"]["n_contrib"], nc_fast)


@pytest.mark.parametrize("path", GOLDEN or [None])
def test_forward_and_backward_match_golden(dev, path):
    if path is None:
        pytest.skip("no golden fixtures committed")
    gold = Hh.golden_case(os.path.basename(path)[:-4])
    a = Hh.resolve(Hh.case_inputs(str(gold["case"])), dev)
    ours = Hh.run_ours(a, for_backward=True)
    R = int(gold["num_rendered"])
    assert np.array_equal(ours["radii"].cpu().numpy(), gold["radii"])
    assert ours["stats"]["num_rendered"] == R
    assert np.array_equal(ours["views"]["point_list"][:R].cpu().numpy(), gold["point_list"])
    assert np.array_equal(ours["views"]["ranges"].cpu().numpy().reshape(-1), gold["ranges"].reshape(-1))
    assert np.array_equal(ours["views"]["n_contrib"].cpu().numpy(), gold["n_contrib"])
    Hh.assert_images_close(ours, gold)
    exact = Hh.run_ours(a, for_backward=True, exact=True)
    for k in ("color", "depth", "alpha"):
        assert np.array_equal(exact[k].cpu().numpy().reshape(gold[k].shape), gold[k]), k
    if "dL_dmeans3D" in gold:
        dc, dd, da = Hh.image_grads(a, device=dev)
        _, g = Hh.ours_backward(a, dc, dd, da)
        pairs = [("means3D", "dL_dmeans3D"), ("means2D", "dL_dmeans2D"), ("opacities", "dL_dopacity")]
        pairs += [("shs", "dL_dsh")] if (a["shs"] is not None and "dL_dsh" in gold) else []
        pairs += [("scales", "dL_dscales"), ("rotations", "dL_drotations")] if a["scales"] is not None else [("cov3D_precomp", "dL_dcov3D")]
        pairs += [("colors_precomp", "dL_dcolors")] if a["colors_precomp"] is not None else []
        for mine, theirs in pairs:
            assert Hh.relerr(g[mine].reshape(gold[theirs].shape), gold[theirs]) < 2e-4, mine


@pytest.mark.parametrize("name", CASES)
def test_backward_matches_cpu_oracle(dev, name):
    a = Hh.resolve(Hh.case_inputs(name), dev)
    dc, dd, da = Hh.image_grads(a, device=dev)
    _, g = Hh.ours_backward(a, dc, dd, da)
    orc = Hh.run_oracle(a)
    og = Hh.oracle_backward(a, orc, dc, dd, da)
    tol = 1e-3  # fp32 sums in different orders; relative to the largest entry of each tensor
    assert Hh.relerr(g["means3D"], og["dL_dmeans3D"]) < tol
    assert Hh.relerr(g["means2D"], og["dL_dmeans2D"]) < tol
    assert Hh.relerr(g["opacities"], og["dL_dopacity"]) < tol
    if a["shs"] is not None:
        assert Hh.relerr(g["shs"], og["dL_dsh"]) < tol
    else:
        assert Hh.relerr(g["colors_precomp"], og["dL_dcolors"]) < tol
    if a["scales"] is not None:
        assert Hh.relerr(g["scales"], og["dL_dscales"]) < tol
        assert Hh.relerr(g["rotations"], og["dL_drotations"]) < tol
    else:
        assert Hh.relerr(g["cov3D_precomp"], og["dL_dcov3D"]) < tol


def test_backward_matches_compiled_reference(dev):
    for name in ("config1", "big_splats", "small_precomp"):
        a = Hh.resolve(Hh.case_inputs(name), dev)
        dc, dd, da = Hh.image_grads(a, device=dev)
        gr = Hh.golden_case(name)  # the reference's backward with the same image gradients (tests/golden/make_golden.py)
        _, g = Hh.ours_backward(a, dc, dd, da)
        assert Hh.relerr(g["means3D"], gr["dL_dmeans3D"]) < 2e-4
        assert Hh.relerr(g["means2D"], gr["dL_dmeans2D"]) < 2e-4
        assert Hh.relerr(g["opacities"], gr["dL_dopacity"]) < 2e-4
        assert torch.equal(g["means2D"][:, 2], torch.zeros_like(g["means2D"][:, 2]))


@pytest.fixture(scope="module")
def scene3m(dev):
    g = scene.config3_scene()
    cams = scene.cameras_from_trajectory(scene.trajectory_dict(num_views=300))
    return g, cams


def test_full_size_3m_1080p_properties_and_reference(dev, scene3m):
    """BASELINE configs 3/4 at full size: size-independent properties + the compiled reference on identical tensors."""
    g, cams = scene3m
    a = Hh.resolve(dict(g=g, cam=cams[42], sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0), dev)
    o1 = Hh.run_ours(a, for_backward=True, sorted_keys=True, debug=False)
    v = o1["views"]
    R, P = o1["stats"]["num_rendered"], a["means3D"].shape[0]
    assert o1["stats"]["overflow"] == 0
    assert int(v["tile_count"].sum()) == R and int((o1["radii"] > 0).sum()) == o1["stats"]["num_visible"]
    rg = v["ranges"].long()
    cnt = rg[:, 1] - rg[:, 0]
    assert int(cnt.sum()) == R and int(cnt.max()) == o1["stats"]["max_tile"]
    # per-tile lists are sorted by (depth bits, id): within a tile the 64-bit pairs increase strictly
    sk = v["sorted_keys"][:R]
    tile_of = torch.repeat_interleave(torch.arange(rg.shape[0], device=dev), cnt)
    same_tile = tile_of[1:] == tile_of[:-1]
    assert bool((sk[1:][same_tile] > sk[:-1][same_tile]).all())
    assert torch.equal(sk & 0xFFFFFFFF, v["point_list"][:R].long() & 0xFFFFFFFF)
    assert float(o1["alpha"].min()) >= 0.0 and float(o1["alpha"].max()) <= 1.0 and bool(torch.isfinite(o1["color"]).all())
    assert bool((v["n_contrib"].view(-1).long() <= cnt.max()).all())
    # idempotence / determinism: a second run is bitwise identical
    imgs1 = [o1[k].clone() for k in ("color", "depth", "alpha")]
    pl1 = v["point_list"][:R].clone()
    o2 = Hh.run_ours(a, for_backward=True, sorted_keys=True, debug=False)
    assert torch.equal(o2["views"]["point_list"][:R], pl1)
    for x, k in zip(imgs1, ("color", "depth", "alpha")):
        assert torch.equal(x, o2[k]), k
    ref = Hh.ref_forward("parity", "full_size_3m", a, state=("point_list", "ranges", "n_contrib"))
    assert Hh.same(o2["radii"], ref["radii"]) and int(ref["num_rendered"]) == R
    assert Hh.same(pl1, ref["point_list"]) and Hh.same(o2["views"]["ranges"], ref["ranges"])
    fast = {k: o2[k].clone() for k in ("color", "depth", "alpha")}
    nc_fast = o2["views"]["n_contrib"].clone()
    redos = o2["stats"]["exact_redos"]
    o3 = Hh.run_ours(a, for_backward=True, debug=False, exact=True)
    for k in ("color", "depth", "alpha"):
        assert Hh.same(o3[k], ref[k]), k
    Hh.assert_images_close(fast, o3)  # = against the reference's images
    assert torch.equal(o3["views"]["n_contrib"], nc_fast) and Hh.same(nc_fast, ref["n_contrib"])
    # the default mode's repair path ran on a small fraction of the 65,280 warps
    assert 0 < redos < 6000 and o3["stats"]["exact_redos"] == 0


def test_full_size_3m_gradients_match_compiled_reference(dev, scene3m):
    """Config 3's backward half at full size (3M Gaussians, 1080p): every gradient against the reference's own CUDA backward.
    Stored of the reference: each gradient's largest magnitude, and its rows for a fixed sample of Gaussians (the 32 largest
    rows of every gradient and 512 seeded picks among the visible ones)."""
    g, cams = scene3m
    pairs = (("means3D", "dL_dmeans3D"), ("means2D", "dL_dmeans2D"), ("opacities", "dL_dopacity"), ("shs", "dL_dsh"), ("scales", "dL_dscales"),
             ("rotations", "dL_drotations"))
    for ci in (42, 171):
        a = Hh.resolve(dict(g=g, cam=cams[ci], sh_degree=3, bg=(0.1, 0.2, 0.3), scale_modifier=1.0), dev)
        dc, dd, da = Hh.image_grads(a, device=dev)

        def compute():
            from oracle import ref_cuda
            fw = Hh.run_ref(a)
            gr = ref_cuda.backward(fw, dc, dd, da)
            P = fw["radii"].shape[0]
            rows = [gr[t].reshape(P, -1).abs().amax(1).topk(32).indices for _, t in pairs]
            vis = torch.nonzero(fw["radii"] > 0).squeeze(1)
            rows.append(vis[torch.randperm(vis.numel(), generator=torch.Generator().manual_seed(ci))[:512].to(dev)])
            idx = torch.unique(torch.cat(rows))
            out = {"idx": idx}
            for _, t in pairs:
                out[t] = gr[t].reshape(P, -1)[idx]
                out[t + "_absmax"] = gr[t].abs().max()
            return out
        gr = Hh.reference("parity_grads", "full_size_3m_grads_%d" % ci, compute, full=[t for _, t in pairs])
        outs, go = Hh.ours_backward(a, dc, dd, da)
        idx = torch.from_numpy(gr["idx"]).to(dev)
        for mine, theirs in pairs:
            m = go[mine].reshape(go[mine].shape[0], -1)
            big = float(gr[theirs + "_absmax"])
            assert abs(float(m.abs().max()) - big) <= 2e-4 * big, (ci, mine)
            assert float((m[idx].cpu() - torch.from_numpy(gr[theirs])).abs().max()) < 2e-4 * big, (ci, mine)
        # Gaussians the frame does not see get exactly zero, like the reference's zero-initialised outputs
        unseen = outs[3] == 0
        assert float(go["shs"][unseen].abs().max()) == 0.0 and float(go["means3D"][unseen].abs().max()) == 0.0
        del gr, go


def test_p_zero_returns_zero_images(dev):
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    a["bg"] = torch.tensor([0.3, 0.3, 0.3], device=dev)
    r = GaussianRasterizer(Hh.settings_from(a))
    e = torch.zeros((0, 3), device=dev)
    color, depth, alpha, radii = r(e, e, torch.zeros((0, 1), device=dev), shs=torch.zeros((0, 16, 3), device=dev),
                                   scales=torch.zeros((0, 3), device=dev), rotations=torch.zeros((0, 4), device=dev))
    assert radii.numel() == 0 and float(color.abs().max()) == 0 and float(depth.abs().max()) == 0 and float(alpha.abs().max()) == 0


def test_capacity_overflow_is_detected_and_recovered(dev):
    from autovfx_b200 import rasterizer as R
    a = Hh.resolve(Hh.case_inputs("config1"), dev)
    want = Hh.run_ours(a)
    st = R._state(dev)
    old = st.capacity
    try:
        st.cache.clear()    # cached binning buffers from earlier tests are larger than the capacity under test
        st.capacity = 1000  # far below R = 41671
        st.ensure_capacity = lambda P, W=0, H=0: None  # keep the tiny capacity for this test
        s = Hh.settings_from(a)
        # async: the frame is incomplete and its ticket says so
        res = R.forward_raw(a["means3D"], a["shs"], None, a["opacities"], a["scales"], a["rotations"], None, s, sync=False)
        assert res[5].stats()["overflow"] == 1 and not res[5].ok()
        assert st.capacity >= 41671  # ok() grew the capacity from the device-side count
        st.cache.clear()
        st.capacity = 1000
        # safe mode: transparently re-runs with a larger binning buffer
        res = R.forward_raw(a["means3D"], a["shs"], None, a["opacities"], a["scales"], a["rotations"], None, s, sync=True)
        assert res[5].stats()["overflow"] == 0
        for i, k in enumerate(("color", "depth", "alpha")):
            assert torch.equal(res[i], want[k])
    finally:
        del st.ensure_capacity
        st.capacity = max(old, st.capacity)


def test_prefiltered_trap(dev):
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("big_splats"), dev)
    r = GaussianRasterizer(Hh.settings_from(a, prefiltered=True))
    with pytest.raises(RuntimeError, match="prefiltered"):
        r(a["means3D"], torch.zeros_like(a["means3D"]), a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])


def test_mark_visible(dev):
    from autovfx_b200.rasterizer import GaussianRasterizer
    from oracle import gsr_oracle as O
    a = Hh.resolve(Hh.case_inputs("big_splats"), dev)
    vis = GaussianRasterizer(Hh.settings_from(a)).markVisible(a["means3D"])
    want = O.mark_visible(a["means3D"].cpu().numpy(), a["view"].cpu().numpy(), a["proj"].cpu().numpy())
    hom = torch.cat([a["means3D"], torch.ones(a["means3D"].shape[0], 1, device=dev)], dim=1)
    safe = ((hom @ a["view"])[:, 2] - 0.2).abs().cpu().numpy() > 1e-5
    assert vis.dtype == torch.bool and np.array_equal(vis.cpu().numpy()[safe], want[safe])

    def compute():
        from oracle import ref_cuda
        return {"visible": ref_cuda.mark_visible(a["means3D"], a["view"], a["proj"])}
    assert Hh.same(vis, Hh.reference("parity", "mark_visible", compute)["visible"])


@pytest.mark.parametrize("P", [1, 7, 1024, 5000, 70000])
def test_dist2_matches_oracle(dev, P):
    from simple_knn._C import distCUDA2
    from oracle import gsr_oracle as O
    gen = torch.Generator().manual_seed(P)
    pts = torch.randn(P, 3, generator=gen) * torch.tensor([2.0, 1.0, 0.3]) + torch.tensor([3.0, -1.0, 0.5])
    d = distCUDA2(pts.to(dev))
    want = torch.from_numpy(O.dist2(pts.numpy()))
    if P >= 4:
        assert torch.allclose(d.cpu(), want, rtol=2e-6, atol=0)
    if P >= 4:  # the reference's simple-knn on the same points: all of them, or a seeded sample of 4096 above that
        idx = torch.randperm(P, generator=torch.Generator().manual_seed(P))[:4096].sort().values if P > 4096 else torch.arange(P)

        def compute():
            from oracle import ref_cuda
            return {"dist2": ref_cuda.dist2(pts.to(dev)).cpu()[idx]}
        ref = torch.from_numpy(Hh.reference("parity", "dist2_%d" % P, compute, full=["dist2"])["dist2"])
        assert torch.allclose(d.cpu()[idx], ref, rtol=2e-6, atol=0)


def test_second_pass_with_precomputed_colors_reuses_geometry(dev):
    """The product frame = two passes with identical geometry (gaussian_renderer/__init__.py:151-185): SH pass, then
    colors_precomp = normal*0.5+0.5.  Depth/alpha/radii of the two passes must be identical."""
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("config1"), dev)
    r = GaussianRasterizer(Hh.settings_from(a))
    m2 = torch.zeros_like(a["means3D"])
    c1, d1, a1, r1 = r(a["means3D"], m2, a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
    normals = torch.nn.functional.normalize(a["means3D"]) * 0.5 + 0.5
    c2, d2, a2, r2 = r(a["means3D"], m2, a["opacities"], colors_precomp=normals, scales=a["scales"], rotations=a["rotations"])
    assert torch.equal(d1, d2) and torch.equal(a1, a2) and torch.equal(r1, r2) and not torch.equal(c1, c2)


def test_misaligned_and_noncontiguous_inputs(dev):
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    want = Hh.run_ours(a)
    P = a["means3D"].shape[0]
    buf = torch.zeros(P * 4 + 1, device=dev)
    buf[1:] = a["rotations"].reshape(-1)
    rot_misaligned = buf[1:].view(P, 4)  # 4-byte aligned only
    shs_nc = torch.zeros(P, 16, 6, device=dev)[:, :, :3]
    shs_nc.copy_(a["shs"])
    r = GaussianRasterizer(Hh.settings_from(a))
    c, d, al, _ = r(a["means3D"], torch.zeros_like(a["means3D"]), a["opacities"], shs=shs_nc, scales=a["scales"], rotations=rot_misaligned)
    assert torch.equal(c, want["color"]) and torch.equal(d, want["depth"]) and torch.equal(al, want["alpha"])


def test_frame_loop_matches_single_calls(dev, scene3m):
    from autovfx_b200 import render_loop as RL
    g, cams = scene3m
    gs = {k: v[:200000] for k, v in g.items()}
    sel = [cams[i] for i in (0, 50, 100, 150, 200)]
    loop = RL.FrameLoop(gs, 3, 1920, 1080, device=dev, ring=2, to_host=True)
    got = {}
    stats = loop.render(RL.pack_cameras(sel), lambda i, f, s: got.__setitem__(i, f.clone()))
    assert len(got) == 5 and all(s["overflow"] == 0 for s in stats)
    for i, cam in enumerate(sel):
        a = Hh.resolve(dict(g=gs, cam=cam, sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0), dev)
        o = Hh.run_ours(a, debug=False)
        assert torch.equal(got[i][0:3], o["color"].cpu()) and torch.equal(got[i][3:4], o["depth"].cpu()) and torch.equal(got[i][4:5], o["alpha"].cpu())
        assert stats[i]["num_rendered"] == o["stats"]["num_rendered"]


def test_training_step_through_module_reduces_loss(dev):
    from diff_gaussian_rasterization import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    target = Hh.run_ours(a)["color"].clone()
    shs = (a["shs"] * 0.5).clone().requires_grad_(True)
    means = a["means3D"].clone().requires_grad_(True)
    opt = torch.optim.Adam([shs, means], lr=1e-2)
    r = GaussianRasterizer(Hh.settings_from(a))
    losses = []
    for _ in range(15):
        m2 = torch.zeros_like(means, requires_grad=True)
        color, _, _, radii = r(means, m2, a["opacities"], shs=shs, scales=a["scales"], rotations=a["rotations"])
        loss = (color - target).abs().mean()
        opt.zero_grad()
        loss.backward()
        assert m2.grad is not None and radii.dtype == torch.int32
        opt.step()
        losses.append(float(loss))
    assert losses[-1] < 0.7 * losses[0]


@pytest.mark.parametrize("name", CASES)
def test_tight_tiles_changes_lists_but_not_images_or_gradients(dev, name):
    """GSR_FLAG_TIGHT_TILES (opt-in): per-tile lists become sub-sequences of the exact-key lists; color/depth/alpha/radii
    are bitwise identical; gradients agree to summation order."""
    from autovfx_b200 import rasterizer as R
    a = Hh.resolve(Hh.case_inputs(name), dev)
    exact = Hh.run_ours(a, for_backward=True, sorted_keys=True, tight=False)
    ex_imgs = [exact[k].clone() for k in ("color", "depth", "alpha")]
    ex_radii = exact["radii"].clone()
    Re = exact["stats"]["num_rendered"]
    ex_list = exact["views"]["point_list"][:Re].clone()
    ex_rg = exact["views"]["ranges"].clone().long()
    tight = Hh.run_ours(a, for_backward=True, sorted_keys=True, tight=True)
    Rt = tight["stats"]["num_rendered"]
    assert Rt <= Re and torch.equal(tight["radii"], ex_radii)
    for x, k in zip(ex_imgs, ("color", "depth", "alpha")):
        assert torch.equal(x, tight[k]), k
    # sub-sequence check per tile (on the host, small cases only)
    tl = tight["views"]["point_list"][:Rt].cpu().numpy()
    tr = tight["views"]["ranges"].cpu().numpy().astype(np.int64)
    el, er = ex_list.cpu().numpy(), ex_rg.cpu().numpy()
    for t in range(0, er.shape[0], max(1, er.shape[0] // 40)):
        full = el[er[t, 0]:er[t, 1]].tolist()
        sub = tl[tr[t, 0]:tr[t, 1]].tolist()
        it = iter(full)
        assert all(any(x == y for y in it) for x in sub), t
    dc, dd, da = Hh.image_grads(a, device=dev)
    _, g_exact = Hh.ours_backward(a, dc, dd, da)
    R.set_tight_tiles(True)
    try:
        _, g_tight = Hh.ours_backward(a, dc, dd, da)
    finally:
        R.set_tight_tiles(False)
    for k in ("means3D", "means2D", "opacities"):
        assert Hh.relerr(g_tight[k], g_exact[k]) < 1e-5, k


def test_geometry_reuse_second_pass_is_bit_identical_to_a_full_forward(dev):
    """§8f(1): the colors_precomp pass that follows an SH pass on the same geometry/camera skips projection+binning
    (GSR_FLAG_REUSE_GEOMETRY).  Its outputs must equal a full forward bit for bit; changing the geometry must miss."""
    from autovfx_b200 import rasterizer as R
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("config1"), dev)
    rast = GaussianRasterizer(Hh.settings_from(a))
    m2 = torch.zeros_like(a["means3D"])
    normals = (torch.nn.functional.normalize(a["means3D"]) * 0.5 + 0.5).contiguous()
    with torch.no_grad():
        R.set_geometry_reuse(False)
        full = rast(a["means3D"], m2, a["opacities"], colors_precomp=normals, scales=a["scales"], rotations=a["rotations"])
        R.set_geometry_reuse(True)
        first = rast(a["means3D"], m2, a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
        calls_before = R._state(dev).geom_cache[torch.cuda.current_stream(dev).cuda_stream][0]
        second = rast(a["means3D"], m2, a["opacities"], colors_precomp=normals, scales=a["scales"], rotations=a["rotations"])
        assert R._state(dev).geom_cache[torch.cuda.current_stream(dev).cuda_stream][0] == calls_before  # hit: cache untouched
        for x, y in zip(full, second):
            assert torch.equal(x, y)
        assert torch.equal(first[1], second[1]) and torch.equal(first[3], second[3])
        # in-place change of the geometry bumps the version counter -> the next precomp pass is a full forward again
        moved = a["means3D"].clone()
        rast(moved, m2, a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
        moved.add_(0.01)
        third = rast(moved, m2, a["opacities"], colors_precomp=normals, scales=a["scales"], rotations=a["rotations"])
        R.set_geometry_reuse(False)
        want = rast(moved, m2, a["opacities"], colors_precomp=normals, scales=a["scales"], rotations=a["rotations"])
        R.set_geometry_reuse(True)
        for x, y in zip(third, want):
            assert torch.equal(x, y)


@pytest.mark.parametrize("W,H", [(1, 1), (16, 16), (17, 1), (33, 47)])
def test_degenerate_image_sizes_match_reference(dev, W, H):
    """Tile grids of 1x1, exact multiples and ragged edges; the same inputs through the compiled reference."""
    case = Hh.case_inputs("small_sh")
    case["cam"] = scene.lookat_camera((0.3, -3.0, 0.4), (0, 0, 0), W, H, 55.0)
    a = Hh.resolve(case, dev)
    ours = Hh.run_ours(a, for_backward=True, exact=True)
    ref = Hh.ref_forward("parity", "size_%dx%d" % (W, H), a, full=("color", "depth", "alpha", "radii"))
    for k in ("color", "depth", "alpha", "radii"):
        assert Hh.same(ours[k], ref[k]), k
    Hh.assert_images_close(Hh.run_ours(a, for_backward=True), {k: torch.from_numpy(ref[k]) for k in ("color", "depth", "alpha")})
    dc, dd, da = Hh.image_grads(a, device=dev)
    _, g = Hh.ours_backward(a, dc, dd, da)
    assert all(torch.isfinite(v).all() for v in g.values() if v is not None)


def test_everything_behind_the_camera(dev):
    """No Gaussian survives the near cull: zero instances, background-only image, zero gradients, no kernel misbehaves."""
    case = Hh.case_inputs("small_sh")
    case["cam"] = scene.lookat_camera((0.0, -3.0, 0.0), (0.0, -6.0, 0.0), 64, 48, 55.0)  # looking away from the cloud
    a = Hh.resolve(case, dev)
    ours = Hh.run_ours(a, for_backward=True)
    assert ours["stats"]["num_rendered"] == 0 and ours["stats"]["num_visible"] == 0
    assert int(ours["radii"].abs().max()) == 0 and float(ours["alpha"].abs().max()) == 0.0
    bg = a["bg"].view(3, 1, 1).expand(3, 48, 64)
    assert torch.equal(ours["color"], bg.contiguous())
    ref = Hh.ref_forward("parity", "behind_camera", a, names=("color",))
    assert Hh.same(ours["color"], ref["color"])
    dc, dd, da = Hh.image_grads(a, device=dev)
    _, g = Hh.ours_backward(a, dc, dd, da)
    for k, v in g.items():
        if v is not None:
            assert float(v.abs().max()) == 0.0, k
    from autovfx_b200 import rasterizer as R
    extra = torch.rand(a["means3D"].shape[0], 3, device=dev)
    res = R.forward_multi(a["means3D"], a["shs"], None, extra, a["opacities"], a["scales"], a["rotations"], None, Hh.settings_from(a), sync=True)
    assert torch.equal(res[3], bg.contiguous())


def test_c_abi_rejects_bad_arguments(dev):
    """Status codes + gsr_last_error for the argument errors the reference raises from C++ (rasterize_points.cu:57-59,
    rasterizer_impl.cu:243-246) and for undersized workspaces."""
    import ctypes as C
    from autovfx_b200 import _lib
    L = _lib.lib
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    P, W, H = a["means3D"].shape[0], a["W"], a["H"]
    buf = lambda n: torch.empty(int(n), dtype=torch.uint8, device=dev)  # noqa: E731
    geom, binning, image = buf(L.gsr_geom_bytes(P)), buf(L.gsr_binning_bytes(1 << 16)), buf(L.gsr_image_bytes(W, H))
    color, depth, alpha = (torch.empty((c, H, W), device=dev) for c in (3, 1, 1))
    radii = torch.empty(P, dtype=torch.int32, device=dev)
    p = lambda t: None if t is None else t.data_ptr()  # noqa: E731

    def frame(**over):
        fr = _lib.gsr_frame(P, 3, 16, W, H, 1.0, a["tanfovx"], a["tanfovy"], 0, 0, p(a["bg"]), p(a["means3D"]), p(a["shs"]), None, p(a["opacities"]),
                            p(a["scales"]), p(a["rotations"]), None, p(a["view"]), p(a["proj"]), p(a["campos"]))
        for k, v in over.items():
            setattr(fr, k, v)
        return fr

    def call(fr, ws, out_color=color):
        return L.gsr_forward(C.byref(fr), C.byref(ws), p(out_color), p(depth), p(alpha), p(radii), 0, None)
    ws = _lib.gsr_workspace(p(geom), geom.numel(), p(binning), binning.numel(), p(image), image.numel())
    assert call(frame(), ws) == 0
    torch.cuda.synchronize()
    assert call(frame(colors_precomp=p(a["means3D"])), ws) == -1 and b"exactly one" in L.gsr_last_error()          # both shs and colors
    assert call(frame(shs=None), ws) == -1                                                                          # neither
    assert call(frame(scales=None), ws) == -1                                                                       # rotations without scales
    assert call(frame(D=3, M=4), ws) == -1 and b"coefficients" in L.gsr_last_error()                                # degree needs 16 coefficients
    assert call(frame(W=0), ws) == -1
    small = _lib.gsr_workspace(p(geom), 16, p(binning), binning.numel(), p(image), image.numel())
    assert call(frame(), small) == -2 and b"geometry workspace" in L.gsr_last_error()
    small = _lib.gsr_workspace(p(geom), geom.numel(), p(binning), binning.numel(), p(image), 64)
    assert call(frame(), small) == -2
    assert call(frame(), ws, out_color=None) == -1
    assert L.gsr_forward_multi(C.byref(frame()), C.byref(ws), p(color), p(depth), p(alpha), p(radii), p(a["means3D"]), None, 0, None) == -1
    assert L.gsr_axis_normals(P, None, None, None, None, 0, None, None) == -1
    assert L.gsr_normal_maps(0, 4, None, None, None, 1.0, 1.0, 0.0, 0.0, None, None, None) == -1
    assert L.gsr_pack_frame(4, 4, None, None, None, None, 3.0, p(color), None, None, None) == -1
    assert L.gsr_activate_gaussians(4, 0, None, None, None, None, None, None, None, None, None, None, None, None, None) == -1


def test_4k_image_and_sugar_storage_against_reference(dev):
    """3840x2160 (32,400 tiles) with 600k Gaussians stored with M=25 coefficients, rendered at degree 3, plus its product frame:
    images, radii, per-tile lists and ranges bit-identical to the compiled reference; the 6-channel pass equals its second pass."""
    from autovfx_b200 import rasterizer as R
    g = scene.synthetic_gaussians(600_000, seed=31, extent=(4, 4, 1), log_scale_mean=math.log(0.008), log_scale_std=0.6,
                                  opacity_mean=0.0, opacity_std=2.0, sh_degree=4)
    cam = scene.lookat_camera((3.0, -5.0, 2.0), (0, 0, 0), 3840, 2160, 60.0)
    a = Hh.resolve(dict(g=g, cam=cam, sh_degree=3, bg=(0.1, 0.2, 0.3), scale_modifier=1.0), dev)
    fast = Hh.run_ours(a, debug=False)
    fast_imgs = {k: fast[k].clone() for k in ("color", "depth", "alpha")}
    ours = Hh.run_ours(a, debug=False, exact=True)
    Rn = ours["stats"]["num_rendered"]
    assert ours["stats"]["overflow"] == 0 and Rn > 1_000_000
    Hh.assert_images_close(fast_imgs, ours)  # ours equals the reference's images (below), so this is the default mode against them
    ref = Hh.ref_forward("parity", "4k_sugar", a, state=("point_list", "ranges"))
    assert int(ref["num_rendered"]) == Rn
    for k in ("color", "depth", "alpha", "radii"):
        assert Hh.same(ours[k], ref[k]), k
    assert Hh.same(ours["views"]["point_list"][:Rn], ref["point_list"]) and Hh.same(ours["views"]["ranges"], ref["ranges"])
    extra = torch.rand(600_000, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    res = R.forward_multi(a["means3D"], a["shs"], None, extra, a["opacities"], a["scales"], a["rotations"], None, Hh.settings_from(a), sync=True,
                          exact=True)
    b = dict(a)
    b["shs"], b["colors_precomp"] = None, extra
    ref2 = Hh.ref_forward("parity", "4k_sugar_second_pass", b, names=("color",))["color"]
    assert Hh.same(res[3], ref2) and Hh.same(res[0], ref["color"])
    resf = R.forward_multi(a["means3D"], a["shs"], None, extra, a["opacities"], a["scales"], a["rotations"], None, Hh.settings_from(a), sync=True)
    assert Hh.maxabs(resf[3], res[3]) <= 1e-5 and Hh.maxabs(resf[0], res[0]) <= 1e-5


def test_debug_mode_dumps_a_snapshot_on_failure(dev, tmp_path, monkeypatch):
    """raster_settings.debug: a failing forward leaves snapshot_fw.dump with CPU copies of the arguments (reference __init__.py:83-90)."""
    from autovfx_b200.rasterizer import GaussianRasterizer
    monkeypatch.chdir(tmp_path)
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    s = Hh.settings_from(a, debug=True)
    rast = GaussianRasterizer(s)
    bad_shs = a["shs"][:, :4].contiguous()  # degree 3 needs 16 coefficients
    with pytest.raises(RuntimeError):
        rast(a["means3D"], torch.zeros_like(a["means3D"]), a["opacities"], shs=bad_shs, scales=a["scales"], rotations=a["rotations"])
    dump = torch.load(tmp_path / "snapshot_fw.dump", weights_only=False)
    assert isinstance(dump, tuple) and len(dump) == 19 and dump[1].shape == a["means3D"].shape and not dump[1].is_cuda
    # and a correct call in debug mode still works (synchronous error checking after every stage)
    out = rast(a["means3D"], torch.zeros_like(a["means3D"]), a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
    assert torch.equal(out[0], Hh.run_ours(a)["color"])


def test_parameters_under_no_grad_take_the_inference_path(dev):
    """The reference's eval loops pass nn.Parameters under torch.no_grad() (scene_representation.py:355): no backward buffers
    are kept and the second pass of the product frame reuses the first pass's geometry."""
    from autovfx_b200 import rasterizer as R
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("config1"), dev)
    par = {k: torch.nn.Parameter(a[k].clone()) for k in ("means3D", "opacities", "shs", "scales", "rotations")}
    rast = GaussianRasterizer(Hh.settings_from(a))
    m2 = torch.zeros_like(a["means3D"])
    normals = (torch.nn.functional.normalize(a["means3D"]) * 0.5 + 0.5).contiguous()
    stream = torch.cuda.current_stream(dev).cuda_stream
    with torch.no_grad():
        first = rast(par["means3D"], m2, par["opacities"], shs=par["shs"], scales=par["scales"], rotations=par["rotations"])
        key = R._state(dev).geom_cache[stream][0]  # the inference path remembered the geometry ...
        second = rast(par["means3D"], m2, par["opacities"], colors_precomp=normals, scales=par["scales"], rotations=par["rotations"])
        assert R._state(dev).geom_cache[stream][0] == key  # ... and the second pass hit it (cache untouched)
    assert not first[0].requires_grad and first[0].grad_fn is None
    assert torch.equal(first[1], second[1]) and torch.equal(first[3], second[3])
    # with gradients enabled the same call keeps its buffers and differentiates
    out = rast(par["means3D"], torch.zeros_like(m2, requires_grad=True), par["opacities"], shs=par["shs"], scales=par["scales"], rotations=par["rotations"])
    out[0].sum().backward()
    assert par["means3D"].grad is not None and torch.equal(out[0].detach(), first[0])


def test_backward_with_no_gaussians_returns_empty_grads(dev):
    from autovfx_b200.rasterizer import GaussianRasterizer
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    r = GaussianRasterizer(Hh.settings_from(a))
    leaf = lambda *s: torch.zeros(s, device=dev, requires_grad=True)  # noqa: E731
    m3, m2, op, sh, sc, ro = leaf(0, 3), leaf(0, 3), leaf(0, 1), leaf(0, 16, 3), leaf(0, 3), leaf(0, 4)
    color, depth, alpha, radii = r(m3, m2, op, shs=sh, scales=sc, rotations=ro)
    (color.sum() + depth.sum() + alpha.sum()).backward()
    for t in (m3, m2, op, sh, sc, ro):
        assert t.grad is not None and t.grad.shape == t.shape


def test_ticket_outlives_the_counter_ring(dev):
    """A FrameTicket read after more than RING later forwards still reports its own frame's counters."""
    from autovfx_b200 import rasterizer as R
    a = Hh.resolve(Hh.case_inputs("small_sh"), dev)
    b = Hh.resolve(Hh.case_inputs("config1"), dev)
    sa, sb = Hh.settings_from(a), Hh.settings_from(b)
    want = Hh.run_ours(a)["stats"]["num_rendered"]
    held = R.forward_raw(a["means3D"], a["shs"], None, a["opacities"], a["scales"], a["rotations"], None, sa, sync=False)[5]
    for _ in range(R._DeviceState.RING + 6):
        R.forward_raw(b["means3D"], b["shs"], None, b["opacities"], b["scales"], b["rotations"], None, sb, sync=False)
    assert held.stats()["num_rendered"] == want


def test_frame_loop_two_streams_and_pack8(dev, scene3m):
    """FrameLoop(streams=2): consecutive frames on alternating CUDA streams, same frames bit for bit; pack8 without the product frame
    hands off RGBA8 + fp32 depth + the 8-bit depth index."""
    from autovfx_b200 import render_loop as RL, renderer as RD
    g, cams = scene3m
    gs = {k: v[:150000] for k, v in g.items()}
    sel = [cams[i] for i in (3, 40, 77, 120, 180, 250, 299)]
    one = RL.FrameLoop(gs, 3, 1920, 1080, device=dev, ring=3, to_host=True)
    want = {}
    one.render(RL.pack_cameras(sel), lambda i, f, s: want.__setitem__(i, f.clone()))
    two = RL.FrameLoop(gs, 3, 1920, 1080, device=dev, ring=3, to_host=True, streams=2)
    assert two.ring == 4
    got = {}
    st = two.render(RL.pack_cameras(sel), lambda i, f, s: got.__setitem__(i, f.clone()))
    assert len(got) == len(sel) and all(s["overflow"] == 0 for s in st)
    for i in range(len(sel)):
        assert torch.equal(got[i], want[i]), i
    p8 = RL.FrameLoop(gs, 3, 1920, 1080, device=dev, ring=4, to_host=True, pack8=True, streams=2)
    got8 = {}
    p8.render(RL.pack_cameras(sel), lambda i, f, s: got8.__setitem__(i, {k: v.clone() for k, v in f.items()}))
    for i in range(len(sel)):
        fr = want[i].to(dev)
        packed = RD.pack_frame(fr[0:3], fr[4], fr[3], None, depth_scale=3.0)
        assert torch.equal(got8[i]["rgba8"].to(dev), packed["rgba8"]) and torch.equal(got8[i]["depth8"].to(dev), packed["depth8"])
        assert torch.equal(got8[i]["depth"], want[i][3])


def test_more_tiles_than_the_fixed_ballot_rows(dev):
    """6144x6144 = 147,456 tiles, more than the 131,072 ballot-matrix rows the fixed part of the binning workspace provides: the
    capacity is raised so that the rows fit, and the image equals the compiled reference's."""
    g = scene.synthetic_gaussians(20000, seed=51, extent=(1.0, 1.0, 0.5), log_scale_mean=math.log(0.01), log_scale_std=0.4)
    cam = scene.lookat_camera((0.2, -2.2, 0.6), (0, 0, 0), 6144, 6144, 50.0, fov_y_deg=50.0)
    a = Hh.resolve(dict(g=g, cam=cam, sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0), dev)
    ours = Hh.run_ours(a, debug=False, exact=True)
    assert ours["stats"]["overflow"] == 0 and ours["stats"]["num_rendered"] > 100000
    ref = Hh.ref_forward("parity", "6144x6144", a, names=("color", "alpha", "radii", "num_rendered"))
    assert int(ref["num_rendered"]) == ours["stats"]["num_rendered"]
    for k in ("color", "alpha", "radii"):
        assert Hh.same(ours[k], ref[k]), k
