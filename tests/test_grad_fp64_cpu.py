"""The C oracle's backward, element by element, against fp64 autograd (tests/torch_ref.py) on scenes built to reach the
special cases of the backward (tests/grad_scenes.py): ragged image borders, the 0.99 alpha clamp and early termination, long
contributor lists, the frustum and colour clamps, and every parametrisation.  The decisions (visible set, tile lists, last
contributors) are the oracle forward's.  This pins the fp64 reference itself on those regimes without a GPU; the CUDA kernels
are held to it by tests/test_gpu_grad_fp64.py.

Criterion, per gradient tensor over the compared Gaussians: |g - r| <= rtol |r| + atol rms(r) with rtol = 1e-3, atol = 1e-4
(r: fp64, g: oracle; atol 1e-3 for the alpha-only loss, see grad_scenes.atol_for), with the fp64 loss weighting each pixel by
the oracle's recovered final transmittance over the exact one (torch_ref.Fp64Render.loss, stored_alpha).  Worst ratio
|g - r| / bound observed per scene (<= 1 passes): ragged 0.50, opaque 0.09, deep 0.19, frustum 0.03, modes 0.13, fused 0.03."""
import numpy as np
import pytest
import torch

from tests import grad_scenes as S
from tests import helpers as Hh
from tests import torch_ref

RTOL, ATOL = 1e-3, 1e-4
GRADS = ("dL_dmeans3D", "dL_dmeans2D", "dL_dopacity", "dL_dsh", "dL_dcolors", "dL_dscales", "dL_drotations", "dL_dcov3D")


def _check(a, kinds=("randn",), extra=None):
    fw = Hh.run_oracle(a)
    r = torch_ref.render_fp64(a, fw, extra=extra)
    for k in ("color", "depth", "alpha"):
        assert Hh.maxabs(getattr(r, k).detach(), fw[k]) <= 1e-4, k
    S.check_masked(r.ambiguous_pixels, r.ambiguous_gaussians, r.visible)
    keep = ~r.ambiguous_gaussians
    worst = {}
    for kind in kinds:
        dc, dd, da, de = S.mask_pixels(S.loss_grads(a, kind, extra=extra is not None), r.ambiguous_pixels)
        og = Hh.oracle_backward(a, fw, dc, dd, da)
        if extra is not None:  # the extra image's backward = a second pass with the extra colours as colors_precomp
            b = dict(a, shs=None, colors_precomp=extra)
            z = torch.zeros_like(dd)
            og2 = Hh.oracle_backward(b, Hh.run_oracle(b), de, z, z)
            og = {k: (v + og2[k] if k in GRADS and k not in ("dL_dsh", "dL_dcolors") else v) for k, v in og.items()}
            og["dL_dextra"] = og2["dL_dcolors"]
        for t in r.leaves.values():
            t.grad = None
        r.loss(dc, dd, da, de, stored_alpha=fw["alpha"]).backward(retain_graph=True)
        want = r.kernel_grads()
        res = S.compare_grads({k: torch.from_numpy(np.asarray(v)) for k, v in og.items()}, want, keep, RTOL, S.atol_for(kind, ATOL))
        for k, v in res.items():
            worst[(kind, k)] = v
    bad = {k: v for k, v in worst.items() if v > 1.0}
    assert not bad, bad
    return r, fw, worst


@pytest.mark.parametrize("W,H", S.RAGGED_SIZES)
def test_ragged_sizes(W, H):
    a = S.ragged(W, H)
    r, fw, _ = _check(a, kinds=S.LOSSES)
    assert r.visible.any()
    if W % 8 or H % 4:
        assert S.partial_footprint_only(r) > 0


def test_opaque():
    a = S.opaque()
    r, fw, _ = _check(a, kinds=S.LOSSES)
    assert r.meta["clamped_pairs"] > 0
    rg = fw["ranges"].astype(np.int64)
    gx = (a["W"] + 15) // 16
    lens = rg[:, 1] - rg[:, 0]
    ys, xs = np.mgrid[0:a["H"], 0:a["W"]]
    assert (fw["n_contrib"] < lens[(ys // 16) * gx + xs // 16]).sum() > 0.1 * a["W"] * a["H"]  # early termination


def test_deep():
    a = S.deep()
    r, fw, _ = _check(a, kinds=("randn", "onehot_tile"))
    assert int(fw["n_contrib"].max()) > 300
    rg = fw["ranges"].astype(np.int64)
    assert int((rg[:, 1] - rg[:, 0]).max()) > 2048


def test_frustum():
    a = S.frustum()
    r, fw, _ = _check(a, kinds=("randn", "color", "depth"))
    assert r.meta["frustum_clamped"] > 0
    assert int((fw["clamped"].any(axis=1) & (fw["radii"] > 0)).sum()) > 0
    assert not r.visible.all()  # points behind the camera are culled


@pytest.mark.parametrize("cov3d", [False, True])
@pytest.mark.parametrize("sh", S.MODES_SH, ids=lambda s: "precomp" if s is None else "D%dM%d" % s)
def test_modes(sh, cov3d):
    _check(S.modes(sh, cov3d))


def test_fused_extra_colours():
    a = S.modes((3, 16), False)
    _check(a, kinds=("randn", "onehot_footprint"), extra=S.extra_colours(a))
