"""Shared helpers for the parity tests and tools: run the same seeded inputs through (a) the product CUDA path
(autovfx_b200, via the C ABI), (b) the compiled reference (oracle/_ref, GPU) and (c) the CPU oracle.  The tests compare with
(b) through ``reference()``: what the reference computed on the test's inputs is stored under tests/golden/ref_*.npz."""
from __future__ import annotations

import hashlib
import math
import os
import sys
from typing import Callable, Dict, Optional

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from autovfx_b200 import scene  # noqa: E402


def case_inputs(name: str) -> Dict:
    """Named deterministic cases.  Returns dict(g=gaussians (cpu tensors), cam=Camera, kw=extra settings)."""
    if name == "config1":  # BASELINE configs[0]: 10k Gaussians, 256x256
        g, cam = scene.config1_scene()
        return dict(g=g, cam=cam, sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0)
    if name == "small_sh":  # tiny, non-multiple-of-16 image, coloured background
        g = scene.synthetic_gaussians(600, seed=3, extent=(1, 1, 1), log_scale_mean=math.log(0.05), log_scale_std=0.6)
        cam = scene.lookat_camera((0.3, -3.0, 0.4), (0, 0, 0), 100, 75, 55.0)
        return dict(g=g, cam=cam, sh_degree=3, bg=(0.2, 0.5, 0.9), scale_modifier=1.0)
    if name == "small_deg1_m25":  # SuGaR-style storage: M=25 (stride 300 B), active degree 1, scale modifier
        g = scene.synthetic_gaussians(500, seed=5, extent=(1, 1, 1), log_scale_mean=math.log(0.06), log_scale_std=0.5, sh_degree=4)
        cam = scene.lookat_camera((-2.0, -2.0, 1.0), (0, 0, 0), 96, 64, 70.0)
        return dict(g=g, cam=cam, sh_degree=1, bg=(1.0, 1.0, 1.0), scale_modifier=0.8)
    if name == "deg3_m25":  # SuGaR storage (M=25, 300-byte rows: only 4-byte aligned) rendered at degree 3 and 2: windowed SH staging
        g = scene.synthetic_gaussians(3000, seed=23, extent=(1, 1, 1), log_scale_mean=math.log(0.04), log_scale_std=0.5, sh_degree=4)
        cam = scene.lookat_camera((1.5, -2.5, 0.8), (0, 0, 0), 144, 96, 65.0)
        return dict(g=g, cam=cam, sh_degree=3, bg=(0.3, 0.3, 0.3), scale_modifier=1.0)
    if name == "deg2_m25":
        g = scene.synthetic_gaussians(2000, seed=29, extent=(1, 1, 1), log_scale_mean=math.log(0.05), log_scale_std=0.5, sh_degree=4)
        cam = scene.lookat_camera((-1.0, -2.8, 0.5), (0, 0, 0), 112, 80, 65.0)
        return dict(g=g, cam=cam, sh_degree=2, bg=(0.0, 0.0, 0.0), scale_modifier=1.0)
    if name == "small_precomp":  # colors_precomp + cov3D_precomp mode
        g = scene.synthetic_gaussians(700, seed=7, extent=(1, 1, 1), log_scale_mean=math.log(0.05), log_scale_std=0.5)
        cam = scene.lookat_camera((0.0, -2.5, 1.5), (0, 0, 0), 80, 80, 60.0)
        return dict(g=g, cam=cam, sh_degree=0, bg=(0.0, 0.0, 0.0), scale_modifier=1.0, precomp=True)
    if name == "big_splats":  # few huge splats (warp-cooperative tile walk) + a camera inside the cloud (near culling)
        g = scene.synthetic_gaussians(300, seed=11, extent=(1.5, 1.5, 1.5), log_scale_mean=math.log(0.4), log_scale_std=0.7)
        cam = scene.lookat_camera((0.2, -0.6, 0.1), (0, 0.5, 0), 128, 112, 80.0)
        return dict(g=g, cam=cam, sh_degree=2, bg=(0.1, 0.1, 0.1), scale_modifier=1.0)
    if name == "dense_tile":  # > 4096 splats on single tiles: exercises the large-bucket sort path
        g = scene.synthetic_gaussians(30000, seed=13, extent=(0.05, 0.05, 1.0), log_scale_mean=math.log(0.004), log_scale_std=0.3,
                                      opacity_mean=-3.0, opacity_std=1.0)
        cam = scene.lookat_camera((0.0, -3.0, 0.0), (0, 0, 0), 64, 64, 40.0)
        return dict(g=g, cam=cam, sh_degree=3, bg=(0.0, 0.0, 0.0), scale_modifier=1.0)
    if name == "coplanar":  # thousands of exactly equal depths: sort ties resolve by Gaussian id; degenerate depth range
        g = scene.synthetic_gaussians(6000, seed=17, extent=(0.6, 0.0, 0.6), log_scale_mean=math.log(0.02), log_scale_std=0.3,
                                      opacity_mean=-2.0, opacity_std=1.0)
        cam = scene.lookat_camera((0.0, -2.0, 0.0), (0, 0, 0), 96, 96, 50.0)
        return dict(g=g, cam=cam, sh_degree=3, bg=(0.0, 0.2, 0.0), scale_modifier=1.0)
    raise KeyError(name)


def cov3d_from(scales: torch.Tensor, rotations: torch.Tensor, mod: float) -> torch.Tensor:
    """Python-side precomputed covariance (what gaussian_model.get_covariance builds, gaussian_model.py:47-52,117-118)."""
    r, x, y, z = rotations.unbind(-1)
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                     2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                     2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], dim=-1).view(-1, 3, 3)
    L = R * (scales * mod).unsqueeze(1)  # R @ diag(s)
    S = L @ L.transpose(1, 2)
    return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], dim=-1).contiguous()


def resolve(case: Dict, device=None) -> Dict:
    """Flatten a case into the exact argument set of one rasterizer call."""
    g, cam = case["g"], case["cam"]
    a = dict(means3D=g["means3D"], opacities=g["opacities"], view=cam.world_view_transform, proj=cam.full_proj_transform,
             campos=cam.camera_center, W=cam.image_width, H=cam.image_height, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
             sh_degree=case["sh_degree"], scale_modifier=case["scale_modifier"], bg=torch.tensor(case["bg"], dtype=torch.float32),
             shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None)
    if case.get("precomp"):
        gen = torch.Generator().manual_seed(99)
        a["colors_precomp"] = torch.rand(g["means3D"].shape[0], 3, generator=gen)
        a["cov3D_precomp"] = cov3d_from(g["scales"], g["rotations"], case["scale_modifier"])
    else:
        a["shs"], a["scales"], a["rotations"] = g["shs"], g["scales"], g["rotations"]
    if device is not None:
        a = {k: (v.to(device) if isinstance(v, torch.Tensor) else v) for k, v in a.items()}
    return a


def settings_from(a: Dict, debug=False, prefiltered=False):
    from autovfx_b200.rasterizer import GaussianRasterizationSettings
    return GaussianRasterizationSettings(image_height=a["H"], image_width=a["W"], tanfovx=a["tanfovx"], tanfovy=a["tanfovy"], bg=a["bg"],
                                         scale_modifier=a["scale_modifier"], viewmatrix=a["view"], projmatrix=a["proj"],
                                         sh_degree=a["sh_degree"], campos=a["campos"], prefiltered=prefiltered, debug=debug)


def run_ours(a: Dict, for_backward=False, sorted_keys=False, debug=True, tight=None, exact=None):
    from autovfx_b200 import rasterizer as R
    s = settings_from(a, debug=debug)
    color, depth, alpha, radii, ws, ticket, keep = R.forward_raw(a["means3D"], a["shs"], a["colors_precomp"], a["opacities"], a["scales"],
                                                                 a["rotations"], a["cov3D_precomp"], s, for_backward=for_backward,
                                                                 sorted_keys=sorted_keys, sync=True, tight=tight, exact=exact)
    views = R.debug_views(ws, a["means3D"].shape[0], a["W"], a["H"])
    return dict(color=color, depth=depth, alpha=alpha, radii=radii, views=views, stats=ticket.stats(), ws=ws, keep=keep)


def run_ref(a: Dict):
    from oracle import ref_cuda
    fw = ref_cuda.forward(a["means3D"], a["opacities"], a["view"], a["proj"], a["campos"], a["W"], a["H"], a["tanfovx"], a["tanfovy"],
                          shs=a["shs"], colors_precomp=a["colors_precomp"], scales=a["scales"], rotations=a["rotations"],
                          cov3D_precomp=a["cov3D_precomp"], sh_degree=a["sh_degree"], scale_modifier=a["scale_modifier"], bg=a["bg"])
    return fw


GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
# A directory: reference() runs the compiled reference and writes what it returned to <dir>/ref_<group>.npz (see
# tests/golden/make_golden.py); unset, reference() reads tests/golden/ref_<group>.npz.
RECORD_DIR = os.environ.get("GSR_RECORD_REFERENCE")
INLINE_BYTES = 1 << 16  # larger arrays are stored as digests unless named in `full`
_golden: Dict[str, Dict] = {}


def _np(x) -> np.ndarray:
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def digest(x) -> str:
    a = _np(x)
    return "sha256:%s:%s:%s" % (a.dtype.str, "x".join(map(str, a.shape)), hashlib.sha256(a.tobytes()).hexdigest())


def reference(group: str, key: str, compute: Callable[[], Dict], full=()) -> Dict:
    """What the reference computed for one test input, {name: np.ndarray or digest string}: ``compute()`` (which runs the
    reference) when recording, the stored values otherwise.  Arrays up to INLINE_BYTES and those named in ``full`` are stored
    whole; a larger one as the SHA-256 of its bytes, dtype and shape, which ``same()`` compares bit for bit."""
    if group not in _golden:
        path = os.path.join(GOLDEN_DIR, "ref_%s.npz" % group)
        _golden[group] = {} if RECORD_DIR else dict(np.load(path))
    st = _golden[group]
    if RECORD_DIR:
        for name, v in compute().items():
            a = _np(v)
            st[key + "::" + name] = a if (a.nbytes <= INLINE_BYTES or name in full) else np.array(digest(a))
        os.makedirs(RECORD_DIR, exist_ok=True)
        np.savez_compressed(os.path.join(RECORD_DIR, "ref_%s.npz" % group), **st)
    pre = key + "::"
    out = {k[len(pre):]: v for k, v in st.items() if k.startswith(pre)}
    assert out, "no stored reference values for %s/%s" % (group, key)
    return {k: (str(v) if v.dtype.kind == "U" else v) for k, v in out.items()}


def same(x, ref) -> bool:
    """x equals, bit for bit (dtype and shape included), a value returned by reference()."""
    if isinstance(ref, str):
        return digest(x) == ref
    a = _np(x)
    return a.dtype == ref.dtype and a.shape == ref.shape and np.array_equal(a, ref)


def ref_forward(group: str, key: str, a: Dict, names=("color", "depth", "alpha", "radii", "num_rendered"), state=(), full=()) -> Dict:
    """reference() of one forward of the compiled reference rasterizer on the call arguments ``a``; ``state`` names entries of
    its internal buffers (oracle.ref_cuda.state) to keep as well."""
    def compute():
        fw = run_ref(a)
        out = {k: fw[k] for k in names}
        if state:
            from oracle import ref_cuda
            rs = ref_cuda.state(a["means3D"].device)
            out.update({k: rs[k] for k in state})
        torch.cuda.synchronize()
        return out
    return reference(group, key, compute, full=full)


def golden_case(name: str) -> Dict:
    """tests/golden/<name>.npz (the reference's forward + backward on a named case), with grads_<name>.npz when the gradients
    are stored apart."""
    gold = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    gp = os.path.join(GOLDEN_DIR, "grads_" + name + ".npz")
    if os.path.exists(gp):
        gold.update(np.load(gp))
    return gold


def run_oracle(a: Dict, stop_after="render"):
    from oracle import gsr_oracle as O
    n = lambda t: None if t is None else t.detach().cpu().numpy()  # noqa: E731
    return O.forward(n(a["means3D"]), n(a["opacities"]), n(a["view"]), n(a["proj"]), n(a["campos"]), a["W"], a["H"], a["tanfovx"],
                     a["tanfovy"], shs=n(a["shs"]), colors_precomp=n(a["colors_precomp"]), scales=n(a["scales"]), rotations=n(a["rotations"]),
                     cov3D_precomp=n(a["cov3D_precomp"]), sh_degree=a["sh_degree"], scale_modifier=a["scale_modifier"],
                     bg=tuple(float(v) for v in a["bg"].cpu()), stop_after=stop_after)


def oracle_backward(a: Dict, fw, dc, dd, da):
    from oracle import gsr_oracle as O
    n = lambda t: None if t is None else t.detach().cpu().numpy()  # noqa: E731
    return O.backward(fw, n(a["means3D"]), n(a["view"]), n(a["proj"]), n(a["campos"]), a["W"], a["H"], a["tanfovx"], a["tanfovy"],
                      n(dc), n(dd), n(da), shs=n(a["shs"]), colors_precomp=n(a["colors_precomp"]), scales=n(a["scales"]),
                      rotations=n(a["rotations"]), cov3D_precomp=n(a["cov3D_precomp"]), sh_degree=a["sh_degree"],
                      scale_modifier=a["scale_modifier"], bg=tuple(float(v) for v in a["bg"].cpu()))


def image_grads(a: Dict, seed=7, device=None):
    """dL/dcolor, dL/ddepth, dL/dalpha ~ N(0,1), seed 7 (SURVEY §8d config 3)."""
    g = torch.Generator().manual_seed(seed)
    H, W = a["H"], a["W"]
    dc, dd, da = torch.randn(3, H, W, generator=g), torch.randn(1, H, W, generator=g), torch.randn(1, H, W, generator=g)
    if device is not None:
        dc, dd, da = dc.to(device), dd.to(device), da.to(device)
    return dc, dd, da


def ours_backward(a: Dict, dc, dd, da):
    """Forward+backward through the public GaussianRasterizer API; returns (outputs, grads dict)."""
    from autovfx_b200.rasterizer import GaussianRasterizer
    leaves = {}
    for k in ("means3D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D_precomp"):
        leaves[k] = None if a[k] is None else a[k].detach().clone().requires_grad_(True)
    means2D = torch.zeros_like(leaves["means3D"], requires_grad=True)
    rast = GaussianRasterizer(settings_from(a))
    color, depth, alpha, radii = rast(leaves["means3D"], means2D, leaves["opacities"], shs=leaves["shs"], colors_precomp=leaves["colors_precomp"],
                                      scales=leaves["scales"], rotations=leaves["rotations"], cov3D_precomp=leaves["cov3D_precomp"])
    loss = (color * dc).sum() + (depth * dd).sum() + (alpha * da).sum()
    loss.backward()
    grads = {k: (None if v is None else v.grad) for k, v in leaves.items()}
    grads["means2D"] = means2D.grad
    return (color, depth, alpha, radii), grads


# default (fast-alpha) blend against exact images: the measured differences are ~1e-6 of the value; BASELINE allows 1e-4
FAST_TOL = {"color": 1e-5, "alpha": 1e-5, "depth": 5e-5}


def assert_images_close(got: Dict, want: Dict, tol=None):
    for k in ("color", "depth", "alpha"):
        t = FAST_TOL[k] if tol is None else tol
        e = maxabs(got[k], want[k])
        assert e <= t, "%s: max abs %.3g > %.3g" % (k, e, t)


def maxabs(a, b) -> float:
    a = torch.as_tensor(a).float().cpu()
    b = torch.as_tensor(b).float().cpu()
    if a.numel() == 0:
        return 0.0
    return float((a - b).abs().max())


def relerr(a, b) -> float:
    """max |a-b| / (max|b| + tiny): scale-aware error for gradient tensors."""
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    if a.numel() == 0:
        return 0.0
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))
