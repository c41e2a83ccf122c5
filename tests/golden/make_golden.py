"""Generates the golden vectors under tests/golden/ by running the reference's OWN CUDA rasterizer
(oracle/_ref/libref_dgr.so = unmodified diff-gaussian-rasterization, built by `AUTOVFX_REFERENCE=<reference checkout>` build())
on a B200.

    python tests/golden/make_golden.py OUT     # then copy OUT/*.npz here (config1 and deg3_m25 keep their gradients in grads_<case>.npz)

Inputs are the deterministic named cases of tests/helpers.py (seeded torch generators), so only outputs are stored.

The other reference values the GPU tests compare with (tests/golden/ref_*.npz) are recorded by the tests themselves: with
oracle/_ref and oracle/_ref_py built,

    GSR_RECORD_REFERENCE=OUT python -m pytest -m gpu tests     # then copy OUT/ref_*.npz here
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import helpers as Hh  # noqa: E402
from oracle import ref_cuda  # noqa: E402

CASES = {  # name -> store gradients?
    "config1": ("fw+small_grads",), "small_sh": ("fw+grads",), "small_deg1_m25": ("fw+grads",), "small_precomp": ("fw+grads",),
    "big_splats": ("fw+grads",), "dense_tile": ("fw",), "coplanar": ("fw",), "deg3_m25": ("fw+grads",), "deg2_m25": ("fw",),
}


def main(outdir):
    os.makedirs(outdir, exist_ok=True)
    dev = torch.device("cuda:0")
    for name, (mode,) in CASES.items():
        a = Hh.resolve(Hh.case_inputs(name), dev)
        fw = ref_cuda.forward(a["means3D"], a["opacities"], a["view"], a["proj"], a["campos"], a["W"], a["H"], a["tanfovx"], a["tanfovy"],
                              shs=a["shs"], colors_precomp=a["colors_precomp"], scales=a["scales"], rotations=a["rotations"],
                              cov3D_precomp=a["cov3D_precomp"], sh_degree=a["sh_degree"], scale_modifier=a["scale_modifier"], bg=a["bg"])
        st = ref_cuda.state(dev)
        torch.cuda.synchronize()
        out = {"case": np.array(name), "radii": fw["radii"].cpu().numpy(), "num_rendered": np.array(fw["num_rendered"]),
               "color": fw["color"].cpu().numpy(), "depth": fw["depth"].cpu().numpy(), "alpha": fw["alpha"].cpu().numpy(),
               "point_list": st["point_list"].cpu().numpy(), "ranges": st["ranges"].cpu().numpy(), "n_contrib": st["n_contrib"].cpu().numpy(),
               "means2D": st["means2D"].cpu().numpy(), "depths": st["depths"].cpu().numpy(), "conic_opacity": st["conic_opacity"].cpu().numpy()}
        if mode != "fw":
            dc, dd, da = Hh.image_grads(a, device=dev)
            g = ref_cuda.backward(fw, dc, dd, da)
            torch.cuda.synchronize()
            keys = ["dL_dmeans3D", "dL_dmeans2D", "dL_dopacity", "dL_dscales", "dL_drotations", "dL_dcolors", "dL_dcov3D"]
            if mode == "fw+grads":
                keys.append("dL_dsh")
            for k in keys:
                out[k] = g[k].cpu().numpy()
        path = os.path.join(outdir, name + ".npz")
        if name in ("config1", "deg3_m25"):  # gradients in a file of their own: each file stays under 1 MB
            np.savez_compressed(os.path.join(outdir, "grads_" + name + ".npz"), **{k: out.pop(k) for k in list(out) if k.startswith("dL_")})
        np.savez_compressed(path, **out)
        print(name, "->", path, "%.0f KB" % (os.path.getsize(path) / 1024), "R =", fw["num_rendered"])


def wrapper_golden(outdir, name="small_sh"):
    """render()-wrapper row: the reference's two rasterizer passes (compiled reference) around the wrapper's helper functions
    restated in torch (tests/wrapper_ref.py; the originals cannot be imported) and executed with torch's CUDA kernels."""
    import math
    from tests import wrapper_ref as WR
    dev = torch.device("cuda:0")
    case = Hh.case_inputs(name)
    a = Hh.resolve(case, dev)
    cam = case["cam"]

    def rasterize(shs=None, colors_precomp=None):
        b = dict(a)
        b["shs"], b["colors_precomp"] = shs, colors_precomp
        fw = Hh.run_ref(b)
        return fw["color"], fw["depth"], fw["alpha"], fw["radii"]
    FoVx, FoVy = 2 * math.atan(cam.tanfovx), 2 * math.atan(cam.tanfovy)
    ref = WR.render_two_pass(rasterize, a["means3D"], a["shs"], a["opacities"], a["scales"], a["rotations"], case["sh_degree"],
                             dict(campos=a["campos"], viewmatrix=a["view"], FoVx=FoVx, FoVy=FoVy), a["bg"])
    rgba8 = WR.save_image_bytes(ref["render"].clone())
    nrm = ref["normal"].cpu().numpy()
    normal8 = (((nrm + 1) / 2) * 255).astype(np.uint8)
    depth8 = (np.clip(ref["depth"].cpu().numpy() / 3.0, a_min=0., a_max=1.) * 255).astype(np.uint8)
    out = {"case": np.array(name), "FoVx": np.array(FoVx), "FoVy": np.array(FoVy), "c2w": a["view"].inverse().cpu().numpy(),
           "normal_normed": ref["normal_normed"].cpu().numpy(), "normal_raw_image": ref["normal_raw_image"].cpu().numpy(),
           "render": ref["render"].cpu().numpy(), "depth": ref["depth"].cpu().numpy(), "normal": nrm,
           "pseudo_normal": ref["pseudo_normal"].cpu().numpy(), "rgba8": rgba8.cpu().numpy(), "normal8": normal8, "depth8": depth8}
    path = os.path.join(outdir, "wrapper_" + name + ".npz")
    np.savez_compressed(path, **out)
    print("wrapper", name, "->", path, "%.0f KB" % (os.path.getsize(path) / 1024))


if __name__ == "__main__":
    out = sys.argv[1]
    main(out)
    wrapper_golden(out)
