"""Times one training step through ``renderer.render()``: the fused path (one ``rasterize_gaussians_multi`` call) against the
two-pass graph (``set_fused_training(False)``: two rasterizer calls on the same geometry), in the same process, alternating.

Scene: 3M Gaussians (``scene.config3_scene``) at 1920x1080, trained from their raw parameters (the GaussianModel fields).
Losses:
  * ``full``: the shape of the 3DGS training loop with normal regularisation: L1 on the RGB image, an L2 depth term and
    ``normal_loss(normal, pseudo_normal.detach())``;
  * ``rgb``: L1 on the RGB image only (the inpainting re-training loop), where the normal image gets no gradient.
One step = render() forward + loss + backward, timed with CUDA events after warm-up.  Writes ``render_training.json`` to
``--out`` and prints the card name and power limit beside the numbers.

    python tools/time_render_training.py --out /tmp/rt
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from autovfx_b200 import scene  # noqa: E402


class TrainableGaussians:
    """The GaussianModel surface render() reads, over raw leaf tensors that require gradients (activations as in the
    reference's gaussian_model.py: exp scales, normalised rotations, sigmoid opacities, cat(dc, rest) features)."""

    def __init__(self, raw, sh_degree: int):
        self.raw = raw
        self.active_sh_degree = self.max_sh_degree = sh_degree

    @classmethod
    def from_activated(cls, g, sh_degree: int, device) -> "TrainableGaussians":
        raw = {"xyz": g["means3D"], "f_dc": g["shs"][:, :1], "f_rest": g["shs"][:, 1:], "opacity": torch.logit(g["opacities"]),
               "scaling": torch.log(g["scales"]), "rotation": g["rotations"]}
        return cls({k: v.to(device).float().contiguous().requires_grad_(True) for k, v in raw.items()}, sh_degree)

    @property
    def get_xyz(self):
        return self.raw["xyz"]

    @property
    def get_features(self):
        return torch.cat((self.raw["f_dc"], self.raw["f_rest"]), dim=1)

    @property
    def get_opacity(self):
        return torch.sigmoid(self.raw["opacity"])

    @property
    def get_scaling(self):
        return torch.exp(self.raw["scaling"])

    @property
    def get_rotation(self):
        return torch.nn.functional.normalize(self.raw["rotation"])

    def get_covariance(self, scaling_modifier=1.0):
        """[P,6] upper triangle of R S S^T R^T."""
        r, x, y, z = self.get_rotation.unbind(-1)
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                         2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                         2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], dim=-1).view(-1, 3, 3)
        L = R * (self.get_scaling * scaling_modifier).unsqueeze(1)
        S = L @ L.transpose(1, 2)
        return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], dim=-1)

    def get_normal(self, dir_pp_normalized):
        """Axis of the smallest scale, turned towards the viewer, unit length (gaussian_model.py get_normal)."""
        from tests import wrapper_ref as WR
        n = WR.get_minimum_axis(self.get_scaling, self.get_rotation)
        n, _ = WR.flip_align_view(n, dir_pp_normalized)
        return n / n.norm(dim=1, keepdim=True)

    def zero_grad(self):
        for v in self.raw.values():
            v.grad = None


def normal_loss(pred, gt):
    """L1 + 0.1 x negative cosine between unit normals [H,W,3] (the normal regulariser of 3DGS training loops)."""
    p = torch.nn.functional.normalize(pred, p=2, dim=-1)
    q = torch.nn.functional.normalize(gt, p=2, dim=-1)
    return (p - q).abs().mean() - 0.1 * (p * q).sum(-1).mean()


def training_loss(out, target_rgb, target_depth, rgb_only: bool = False):
    loss = (out["render"][:3] - target_rgb).abs().mean()
    if rgb_only:
        return loss
    return loss + 0.1 * ((out["depth"] - target_depth) ** 2).mean() + 0.05 * normal_loss(out["normal"], out["pseudo_normal"].detach())


PIPE = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)


def _card() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % ex}


def _pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, max(0, int(round(q * (len(xs) - 1)))))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gaussians", type=int, default=3_000_000)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_render_training: needs a CUDA device")
    from autovfx_b200 import renderer as RD
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    card = _card()
    print("card: %s, power limit %s" % (card["name"], card["power_limit"]))

    pc = TrainableGaussians.from_activated(scene.config3_scene(P=args.gaussians), 3, dev)
    traj = scene.trajectory_dict(num_views=300, w=args.width, h=args.height)
    cams = [c.to(dev) for c in scene.cameras_from_trajectory(traj)]
    bg = torch.zeros(3, device=dev)
    gen = torch.Generator().manual_seed(0)
    H, W = args.height, args.width
    target_rgb = torch.rand(3, H, W, generator=gen).to(dev)
    target_depth = (torch.rand(H, W, generator=gen) * 4 + 2).to(dev)

    def step(cam, fused, rgb_only):
        RD.set_fused_training(fused)
        pc.zero_grad()
        out = RD.render(cam, pc, PIPE, bg)
        training_loss(out, target_rgb, target_depth, rgb_only).backward()
        return out

    times = {loss: {"fused": [], "two_pass": []} for loss in ("full", "rgb")}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    try:
        for it in range(args.warmup + args.iters):
            cam = cams[(it * 7) % len(cams)]
            for loss in ("full", "rgb"):
                for fused in ((True, False) if it % 2 == 0 else (False, True)):
                    torch.cuda.synchronize()
                    ev[0].record()
                    step(cam, fused, loss == "rgb")
                    ev[1].record()
                    torch.cuda.synchronize()
                    if it >= args.warmup:
                        times[loss]["fused" if fused else "two_pass"].append(ev[0].elapsed_time(ev[1]))
        # the gradients of one step, fused against two-pass, on the timed size
        agree = {}
        for loss in ("full", "rgb"):
            grads = {}
            for fused in (True, False):
                step(cams[42], fused, loss == "rgb")
                grads[fused] = {k: v.grad.detach().clone() for k, v in pc.raw.items()}
            agree[loss] = {k: float((grads[True][k] - grads[False][k]).abs().max() / (grads[False][k].abs().max() + 1e-30))
                           for k in grads[True]}
    finally:
        RD.set_fused_training(True)

    res = {"workload": "render() forward + loss + backward, %d Gaussians (config3_scene), %dx%d, SH degree 3" % (args.gaussians, W, H),
           "card": card, "iters": args.iters, "warmup": args.warmup, "losses": {}}
    for loss, d in times.items():
        entry = {m: {"median_ms": _pct(v, 0.5), "p10_ms": _pct(v, 0.1), "p90_ms": _pct(v, 0.9)} for m, v in d.items()}
        entry["fused_over_two_pass_median"] = entry["fused"]["median_ms"] / entry["two_pass"]["median_ms"]
        entry["grad_relerr_fused_vs_two_pass"] = agree[loss]
        res["losses"][loss] = entry
        print("%-4s fused %.3f ms (p10 %.3f, p90 %.3f)  two-pass %.3f ms (p10 %.3f, p90 %.3f)  ratio %.3f  max grad relerr %.2e" % (
            loss, entry["fused"]["median_ms"], entry["fused"]["p10_ms"], entry["fused"]["p90_ms"], entry["two_pass"]["median_ms"],
            entry["two_pass"]["p10_ms"], entry["two_pass"]["p90_ms"], entry["fused_over_two_pass_median"], max(agree[loss].values())))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "render_training.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
