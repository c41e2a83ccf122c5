"""CPU checks of the test harness that runs the reference's Python callers (oracle/ref_py.py): the third-party stand-ins it
installs (kornia.create_meshgrid, plyfile) behave as the reference code expects, and the .ply layout helpers of
autovfx_b200.scene are byte-compatible with what `GaussianModel.save_ply` produces through the plyfile API."""
import os

import numpy as np
import torch

from autovfx_b200 import scene
from oracle import ref_py


def test_meshgrid_stand_in_matches_kornia_convention():
    g = ref_py._create_meshgrid(3, 5, False)
    assert g.shape == (1, 3, 5, 2)
    assert g[0, 0, :, 0].tolist() == [0.0, 1.0, 2.0, 3.0, 4.0] and g[0, :, 0, 1].tolist() == [0.0, 1.0, 2.0]
    gn = ref_py._create_meshgrid(3, 5, True)
    assert float(gn.min()) == -1.0 and float(gn.max()) == 1.0


def test_plyfile_stand_in_round_trips_the_3dgs_layout(tmp_path):
    raw = scene.config2_raw(P=2000, seed=3)
    n = lambda t: t.numpy()  # noqa: E731
    p = str(tmp_path / "a.ply")
    scene.save_ply(p, n(raw["xyz"]), n(raw["f_dc"]), n(raw["f_rest"]), n(raw["opacity"]), n(raw["scaling"]), n(raw["rotation"]))
    pd = ref_py.PlyData.read(p)
    el = pd.elements[0]
    names = [q.name for q in el.properties]
    assert names[:6] == ["x", "y", "z", "nx", "ny", "nz"] and names[-4:] == ["rot_0", "rot_1", "rot_2", "rot_3"] and len(names) == 62
    assert np.array_equal(np.asarray(el["x"]), n(raw["xyz"])[:, 0]) and np.array_equal(np.asarray(el["opacity"]), n(raw["opacity"])[:, 0])
    # f_rest is stored channel-major: f_rest_k = coefficient k % 15 + 1 of channel k // 15 (gaussian_model.py:206-207)
    assert np.array_equal(np.asarray(el["f_rest_16"]), n(raw["f_rest"])[:, 1, 1])
    # describe() + write() reproduce the file byte for byte (what GaussianModel.save_ply does with the real plyfile)
    q = str(tmp_path / "b.ply")
    ref_py.PlyData([ref_py.PlyElement.describe(el.data, "vertex")]).write(q)
    assert open(p, "rb").read() == open(q, "rb").read()
    back = scene.load_ply(q)
    assert np.array_equal(back["f_rest"], n(raw["f_rest"])) and np.array_equal(back["rot"], n(raw["rotation"]))


def test_reference_modules_import_against_the_drop_in():
    # the import lines of the reference's callers (gaussian_renderer/__init__.py, scene/gaussian_model.py) resolve to the drop-in
    ns = {}
    exec("from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer\n"
         "from simple_knn._C import distCUDA2", ns)
    from autovfx_b200 import knn, rasterizer
    assert ns["GaussianRasterizer"] is rasterizer.GaussianRasterizer and ns["GaussianRasterizationSettings"] is rasterizer.GaussianRasterizationSettings
    assert ns["distCUDA2"] is knn.distCUDA2
    if os.path.isdir(ref_py.GS):  # the staged reference modules, where they are staged
        mods = ref_py.load("ours")
        assert mods.renderer.GaussianRasterizer is rasterizer.GaussianRasterizer
        assert callable(mods.renderer.render) and callable(mods.gaussians_utils.transform_gaussians)
