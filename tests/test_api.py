"""Python surface of the drop-in (no GPU needed): names, settings tuple, validation, alias packages, no CPU fallback,
and the outputs of the reference's own `GaussianRenderer.forward` source, executed verbatim against this package's
interface (stored in tests/golden/renderer.npz)."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from exavatar_release_b200 import GaussianRasterizationSettings, GaussianRasterizer
from util import kat_settings, pack, splat


def test_settings_tuple_matches_call_site():
    # field names and order of module.py:609-622
    assert GaussianRasterizationSettings._fields == (
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix", "sh_degree",
        "campos", "prefiltered", "debug")
    st = kat_settings(settings_cls=GaussianRasterizationSettings)
    assert isinstance(st, tuple) and st.image_height == 32 and st.debug is False


def test_alias_packages_resolve_to_the_same_classes():
    import diff_gaussian_rasterization as vanilla
    import diff_gaussian_rasterization_depth as depth
    assert depth.GaussianRasterizer is GaussianRasterizer and vanilla.GaussianRasterizer is GaussianRasterizer
    assert depth.GaussianRasterizationSettings is GaussianRasterizationSettings


def test_argument_validation_same_messages_as_upstream():
    st = kat_settings(settings_cls=GaussianRasterizationSettings)
    a = pack([splat((0, 0, 2.0))])
    m2 = torch.zeros(1, 3)
    r = GaussianRasterizer(raster_settings=st)
    with pytest.raises(Exception, match="Please provide excatly one of either SHs or precomputed colors!"):
        r(means3D=a["means3D"], means2D=m2, opacities=a["opacities"], scales=a["scales"], rotations=a["rotations"])
    with pytest.raises(Exception, match="Please provide excatly one of either SHs or precomputed colors!"):
        r(means3D=a["means3D"], means2D=m2, opacities=a["opacities"], shs=torch.zeros(1, 16, 3),
          colors_precomp=a["colors_precomp"], scales=a["scales"], rotations=a["rotations"])
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair or precomputed 3D covariance"):
        r(means3D=a["means3D"], means2D=m2, opacities=a["opacities"], colors_precomp=a["colors_precomp"])
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair or precomputed 3D covariance"):
        r(means3D=a["means3D"], means2D=m2, opacities=a["opacities"], colors_precomp=a["colors_precomp"],
          scales=a["scales"], rotations=a["rotations"], cov3D_precomp=torch.zeros(1, 6))


def test_product_path_has_no_cpu_fallback():
    st = kat_settings(settings_cls=GaussianRasterizationSettings)
    a = pack([splat((0, 0, 2.0))])
    r = GaussianRasterizer(raster_settings=st)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        r(means3D=a["means3D"], means2D=torch.zeros(1, 3), opacities=a["opacities"], colors_precomp=a["colors_precomp"],
          scales=a["scales"], rotations=a["rotations"])


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "exavatar_release_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "gs_oracle" not in src, f


def test_missing_library_raises(monkeypatch):
    from exavatar_release_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libb200raster.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()


def test_reference_renderer_source_runs_unmodified_against_our_interface():
    """tests/golden/renderer.npz holds what the reference's `class GaussianRenderer`, executed as-is with this repo's
    camera helpers and the oracle's settings / rasteriser classes, returned for a T0 scene (tests/golden/make_golden.py).
    This package's `GaussianRenderer` over the same rasteriser must reproduce it bit for bit, gradients included."""
    from oracle import oracle as O
    from exavatar_release_b200.renderer import GaussianRenderer

    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "renderer.npz"))
    t = lambda k: torch.from_numpy(z[k])
    assets = {k[len("asset_"):]: t(k).requires_grad_() for k in z.files if k.startswith("asset_")}
    cam = {k[len("cam_"):]: t(k) for k in z.files if k.startswith("cam_")}
    assert set(assets) == {"mean_3d", "opacity", "scale", "rotation", "rgb"}
    assert set(cam) == {"R", "t", "focal", "princpt"}
    mine = GaussianRenderer(rasterizer_cls=O.OracleRasterizer, settings_cls=O.OracleSettings)
    out = mine(assets, (int(z["H"]), int(z["W"])), cam, t("bg"))
    assert 0 < int(z["is_vis"].sum()) < len(z["is_vis"])  # the fixture exercises visible and culled splats
    for k in ("img", "depthmap", "mask", "radius", "is_vis"):
        assert torch.equal(out[k], t(k)), k
    out["img"].sum().backward()
    assert torch.equal(out["mean_2d"].grad, t("grad_mean_2d"))
    assert torch.equal(assets["mean_3d"].grad, t("grad_mean_3d"))
