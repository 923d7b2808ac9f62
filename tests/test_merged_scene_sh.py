"""A scene with two colour sources (B2RScene.sh_rows): SH rows first, rgb rows after -- the merged five-render frame with
its scene Gaussians coloured from SH in the projection kernel.  Host-side checks that need no GPU: the field's place in
the header's struct, the argument validation of the C ABI (before any CUDA call), and the front end's ValueErrors."""
import ctypes as C
import os
import shutil
import subprocess

import pytest
import torch

from util import ROOT  # noqa: F401  (path setup)
from exavatar_release_b200 import _lib as L
from exavatar_release_b200.fused import scene_sh_degree
from exavatar_release_b200.renderer import scene_gaussian_assets
from exavatar_release_b200.synthetic import make_population_assets, make_scene_sh_params

FAKE = 0x1000  # never dereferenced on the host


def test_sh_rows_sits_at_the_header_offset(tmp_path):
    cc = shutil.which(os.environ.get("CC", "cc")) or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "b200raster.h"\n'
                   'int main(void) { printf("%zu %zu %zu\\n", offsetof(B2RScene, sh_rows), offsetof(B2RScene, skin_J), '
                   'sizeof(B2RScene)); return 0; }\n')
    exe = tmp_path / "off"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    off, off_j, size = (int(v) for v in subprocess.check_output([str(exe)]).split())
    assert L.B2RScene.sh_rows.offset == off == off_j + 4
    assert C.sizeof(L.B2RScene) == size == L.load().b2r_sizeof(0)
    assert L.B2RScene.sh_rows.size == 4


def _scene(P=40):
    sc = L.B2RScene()
    sc.P, sc.width, sc.height, sc.tanfovx, sc.tanfovy = P, 32, 32, 0.5, 0.5
    sc.bg = sc.viewmatrix = sc.projmatrix = sc.campos = FAKE
    sc.means3D = sc.opacities = sc.scales = sc.rotations = FAKE
    sc.shs, sc.colors_precomp = FAKE, FAKE
    sc.sh_degree, sc.sh_coeffs, sc.sh_rows = 3, 16, 33  # a warp straddles the boundary
    return sc


def test_forward_validation_of_sh_rows_without_touching_cuda():
    lib = L.load()
    sc = _scene()
    ws = L.B2RWorkspace()
    ws.ctx, ws.ctx_bytes = FAKE, 16  # too small on purpose: a scene that validates reaches the workspace check (-2)
    out = L.B2RForwardOutputs()
    fwd = lambda: lib.b2r_forward(C.byref(sc), C.byref(ws), C.byref(out), None)
    proj = lambda: lib.b2r_forward_project(C.byref(sc), C.byref(ws), FAKE, None)
    assert fwd() == -2 and proj() == -2          # both sources, SH rows [0, 33), colours for the rest
    sc.sh_rows = -1
    assert fwd() == -1 and proj() == -1
    sc.sh_rows = 41
    assert fwd() == -1 and proj() == -1          # beyond P
    sc.sh_rows = 40
    assert fwd() == -2                           # every row from SH: the colours are not read, may be given
    sc.colors_precomp = None
    assert fwd() == -2                           # ... or not
    sc.sh_rows = 39
    assert fwd() == -1 and proj() == -1          # colour rows without colours
    sc.colors_precomp = FAKE
    sc.shs = None
    assert fwd() == -1                           # SH rows without coefficients
    sc.shs = FAKE
    sc.sh_degree, sc.sh_coeffs = 3, 9
    assert fwd() == -1                           # the degree rules of `shs` still hold for the SH rows
    sc.sh_degree, sc.sh_coeffs = 1, 9
    assert fwd() == -2
    sc.skin_xyz = sc.skin_weights = sc.skin_joint_mats = sc.skin_trans = FAKE
    sc.skin_J = 55
    assert fwd() == -1                           # not with fused skinning
    sc.sh_rows = 0
    assert fwd() == -1                           # sh_rows == 0: exactly one colour source, as before
    sc.colors_precomp = None
    assert fwd() == -2
    sc.P, sc.sh_rows = 0, 1
    assert fwd() == -1                           # sh_rows > P also for an empty scene
    assert lib.b2r_launch_count() == 0


def test_backward_validation_of_sh_rows_without_touching_cuda():
    lib = L.load()
    sc = _scene()
    ws = L.B2RWorkspace()
    ws.ctx, ws.ctx_bytes = FAKE, lib.b2r_ctx_bytes(40, 32, 32)
    args = L.B2RBackwardArgs()
    args.dL_dcolor = FAKE
    # a scratch of 8 bytes is too small: arguments that validate return -2 and nothing is launched
    bwd = lambda: lib.b2r_backward(C.byref(sc), C.byref(ws), C.byref(args), FAKE, 8, None)
    bp = lambda: lib.b2r_backward_project(C.byref(sc), C.byref(ws), C.byref(args), FAKE, 8, None)
    both = lambda: (bwd(), bp())
    assert both() == (-1, -1)                    # SH rows past first_row need dL_dshs
    args.dL_dshs = FAKE
    assert both() == (-2, -2)
    for fr in (1, 20, 32):
        args.first_row = fr
        assert both() == (-1, -1), fr            # a detached prefix may not cut the SH rows
    for fr in (33, 40):
        args.first_row = fr
        assert both() == (-2, -2), fr
    args.dL_dshs = None
    assert both() == (-2, -2)                    # first_row >= sh_rows: no SH row takes part, dL_dshs may be NULL
    args.first_row = 0
    sc.sh_rows = 0
    sc.colors_precomp = None
    assert both() == (-1, -1)                    # one source (SH): dL_dshs is needed, as before
    args.dL_dshs = FAKE
    assert both() == (-2, -2)
    assert lib.b2r_launch_count() == 0


def test_scene_colour_source_must_match_the_frame_renderer():
    p = make_scene_sh_params("T0", seed=0)
    cam = {"R": torch.eye(3), "t": torch.zeros(3)}
    sh = scene_gaussian_assets(p["mean"], p["opacity_logit"], p["log_scale"], p["rotation"], p["feature_dc"],
                               p["feature_rest"], 3, cam, in_kernel_sh=True)
    rgb = scene_gaussian_assets(p["mean"], p["opacity_logit"], p["log_scale"], p["rotation"], p["feature_dc"],
                                p["feature_rest"], 3, cam, in_kernel_sh=False)
    assert scene_sh_degree(rgb, 0) is None
    assert scene_sh_degree(sh, 16) == 3
    assert scene_sh_degree(dict(sh, sh_degree=1), 16) == 1
    with pytest.raises(ValueError, match="needs rgb"):
        scene_sh_degree(sh, 0)                   # SH scene, rgb instance
    with pytest.raises(ValueError, match="needs shs"):
        scene_sh_degree(rgb, 16)                 # rgb scene, SH instance
    with pytest.raises(ValueError, match=r"\(P, 9, 3\)"):
        scene_sh_degree(sh, 9)                   # coefficient count differs
    with pytest.raises(ValueError, match="sh_degree"):
        scene_sh_degree(dict(sh, sh_degree=4), 16)
    with pytest.raises(ValueError, match="sh_degree"):
        scene_sh_degree({k: v for k, v in sh.items() if k != "sh_degree"}, 16)
    # GaussianRenderer's rule: with both present, rgb wins
    assert scene_sh_degree(dict(sh, rgb=rgb["rgb"]), 0) is None


def test_merged_plan_rejects_bad_coefficient_counts():
    from exavatar_release_b200.plan import MergedFivePlan
    for M, Ps in ((17, 10), (-1, 10), (16, 0)):
        with pytest.raises(ValueError, match="scene_sh_coeffs"):
            MergedFivePlan(Ps, 10, 32, 32, None, "cpu", scene_sh_coeffs=M)


def test_scene_sh_generator_leaves_the_other_generators_alone():
    p = make_scene_sh_params("T1", seed=0)
    scene, _, _ = make_population_assets("T1", seed=0)
    again, _, _ = make_population_assets("T1", seed=0)
    for k in scene:
        assert torch.equal(scene[k], again[k])
    Ps = scene["mean_3d"].shape[0]
    assert p["feature_dc"].shape == (Ps, 1, 3) and p["feature_rest"].shape == (Ps, 15, 3)
    assert torch.equal(p["mean"], scene["mean_3d"])
    # DC term alone reproduces the population's rgb (RGB2SH)
    assert torch.allclose(0.28209479177387814 * p["feature_dc"][:, 0] + 0.5, scene["rgb"], atol=1e-6)
    assert torch.equal(make_scene_sh_params("T1", seed=0)["feature_rest"], p["feature_rest"])
    assert not torch.equal(make_scene_sh_params("T1", seed=1)["feature_rest"], p["feature_rest"])
