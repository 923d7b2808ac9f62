"""Generates tests/golden/*.npz from the REFERENCE's own Python code.

    python tests/golden/make_golden.py <checkout of ExAvatar_RELEASE>

The tests run without the reference, so its outputs are committed as fixtures:
  camera.npz   : get_fov / get_view_matrix / get_proj_matrix of avatar/common/utils/transforms.py:38-70
                 and the derived rasteriser settings of module.py:604-622, for a few cameras
  sh.npz       : eval_sh (transforms.py:112-167) + 0.5, clamp_min 0 (module.py:265-266) for degrees 0..3
  renderer.npz : `GaussianRenderer` of avatar/common/nets/module.py executed as-is with this repo's camera helpers
                 and the CPU oracle behind its settings / rasteriser names: inputs, outputs, and the gradients of
                 img.sum() at mean_2d and mean_3d (tests/test_api.py)
`.cuda()` is patched to the identity because the reference hard-codes it (transforms.py:40,56,69, module.py:592,625).
"""
import ast
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
REF_ROOT = None  # the reference checkout, from the command line
REF_TRANSFORMS = os.path.join("avatar", "common", "utils", "transforms.py")
REF_MODULE = os.path.join("avatar", "common", "nets", "module.py")


def load_ref():
    torch.Tensor.cuda = lambda self, *a, **k: self
    spec = importlib.util.spec_from_file_location("ref_transforms", os.path.join(REF_ROOT, REF_TRANSFORMS))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def main():
    T = load_ref()
    g = torch.Generator().manual_seed(7)
    cams = []
    for (H, W, fx, fy) in [(512, 512, 750.08, 750.08), (1080, 1920, 1700.0, 1690.5), (256, 256, 375.04, 375.04),
                           (136, 200, 199.24, 199.24), (1024, 1024, 1500.0, 1500.0)]:
        A = torch.randn(3, 3, generator=g)
        R, _ = torch.linalg.qr(A)
        if torch.det(R) < 0:
            R[:, 0] = -R[:, 0]
        t = torch.randn(3, generator=g) * 0.5 + torch.tensor([0.0, 0.0, 3.0])
        focal = torch.tensor([fx, fy])
        princpt = torch.tensor([W / 2.0 + 3.0, H / 2.0 - 5.0])  # off-centre on purpose: the reference ignores it
        fov = T.get_fov(focal, princpt, (H, W))
        view = T.get_view_matrix(R, t).permute(1, 0)
        proj = T.get_proj_matrix(focal, princpt, (H, W), 0.01, 100, 1.0).permute(1, 0)
        full = torch.mm(view, proj)
        campos = view.inverse()[3, :3]
        cams.append(dict(H=H, W=W, R=R.numpy(), t=t.numpy(), focal=focal.numpy(), princpt=princpt.numpy(), fov=fov.numpy(),
                         view=view.contiguous().numpy(), proj=proj.contiguous().numpy(), full=full.contiguous().numpy(),
                         campos=campos.numpy(), tanfovx=float(torch.tan(fov[0] / 2)), tanfovy=float(torch.tan(fov[1] / 2))))
    np.savez(os.path.join(HERE, "camera.npz"), **{f"{k}_{i}": np.asarray(v) for i, c in enumerate(cams) for k, v in c.items()},
             n=len(cams))

    P = 64
    pos = torch.randn(P, 3, generator=g) * 2.0
    campos = torch.tensor([0.3, -0.2, -4.0])
    shs = torch.randn(P, 16, 3, generator=g) * 0.6
    d = pos - campos[None]
    dirs = d / d.norm(dim=1, keepdim=True)
    out = {}
    for deg in range(4):
        # reference layout is (..., C, coeffs): module.py:264 transposes (P,16,3) -> (P,3,16)
        rgb = T.eval_sh(deg, shs.permute(0, 2, 1), dirs)
        out[f"rgb_deg{deg}"] = torch.clamp_min(rgb + 0.5, 0.0).numpy()
    np.savez(os.path.join(HERE, "sh.npz"), pos=pos.numpy(), campos=campos.numpy(), shs=shs.numpy(), **out)
    renderer_golden()
    print("wrote camera.npz, sh.npz, renderer.npz")


def renderer_golden():
    """The reference's `class GaussianRenderer` source, executed unmodified: its free names are satisfied by this repo
    (camera helpers; settings / rasteriser classes with the CPU oracle behind them)."""
    from exavatar_release_b200 import camera
    from exavatar_release_b200.synthetic import make_assets
    from oracle import build as obuild
    obuild.build()
    from oracle import oracle as O

    path = os.path.join(REF_ROOT, REF_MODULE)
    src = open(path).read()
    cls = next(n for n in ast.parse(src).body if isinstance(n, ast.ClassDef) and n.name == "GaussianRenderer")
    ns = {"torch": torch, "nn": torch.nn, "get_fov": camera.get_fov, "get_view_matrix": camera.get_view_matrix,
          "get_proj_matrix": camera.get_proj_matrix, "GaussianRasterizationSettings": O.OracleSettings,
          "GaussianRasterizer": O.OracleRasterizer}
    exec(compile(ast.get_source_segment(src, cls), path, "exec"), ns)
    ref_renderer = ns["GaussianRenderer"]()

    assets = {k: v.requires_grad_() for k, v in make_assets("T0", seed=5).items()}
    cam = {"R": torch.eye(3), "t": torch.zeros(3), "focal": torch.tensor([93.76, 93.76]),
           "princpt": torch.tensor([32.0, 32.0])}
    bg = torch.tensor([0.2, 0.4, 0.6])
    out = ref_renderer(assets, (64, 64), cam, bg)
    out["img"].sum().backward()
    arr = lambda t: t.detach().numpy()
    np.savez(os.path.join(HERE, "renderer.npz"), H=64, W=64, bg=arr(bg),
             **{f"asset_{k}": arr(v) for k, v in assets.items()}, **{f"cam_{k}": arr(v) for k, v in cam.items()},
             **{k: arr(out[k]) for k in ("img", "depthmap", "mask", "radius", "is_vis")},
             grad_mean_2d=arr(out["mean_2d"].grad), grad_mean_3d=arr(assets["mean_3d"].grad))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    REF_ROOT = sys.argv[1]
    main()
