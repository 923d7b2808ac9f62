"""Shared helpers for the test-suite."""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from exavatar_release_b200.camera import look_at_cam_param  # noqa: E402
from exavatar_release_b200.renderer import render_settings  # noqa: E402
from exavatar_release_b200.synthetic import WORKLOADS, make_assets, make_grad_image  # noqa: E402
from oracle.oracle import OracleSettings  # noqa: E402


def kat_settings(W=32, H=32, f=32.0, bg=(0.0, 0.0, 0.0), R=None, t=None, device="cpu", settings_cls=OracleSettings):
    """App. B camera: R = I, t = 0, fx = fy = f (tanfov = W / 2f)."""
    cam = {
        "R": torch.eye(3) if R is None else R,
        "t": torch.zeros(3) if t is None else t,
        "focal": torch.tensor([f, f], dtype=torch.float32),
        "princpt": torch.tensor([W / 2.0, H / 2.0], dtype=torch.float32),
    }
    cam = {k: v.to(device) for k, v in cam.items()}
    return render_settings((H, W), cam, torch.tensor(bg, dtype=torch.float32, device=device), settings_cls)


def workload_settings(name, yaw=0.0, bg=(1.0, 1.0, 1.0), device="cpu", settings_cls=OracleSettings):
    wl = WORKLOADS[name]
    cam = look_at_cam_param(yaw, (wl.height, wl.width), device=device)
    return render_settings((wl.height, wl.width), cam, torch.tensor(bg, dtype=torch.float32, device=device), settings_cls)


def splat(p, scale=0.1, q=(1.0, 0.0, 0.0, 0.0), o=0.5, rgb=(1.0, 0.0, 0.0)):
    s = (scale, scale, scale) if np.isscalar(scale) else scale
    return dict(p=p, s=s, q=q, o=o, rgb=rgb)


def pack(splats, device="cpu", dtype=torch.float32):
    t = lambda k, n: torch.tensor([list(s[k]) if n > 1 else [s[k]] for s in splats], dtype=dtype, device=device).reshape(-1, n)
    return dict(means3D=t("p", 3), scales=t("s", 3), rotations=t("q", 4), opacities=t("o", 1), colors_precomp=t("rgb", 3))


def rel_err(x, y, floor):
    """max |x-y| / max(|y|, floor)  (SURVEY section 8c tolerance form)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    if x.size == 0:
        return 0.0
    return float(np.max(np.abs(x - y) / np.maximum(np.abs(y), floor)))


def ctx_arrays(lib, ws_owner, P, W, H):
    """(ranges (Tn,2) uint32, ids uint32, n_contrib (H,W) uint32, final_T (H,W) float32) of the last projection +
    binning (and, for a FramePlan, forward composite) that ran in `ws_owner`'s workspace: a FramePlan or a pass of a
    MergedFivePlan (whose views keep their per-pixel state outside the ctx, so there only ranges and ids are theirs)."""
    import ctypes as C
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    buf = ws_owner.ctx_buf.cpu().numpy()
    base = ws_owner.ctx_buf.data_ptr()
    off = lambda fn: fn(C.byref(ws_owner.ws), P, W, H) - base
    take = lambda o, n, dt: np.frombuffer(buf[o:o + n].tobytes(), dt)
    ranges = take(off(lib.b2r_ctx_ranges), tiles * 8, np.uint32).reshape(tiles, 2)
    ncon = take(off(lib.b2r_ctx_n_contrib), W * H * 4, np.uint32).reshape(H, W)
    fT = take(off(lib.b2r_ctx_final_T), W * H * 4, np.float32).reshape(H, W)
    ids = ws_owner.ids.cpu().numpy().view(np.uint32)
    return ranges, ids, ncon, fT


def settings_on(st, device, settings_cls):
    """The SAME settings (bit for bit) with their tensors on `device`, as another settings class.  Camera matrices built
    on different devices can differ in the last bit (atan / tan / inverse / mm), which flips radius and tile-rect
    decisions for a few of 10^5 Gaussians; parity tests therefore build them once (CPU) and hand both paths the same bits."""
    import torch
    d = st._asdict()
    for k, v in d.items():
        if isinstance(v, torch.Tensor):
            d[k] = v.to(device)
    return settings_cls(**d)
