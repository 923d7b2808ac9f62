"""Seeded synthetic Gaussian assets for parity tests and bench.py (no dataset / SMPL-X files offline).

Generator of SURVEY.md section 8(d).  Two populations:
  * "avatar": what `HumanGaussian.forward` emits (module.py:516-586): isotropic scale (module.py:532),
    identity quaternion (module.py:564), opacity == 1 (module.py:565), on a body-sized ellipsoid shell;
  * "scene": what `SceneGaussian.forward` emits (module.py:253-272): anisotropic, random rotation,
    sigmoid opacity, scattered through the view frustum.
Workloads follow BASELINE.json `configs` (C1..C5).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

SH_C0 = 0.28209479177387814


@dataclass(frozen=True)
class Workload:
    name: str
    height: int
    width: int
    n_avatar: int
    n_scene: int
    sh_degree: int  # 0 => colours precomputed (ExAvatar's real call, module.py:618,635-636)
    backward: bool


WORKLOADS = {
    # BASELINE.json configs[0..4]
    "C1": Workload("C1:256x256,10475 avatar splats,fwd", 256, 256, 10475, 0, 0, False),
    "C2": Workload("C2:512x512,100k splats (56k avatar+44k scene),fwd+bwd", 512, 512, 56000, 44000, 0, True),
    "C3": Workload("C3:1024x1024,300k splats,SH deg 3,fwd+bwd", 1024, 1024, 167000, 133000, 3, True),
    "C4": Workload("C4:512x512 train frame,167k avatar+130k scene,fwd+bwd", 512, 512, 167000, 130000, 0, True),
    "C5": Workload("C5:1920x1080,500k splats (167k avatar+333k scene),fwd", 1080, 1920, 167000, 333000, 0, False),
    # small cases for tests
    "T0": Workload("T0:64x64,300 splats", 64, 64, 150, 150, 0, True),
    "T1": Workload("T1:128x96,4k splats", 96, 128, 2000, 2000, 0, True),
    "T2": Workload("T2:200x136,6k splats,SH3", 136, 200, 3000, 3000, 3, True),
    # odd image sizes (ExAvatar renders at the size of the input frame): T3's width is not a multiple of 4 (scalar
    # output stores) and its right / bottom quarter tiles are cut off; T4's right-hand tiles have a half-inside quarter
    # and a quarter wholly outside, and its bottom tile row a warp whose 8x4 pixel rect lies wholly below the image
    "T3": Workload("T3:101x77,4k splats", 77, 101, 2000, 2000, 0, True),
    "T4": Workload("T4:100x68,4k splats", 68, 100, 2000, 2000, 0, True),
}


def _avatar(n, g, tiny_scale=False):
    # points on a 0.5 x 1.7 x 0.3 m ellipsoid shell centred 4.24 m in front of the camera
    u = torch.randn(n, 3, generator=g)
    u = u / u.norm(dim=1, keepdim=True)
    semi = torch.tensor([0.25, 0.85, 0.15])
    pos = u * semi
    normal = u / semi
    normal = normal / normal.norm(dim=1, keepdim=True)
    pos = pos + normal * (0.005 * torch.randn(n, 1, generator=g))
    pos[:, 2] += 4.24
    s = torch.exp(math.log(0.004) + 0.4 * torch.randn(n, 1, generator=g))
    if tiny_scale:  # warm-up clamp of model.py:90-97
        s = s.clamp(max=1e-3)
    scale = s.repeat(1, 3)
    rot = torch.tensor([[1.0, 0.0, 0.0, 0.0]]).repeat(n, 1)
    opacity = torch.ones(n, 1)
    rgb = torch.rand(n, 3, generator=g)
    return pos, scale, rot, opacity, rgb


def _scene(n, g, tan_half_x, tan_half_y):
    z = 2.0 + 10.0 * torch.rand(n, generator=g)
    x = (2 * torch.rand(n, generator=g) - 1) * 1.2 * tan_half_x * z
    y = (2 * torch.rand(n, generator=g) - 1) * 1.2 * tan_half_y * z
    pos = torch.stack([x, y, z], 1)
    scale = torch.exp(math.log(0.02) + 0.7 * torch.randn(n, 3, generator=g))
    q = torch.randn(n, 4, generator=g)
    rot = q / q.norm(dim=1, keepdim=True)
    opacity = torch.sigmoid(2.0 * torch.randn(n, 1, generator=g))
    rgb = torch.rand(n, 3, generator=g)
    return pos, scale, rot, opacity, rgb


def make_assets(workload, seed=0, device="cpu", focal_ratio=1.465, tiny_scale=False):
    """Returns the dict `GaussianRenderer.forward` consumes (module.py:594-598) plus `shs` when sh_degree > 0."""
    wl = WORKLOADS[workload] if isinstance(workload, str) else workload
    g = torch.Generator().manual_seed(seed)
    tan_x = wl.width / (2 * focal_ratio * wl.height)
    tan_y = 1.0 / (2 * focal_ratio)
    parts = []
    if wl.n_avatar:
        parts.append(_avatar(wl.n_avatar, g, tiny_scale))
    if wl.n_scene:
        parts.append(_scene(wl.n_scene, g, tan_x, tan_y))
    pos, scale, rot, opacity, rgb = (torch.cat([p[i] for p in parts]) for i in range(5))
    # interleave the populations so depth order is not the input order
    perm = torch.randperm(pos.shape[0], generator=g)
    assets = {
        "mean_3d": pos[perm].contiguous(), "scale": scale[perm].contiguous(), "rotation": rot[perm].contiguous(),
        "opacity": opacity[perm].contiguous(), "rgb": rgb[perm].contiguous(),
    }
    if wl.sh_degree > 0:
        m = (wl.sh_degree + 1) ** 2
        shs = 0.3 * torch.randn(pos.shape[0], m, 3, generator=g)
        shs[:, 0, :] = (assets["rgb"] - 0.5) / SH_C0  # RGB2SH, transforms.py:169-170
        assets["shs"] = shs.contiguous()
    return {k: v.to(device) for k, v in assets.items()}


def make_grad_image(workload, seed=0, device="cpu"):
    """Upstream gradient dL/dcolor ~ N(0,1), fixed per seed (SURVEY section 8d)."""
    wl = WORKLOADS[workload] if isinstance(workload, str) else workload
    g = torch.Generator().manual_seed(1000 + seed)
    return torch.randn(3, wl.height, wl.width, generator=g).to(device)


def make_population_assets(workload, seed=0, device="cpu", focal_ratio=1.465):
    """The two populations of a workload as separate asset dicts, for ExAvatar's five-render training frame
    (avatar/main/model.py:81-162): `scene` (SceneGaussian), `human` (HumanGaussian) and `human_refined` (the same
    anchors with the pose-dependent mean / scale / colour offsets applied, module.py:531-534,561-562)."""
    wl = WORKLOADS[workload] if isinstance(workload, str) else workload
    g = torch.Generator().manual_seed(seed)
    tan_x = wl.width / (2 * focal_ratio * wl.height)
    tan_y = 1.0 / (2 * focal_ratio)
    keys = ("mean_3d", "scale", "rotation", "opacity", "rgb")
    human = dict(zip(keys, (t.contiguous() for t in _avatar(wl.n_avatar, g))))
    scene = dict(zip(keys, (t.contiguous() for t in _scene(wl.n_scene, g, tan_x, tan_y))))
    refined = {k: v.clone() for k, v in human.items()}
    refined["mean_3d"] = human["mean_3d"] + 0.002 * torch.randn(wl.n_avatar, 3, generator=g)
    refined["scale"] = human["scale"] * torch.exp(0.1 * torch.randn(wl.n_avatar, 1, generator=g))
    refined["rgb"] = (human["rgb"] + 0.05 * torch.randn(wl.n_avatar, 3, generator=g)).clamp(0, 1)
    to = lambda d: {k: v.to(device) for k, v in d.items()}
    return to(scene), to(human), to(refined)


def make_scene_sh_params(workload, seed=0, device="cpu", focal_ratio=1.465):
    """The scene population of `make_population_assets(workload, seed)` as SceneGaussian stores it (module.py:103-108):
    mean, opacity_logit, log_scale, rotation (activated), feature_dc (P,1,3) and feature_rest (P,15,3) -- degree-3
    SH as `max_sh_degree = 3` trains it (config.py:15-16).  feature_dc is RGB2SH of the population's rgb
    (transforms.py:169-170); feature_rest is drawn from a generator of its own, so the other generators' outputs do not
    change.  Feed them to `renderer.scene_gaussian_assets`."""
    scene, _, _ = make_population_assets(workload, seed=seed, focal_ratio=focal_ratio)
    n = scene["mean_3d"].shape[0]
    g = torch.Generator().manual_seed(3000 + seed)
    p = {
        "mean": scene["mean_3d"],
        "opacity_logit": torch.logit(scene["opacity"].clamp(1e-4, 1 - 1e-4)),
        "log_scale": torch.log(scene["scale"]),
        "rotation": scene["rotation"],
        "feature_dc": ((scene["rgb"] - 0.5) / SH_C0)[:, None, :],
        "feature_rest": 0.2 * torch.randn(n, 15, 3, generator=g),
    }
    return {k: v.contiguous().to(device) for k, v in p.items()}
