"""`TrainingFrameRenderer`: ExAvatar's five renders of a training frame as ONE autograd call (SURVEY.md section 8f-3).

`Model.forward` renders every frame five times with the same camera (avatar/main/model.py:117-162):

    scene_render                = gaussian_renderer(scene_asset, ...)
    human_render                = gaussian_renderer(human_asset, ..., bg)
    scene_human_render          = gaussian_renderer(cat(scene_asset.detach(), human_asset), ...)
    human_render_refined        = gaussian_renderer(human_asset_refined, ..., bg)
    scene_human_render_refined  = gaussian_renderer(cat(scene_asset.detach(), human_asset_refined), ...)

Through the drop-in `GaussianRasterizer` those are five full projection / binning / sort / composite pipelines.  This
module renders the same five images from TWO projection + binning passes (`plan.MergedFivePlan`: views of
cat(scene, human) and cat(scene, human_refined), human-free tiles of the human-only and combined views skipped) and
back-propagates into the three asset dicts exactly what `loss.backward()` leaves there: the scene render's gradient in the
scene assets, human-only + combined render in the human assets (the scene part of the combined renders is detached, as in
the reference), likewise for the refined set.  INTEGRATION.md shows the replacement of model.py:117-162.

    frame = TrainingFrameRenderer(P_scene, P_human, (H, W), device, dup_capacity)
    out = frame(scene_asset, human_asset, human_asset_refined, cam_param, bg_human)
    out["scene"]["img"], out["human"]["mask"], out["scene_human"]["img"], ...      # same keys as GaussianRenderer
    out["scene"]["mean_2d"].grad                                                   # after backward (train.py:51)

The duplicate capacity is fixed per instance (every buffer is resident; nothing is polled or synchronised, so the call
is capturable in a CUDA graph); `overflowed()` reports if a frame needed more (its lists were truncated, never corrupt).
One frame may be in flight per instance: run backward (or drop the outputs) before the next call.

`use_graph=True`: the first frame captures the forward and the backward of the plan into two CUDA graphs; later frames
copy their inputs into the plan's resident buffers (assets, camera, dL/dimage) and replay.  The Python cost of a frame
drops from ~2.9 ms (hundreds of stream switches, ctypes calls and small copies) to a few copies and two graph launches,
so an otherwise EAGER training loop runs the raster part at graph speed.  Kernel arguments passed by value are frozen in
the graphs, so a change of the intrinsics (tan fov) re-captures; every render's backward runs (a render left out of the
loss contributes zeros).

`scene_sh_coeffs=M > 0`: the scene asset dict carries `shs` (P_scene, M, 3) + `sh_degree` in place of `rgb` -- what
`renderer.scene_gaussian_assets(in_kernel_sh=True)` returns -- and the projection kernel colours the scene Gaussians from
it (SURVEY.md section 8f-4), in both merged passes.  The gradient reaches `shs` (and through it feature_dc /
feature_rest) and the scene `mean_3d` gets the view-direction term, as with `GaussianRenderer`.  As there, `shs` is used
iff `rgb` is absent; a scene whose colour source or M does not match the instance raises a ValueError.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
from torch import nn

from .plan import RENDERS, MergedFivePlan
from .rasterizer import GaussianRasterizationSettings, _f32c
from .renderer import render_settings

_KEYS = ("mean_3d", "opacity", "scale", "rotation", "rgb")
_SH_KEYS = ("mean_3d", "opacity", "scale", "rotation", "shs")  # a scene coloured in the kernel
_GRAD_OF = {"mean_3d": "means3D", "opacity": "opacities", "scale": "scales", "rotation": "rotations", "rgb": "colors",
            "shs": "shs"}


def scene_sh_degree(scene_asset, M: int) -> Optional[int]:
    """The SH degree of a scene asset dict for a frame renderer built with scene_sh_coeffs = M, or None for an rgb scene.
    `shs` is used iff `rgb` is absent (GaussianRenderer's rule); a colour source or coefficient count the instance was
    not built for raises a ValueError."""
    sh_scene = "rgb" not in scene_asset
    if sh_scene != (M > 0):
        raise ValueError(f"TrainingFrameRenderer(scene_sh_coeffs={M}): the scene asset dict carries "
                         f"{'no rgb' if sh_scene else 'rgb'}; this instance needs {'shs + sh_degree' if M else 'rgb'}")
    if not sh_scene:
        return None
    shs = scene_asset.get("shs")
    if shs is None or "sh_degree" not in scene_asset or shs.dim() != 3 or tuple(shs.shape[1:]) != (M, 3):
        raise ValueError(f"TrainingFrameRenderer(scene_sh_coeffs={M}): the scene needs shs of shape (P, {M}, 3) and "
                         f"sh_degree, got shs {None if shs is None else tuple(shs.shape)}")
    deg = int(scene_asset["sh_degree"])
    if not 0 <= deg <= 3 or (deg + 1) ** 2 > M:
        raise ValueError(f"TrainingFrameRenderer(scene_sh_coeffs={M}): sh_degree {deg} is not in [0, 3] or needs more "
                         f"than {M} coefficients")
    return deg


class _FrameFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, settings, settings_h, scene_m2d, *tensors):
        plan: MergedFivePlan = mod.plan
        keys = (mod._scene_keys, _KEYS, _KEYS)
        scene, human, refined = (dict(zip(keys[i], (_f32c(t.detach(), k) for k, t in zip(keys[i], tensors[i * 5:i * 5 + 5]))))
                                 for i in range(3))
        mod._frame_no += 1
        if mod.use_graph:
            mod._graph_forward(settings, settings_h, scene, human, refined)
        else:
            plan.set_scene(scene)
            plan.forward_frame(None, settings, settings_h, scene, human, refined)  # no descriptor cache: cameras change
        outs = []
        for r in RENDERS:  # fresh tensors: the plan's image buffers are overwritten by the next frame
            pk = "A" if r in plan.VIEWS["A"] else "B"
            color, depth, alpha = plan.passes[pk].img[plan.VIEWS[pk].index(r)]
            outs += [color.clone(), depth.clone(), alpha.clone()]
        radii_a, radii_b = plan.passes["A"].radii.clone(), plan.passes["B"].radii.clone()
        ctx.mod = mod
        ctx.shapes = [t.shape for t in tensors]
        ctx.m2d_shape = scene_m2d.shape
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(radii_a, radii_b)
        return (*outs, radii_a, radii_b)

    @staticmethod
    def backward(ctx, *grads):
        mod = ctx.mod
        plan: MergedFivePlan = mod.plan
        g = grads[:15]
        gc = {r: (None if g[3 * i] is None else _f32c(g[3 * i], "grad_color")) for i, r in enumerate(RENDERS)}
        gd = {r: (None if g[3 * i + 1] is None else _f32c(g[3 * i + 1], "grad_depth")) for i, r in enumerate(RENDERS)}
        ga = {r: (None if g[3 * i + 2] is None else _f32c(g[3 * i + 2], "grad_alpha")) for i, r in enumerate(RENDERS)}
        dev = plan.device
        if mod.use_graph:
            flat_a, flat_b = mod._graph_backward(gc, gd, ga)  # fresh copies of the resident gradient buffers
        else:
            flat_a = torch.empty(plan.nA, dtype=torch.float32, device=dev)
            flat_b = torch.empty(plan.nB, dtype=torch.float32, device=dev)
        va, vb = plan.grad_views(flat_a, flat_b)
        if not mod.use_graph:
            plan.backward_frame(gc, va, vb, g_depths=gd, g_alphas=ga, densify=mod.densify)
        Ps = plan.Ps
        out = [None, None, None, va["means2D"][:Ps].reshape(ctx.m2d_shape)]
        for keys, part in ((mod._scene_keys, lambda v: v[:Ps]), (_KEYS, lambda v: v[Ps:])):
            for k in keys:
                out.append(part(va[_GRAD_OF[k]]))
        for k in _KEYS:
            out.append(vb[_GRAD_OF[k]])
        for i, shp in enumerate(ctx.shapes):
            out[4 + i] = out[4 + i].reshape(shp)
        return tuple(out)


class TrainingFrameRenderer(nn.Module):
    def __init__(self, P_scene: int, P_human: int, img_shape, device, dup_capacity: Optional[Dict[str, int]] = None,
                 use_graph: bool = False, graph_depth_alpha: bool = False, scene_sh_coeffs: int = 0):
        super().__init__()
        self.img_shape = (int(img_shape[0]), int(img_shape[1]))
        self.plan = MergedFivePlan(P_scene, P_human, self.img_shape[1], self.img_shape[0], dup_capacity, device,
                                   scene_sh_coeffs=scene_sh_coeffs)
        self._scene_keys = _SH_KEYS if self.plan.M else _KEYS
        self.densify = None  # optional {'grad_accum','count','radius_max'} (P_scene) tensors updated by the backward
        self._frame_no = 0
        self.use_graph = bool(use_graph)
        if self.use_graph:
            dev, (H, W), plan = self.plan.device, self.img_shape, self.plan
            # resident camera / background block the captured kernels read: view (16) | full projection (16) | campos (3) |
            # bg (3) | bg of the human-only renders (3)
            self._cam = torch.zeros(41, dtype=torch.float32, device=dev)
            self._gin = {r: torch.zeros(3, H, W, dtype=torch.float32, device=dev) for r in RENDERS}
            # dL/ddepth and dL/dalpha inputs only when asked for: their backward variant is the slower one
            self._gin_d = {r: torch.zeros(1, H, W, dtype=torch.float32, device=dev) for r in RENDERS} if graph_depth_alpha else None
            self._gin_a = {r: torch.zeros(1, H, W, dtype=torch.float32, device=dev) for r in RENDERS} if graph_depth_alpha else None
            self._flat_a = torch.zeros(plan.nA, dtype=torch.float32, device=dev)
            self._flat_b = torch.zeros(plan.nB, dtype=torch.float32, device=dev)
            # (tanfovx, tanfovy, scale modifier, densify buffers, SH degree) -> (settings, settings_h, forward graph,
            # backward graph); the SH degree is a by-value kernel argument that grows during training
            self._graphs = {}
            self._cur = None

    # ---- use_graph=True ----
    def _resident_settings(self, settings, settings_h):
        c = self._cam
        mk = lambda bg: GaussianRasterizationSettings(
            image_height=settings.image_height, image_width=settings.image_width, tanfovx=settings.tanfovx,
            tanfovy=settings.tanfovy, bg=bg, scale_modifier=settings.scale_modifier, viewmatrix=c[0:16].view(4, 4),
            projmatrix=c[16:32].view(4, 4), sh_degree=settings.sh_degree, campos=c[32:35], prefiltered=False, debug=False)
        return mk(c[35:38]), mk(c[38:41])

    def _load_inputs(self, settings, settings_h, scene, human, refined):
        plan, c = self.plan, self._cam
        c[0:16].copy_(settings.viewmatrix.reshape(16))
        c[16:32].copy_(settings.projmatrix.reshape(16))
        c[32:35].copy_(settings.campos.reshape(3))
        c[35:38].copy_(settings.bg.reshape(3))
        c[38:41].copy_(settings_h.bg.reshape(3))
        pa, pb = plan.passes["A"], plan.passes["B"]
        for k in _KEYS:
            if not (plan.M and k == "rgb"):
                pa.cat[k][: plan.Ps].copy_(scene[k].reshape(plan.Ps, -1))
            pa.cat[k][plan.Ps:].copy_(human[k].reshape(plan.Ph, -1))
            pb.cat[k][plan.Ps:].copy_(refined[k].reshape(plan.Ph, -1))
        if plan.M:
            plan.shs.copy_(scene["shs"].reshape(plan.Ps, plan.M, 3))

    def _graph_forward(self, settings, settings_h, scene, human, refined):
        plan = self.plan
        self._load_inputs(settings, settings_h, scene, human, refined)
        dn = self.densify or {}
        key = (float(settings.tanfovx), float(settings.tanfovy), float(settings.scale_modifier),
               tuple(0 if dn.get(k) is None else dn[k].data_ptr() for k in ("grad_accum", "count", "radius_max")))
        if plan.M:
            key += (int(settings.sh_degree),)
        if key not in self._graphs:
            st, st_h = self._resident_settings(settings, settings_h)
            pa, pb = plan.passes["A"], plan.passes["B"]
            va, vb = plan.grad_views(self._flat_a, self._flat_b)

            def fwd():
                for k in _KEYS:  # the scene rows of pass B come from pass A's copy (SH: both read plan.shs)
                    if not (plan.M and k == "rgb"):
                        pb.cat[k][: plan.Ps].copy_(pa.cat[k][: plan.Ps])
                plan.forward_frame(("graph", key), st, st_h, None, None, None, copy_inputs=False)

            def bwd():
                plan.backward_frame(self._gin, va, vb, g_depths=self._gin_d, g_alphas=self._gin_a, densify=self.densify)

            cur = torch.cuda.current_stream(plan.device)
            side = torch.cuda.Stream(plan.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):  # warm-up (also primes the ctx counters), then capture
                fwd()
                bwd()
            cur.wait_stream(side)
            torch.cuda.synchronize(plan.device)
            gf, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(gf):
                fwd()
            with torch.cuda.graph(gb, pool=gf.pool()):
                bwd()
            self._graphs[key] = (st, st_h, gf, gb)
        self._cur = self._graphs[key]
        self._cur[2].replay()

    def _graph_backward(self, gc, gd, ga):
        for dst, src in ((self._gin, gc), (self._gin_d, gd), (self._gin_a, ga)):
            if dst is None:
                if any(v is not None for v in src.values()):
                    raise RuntimeError("TrainingFrameRenderer(use_graph=True): gradients of depthmap / mask need "
                                       "graph_depth_alpha=True")
                continue
            for r in RENDERS:
                if src[r] is None:
                    dst[r].zero_()
                else:
                    dst[r].copy_(src[r].reshape(dst[r].shape))
        self._cur[3].replay()
        return self._flat_a.clone(), self._flat_b.clone()

    def overflowed(self) -> bool:
        return self.plan.overflowed()

    def forward(self, scene_asset, human_asset, human_asset_refined, cam_param, bg_human, bg=None, raster_settings=None,
                raster_settings_human=None):
        """Asset dicts as `GaussianRenderer.forward` takes them (mean_3d, opacity, scale, rotation, rgb -- or, for the scene
        of an instance built with scene_sh_coeffs > 0, shs + sh_degree in place of rgb); `bg_human` is the
        background of the two human-only renders (model.py:72), `bg` of the others (white by default, module.py:592).
        Returns {render name: {img, depthmap, mask, radius, is_vis[, mean_2d]}} for the five renders of plan.RENDERS."""
        dev = scene_asset["mean_3d"].device
        deg = scene_sh_degree(scene_asset, self.plan.M)  # raises before anything is enqueued
        if bg is None:
            bg = torch.ones(3, dtype=torch.float32, device=dev)
        st = raster_settings or render_settings(self.img_shape, cam_param, bg, GaussianRasterizationSettings)
        if deg is not None:
            st = st._replace(sh_degree=deg)
        st_h = raster_settings_human or st._replace(bg=bg_human)
        Ps = scene_asset["mean_3d"].shape[0]
        mean_2d = torch.zeros((Ps, 3), dtype=torch.float32, device=dev, requires_grad=True)  # module.py:626-629
        flat = [a[k] for a, keys in ((scene_asset, self._scene_keys), (human_asset, _KEYS), (human_asset_refined, _KEYS))
                for k in keys]
        res = _FrameFn.apply(self, st, st_h, mean_2d, *flat)
        radii_a, radii_b = res[15], res[16]
        radius = {"scene": radii_a[:Ps], "human": radii_a[Ps:], "scene_human": radii_a, "human_refined": radii_b[Ps:],
                  "scene_human_refined": radii_b}
        out = {}
        for i, r in enumerate(RENDERS):
            out[r] = {"img": res[3 * i], "depthmap": res[3 * i + 1], "mask": res[3 * i + 2], "radius": radius[r],
                      "is_vis": radius[r] > 0}
        out["scene"]["mean_2d"] = mean_2d
        return out
