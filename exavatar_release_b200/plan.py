"""`FramePlan`: allocation-free, sync-free, CUDA-graph-capturable use of the C ABI.

The autograd front-end (`rasterizer.py`) must size buffers per call because it cannot know the caller's next scene.
A training loop that renders the same Gaussian set frame after frame (ExAvatar: avatar/main/train.py:24-57) can do
better: fix the duplicate capacity once, keep every buffer resident, and enqueue forward + backward with no host
round-trip at all -- which also makes the whole step capturable in a CUDA graph (`torch.cuda.graph`), so a step of F
frames costs one graph launch instead of ~9 F kernel launches.  Overflow of the fixed capacity is detected from the
device status block (`status()`), checked by the caller outside the hot loop.

Gradients are written (or, with `accumulate=True`, summed) into caller-provided tensors, e.g. views of the flat
bucket that is all-reduced once per step (SURVEY.md section 8e).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch

from . import _lib as L
from .rasterizer import _f32c, _make_scene, _ptr


class _Workspace:
    """The resident workspace of one projection + binning of P Gaussians with a fixed duplicate capacity: ctx block,
    duplicate ids, scratch, backward scratch, `n_ckpts` checkpoint buffers and the B2RWorkspace over them."""

    def __init__(self, lib, P: int, width: int, height: int, dup_capacity: int, device, n_ckpts: int = 1):
        self.capacity = int(dup_capacity)
        self.ctx_bytes = lib.b2r_ctx_bytes(P, width, height)
        self.ctx_buf = torch.empty(self.ctx_bytes, dtype=torch.uint8, device=device)
        self.ids = torch.empty(max(self.capacity, 1), dtype=torch.int32, device=device)
        self.scratch_bytes = lib.b2r_scratch_bytes(P, width, height, self.capacity)
        self.scratch = torch.empty(self.scratch_bytes, dtype=torch.uint8, device=device)
        self.bwd_bytes = lib.b2r_backward_scratch_bytes(P)
        # zero once: every backward leaves it zero again (B2R_BWD_SCRATCH_ZEROED), so no memset node per render
        self.bwd_scratch = torch.zeros(self.bwd_bytes, dtype=torch.uint8, device=device)
        # segment table + blend-state checkpoints of a forward composite (lets the backward replay 512-entry list
        # segments as independent work items); one buffer per view composited from the same lists
        self.ckpt_bytes = lib.b2r_checkpoint_bytes(width, height, self.capacity)
        self.ckpts = [torch.empty(self.ckpt_bytes, dtype=torch.uint8, device=device) for _ in range(n_ckpts)]
        self.ws = L.B2RWorkspace(self.ctx_buf.data_ptr(), self.ctx_bytes, self.ids.data_ptr(), self.capacity,
                                 self.scratch.data_ptr(), self.scratch_bytes, None, 0, self.ckpts[0].data_ptr(),
                                 self.ckpt_bytes)

    def status(self) -> dict:
        return L.read_status(self.ctx_buf)


class FramePlan(_Workspace):
    def __init__(self, P: int, width: int, height: int, dup_capacity: int, device, sh_coeffs: int = 0):
        self.lib = L.load()
        self.P, self.W, self.H, self.M = int(P), int(width), int(height), int(sh_coeffs)
        self.device = torch.device(device)
        dev = self.device
        f = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        self.color, self.depth, self.alpha = f(3, height, width), f(1, height, width), f(1, height, width)
        self.radii = torch.empty(P, dtype=torch.int32, device=dev)
        super().__init__(self.lib, self.P, self.W, self.H, dup_capacity, dev)
        self.out = L.B2RForwardOutputs(self.color.data_ptr(), self.depth.data_ptr(), self.alpha.data_ptr(),
                                       self.radii.data_ptr())
        self._scenes = {}
        self._primed = False

    def scene(self, key, settings, assets: Dict[str, torch.Tensor], flags: int = 0):
        """Builds (and caches under `key`) the B2RScene for one frame; tensors must stay alive and in place."""
        if key in self._scenes:
            return self._scenes[key][0]
        g = lambda k: None if assets.get(k) is None else _f32c(assets[k], k)
        shs = g("shs") if self.M > 0 else None
        sc, keep = _make_scene(settings, g("mean_3d"), shs, None if shs is not None else g("rgb"), g("opacity"),
                               g("scale"), g("rotation"), None, flags)
        self._scenes[key] = (sc, keep)
        return sc

    def forward(self, sc) -> None:
        # from the second forward on the ctx counters are known to be zero (every forward leaves them so): no reset launch
        base = sc.flags & ~L.B2R_FLAG_CTX_CLEAN
        sc.flags = base | (L.B2R_FLAG_CTX_CLEAN if self._primed else 0)
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            L.check(self.lib.b2r_forward(C.byref(sc), C.byref(self.ws), C.byref(self.out), st), "b2r_forward")
        sc.flags = base
        self._primed = True

    def backward(self, sc, g_color: torch.Tensor, grads: Dict[str, Optional[torch.Tensor]], accumulate: bool = False,
                 g_depth: Optional[torch.Tensor] = None, g_alpha: Optional[torch.Tensor] = None,
                 densify: Optional[Dict[str, torch.Tensor]] = None, first_row: int = 0) -> None:
        """grads keys: means3D, means2D, shs, colors, opacities, scales, rotations, cov3D (missing -> not written).
        densify (optional): {'grad_accum', 'count', 'radius_max'} fp32 (P) tensors updated in place by the backward
        projection kernel -- ExAvatar's `track_stats` + `radius_max` update (module.py:155-157, model.py:283-285).
        first_row: Gaussians [0, first_row) are a detached prefix (cat(scene.detach(), human), model.py:117-125): the
        `grads` tensors then have P - first_row rows and receive the gradient of the remaining Gaussians only."""
        a = L.B2RBackwardArgs(_ptr(g_color), _ptr(g_depth), _ptr(g_alpha), _ptr(grads.get("means3D")),
                              _ptr(grads.get("means2D")), _ptr(grads.get("shs")), _ptr(grads.get("colors")),
                              _ptr(grads.get("opacities")), _ptr(grads.get("scales")), _ptr(grads.get("rotations")),
                              _ptr(grads.get("cov3D")), (L.B2R_BWD_ACCUMULATE if accumulate else 0) | L.B2R_BWD_SCRATCH_ZEROED, int(first_row),
                              _ptr((densify or {}).get("grad_accum")), _ptr((densify or {}).get("count")),
                              _ptr((densify or {}).get("radius_max")))
        with torch.cuda.device(self.device):
            st = torch.cuda.current_stream(self.device).cuda_stream
            L.check(self.lib.b2r_backward(C.byref(sc), C.byref(self.ws), C.byref(a), self.bwd_scratch.data_ptr(),
                                          self.bwd_bytes, st), "b2r_backward")


def grad_bucket(P: int, device, sh_coeffs: int = 0):
    """One flat fp32 buffer holding every per-Gaussian gradient, plus named views into it."""
    per = 3 + 3 + 1 + 3 + 4 + (3 * sh_coeffs if sh_coeffs > 0 else 3)
    return _views_of(torch.zeros(per * P, dtype=torch.float32, device=device), P, sh_coeffs)


class FrameLanes:
    """S concurrent `FramePlan`s ("lanes"), each on its own CUDA stream with its own workspace and gradient bucket.

    Frames of a training batch are independent (SURVEY.md section 8e; avatar/main/model.py:81 loops over them), and at
    ExAvatar's sizes a single frame cannot fill a B200: the scan / sort kernels are latency-bound single-wave launches
    and the composites end in a tail of long tile lists.  Running frame f on lane f mod S lets the hardware fill those
    holes with another frame's kernels.  The lanes fork from and join back into the caller's current stream, so the
    whole step is still one CUDA-graph capture.  Gradients of the frames of one lane are summed inside the backward
    projection kernel (`accumulate`); the S lane buckets are then added in a fixed order (deterministic result) into
    `bucket`, the tensor that is all-reduced once per step.
    """

    def __init__(self, lanes: int, P: int, width: int, height: int, dup_capacity: int, device, sh_coeffs: int = 0):
        self.S = max(1, int(lanes))
        self.device = torch.device(device)
        self.plans = [FramePlan(P, width, height, dup_capacity, device, sh_coeffs) for _ in range(self.S)]
        self.streams = [torch.cuda.Stream(self.device) for _ in range(self.S)]
        flat0, _ = grad_bucket(P, device, sh_coeffs)
        self.lane_flat = torch.zeros(self.S, flat0.numel(), dtype=torch.float32, device=device)
        self.lane_views = []
        for s in range(self.S):
            _, v = _views_of(self.lane_flat[s], P, sh_coeffs)
            self.lane_views.append(v)
        self.bucket = self.lane_flat[0] if self.S == 1 else flat0
        _, self.views = _views_of(self.bucket, P, sh_coeffs)

    def scene(self, key, settings, assets, flags: int = 0):
        return self.plans[0].scene(key, settings, assets, flags)

    def step(self, scenes, g_colors, backward: bool = True) -> None:
        """Forward (+ backward) of every frame in `scenes`; on return (stream order) `bucket` holds the summed gradients."""
        cur = torch.cuda.current_stream(self.device)
        F = len(scenes)
        for s in range(self.S):
            st = self.streams[s]
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                plan = self.plans[s]
                for j, f in enumerate(range(s, F, self.S)):
                    plan.forward(scenes[f])
                    if backward:
                        plan.backward(scenes[f], g_colors[f], self.lane_views[s], accumulate=(j > 0))
        for st in self.streams:
            cur.wait_stream(st)
        if backward and self.S > 1:
            torch.sum(self.lane_flat[: min(self.S, F)], dim=0, out=self.bucket)

    def status(self) -> dict:
        sts = [p.status() for p in self.plans]
        out = dict(sts[0])
        out["overflow"] = int(any(s["overflow"] for s in sts))
        return out


def _views_of(flat: torch.Tensor, P: int, sh_coeffs: int = 0):
    widths = [("means3D", 3), ("means2D", 3), ("opacities", 1), ("scales", 3), ("rotations", 4)]
    widths.append(("shs", 3 * sh_coeffs) if sh_coeffs > 0 else ("colors", 3))
    views, o = {}, 0
    for name, w in widths:
        views[name] = flat[o:o + w * P].view(P, w) if name != "shs" else flat[o:o + w * P].view(P, sh_coeffs, 3)
        o += w * P
    return flat, views


RENDERS = ("scene", "human", "scene_human", "human_refined", "scene_human_refined")


class FiveRenderPlan:
    """One ExAvatar training frame = five rasteriser calls with one camera (avatar/main/model.py:81-162):

        scene                      -> gradients to the scene Gaussians
        human            (bg rand) -> gradients to the human Gaussians
        cat(scene.detach(), human) -> gradients to the human Gaussians only        (model.py:117-125)
        human_refined    (bg rand) -> gradients to the refined human Gaussians
        cat(scene.detach(), human_refined) -> gradients to the refined human Gaussians only

    The reference runs them one after the other, each with its own device->host sync.  Here the five renders are
    independent until their gradients meet, so each runs on its own CUDA stream (fork / join inside the caller's
    stream: capturable in one CUDA graph with the rest of the step); the "detached prefix" of the combined renders is a
    field of the backward call (`first_row`), so the human part of their gradient is written straight into a
    human-sized bucket and nothing is computed-then-discarded on the host side.  Frames of a step accumulate into the
    same five buckets; `reduce()` folds them into the three parameter sets (scene, human, human_refined).

    All gradients live in ONE flat fp32 buffer (`flat_bucket()`: scene | human | human_refined after `reduce()`), the
    tensor a multi-GPU step all-reduces once (SURVEY.md section 8e).  `MergedFivePlan` below produces the same results
    from two projection / binning passes instead of five (SURVEY.md section 8f-3).
    """
    PER = 3 + 3 + 1 + 3 + 4 + 3  # floats per Gaussian in a bucket

    def __init__(self, P_scene: int, P_human: int, width: int, height: int, caps: Optional[Dict[str, int]], device):
        self.Ps, self.Ph = int(P_scene), int(P_human)
        self.device = torch.device(device)
        caps = caps or {r: 8_000_000 for r in RENDERS}
        sizes = {"scene": self.Ps, "human": self.Ph, "scene_human": self.Ps + self.Ph, "human_refined": self.Ph,
                 "scene_human_refined": self.Ps + self.Ph}
        self.plans = {r: FramePlan(sizes[r], width, height, caps[r], device) for r in RENDERS}
        self.streams = {r: torch.cuda.Stream(self.device) for r in RENDERS}
        self.first_row = {"scene": 0, "human": 0, "scene_human": self.Ps, "human_refined": 0, "scene_human_refined": self.Ps}
        out_rows = {"scene": self.Ps, "human": self.Ph, "scene_human": self.Ph, "human_refined": self.Ph,
                    "scene_human_refined": self.Ph}
        # one allocation: [scene | human | human_refined | scene_human | scene_human_refined]; the first three segments
        # are what reduce() leaves the step's gradients in
        order = ("scene", "human", "human_refined", "scene_human", "scene_human_refined")
        tail = 2 * self.Ps  # per-step densification sums of the scene Gaussians ride in the all-reduced buffer (stats())
        self.all_flat = torch.zeros(self.PER * sum(out_rows[r] for r in order) + tail, dtype=torch.float32, device=device)
        self.flat, self.views, o = {}, {}, 0
        for r in order:
            n = self.PER * out_rows[r]
            self.flat[r], self.views[r] = _views_of(self.all_flat[o:o + n], out_rows[r])
            o += n
            if r == "human_refined":
                self._stats = self.all_flat[o:o + tail]
                o += tail
        self._reduced = self.PER * (self.Ps + 2 * self.Ph) + tail
        f = lambda w: torch.empty(self.Ps + self.Ph, w, dtype=torch.float32, device=device)
        widths = {"mean_3d": 3, "opacity": 1, "scale": 3, "rotation": 4, "rgb": 3}
        self.cat = {r: {k: f(w) for k, w in widths.items()} for r in ("scene_human", "scene_human_refined")}

    def describe(self) -> str:
        return "five independent renders (project+bin+sort+composite each) on five CUDA streams per frame"

    def set_scene(self, scene_assets: Dict[str, torch.Tensor]) -> None:
        """Copies the (detached) scene Gaussians into the prefix of the two combined asset sets; once per step."""
        for r in self.cat:
            for k, buf in self.cat[r].items():
                buf[: self.Ps].copy_(scene_assets[k].reshape(self.Ps, -1))

    def assets_of(self, render: str, scene, human, refined):
        if render == "scene":
            return scene
        if render in ("human", "human_refined"):
            return human if render == "human" else refined
        src = human if render == "scene_human" else refined
        for k, buf in self.cat[render].items():
            buf[self.Ps:].copy_(src[k].reshape(self.Ph, -1))
        return self.cat[render]

    def frame(self, key, settings, settings_human_bg, scene, human, refined, g_colors: Dict[str, torch.Tensor],
              accumulate: bool, densify: Optional[Dict[str, torch.Tensor]] = None, serial: bool = False) -> None:
        """Forward + backward of the five renders of one frame.  `settings_human_bg` carries the random background of
        the human-only renders (model.py:72).  `key` caches the per-(frame, render) scene descriptors.  `densify`:
        ExAvatar's densification statistics of the SCENE Gaussians, fed by the scene render (model.py:193, 279-285).
        `serial`: all five on the caller's stream, one after the other (per-kernel profiling)."""
        cur = torch.cuda.current_stream(self.device)
        for r in RENDERS:
            st = cur if serial else self.streams[r]
            if not serial:
                st.wait_stream(cur)
            with torch.cuda.stream(st):
                plan = self.plans[r]
                assets = self.assets_of(r, scene, human, refined)
                sc = plan.scene((key, r), settings_human_bg if r in ("human", "human_refined") else settings, assets)
                plan.forward(sc)
                plan.backward(sc, g_colors[r], self.views[r], accumulate=accumulate, first_row=self.first_row[r],
                              densify=densify if r == "scene" else None)
        if not serial:
            for r in RENDERS:
                cur.wait_stream(self.streams[r])

    def render_outputs(self, render: str):
        """(color (3,H,W), alpha (1,H,W), radii) of one of the five renders of the last frame (valid until the next)."""
        p = self.plans[render]
        return p.color, p.alpha, p.radii

    def reduce(self):
        """(scene, human, human_refined) flat gradient buckets of the step (the first three segments of the flat bucket;
        the combined renders' human rows are folded in, in a fixed order)."""
        self.flat["human"].add_(self.flat["scene_human"])
        self.flat["human_refined"].add_(self.flat["scene_human_refined"])
        return self.flat["scene"], self.flat["human"], self.flat["human_refined"]

    def grads(self, which: str) -> Dict[str, torch.Tensor]:
        """Named gradient tensors of one parameter set ("scene" | "human" | "human_refined"), valid after reduce()."""
        return dict(self.views[which])

    def flat_bucket(self) -> torch.Tensor:
        return self.all_flat[: self._reduced]

    def stats(self) -> Dict[str, torch.Tensor]:
        """Per-step sums of ExAvatar's densification statistics (module.py:155-157), stored at the tail of the flat
        bucket so the step's ONE sum all-reduce covers them; zero them at the start of a step (`zero_stats`)."""
        return {"grad_accum": self._stats[: self.Ps], "count": self._stats[self.Ps:]}

    def zero_stats(self) -> None:
        self._stats.zero_()

    def dups(self) -> Dict[str, int]:
        return {r: p.status()["num_dups"] for r, p in self.plans.items()}

    def consumed(self) -> Dict[str, list]:
        st = [self.plans[r].status() for r in RENDERS]
        return {"fwd": [s["consumed_fwd"] / s["consumed_fwd_div"] for s in st],
                "bwd": [s["consumed_bwd"] / s["consumed_bwd_div"] for s in st]}

    def overflowed(self) -> bool:
        return any(p.status()["overflow"] for p in self.plans.values())


class _Pass(_Workspace):
    """One projection + binning of cat(scene, X) and the views composited from it (MergedFivePlan)."""

    def __init__(self, lib, P, W, H, dup_capacity, n_views, device):
        dev = device
        super().__init__(lib, P, W, H, dup_capacity, dev, n_views)
        self.P = P
        self.radii = torch.empty(P, dtype=torch.int32, device=dev)
        f = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        self.img = [(f(3, H, W), f(1, H, W), f(1, H, W)) for _ in range(n_views)]
        self.state = [(f(H * W), torch.empty(H * W, dtype=torch.int32, device=dev)) for _ in range(n_views)]
        widths = {"mean_3d": 3, "opacity": 1, "scale": 3, "rotation": 4, "rgb": 3}
        self.cat = {k: f(P, w) for k, w in widths.items()}
        self.streams = [torch.cuda.Stream(dev) for _ in range(n_views)]
        self.primed = False


class MergedFivePlan:
    """ExAvatar's five renders per training frame (avatar/main/model.py:81-162) from TWO projection + binning passes
    instead of five (SURVEY.md section 8f-3, kernel half):

        pass A  Gaussians cat(scene, human)          views  scene-only | human-only (random bg) | both
        pass B  Gaussians cat(scene, human_refined)  views               human-only (random bg) | both

    The five renders share one camera, so the scene Gaussians project, bin and depth-sort identically in renders 1, 3, 5
    and the human Gaussians in 2, 3 (refined: 4, 5).  A view (B2RView) composites the merged per-tile lists keeping only
    one index range -- entries of the other population are dropped when a batch is staged -- with its own background and
    per-pixel state.  Backward: the views of a pass accumulate their screen-space gradients into ONE scratch (the
    combined view skips the detached scene prefix, `first_row`), and the backward projection runs once per pass: scene
    rows carry the scene render's gradient, human rows the sum of the human-only and the combined render's -- what
    `loss.backward()` leaves in the leaves of model.py:117-125.  Same results as five separate renders (tests/), 2/5 of
    the projection / scatter / sort work.  Interface of FiveRenderPlan.

    scene_sh_coeffs = M > 0 (SURVEY.md section 8f-4 inside the merged frame): the scene Gaussians are coloured from their
    (P_scene, M, 3) SH coefficients in the projection kernel, as SceneGaussian does in PyTorch (module.py:253-272); the
    human rows keep their rgb.  One resident SH buffer serves both passes (their scene rows are identical; `set_scene`
    takes `shs`), each pass is described with B2RScene.sh_rows = P_scene and the frame's `settings.sh_degree`.  Pass A's
    backward projection writes the SH gradient of the scene rows (`grads("scene")["shs"]`, in place of "colors") and
    adds the view-direction term to their mean gradient; pass B's scene rows are detached and get nothing."""
    PER = FiveRenderPlan.PER
    VIEWS = {"A": ("scene", "human", "scene_human"), "B": ("human_refined", "scene_human_refined")}

    def __init__(self, P_scene: int, P_human: int, width: int, height: int, caps: Optional[Dict[str, int]], device,
                 scene_sh_coeffs: int = 0):
        self.lib = L.load()
        self.Ps, self.Ph, self.P = int(P_scene), int(P_human), int(P_scene) + int(P_human)
        self.M = int(scene_sh_coeffs)
        if not 0 <= self.M <= 16 or (self.M > 0 and self.Ps == 0):
            raise ValueError(f"MergedFivePlan: scene_sh_coeffs must be in [0, 16] with a non-empty scene, got {self.M}")
        self.W, self.H = int(width), int(height)
        self.device = torch.device(device)
        caps = caps or {"A": 8_000_000, "B": 8_000_000}
        self.passes = {k: _Pass(self.lib, self.P, self.W, self.H, caps[k], len(v), self.device) for k, v in self.VIEWS.items()}
        self.pass_streams = {k: torch.cuda.Stream(self.device) for k in self.passes}
        # the scene's SH coefficients, read by the projection of both passes
        self.shs = torch.zeros(self.Ps, self.M, 3, dtype=torch.float32, device=device) if self.M else None
        # one flat gradient buffer: [pass A: scene rows | human rows (| scene SH)][pass B: refined rows]
        self.nA, self.nB = self.PER * self.P + 3 * self.M * self.Ps, self.PER * self.Ph
        nA, nB = self.nA, self.nB
        self.all_flat = torch.zeros(nA + nB + 2 * self.Ps, dtype=torch.float32, device=device)
        self._stats = self.all_flat[nA + nB:]  # per-step densification sums ride in the all-reduced buffer (stats())
        self.views_A, self.views_B = self.grad_views(self.all_flat[:nA], self.all_flat[nA:nA + nB])
        Ps, P = self.Ps, self.P
        self.ranges = {"scene": (0, Ps), "human": (Ps, P), "scene_human": (0, P), "human_refined": (Ps, P),
                       "scene_human_refined": (0, P)}
        self.first_row = {"scene": 0, "human": Ps, "scene_human": Ps, "human_refined": Ps, "scene_human_refined": Ps}
        self._scenes = {}
        self._keep = []

    def describe(self) -> str:
        return ("two merged passes per frame (cat(scene,human): 3 views; cat(scene,refined): 2 views), each one "
                "projection + binning + sort; composites of a pass on parallel CUDA streams")

    def grad_views(self, flat_a: torch.Tensor, flat_b: torch.Tensor):
        """`_views_of`-style dicts over flat pass-A / pass-B gradient buffers of `nA` / `nB` floats.  Pass A: scene rows
        then human rows, and with an SH scene its (P_scene, M, 3) coefficient gradient under "shs"; pass B: refined rows."""
        _, va = _views_of(flat_a[: self.PER * self.P], self.P)
        if self.M:
            va["shs"] = flat_a[self.PER * self.P:].view(self.Ps, self.M, 3)
        _, vb = _views_of(flat_b, self.Ph)
        return va, vb

    def set_scene(self, scene_assets: Dict[str, torch.Tensor]) -> None:
        """Copies the scene Gaussians into the prefix of both passes; with scene_sh_coeffs > 0 `scene_assets` carries
        `shs` (P_scene, M, 3) in place of `rgb`."""
        for ps in self.passes.values():
            for k, buf in ps.cat.items():
                if self.M and k == "rgb":
                    continue
                buf[: self.Ps].copy_(scene_assets[k].reshape(self.Ps, -1))
        if self.M:
            self.shs.copy_(scene_assets["shs"].reshape(self.Ps, self.M, 3))

    def _scene_desc(self, key, ps, settings):
        """B2RScene of a pass for one camera; cached under `key` (the settings' tensors are then kept alive), or, when
        key[0] is None (a caller with a new camera every frame), kept only until the pass is used again."""
        if key[0] is not None and key in self._scenes:
            return self._scenes[key][0]
        entry = _make_scene(settings, ps.cat["mean_3d"], self.shs, ps.cat["rgb"], ps.cat["opacity"], ps.cat["scale"],
                            ps.cat["rotation"], None, 0)
        if self.M:
            entry[0].sh_rows = self.Ps  # scene rows from SH, human rows from rgb
        if key[0] is None:
            ps.last_scene = entry
        else:
            self._scenes[key] = entry
        return entry[0]

    def _human_bg(self, settings_human_bg) -> torch.Tensor:
        bg_h = _f32c(settings_human_bg.bg.to(self.device), "bg")
        self._keep.append(bg_h)  # the human-only views point at it until their composites have run
        del self._keep[:-64]
        return bg_h

    # ---- the stages of a frame; each enqueues on the stream that is current when it is called ----
    def _project_bin(self, pk, key, settings, src):
        """Projection + binning of pass `pk`; returns its B2RScene.  `src`: the human (A) or refined (B) assets, copied
        into the rows after the scene prefix; None when the caller already wrote them into `passes[pk].cat`."""
        ps = self.passes[pk]
        if src is not None:
            for k, buf in ps.cat.items():
                buf[self.Ps:].copy_(src[k].reshape(self.Ph, -1))
        sc = self._scene_desc((key, pk), ps, settings)
        sc.flags = L.B2R_FLAG_CTX_CLEAN if ps.primed else 0  # every pass leaves its ctx counters zero
        ps.primed = True
        st = torch.cuda.current_stream(self.device).cuda_stream
        L.check(self.lib.b2r_forward_project(C.byref(sc), C.byref(ps.ws), ps.radii.data_ptr(), st), "b2r_forward_project")
        L.check(self.lib.b2r_forward_bin(C.byref(sc), C.byref(ps.ws), st), "b2r_forward_bin")
        return sc

    def _forward_composite(self, pk, v, sc, bg_h, scene_done):
        """Forward composite of view `v` of pass `pk`; returns its B2RView, which the view's backward needs.  Every view
        but the scene-only one skips the tiles no human Gaussian reaches: a combined view equals the scene-only view
        there and carries no gradient; a human-only view shows the bare background there.  Both are pre-filled here.
        `scene_done` is recorded after the scene-only view and waited on before a combined view's pre-fill."""
        ps, name = self.passes[pk], self.VIEWS[pk][v]
        st = torch.cuda.current_stream(self.device)
        color, depth, alpha = ps.img[v]
        human_only = name in ("human", "human_refined")
        if human_only:  # bare background, no depth / alpha
            color.copy_(bg_h.view(3, 1, 1).expand_as(color))
            depth.zero_()
            alpha.zero_()
        elif name != "scene":  # the scene-only render; the composite overwrites the tiles a human Gaussian reaches
            st.wait_event(scene_done)
            for dst, src in zip(ps.img[v], self.passes["A"].img[0]):
                dst.copy_(src)
        lo, hi = self.ranges[name]
        fT, nc = ps.state[v]
        view = L.B2RView(lo, hi, _ptr(bg_h if human_only else None), fT.data_ptr(), nc.data_ptr(),
                         ps.ckpts[v].data_ptr(), ps.ckpt_bytes, 0 if name == "scene" else self.Ps, 0)
        out = L.B2RForwardOutputs(color.data_ptr(), depth.data_ptr(), alpha.data_ptr(), ps.radii.data_ptr())
        L.check(self.lib.b2r_forward_composite(C.byref(sc), C.byref(ps.ws), C.byref(view), C.byref(out), st.cuda_stream),
                "b2r_forward_composite")
        if name == "scene":
            scene_done.record(st)
        return view

    def _backward_composite(self, pk, v, sc, view, g_color, g_depth=None, g_alpha=None):
        """Backward composite of view `v` of pass `pk`: adds the view's screen-space gradients into the pass's scratch."""
        ps = self.passes[pk]
        a = L.B2RBackwardArgs(_ptr(g_color), _ptr(g_depth), _ptr(g_alpha))
        a.flags = L.B2R_BWD_SCRATCH_ZEROED
        a.first_row = self.first_row[self.VIEWS[pk][v]]
        L.check(self.lib.b2r_backward_composite(C.byref(sc), C.byref(ps.ws), C.byref(view), C.byref(a),
                                                ps.bwd_scratch.data_ptr(), ps.bwd_bytes,
                                                torch.cuda.current_stream(self.device).cuda_stream),
                "b2r_backward_composite")

    def _backward_project(self, pk, sc, g, accumulate, densify):
        """Backward projection of pass `pk`: writes (accumulate: adds) the gradients of its rows into the `_views_of`
        dict `g` (pass A: scene rows then human rows; pass B: refined rows).  `densify` is fed by pass A's scene rows."""
        ps = self.passes[pk]
        a = L.B2RBackwardArgs(None, None, None, _ptr(g["means3D"]), _ptr(g["means2D"]), _ptr(g.get("shs")), _ptr(g["colors"]),
                              _ptr(g["opacities"]), _ptr(g["scales"]), _ptr(g["rotations"]), None)
        a.flags = (L.B2R_BWD_ACCUMULATE if accumulate else 0) | L.B2R_BWD_SCRATCH_ZEROED
        a.first_row = 0 if pk == "A" else self.Ps
        if pk == "A" and densify is not None:
            a.densify_grad_accum, a.densify_count = _ptr(densify.get("grad_accum")), _ptr(densify.get("count"))
            a.densify_radius_max = _ptr(densify.get("radius_max"))
            a.densify_rows = self.Ps
        L.check(self.lib.b2r_backward_project(C.byref(sc), C.byref(ps.ws), C.byref(a), ps.bwd_scratch.data_ptr(),
                                              ps.bwd_bytes, torch.cuda.current_stream(self.device).cuda_stream),
                "b2r_backward_project")

    def frame(self, key, settings, settings_human_bg, scene, human, refined, g_colors: Dict[str, torch.Tensor],
              accumulate: bool, densify: Optional[Dict[str, torch.Tensor]] = None, serial: bool = False, probe=None) -> None:
        """Forward + backward of the five renders of one frame.  `serial`: everything on the caller's stream, one stage
        after the other.  `probe(label)` (serial mode only) is called after every stage with the label "{pass}:bin",
        "{pass}:{view}:fwd", "{pass}:{view}:bwd" or "{pass}:project_bwd" -- bench.py reads the in-library profiler
        there to get per-view kernel times."""
        probe = probe if (probe is not None and serial) else (lambda label: None)
        cur = torch.cuda.current_stream(self.device)
        bg_h = self._human_bg(settings_human_bg)
        scene_done = torch.cuda.Event()
        for pk, names in self.VIEWS.items():
            ps = self.passes[pk]
            st = cur if serial else self.pass_streams[pk]
            if not serial:
                st.wait_stream(cur)
            with torch.cuda.stream(st):
                sc = self._project_bin(pk, key, settings, human if pk == "A" else refined)
                probe(f"{pk}:bin")
                # forward + backward composite of every view; the views of a pass are independent of each other
                for v, n in enumerate(names):
                    vs = st if serial else ps.streams[v]
                    if not serial:
                        vs.wait_stream(st)
                    with torch.cuda.stream(vs):
                        view = self._forward_composite(pk, v, sc, bg_h, scene_done)
                        probe(f"{pk}:{n}:fwd")
                        self._backward_composite(pk, v, sc, view, g_colors[n])
                        probe(f"{pk}:{n}:bwd")
                if not serial:
                    for vs in ps.streams:
                        st.wait_stream(vs)
                self._backward_project(pk, sc, self.views_A if pk == "A" else self.views_B, accumulate, densify)
                probe(f"{pk}:project_bwd")
        if not serial:
            for pk in self.passes:
                cur.wait_stream(self.pass_streams[pk])

    # ---- the same frame in two halves (forward now, backward when the caller's gradients exist): fused.py ----
    def forward_frame(self, key, settings, settings_human_bg, scene, human, refined, copy_inputs: bool = True) -> None:
        """Forward of the five renders; images in `render_outputs()`, per-pixel state and checkpoints stay in the plan
        until `backward_frame` (so the plan must not start another frame in between).  copy_inputs=False: the caller
        already wrote the human / refined rows into `passes[*].cat` (a captured graph keeps the copies outside)."""
        cur = torch.cuda.current_stream(self.device)
        bg_h = self._human_bg(settings_human_bg)
        scene_done = torch.cuda.Event()
        self._pending = {}
        for pk in self.VIEWS:
            ps = self.passes[pk]
            st = self.pass_streams[pk]
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                sc = self._project_bin(pk, key, settings, (human if pk == "A" else refined) if copy_inputs else None)
                views = []
                for v, vs in enumerate(ps.streams):
                    vs.wait_stream(st)
                    with torch.cuda.stream(vs):
                        views.append(self._forward_composite(pk, v, sc, bg_h, scene_done))
                self._pending[pk] = (sc, views)
                for vs in ps.streams:
                    st.wait_stream(vs)
        for pk in self.passes:
            cur.wait_stream(self.pass_streams[pk])

    def backward_frame(self, g_colors: Dict[str, Optional[torch.Tensor]], grads_A: Dict[str, torch.Tensor],
                       grads_B: Dict[str, torch.Tensor], g_depths: Optional[Dict[str, torch.Tensor]] = None,
                       g_alphas: Optional[Dict[str, torch.Tensor]] = None, accumulate: bool = False,
                       densify: Optional[Dict[str, torch.Tensor]] = None) -> None:
        """Backward of the frame `forward_frame` rendered.  g_colors[name] = dL/dimage of a render, or None when the render
        was not used downstream.  grads_A / grads_B: `_views_of`-style dicts with P / P_human rows (pass A: scene rows then
        human rows; pass B: refined rows)."""
        cur = torch.cuda.current_stream(self.device)
        for pk, names in self.VIEWS.items():
            ps = self.passes[pk]
            sc, views = self._pending[pk]
            st = self.pass_streams[pk]
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                for v, n in enumerate(names):
                    gc, gd, ga = g_colors.get(n), (g_depths or {}).get(n), (g_alphas or {}).get(n)
                    if gc is None and gd is None and ga is None:
                        continue  # this render was not used downstream
                    vs = ps.streams[v]
                    vs.wait_stream(st)
                    with torch.cuda.stream(vs):
                        if gc is None:
                            gc = torch.zeros(3, self.H, self.W, dtype=torch.float32, device=self.device)
                        self._backward_composite(pk, v, sc, views[v], gc, gd, ga)
                        self._keep.append((gc, gd, ga))
                for vs in ps.streams:
                    st.wait_stream(vs)
                self._backward_project(pk, sc, grads_A if pk == "A" else grads_B, accumulate, densify)
        for pk in self.passes:
            cur.wait_stream(self.pass_streams[pk])

    def render_outputs(self, render: str):
        pk = "A" if render in self.VIEWS["A"] else "B"
        ps = self.passes[pk]
        color, _, alpha = ps.img[self.VIEWS[pk].index(render)]
        lo, hi = self.ranges[render]
        return color, alpha, ps.radii[lo:hi]

    def reduce(self):
        """(scene, human, human_refined) flat gradient buckets of the step.  Nothing to fold: the backward projection of
        a pass already summed the renders that share a parameter set.  NOTE the buckets are row-interleaved views of the
        pass buffers (means3D of all rows, then means2D ...); `grads(which)` gives named per-set tensors."""
        return self.grads("scene"), self.grads("human"), self.grads("human_refined")

    def grads(self, which: str) -> Dict[str, torch.Tensor]:
        if which == "scene":
            g = {k: v[: self.Ps] for k, v in self.views_A.items()}
            if self.M:
                del g["colors"]  # the scene rows' colour gradient went to their SH coefficients
            return g
        if which == "human":
            return {k: v[self.Ps:] for k, v in self.views_A.items() if k != "shs"}
        return dict(self.views_B)

    def flat_bucket(self) -> torch.Tensor:
        return self.all_flat

    def stats(self) -> Dict[str, torch.Tensor]:
        """Per-step sums of the densification statistics at the tail of the flat bucket (see FiveRenderPlan.stats)."""
        return {"grad_accum": self._stats[: self.Ps], "count": self._stats[self.Ps:]}

    def zero_stats(self) -> None:
        self._stats.zero_()

    def dups(self) -> Dict[str, int]:
        return {k: ps.status()["num_dups"] for k, ps in self.passes.items()}

    def consumed(self) -> Dict[str, list]:
        fwd, bwd = [], []
        for pk, names in self.VIEWS.items():  # the views of a pass add into the same counters: per-launch averages
            s = self.passes[pk].status()
            fwd += [s["consumed_fwd"] / L.CONSUMED_FWD_DIV / len(names)] * len(names)
            bwd += [s["consumed_bwd"] / L.CONSUMED_BWD_DIV / len(names)] * len(names)
        return {"fwd": fwd, "bwd": bwd}

    def overflowed(self) -> bool:
        return any(ps.status()["overflow"] for ps in self.passes.values())
