"""`GaussianRasterizationSettings` / `GaussianRasterizer` -- the Python surface ExAvatar imports.

Drop-in for `from diff_gaussian_rasterization_depth import GaussianRasterizationSettings, GaussianRasterizer`
(/root/reference/avatar/common/nets/module.py:11): same 12-field settings tuple in the order of the call site
(module.py:609-622), same keyword call (module.py:632-640), same 4-tuple `(color, radii, depth, alpha)` (module.py:632),
same argument-validation exceptions, gradients for the same eight tensor inputs.  The compute is the hand-written
sm_100a library behind include/b200raster.h, reached through ctypes with raw device pointers on the caller's current
CUDA stream; PyTorch only owns memory, streams and autograd.

No CPU path exists here on purpose: CPU tensors or a missing libb200raster.so raise.

Duplicate-capacity policy (the reference rasteriser stalls on a device->host copy of the duplicate count every
render, SURVEY.md section 2.3 row 3):
  * "exact": run the projection phase, learn the count from a pinned-host mirror the scan kernel writes (polling, no
    stream synchronise), size the lists exactly, run the render phase;
  * "speculative" (default once a count has been seen for this shape): enqueue BOTH phases with a capacity predicted
    from the previous render of the same (P, W, H); the poll then only confirms the prediction while the GPU is
    already compositing.  A misprediction re-runs the render phase with the exact size -- outputs are never truncated.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import time
from typing import NamedTuple, Optional

import numpy as np
import torch
from torch import nn

from . import _lib as L


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


# ---------------------------------------------------------------------------------------------------------------
# per-device host state: pinned status mirror, call counter, capacity predictions
# ---------------------------------------------------------------------------------------------------------------
class _DeviceState:
    def __init__(self, device: torch.device):
        self.lock = threading.Lock()
        self.mirror = torch.zeros(2, dtype=torch.int64).pin_memory()
        self.mirror_np = self.mirror.numpy()
        self.token = 0
        self.predicted = {}  # (P, W, H) -> last duplicate count

    def next_token(self) -> int:
        self.token += 1
        return self.token


_STATES = {}
_STATES_LOCK = threading.Lock()
CAPACITY_MODE = os.environ.get("B2R_CAPACITY_MODE", "speculative")  # or "exact"
CAPACITY_HEADROOM = 1.25
TILE_CULL = os.environ.get("B2R_TILE_CULL", "1") != "0"
SEGMENTED = os.environ.get("B2R_SEGMENTED", "1") != "0"  # checkpointed forward + segment-parallel backward
# Fixed-capacity mode: every render uses this many list entries, nothing is polled or synchronised, so the call is
# capturable in a CUDA graph (torch.cuda.graph) together with the caller's loss, backward and copies.  Overflow is
# not repaired on the fly in this mode: check `overflowed()` after the step (outputs are truncated, never corrupt).
FIXED_CAPACITY = None
RECENT_CONTEXTS = []  # contexts created in fixed-capacity mode (bounded), for the deferred overflow check
LAST_STATS = {}  # filled when a caller asks for stats (bench / tests)


def _state(device: torch.device) -> _DeviceState:
    key = device.index if device.index is not None else torch.cuda.current_device()
    with _STATES_LOCK:
        st = _STATES.get(key)
        if st is None:
            st = _STATES[key] = _DeviceState(device)
        return st


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None or t.numel() == 0 else t.data_ptr()


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"b200raster: `{name}` must be a CUDA tensor (got {t.device}); there is no CPU fallback")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _wait_mirror(st: _DeviceState, token: int, stream: torch.cuda.Stream, timeout_s: float = 20.0) -> int:
    """Spin until the scan kernel has published {num_dups, token}; returns num_dups."""
    m = st.mirror_np
    t0 = time.perf_counter()
    spins = 0
    while int(m[1]) != token:
        spins += 1
        if spins % 4096 == 0 and time.perf_counter() - t0 > timeout_s:
            stream.synchronize()  # surfaces a sticky CUDA error if the kernels died
            if int(m[1]) != token:
                raise RuntimeError("b200raster: projection phase never published its duplicate count")
    return int(m[0])


class _Context:
    """What must survive from forward to backward (SURVEY.md section 8b 'Ownership')."""
    __slots__ = ("scene", "ws", "keep", "ctx_buf", "dup_ids", "num_dups", "P", "W", "H", "M", "flags", "ckpt")


def _make_scene(settings: GaussianRasterizationSettings, means3D, shs, colors, opac, scales, rots, cov, flags, skin=None):
    """`skin` (fused skinning, SURVEY section 8f-2): dict(xyz, weights, joint_mats, trans, Rinv, t); `means3D` is then the
    (P,3) tensor that RECEIVES the posed positions."""
    dev = means3D.device
    keep = {
        "bg": _f32c(settings.bg.to(dev), "bg"),
        "view": _f32c(settings.viewmatrix.to(dev), "viewmatrix"),
        "proj": _f32c(settings.projmatrix.to(dev), "projmatrix"),
        "campos": _f32c(settings.campos.to(dev), "campos"),
        "means3D": means3D, "shs": shs, "colors": colors, "opac": opac, "scales": scales, "rots": rots, "cov": cov,
    }
    sc = L.B2RScene()
    sc.P = means3D.shape[0]
    sc.width = int(settings.image_width)
    sc.height = int(settings.image_height)
    sc.sh_degree = int(settings.sh_degree)
    sc.sh_coeffs = 0 if shs is None or shs.numel() == 0 else int(shs.shape[1])
    sc.flags = flags
    sc.scale_modifier = float(settings.scale_modifier)
    sc.tanfovx = float(settings.tanfovx)
    sc.tanfovy = float(settings.tanfovy)
    sc.bg = _ptr(keep["bg"])
    sc.viewmatrix = _ptr(keep["view"])
    sc.projmatrix = _ptr(keep["proj"])
    sc.campos = _ptr(keep["campos"])
    sc.means3D = None if skin is not None else _ptr(means3D)
    if skin is not None:
        keep["skin"] = skin
        sc.skin_xyz, sc.skin_weights = _ptr(skin["xyz"]), _ptr(skin["weights"])
        sc.skin_joint_mats, sc.skin_trans = _ptr(skin["joint_mats"]), _ptr(skin["trans"])
        sc.skin_cam_Rinv, sc.skin_cam_t = _ptr(skin.get("Rinv")), _ptr(skin.get("t"))
        sc.skin_means_out = _ptr(means3D)
        sc.skin_J = int(skin["weights"].shape[1])
    sc.shs = _ptr(shs)
    sc.colors_precomp = _ptr(colors)
    sc.opacities = _ptr(opac)
    sc.scales = _ptr(scales)
    sc.rotations = _ptr(rots)
    sc.cov3D_precomp = _ptr(cov)
    return sc, keep


def _forward_impl(settings, means3D, shs, colors, opac, scales, rots, cov, want_stats=False, skin=None, need_grad=True):
    """need_grad: a backward may follow, so the forward composite also stores its blend-state checkpoints (the segmented
    backward replays 512-entry list segments independently from them); inference calls skip that buffer."""
    lib = L.load()
    dev = means3D.device
    P = int(means3D.shape[0])
    H, W = int(settings.image_height), int(settings.image_width)
    flags = (0 if TILE_CULL else L.B2R_FLAG_NO_TILE_CULL) | (L.B2R_FLAG_DEBUG if settings.debug else 0)
    color = torch.empty((3, H, W), dtype=torch.float32, device=dev)
    depth = torch.empty((1, H, W), dtype=torch.float32, device=dev)
    alpha = torch.empty((1, H, W), dtype=torch.float32, device=dev)
    radii = torch.empty((P,), dtype=torch.int32, device=dev)
    if P == 0:  # upstream returns a zero image without launching anything [EXT]
        color.zero_(); depth.zero_(); alpha.zero_()
        return color, radii, depth, alpha, None

    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        sptr = stream.cuda_stream
        sc, keep = _make_scene(settings, means3D, shs, colors, opac, scales, rots, cov, flags, skin)
        st = None if FIXED_CAPACITY is not None else _state(dev)  # no pinned allocation inside a graph capture
        ctx_bytes = lib.b2r_ctx_bytes(P, W, H)
        ctx_buf = torch.empty(ctx_bytes, dtype=torch.uint8, device=dev)
        out = L.B2RForwardOutputs(color.data_ptr(), depth.data_ptr(), alpha.data_ptr(), radii.data_ptr())

        def checkpoints(cap):
            if not (need_grad and SEGMENTED):
                return None, 0
            nbytes = lib.b2r_checkpoint_bytes(W, H, cap)
            return torch.empty(nbytes, dtype=torch.uint8, device=dev), nbytes

        def workspace(cap, token):
            ids = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
            sbytes = lib.b2r_scratch_bytes(P, W, H, cap)
            scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
            ck, ckb = checkpoints(cap)
            ws = L.B2RWorkspace(ctx_buf.data_ptr(), ctx_bytes, ids.data_ptr(), cap, scratch.data_ptr(), sbytes,
                                st.mirror.data_ptr(), token, _ptr(ck), ckb)
            return ws, ids, scratch, ck

        key = (P, W, H)
        if FIXED_CAPACITY is not None:
            cap = int(FIXED_CAPACITY)
            ids = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
            sbytes = lib.b2r_scratch_bytes(P, W, H, cap)
            scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
            ck, ckb = checkpoints(cap)
            ws = L.B2RWorkspace(ctx_buf.data_ptr(), ctx_bytes, ids.data_ptr(), cap, scratch.data_ptr(), sbytes, None, 0,
                                _ptr(ck), ckb)
            L.check(lib.b2r_forward(C.byref(sc), C.byref(ws), C.byref(out), sptr), "b2r_forward")
            num = -1
        else:
          with st.lock:
              token = st.next_token()
              predicted = st.predicted.get(key) if CAPACITY_MODE == "speculative" else None
              if predicted is not None:
                  cap = int(predicted * CAPACITY_HEADROOM) + 4096
                  ws, ids, scratch, ck = workspace(cap, token)
                  L.check(lib.b2r_forward(C.byref(sc), C.byref(ws), C.byref(out), sptr), "b2r_forward")
                  num = _wait_mirror(st, token, stream)
                  if num > cap:  # misprediction: the whole forward again with the exact size (a forward that was given
                      # a capacity consumes the tile counters, so the render phase alone cannot be repeated)
                      token = st.next_token()
                      ws, ids, scratch, ck = workspace(num, token)
                      L.check(lib.b2r_forward(C.byref(sc), C.byref(ws), C.byref(out), sptr), "b2r_forward")
                      num = _wait_mirror(st, token, stream)
              else:
                  ws0 = L.B2RWorkspace(ctx_buf.data_ptr(), ctx_bytes, None, 0, None, 0, st.mirror.data_ptr(), token, None, 0)
                  L.check(lib.b2r_forward_project(C.byref(sc), C.byref(ws0), radii.data_ptr(), sptr), "b2r_forward_project")
                  num = _wait_mirror(st, token, stream)
                  ws, ids, scratch, ck = workspace(num, token)
                  L.check(lib.b2r_forward_render(C.byref(sc), C.byref(ws), C.byref(out), sptr), "b2r_forward_render")
              st.predicted[key] = num
        # `scratch` may be recycled by the caching allocator as soon as we drop it: same-stream ordering makes that safe
        if settings.debug:
            stream.synchronize()

        cx = _Context()
        cx.scene, cx.ws, cx.keep, cx.ctx_buf, cx.dup_ids, cx.num_dups = sc, ws, keep, ctx_buf, ids, num
        cx.P, cx.W, cx.H, cx.M, cx.flags = P, W, H, sc.sh_coeffs, flags
        # the saved workspace must not point at the recycled scratch
        cx.ckpt = ck
        cx.ws = L.B2RWorkspace(ctx_buf.data_ptr(), ctx_bytes, ids.data_ptr(), ws.dup_capacity, None, 0, None, 0,
                               ws.checkpoints, ws.checkpoint_bytes)
        if FIXED_CAPACITY is not None:
            RECENT_CONTEXTS.append(cx)
            del RECENT_CONTEXTS[:-64]
        if want_stats:
            LAST_STATS.clear()
            LAST_STATS.update(read_status(cx))
    return color, radii, depth, alpha, cx


def set_fixed_capacity(cap: Optional[int]) -> None:
    """None restores the adaptive (polling) policy."""
    global FIXED_CAPACITY
    FIXED_CAPACITY = None if cap is None else int(cap)
    RECENT_CONTEXTS.clear()


def overflowed() -> bool:
    """Deferred check for fixed-capacity mode: did any recent render need more list entries than it was given?"""
    return any(read_status(cx)["overflow"] for cx in RECENT_CONTEXTS)


def read_status(cx: _Context) -> dict:
    """Copies the device status block back (synchronises); for tests, bench accounting and debugging."""
    return L.read_status(cx.ctx_buf)


def _backward_impl(cx: _Context, g_color, g_depth, g_alpha, g_posed=None):
    lib = L.load()
    keep = cx.keep
    dev = keep["means3D"].device
    P, M = cx.P, cx.M
    f = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    d_means3D, d_means2D, d_colors, d_opac = f(P, 3), f(P, 3), f(P, 3), f(P, 1)
    d_scales, d_rots, d_cov = f(P, 3), f(P, 4), f(P, 6)
    d_shs = f(P, M, 3) if M > 0 else None
    skin = keep.get("skin")
    d_xyz, d_G = (f(P, 3), f(P, 12)) if skin is not None else (None, None)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        g_color = _f32c(g_color, "grad_color")
        g_depth = None if g_depth is None else _f32c(g_depth, "grad_depth")
        g_alpha = None if g_alpha is None else _f32c(g_alpha, "grad_alpha")
        sbytes = lib.b2r_backward_scratch_bytes(P)
        scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
        args = L.B2RBackwardArgs(_ptr(g_color), _ptr(g_depth), _ptr(g_alpha), _ptr(d_means3D), _ptr(d_means2D),
                                 _ptr(d_shs), _ptr(d_colors), _ptr(d_opac), _ptr(d_scales), _ptr(d_rots), _ptr(d_cov),
                                 0, 0, None, None, None, _ptr(d_xyz), _ptr(d_G),
                                 None if g_posed is None else _ptr(_f32c(g_posed, "grad_posed")))
        L.check(lib.b2r_backward(C.byref(cx.scene), C.byref(cx.ws), C.byref(args), scratch.data_ptr(), sbytes,
                                 stream.cuda_stream), "b2r_backward")
        if cx.flags & L.B2R_FLAG_DEBUG:
            stream.synchronize()
    if skin is not None:
        return d_means3D, d_means2D, d_shs, d_colors, d_opac, d_scales, d_rots, d_cov, d_xyz, d_G
    return d_means3D, d_means2D, d_shs, d_colors, d_opac, d_scales, d_rots, d_cov


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings):
        opt = lambda t, n: None if t is None or t.numel() == 0 else _f32c(t, n)
        m3 = _f32c(means3D, "means3D")
        args = (m3, opt(sh, "shs"), opt(colors_precomp, "colors_precomp"), _f32c(opacities, "opacities"),
                opt(scales, "scales"), opt(rotations, "rotations"), opt(cov3Ds_precomp, "cov3D_precomp"))
        try:
            color, radii, depth, alpha, cx = _forward_impl(raster_settings, *args, need_grad=any(ctx.needs_input_grad))
        except Exception:
            if raster_settings.debug:  # reference behaviour with debug=True: dump the arguments, re-raise
                torch.save(tuple(None if a is None else a.cpu() for a in args), "snapshot_fw.dump")
            raise
        ctx.set_materialize_grads(False)  # unused outputs (depth, alpha) arrive as None, not as zero images
        ctx.cx = cx
        ctx.has = (sh is not None and sh.numel() > 0, colors_precomp is not None and colors_precomp.numel() > 0,
                   scales is not None and scales.numel() > 0, rotations is not None and rotations.numel() > 0,
                   cov3Ds_precomp is not None and cov3Ds_precomp.numel() > 0)
        ctx.shapes = (means3D.shape, means2D.shape, opacities.shape)
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_color, grad_radii, grad_depth, grad_alpha):
        cx = ctx.cx
        m3s, m2s, ops = ctx.shapes
        if grad_color is None and grad_depth is None and grad_alpha is None:
            return (None,) * 9
        if grad_color is None:  # only depth / alpha were used downstream
            ref = grad_depth if grad_depth is not None else grad_alpha
            grad_color = torch.zeros((3,) + tuple(ref.shape[-2:]), dtype=torch.float32, device=ref.device)
        if cx is None:  # P == 0
            z = lambda s: torch.zeros(s, dtype=torch.float32, device=grad_color.device)
            return z(m3s), z(m2s), None, None, z(ops), None, None, None, None
        d_means3D, d_means2D, d_shs, d_colors, d_opac, d_scales, d_rots, d_cov = _backward_impl(
            cx, grad_color, grad_depth, grad_alpha)
        has_sh, has_col, has_sc, has_rot, has_cov = ctx.has
        return (d_means3D, d_means2D.reshape(m2s) if d_means2D.shape == tuple(m2s) else d_means2D,
                d_shs if has_sh else None, d_colors if has_col else None, d_opac.reshape(ops),
                d_scales if has_sc else None, d_rots if has_rot else None, d_cov if has_cov else None, None)


# The compiled binding of this call (csrc_torch/b2r_torch.cpp, built by build_ext.build_torch_ext): the same host logic
# as _RasterizeGaussians / _forward_impl / _backward_impl as a C++ autograd Function over the same C ABI -- it removes
# ~0.2 ms of Python per render from the eager path.  B2R_COMPILED_BINDING=0 keeps the Python route (also used for
# debug=True, fixed-capacity / graph capture and when the extension has not been built).
COMPILED_BINDING = os.environ.get("B2R_COMPILED_BINDING", "1") != "0"
_COMPILED = None


def _compiled_binding():
    global _COMPILED
    if _COMPILED is None:
        _COMPILED = False
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_b2r_torch.so")
        if COMPILED_BINDING and os.path.exists(path):
            import importlib.util
            L.load()  # libb200raster.so first: the extension links against it
            spec = importlib.util.spec_from_file_location("_b2r_torch", path)
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            if mod.abi_version() != L.ABI_VERSION:
                raise RuntimeError("b200raster: _b2r_torch.so was built against another ABI version; rebuild it")
            _COMPILED = mod
    return _COMPILED


def last_duplicate_count(device: torch.device, P: int, W: int, H: int) -> int:
    """Duplicate count of the most recent adaptive-capacity render of this shape on `device` (whichever host route ran
    it); KeyError when there was none.  Callers size fixed-capacity plans with it."""
    ext = _compiled_binding()
    idx = device.index if device.index is not None else torch.cuda.current_device()
    n = ext.get_predicted(idx, P, W, H) if ext else -1
    if n >= 0:
        return int(n)
    return int(_state(device).predicted[(P, W, H)])


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings):
    st = raster_settings
    ext = _compiled_binding() if (FIXED_CAPACITY is None and not st.debug) else False
    if ext:
        return tuple(ext.rasterize(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                   int(st.image_height), int(st.image_width), float(st.tanfovx), float(st.tanfovy), st.bg,
                                   float(st.scale_modifier), st.viewmatrix, st.projmatrix, int(st.sh_degree), st.campos,
                                   TILE_CULL, CAPACITY_MODE == "speculative", CAPACITY_HEADROOM, SEGMENTED))
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                     raster_settings)


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        """bool (P): Gaussians in front of the near plane (z_view > 0.2).  Unused by ExAvatar; kept for API parity."""
        lib = L.load()
        with torch.no_grad():
            p = _f32c(positions, "positions")
            view = _f32c(self.raster_settings.viewmatrix.to(p.device), "viewmatrix")
            present = torch.empty(p.shape[0], dtype=torch.uint8, device=p.device)
            with torch.cuda.device(p.device):
                L.check(lib.b2r_mark_visible(p.shape[0], _ptr(p), _ptr(view), _ptr(present),
                                             torch.cuda.current_stream(p.device).cuda_stream), "b2r_mark_visible")
            return present.bool()

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None):
        raster_settings = self.raster_settings
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception("Please provide excatly one of either SHs or precomputed colors!")
        if ((scales is None or rotations is None) and cov3D_precomp is None) or (
                (scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!")
        empty = torch.empty(0, dtype=torch.float32, device=means3D.device)
        if shs is None:
            shs = empty
        if colors_precomp is None:
            colors_precomp = empty
        if scales is None:
            scales = empty
        if rotations is None:
            rotations = empty
        if cov3D_precomp is None:
            cov3D_precomp = empty
        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp,
                                   raster_settings)


# ---------------------------------------------------------------------------------------------------------------
# SURVEY.md section 8f-2: linear-blend skinning fused into the projection kernels
# ---------------------------------------------------------------------------------------------------------------
class _RasterizeSkinned(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, skin_weights, joint_mats, trans, cam_R, cam_t, means2D, colors_precomp, opacities, scales,
                rotations, raster_settings):
        dev = xyz.device
        P = xyz.shape[0]
        skin = {"xyz": _f32c(xyz, "xyz"), "weights": _f32c(skin_weights, "skin_weights"),
                "joint_mats": _f32c(joint_mats, "joint_mats").reshape(-1, 16), "trans": _f32c(trans.reshape(3), "trans")}
        if cam_R is not None:
            skin["Rinv"] = _f32c(_inv3(cam_R), "cam_R")
            skin["t"] = _f32c(cam_t.reshape(3), "cam_t")
        posed = torch.empty((P, 3), dtype=torch.float32, device=dev)
        color, radii, depth, alpha, cx = _forward_impl(raster_settings, posed, None, _f32c(colors_precomp, "colors_precomp"),
                                                       _f32c(opacities, "opacities"), _f32c(scales, "scales"),
                                                       _f32c(rotations, "rotations"), None, skin=skin,
                                                       need_grad=any(ctx.needs_input_grad))
        ctx.set_materialize_grads(False)
        ctx.cx = cx
        ctx.shapes = (means2D.shape, opacities.shape, joint_mats.shape, trans.shape)
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha, posed

    @staticmethod
    def backward(ctx, grad_color, grad_radii, grad_depth, grad_alpha, grad_posed):
        cx = ctx.cx
        if grad_color is None and grad_depth is None and grad_alpha is None and grad_posed is None:
            return (None,) * 12
        if grad_color is None:  # only depth / alpha / the posed positions were used downstream
            grad_color = torch.zeros((3, cx.H, cx.W), dtype=torch.float32, device=cx.keep["means3D"].device)
        m2s, ops, js, ts = ctx.shapes
        # `posed` is differentiable: ExAvatar reads the posed mean_3d elsewhere (face_mesh_renderer, model.py:172-173, and
        # the cat(scene.detach(), human) renders, model.py:117-125); its gradient joins dL/dworld inside the backward
        # projection kernel, i.e. d_xyz += M^T Rinv^T g, d_G += (Rinv^T g) [x, 1]^T
        _, d_m2, _, d_col, d_op, d_sc, d_rot, _, d_xyz, d_G = _backward_impl(cx, grad_color, grad_depth, grad_alpha, grad_posed)
        W = cx.keep["skin"]["weights"]
        J = W.shape[1]
        d_joint = torch.zeros((J, 4, 4), dtype=torch.float32, device=W.device)
        d_joint[:, :3, :] = _tall_skinny_tn(W, d_G).view(J, 3, 4)  # the one dense contraction of this path: library GEMMs
        d_trans = d_G.view(-1, 3, 4)[:, :, 3].sum(0)
        return (d_xyz, None, d_joint.reshape(js), d_trans.reshape(ts), None, None, d_m2.reshape(m2s), d_col,
                d_op.reshape(ops), d_sc, d_rot, None)


class SkinnedGaussianRasterizer(nn.Module):
    """`GaussianRasterizer` with ExAvatar's linear-blend skinning in front of it, evaluated inside the projection
    kernels: replaces `get_transform_mat_vertex` + `lbs` + the camera->world transform
    (avatar/common/nets/module.py:413-422, 549-557) AND the rasteriser call (module.py:632-640) for the human Gaussians.

        color, radii, depth, alpha, posed = SkinnedGaussianRasterizer(settings)(
            xyz, skin_weights, joint_mats, trans, cam_R, cam_t, means2D, opacities, colors_precomp, scales, rotations)

    xyz (P,3) canonical positions; skin_weights (P,J) rows gathered per Gaussian (module.py:414); joint_mats (J,4,4);
    trans (3); cam_R (3,3) / cam_t (3) or None to stay in the posed frame (`is_world_coord=True`).  `posed` (P,3) is the
    world position ExAvatar's other modules read; it is a differentiable output: a gradient arriving at it is added to
    dL/dworld inside the backward projection kernel and reaches xyz, joint_mats and trans like the render's own."""

    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def forward(self, xyz, skin_weights, joint_mats, trans, cam_R, cam_t, means2D, opacities, colors_precomp, scales,
                rotations):
        return _RasterizeSkinned.apply(xyz, skin_weights, joint_mats, trans, cam_R, cam_t, means2D, colors_precomp,
                                       opacities, scales, rotations, self.raster_settings)


def _tall_skinny_tn(W: torch.Tensor, G: torch.Tensor, chunks: int = 64) -> torch.Tensor:
    """W^T G for W (P,J), G (P,n) with P ~ 10^5 and J, n ~ 10: a batched GEMM over `chunks` row blocks plus a tiny sum.
    A single (J x P)(P x n) GEMM leaves the library with one long-K tile and, depending on its heuristic, almost no
    parallelism; the batched form always fills the machine."""
    P, J = W.shape
    n = G.shape[1]
    pad = (-P) % chunks
    if pad:
        W = torch.cat((W, W.new_zeros(pad, J)))
        G = torch.cat((G, G.new_zeros(pad, n)))
    Wc = W.view(chunks, -1, J)
    Gc = G.view(chunks, -1, n)
    return torch.bmm(Wc.transpose(1, 2), Gc).sum(0)


def _inv3(R: torch.Tensor) -> torch.Tensor:
    """3x3 inverse by cofactors: a handful of elementwise kernels, no cuSOLVER call -- capturable in a CUDA graph
    (`torch.inverse`, which the reference uses at module.py:556, synchronises)."""
    a, b, c, d, e, f, g, h, i = R.reshape(9).unbind()
    adj = torch.stack((e * i - f * h, c * h - b * i, b * f - c * e,
                       f * g - d * i, a * i - c * g, c * d - a * f,
                       d * h - e * g, b * g - a * h, a * e - b * d)).reshape(3, 3)
    return adj / (a * (e * i - f * h) - b * (d * i - f * g) + c * (d * h - e * g))
