"""The merged five-render frame with its scene Gaussians coloured from SH in the projection kernel (B2RScene.sh_rows:
SH rows first, rgb rows after), on the B200.

  * one merged pass cat(scene, human) through the C ABI against the CPU oracle's all-SH render of the same Gaussians,
    the human rows given DC-only coefficients (rgb - 0.5) / C0 (their SH colour is then their rgb and no view-direction
    term arises); write and accumulate mode, and the detached scene prefix (first_row = P_scene, no dL_dshs);
  * sh_rows = P against the one-source SH path, bit for bit;
  * `TrainingFrameRenderer(scene_sh_coeffs=16)` against ExAvatar's five `GaussianRenderer` calls with the scene
    coloured caller-side, eager and in CUDA graphs, the SH degree changing between frames;
  * the merged plan's densification statistics with an SH scene and with its rgb equivalent.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from parity import compare
from util import settings_on, workload_settings
from exavatar_release_b200.synthetic import WORKLOADS, make_grad_image, make_population_assets, make_scene_sh_params
from oracle import oracle as O

pytestmark = pytest.mark.gpu

C0 = 0.28209479177387814
CUT = 7  # scene rows dropped from T1's 2000, so that P_scene is not a multiple of 32 and a warp straddles sh_rows


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _merged_population(M):
    """cat(scene, human) of T1 with the scene's SH coefficients (P_scene, M, 3) and the human rgb kept in [0.1, 0.9]
    (away from the clamp).  Returns (assets with rgb, scene shs, all-SH coefficients of the oracle reference, Ps)."""
    scene, human, _ = make_population_assets("T1", seed=0)
    p = make_scene_sh_params("T1", seed=0)
    Ps = scene["mean_3d"].shape[0] - CUT
    shs_s = torch.cat((p["feature_dc"], p["feature_rest"]), 1)[:Ps, :M].contiguous()
    h_rgb = 0.1 + 0.8 * human["rgb"]
    a = {k: torch.cat((scene[k][:Ps], human[k])).contiguous() for k in ("mean_3d", "opacity", "scale", "rotation")}
    # the colour rows of the SH rows are never read: NaN there would show up in every output
    a["rgb"] = torch.cat((torch.full((Ps, 3), float("nan")), h_rgb)).contiguous()
    h_sh = torch.zeros(h_rgb.shape[0], M, 3)
    h_sh[:, 0, :] = (h_rgb - 0.5) / C0
    return a, shs_s, torch.cat((shs_s, h_sh)).contiguous(), Ps


def _plan_scene(plan, st, a, shs, colors, sh_rows):
    from exavatar_release_b200.rasterizer import _make_scene
    sc, keep = _make_scene(st, a["mean_3d"], shs, colors, a["opacity"], a["scale"], a["rotation"], None, 0)
    sc.sh_rows = sh_rows
    plan._keep_scene = keep
    return sc


def _grads(P, rows, Ps_sh, M, dev, with_sh):
    nan = lambda *s: torch.full(s, float("nan"), device=dev)
    g = {"means3D": nan(rows, 3), "means2D": nan(rows, 3), "colors": nan(rows, 3), "opacities": nan(rows, 1),
         "scales": nan(rows, 3), "rotations": nan(rows, 4)}
    if with_sh:
        g["shs"] = nan(Ps_sh, M, 3)
    return g


@pytest.mark.parametrize("deg,M", [(1, 16), (3, 16), (1, 9), (2, 9)])
def test_merged_pass_with_sh_rows_matches_the_all_sh_oracle(dev, deg, M):
    from exavatar_release_b200.plan import FramePlan
    from exavatar_release_b200.rasterizer import GaussianRasterizationSettings
    wl = WORKLOADS["T1"]
    a, shs_s, shs_all, Ps = _merged_population(M)
    P = a["mean_3d"].shape[0]
    st_c = workload_settings("T1", yaw=10.0, bg=(0.2, 0.6, 0.9))._replace(sh_degree=deg)
    st_g = settings_on(st_c, dev, GaussianRasterizationSettings)
    oc, orad, od, oa, octx = O.forward(st_c, a["mean_3d"], a["opacity"], shs=shs_all, scales=a["scale"],
                                       rotations=a["rotation"])
    gi = make_grad_image("T1", 3)
    og = O.backward(octx, gi.numpy())
    pm, gm = O.fragility(octx)
    og["colors_h"] = og["shs"][:, 0, :] / C0  # human rows: dL/drgb of a DC-only colour

    plan = FramePlan(P, wl.width, wl.height, 2_000_000, dev)
    g = {k: v.to(dev) for k, v in a.items()}
    sc = _plan_scene(plan, st_g, g, shs_s.to(dev), g["rgb"], Ps)
    row = lambda y, lo=0: np.broadcast_to(gm[lo:].reshape((-1,) + (1,) * (y.ndim - 1)), y.shape)
    case = f"merged_sh_rows/deg{deg}/M{M}"

    def check(grads, scale, lo):
        for k in ("means3D", "means2D", "opacities", "scales", "rotations"):
            y = og[k][lo:] * scale
            compare(case, f"d_{k}/x{scale}/from{lo}", grads[k].cpu().numpy(), y, row(y, lo))
        y = og["colors_h"][Ps:] * scale
        compare(case, f"d_colors/x{scale}/from{lo}", grads["colors"][Ps - lo:].cpu().numpy(), y, row(y, Ps))
        if "shs" in grads:
            y = og["shs"][:Ps] * scale
            compare(case, f"d_shs/x{scale}", grads["shs"].cpu().numpy(), y, np.broadcast_to(gm[:Ps, None, None], y.shape))

    # write mode: every element written, the colour rows of the SH rows zero
    plan.forward(sc)
    gw = _grads(P, P, Ps, M, dev, True)
    plan.backward(sc, gi.to(dev), gw)
    torch.cuda.synchronize()
    assert np.array_equal(plan.radii.cpu().numpy(), orad), "radii must be identical"
    compare(case, "color", plan.color.cpu().numpy(), oc, np.broadcast_to(pm, oc.shape), kind="image")
    compare(case, "alpha", plan.alpha.cpu().numpy(), oa, pm[None], kind="image")
    for k, t in gw.items():
        assert bool(torch.isfinite(t).all()), k
    assert float(gw["colors"][:Ps].abs().max()) == 0.0
    if (deg + 1) ** 2 < M:  # coefficients above the active degree receive exactly zero
        assert float(gw["shs"][:, (deg + 1) ** 2:].abs().max()) == 0.0
    check(gw, 1, 0)
    assert float(gw["shs"][:, 1:].abs().max()) > 0 and float(gw["colors"][Ps:].abs().max()) > 0

    # accumulate mode: everything doubles, the colour rows of the SH rows are left as they are
    gw["colors"][:Ps] = 7.0
    plan.forward(sc)
    plan.backward(sc, gi.to(dev), gw, accumulate=True)
    torch.cuda.synchronize()
    assert bool((gw["colors"][:Ps] == 7.0).all())
    check(gw, 2, 0)

    # the detached scene prefix (pass B of the merged frame): first_row = P_scene, no SH gradient buffer
    plan.forward(sc)
    gb = _grads(P, P - Ps, 0, M, dev, False)
    plan.backward(sc, gi.to(dev), gb, first_row=Ps)
    torch.cuda.synchronize()
    for k, t in gb.items():
        assert bool(torch.isfinite(t).all()), k
    check(gb, 1, Ps)


def test_sh_rows_equal_to_P_is_the_sh_path_bit_for_bit(dev):
    """sh_rows = P (colour pointer set, never read) and sh_rows = 0 run the same arithmetic: forward outputs and the
    projection's ctx records bit for bit; the backward projection, fed the same screen-space gradients, writes the same
    bits into every gradient."""
    from exavatar_release_b200 import _lib as L
    from exavatar_release_b200.plan import FramePlan
    from exavatar_release_b200.rasterizer import GaussianRasterizationSettings
    wl = WORKLOADS["T1"]
    a, _, shs_all, _ = _merged_population(16)
    P = a["mean_3d"].shape[0]
    st = settings_on(workload_settings("T1", yaw=-7.0)._replace(sh_degree=3), dev, GaussianRasterizationSettings)
    g = {k: v.to(dev) for k, v in a.items()}
    shs = shs_all.to(dev)
    plan = FramePlan(P, wl.width, wl.height, 2_000_000, dev)
    lib = plan.lib
    sc_one = _plan_scene(plan, st, g, shs, None, 0)
    keep_one = plan._keep_scene
    sc_two = _plan_scene(plan, st, g, shs, g["rgb"], P)
    geom = lambda: plan.ctx_buf[lib.b2r_ctx_geom(C.byref(plan.ws), P, wl.width, wl.height) - plan.ctx_buf.data_ptr():][:P * 48].clone()
    outs = {}
    for name, sc in (("one", sc_one), ("two", sc_two)):
        plan.forward(sc)
        torch.cuda.synchronize()
        outs[name] = [t.clone() for t in (plan.color, plan.depth, plan.alpha, plan.radii)] + [geom()]
    for x, y in zip(outs["one"], outs["two"]):
        assert torch.equal(x, y)
    # screen-space gradients once (backward composite), then the backward projection of each scene from a copy
    gi = make_grad_image("T1", 5).to(dev)
    scratch = torch.zeros(plan.bwd_bytes, dtype=torch.uint8, device=dev)
    args = L.B2RBackwardArgs(gi.data_ptr())
    st_ = torch.cuda.current_stream(dev).cuda_stream
    L.check(lib.b2r_backward_composite(C.byref(sc_two), C.byref(plan.ws), None, C.byref(args), scratch.data_ptr(),
                                       plan.bwd_bytes, st_), "b2r_backward_composite")
    res = {}
    for name, sc in (("one", sc_one), ("two", sc_two)):
        s = scratch.clone()
        gr = _grads(P, P, P, 16, dev, True)
        gr["colors"].zero_()
        b = L.B2RBackwardArgs(None, None, None, *(gr[k].data_ptr() for k in ("means3D", "means2D", "shs")),
                              gr["colors"].data_ptr() if name == "two" else None,
                              *(gr[k].data_ptr() for k in ("opacities", "scales", "rotations")), None)
        L.check(lib.b2r_backward_project(C.byref(sc), C.byref(plan.ws), C.byref(b), s.data_ptr(), plan.bwd_bytes, st_),
                "b2r_backward_project")
        res[name] = gr
    torch.cuda.synchronize()
    del keep_one
    for k in ("means3D", "means2D", "shs", "opacities", "scales", "rotations"):
        assert torch.equal(res["one"][k], res["two"][k]), k
    assert float(res["two"]["colors"].abs().max()) == 0.0
    assert float(res["one"]["shs"].abs().max()) > 0


@pytest.mark.parametrize("use_graph,wl_name", [(False, "T1"), (True, "T1"), (False, "T3"), (True, "T3")])
def test_training_frame_renderer_with_sh_scene_equals_five_renderer_calls(dev, use_graph, wl_name):
    """`TrainingFrameRenderer(scene_sh_coeffs=16)` given scene_gaussian_assets(in_kernel_sh=True) against the five
    `GaussianRenderer` calls of ExAvatar with the scene coloured caller-side (in_kernel_sh=False): images, masks, radii
    and every gradient -- feature_dc / feature_rest, mean (view direction included), opacity / scale, the human and
    refined assets and the scene mean_2d -- over frames with a new camera and SH degree each (0, 1, 3), then degree 1 again with another camera."""
    from exavatar_release_b200 import GaussianRenderer, TrainingFrameRenderer
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS
    from exavatar_release_b200.renderer import scene_gaussian_assets
    wl = WORKLOADS[wl_name]
    H, W = wl.height, wl.width
    _, human, refined = make_population_assets(wl_name, seed=0, device=dev)
    p0 = make_scene_sh_params(wl_name, seed=0, device=dev)
    Ps, Ph = p0["mean"].shape[0], human["mean_3d"].shape[0]
    bg_r = torch.tensor([0.3, 0.7, 0.2], device=dev)
    gcol = {r: make_grad_image(wl_name, 70 + j).to(dev) for j, r in enumerate(RENDERS)}
    gmask = make_grad_image(wl_name, 80).to(dev)[:1]
    used = ("scene", "human", "scene_human", "scene_human_refined")
    frame = TrainingFrameRenderer(Ps, Ph, (H, W), dev, {"A": 2_000_000, "B": 2_000_000}, use_graph=use_graph,
                                  graph_depth_alpha=use_graph, scene_sh_coeffs=16)

    def leaves():
        p = {k: v.clone().requires_grad_() for k, v in p0.items()}
        hr = {n: {k: v.clone().requires_grad_() for k, v in a.items()} for n, a in (("human", human), ("refined", refined))}
        return p, hr

    def scene_of(p, deg, cam, in_kernel):
        return scene_gaussian_assets(p["mean"], p["opacity_logit"], p["log_scale"], p["rotation"], p["feature_dc"],
                                     p["feature_rest"], deg, cam, in_kernel_sh=in_kernel)

    for yaw, deg in ((-9.0, 0), (6.0, 1), (14.0, 3), (-3.0, 1)):  # graphs: three captures, then a replay
        cam = look_at_cam_param(yaw, (H, W), device=dev)
        pa, ha = leaves()
        R = GaussianRenderer()
        sa = scene_of(pa, deg, cam, False)
        cat = lambda x, y: {k: torch.cat((x[k].detach(), y[k])) for k in y}
        ref = {"scene": R(sa, (H, W), cam), "human": R(ha["human"], (H, W), cam, bg_r),
               "scene_human": R(cat(sa, ha["human"]), (H, W), cam), "human_refined": R(ha["refined"], (H, W), cam, bg_r),
               "scene_human_refined": R(cat(sa, ha["refined"]), (H, W), cam)}
        (sum((ref[r]["img"] * gcol[r]).sum() for r in used) + (ref["human"]["mask"] * gmask).sum()).backward()
        pb, hb = leaves()
        out = frame(scene_of(pb, deg, cam, True), hb["human"], hb["refined"], cam, bg_r)
        (sum((out[r]["img"] * gcol[r]).sum() for r in used) + (out["human"]["mask"] * gmask).sum()).backward()
        torch.cuda.synchronize()
        assert not frame.overflowed()
        near = lambda x, y: float((x - y).abs().max()) <= 1e-4 * float(y.abs().max()) + 1e-12
        for r in RENDERS:
            assert torch.equal(out[r]["radius"], ref[r]["radius"]) and torch.equal(out[r]["is_vis"], ref[r]["is_vis"]), r
            assert near(out[r]["img"], ref[r]["img"]), (r, deg)
            assert near(out[r]["mask"], ref[r]["mask"]) and near(out[r]["depthmap"], ref[r]["depthmap"]), (r, deg)
        for k in pa:
            assert pb[k].grad is not None and near(pb[k].grad, pa[k].grad), ("scene", k, deg)
        for n in ha:
            for k in ha[n]:
                assert hb[n][k].grad is not None and near(hb[n][k].grad, ha[n][k].grad), (n, k, deg)
        assert near(out["scene"]["mean_2d"].grad, ref["scene"]["mean_2d"].grad)
        assert float(pa["feature_dc"].grad.abs().max()) > 0
        if deg > 0:
            assert float(pb["feature_rest"].grad.abs().max()) > 0
        else:
            assert float(pb["feature_rest"].grad.abs().max()) == 0.0


def test_frame_renderer_rejects_a_mismatched_scene_before_enqueueing(dev):
    from exavatar_release_b200 import TrainingFrameRenderer
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.renderer import scene_gaussian_assets
    wl = WORKLOADS["T0"]
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets("T0", seed=0, device=dev)
    p = make_scene_sh_params("T0", seed=0, device=dev)
    cam = look_at_cam_param(0.0, (H, W), device=dev)
    sh = scene_gaussian_assets(p["mean"], p["opacity_logit"], p["log_scale"], p["rotation"], p["feature_dc"],
                               p["feature_rest"], 3, cam, in_kernel_sh=True)
    Ps, Ph = scene["mean_3d"].shape[0], human["mean_3d"].shape[0]
    bg = torch.zeros(3, device=dev)
    for M, s in ((16, scene), (0, sh), (9, sh)):
        frame = TrainingFrameRenderer(Ps, Ph, (H, W), dev, {"A": 100_000, "B": 100_000}, scene_sh_coeffs=M)
        with pytest.raises(ValueError):
            frame(s, human, refined, cam, bg)
        assert frame._frame_no == 0 and not any(ps.primed for ps in frame.plan.passes.values())


def test_densification_statistics_of_an_sh_scene_equal_its_rgb_equivalent(dev):
    """The merged plan's densification statistics over three frames: an SH scene (coloured in the kernel) and the same
    scene with the colours computed caller-side.  The radii and so the counts and radius maxima are identical; the
    accumulated screen-space gradient norms agree to the rounding of the two colour evaluations."""
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS, MergedFivePlan
    from exavatar_release_b200.rasterizer import GaussianRasterizationSettings
    from exavatar_release_b200.renderer import render_settings, scene_gaussian_assets
    wl = WORKLOADS["T1"]
    H, W = wl.height, wl.width
    _, human, refined = make_population_assets("T1", seed=0, device=dev)
    p = make_scene_sh_params("T1", seed=0, device=dev)
    Ps, Ph = p["mean"].shape[0], human["mean_3d"].shape[0]
    plans = {"sh": MergedFivePlan(Ps, Ph, W, H, None, dev, scene_sh_coeffs=16), "rgb": MergedFivePlan(Ps, Ph, W, H, None, dev)}
    stats = {k: {n: torch.zeros(Ps, device=dev) for n in ("grad_accum", "count", "radius_max")} for k in plans}
    bg_w, bg_r = torch.ones(3, device=dev), torch.tensor([0.3, 0.7, 0.2], device=dev)
    for f, yaw in enumerate((-12.0, 0.0, 14.0)):
        cam = look_at_cam_param(yaw, (H, W), device=dev)
        gcol = {r: make_grad_image("T1", 90 + 5 * f + j).to(dev) for j, r in enumerate(RENDERS)}
        for k, plan in plans.items():
            s = scene_gaussian_assets(p["mean"], p["opacity_logit"], p["log_scale"], p["rotation"], p["feature_dc"],
                                      p["feature_rest"], 3, cam, in_kernel_sh=(k == "sh"))
            plan.set_scene(s)
            st_w = render_settings((H, W), cam, bg_w, GaussianRasterizationSettings)
            st_r = render_settings((H, W), cam, bg_r, GaussianRasterizationSettings)
            if k == "sh":
                st_w, st_r = st_w._replace(sh_degree=3), st_r._replace(sh_degree=3)
            plan.frame(None, st_w, st_r, None, human, refined, gcol, accumulate=(f > 0), densify=stats[k])
    torch.cuda.synchronize()
    assert torch.equal(stats["sh"]["count"], stats["rgb"]["count"])
    assert torch.equal(stats["sh"]["radius_max"], stats["rgb"]["radius_max"])
    ref = stats["rgb"]["grad_accum"]
    assert float((stats["sh"]["grad_accum"] - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    assert float(stats["sh"]["count"].max()) == 3.0 and float(ref.max()) > 0
    gs, gr = plans["sh"].grads("scene"), plans["rgb"].grads("scene")
    assert "shs" in gs and "colors" not in gs and gs["shs"].shape == (Ps, 16, 3)
    assert plans["sh"].flat_bucket().numel() == plans["rgb"].flat_bucket().numel() + 48 * Ps
    for k in ("means2D", "opacities", "scales", "rotations"):
        assert float((gs[k] - gr[k]).abs().max()) <= 1e-4 * float(gr[k].abs().max()) + 1e-12, k
    for w in ("human", "human_refined"):
        a, b = plans["sh"].grads(w), plans["rgb"].grads(w)
        assert set(a) == set(b)
        for k in a:
            assert float((a[k] - b[k]).abs().max()) <= 1e-4 * float(b[k].abs().max()) + 1e-12, (w, k)
