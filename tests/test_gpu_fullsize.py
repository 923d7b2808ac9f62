"""Full-size GPU-vs-oracle parity on every BASELINE.json config (C2..C5), driven through the C ABI (FramePlan /
FiveRenderPlan), with the tightness report of tests/parity.py, plus bit-exact per-tile lists for every sort class.

VERDICT r01 item 1: C3 (1024x1024, 300 k, SH-3, fwd+bwd), C4 (each of the five renders of avatar/main/model.py:130-162
against its OWN oracle render, including the detached scene prefix), C5 (1080p, 500 k, fwd), long lists of 600 / 3000 /
20000 entries in one tile (CTA class, 2-chunk merge, 10-chunk merge).
"""
import numpy as np
import pytest
import torch

from parity import compare, contributor_report, last_contributor
from util import ctx_arrays, kat_settings, settings_on, workload_settings
from exavatar_release_b200.synthetic import WORKLOADS, make_assets, make_grad_image, make_population_assets
from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _oracle_last(octx):
    return last_contributor(octx.sorted_ids(), octx.ranges(), octx.n_contrib(), octx.W, octx.H)


def _plan_vs_oracle(dev, case, wl_name, yaw, seed=0, cap=12_000_000, with_da=False):
    """One frame of a workload through FramePlan (C ABI) against the oracle; returns nothing, asserts + reports."""
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    wl = WORKLOADS[wl_name]
    assets = make_assets(wl_name, seed=seed)
    bg = (0.2, 0.6, 0.9)
    st_c = workload_settings(wl_name, yaw=yaw, bg=bg)
    use_sh = wl.sh_degree > 0
    M = (wl.sh_degree + 1) ** 2 if use_sh else 0
    if use_sh:
        st_c = st_c._replace(sh_degree=wl.sh_degree)
    st_g = settings_on(st_c, dev, rz.GaussianRasterizationSettings)
    kw = dict(shs=assets["shs"]) if use_sh else dict(colors_precomp=assets["rgb"])
    oc, orad, od, oa, octx = O.forward(st_c, assets["mean_3d"], assets["opacity"], scales=assets["scale"],
                                       rotations=assets["rotation"], **kw)
    pm, gm = O.fragility(octx)
    P = assets["mean_3d"].shape[0]
    g_assets = {k: v.to(dev) for k, v in assets.items()}
    plan = FramePlan(P, wl.width, wl.height, cap, dev, sh_coeffs=M)
    sc = plan.scene(0, st_g, g_assets)
    plan.forward(sc)
    torch.cuda.synchronize()
    stt = plan.status()
    assert stt["overflow"] == 0, stt
    assert np.array_equal(plan.radii.cpu().numpy(), orad), "radii must be identical"
    compare(case, "color", plan.color.cpu().numpy(), oc, pm[None], kind="image")
    compare(case, "depth", plan.depth.cpu().numpy(), od, pm[None], kind="image")
    compare(case, "alpha", plan.alpha.cpu().numpy(), oa, pm[None], kind="image")
    ranges, ids, ncon, fT = ctx_arrays(plan.lib, plan, plan.P, plan.W, plan.H)
    contributor_report(case, last_contributor(ids, ranges, ncon, wl.width, wl.height), fT, _oracle_last(octx),
                       octx.final_T(), pm)
    if not wl.backward:
        return
    gi = make_grad_image(wl_name, seed)
    gd = ga = None
    if with_da:
        gen = torch.Generator().manual_seed(77)
        gd = torch.randn(1, wl.height, wl.width, generator=gen)
        ga = torch.randn(1, wl.height, wl.width, generator=gen)
    flat, views = grad_bucket(P, dev, M)
    plan.backward(sc, gi.to(dev), views, g_depth=None if gd is None else gd.to(dev),
                  g_alpha=None if ga is None else ga.to(dev))
    torch.cuda.synchronize()
    og = O.backward(octx, gi.numpy(), None if gd is None else gd.numpy()[0], None if ga is None else ga.numpy()[0])
    names = ["means3D", "means2D", "opacities", "scales", "rotations", "shs" if use_sh else "colors"]
    for k in names:
        y = og[k]
        x = views[k].cpu().numpy().reshape(y.shape)
        compare(case, "d_" + k, x, y, gm.reshape((-1,) + (1,) * (y.ndim - 1)), kind="grad")
    assert float(views["means2D"][:, 2].abs().max()) == 0.0


def test_c2_full_size_with_depth_alpha_grads(dev):
    """BASELINE configs[1] again, through the C ABI, with depth / alpha gradients and the contributor report."""
    _plan_vs_oracle(dev, "C2", "C2", yaw=-7.0, seed=1, with_da=True)


def test_c3_full_size_parity(dev):
    """BASELINE configs[2]: 1024x1024, 300 k Gaussians, SH degree 3, forward + backward."""
    _plan_vs_oracle(dev, "C3", "C3", yaw=9.0)


def test_c5_full_size_forward(dev):
    """BASELINE configs[4]: 1920x1080, 500 k Gaussians, forward only."""
    _plan_vs_oracle(dev, "C5", "C5", yaw=-4.0)


def test_c4_single_render_parity(dev):
    """The C4 Gaussian set (167 k avatar + 130 k scene) as one render, forward + backward."""
    _plan_vs_oracle(dev, "C4", "C4", yaw=15.0)


@pytest.mark.parametrize("engine", ["merged", "separate"])
def test_c4_five_render_frame_vs_five_oracle_renders(dev, engine):
    """BASELINE configs[3]: one training frame of avatar/main/model.py:81-162 at full size (167 k human + 130 k scene
    Gaussians, 512x512) on FiveRenderPlan, every render against ITS OWN oracle render: scene | human (random bg) |
    cat(scene.detach(), human) | human_refined | cat(scene.detach(), human_refined).  Gradients: the scene bucket is the
    scene render's; the human bucket is render 2 + the human rows of render 3 (the detached prefix gets nothing).
    engine "merged": MergedFivePlan (two projection / binning passes, five views -- SURVEY 8f-3); "separate": five
    independent renders (FiveRenderPlan)."""
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS, FiveRenderPlan, MergedFivePlan
    from exavatar_release_b200.renderer import render_settings
    wl = WORKLOADS["C4"]
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets("C4", seed=0)
    Ps, Ph = scene["mean_3d"].shape[0], human["mean_3d"].shape[0]
    bg_w, bg_r = torch.ones(3), torch.tensor([0.3, 0.7, 0.2])
    cam = look_at_cam_param(-6.0, (H, W))
    gcol = {r: make_grad_image("C4", 40 + j) for j, r in enumerate(RENDERS)}
    cat = lambda a, b: {k: torch.cat((a[k], b[k])) for k in a}
    sets = {"scene": (scene, bg_w), "human": (human, bg_r), "scene_human": (cat(scene, human), bg_w),
            "human_refined": (refined, bg_r), "scene_human_refined": (cat(scene, refined), bg_w)}
    ora = {}
    for r, (a, bg) in sets.items():
        st = render_settings((H, W), cam, bg, O.OracleSettings)
        oc, orad, od, oa, octx = O.forward(st, a["mean_3d"], a["opacity"], colors_precomp=a["rgb"], scales=a["scale"],
                                           rotations=a["rotation"])
        og = O.backward(octx, gcol[r].numpy())
        ora[r] = dict(color=oc, radii=orad, alpha=oa, grads=og, frag=O.fragility(octx), ctx=octx)

    to = lambda d: {k: v.to(dev) for k, v in d.items()}
    plan = (MergedFivePlan if engine == "merged" else FiveRenderPlan)(Ps, Ph, W, H, None, dev)
    plan.set_scene(to(scene))
    st_w = settings_on(render_settings((H, W), cam, bg_w, O.OracleSettings), dev, rz.GaussianRasterizationSettings)
    st_r = settings_on(render_settings((H, W), cam, bg_r, O.OracleSettings), dev, rz.GaussianRasterizationSettings)
    plan.frame(0, st_w, st_r, to(scene), to(human), to(refined), {r: g.to(dev) for r, g in gcol.items()}, accumulate=False)
    torch.cuda.synchronize()
    assert not plan.overflowed()
    # forward images and radii, render by render
    for r in RENDERS:
        pm, _ = ora[r]["frag"]
        img, alpha, radii = plan.render_outputs(r)
        assert np.array_equal(radii.cpu().numpy(), ora[r]["radii"]), r
        compare(f"C4-{engine}/" + r, "color", img.cpu().numpy(), ora[r]["color"], pm[None], kind="image")
        compare(f"C4-{engine}/" + r, "alpha", alpha.cpu().numpy(), ora[r]["alpha"], pm[None], kind="image")
    # gradients: three parameter sets
    names = {"means3D": "means3D", "means2D": "means2D", "opacities": "opacities", "scales": "scales",
             "rotations": "rotations", "colors": "colors"}
    plan.reduce()

    def expect(parts):
        out, flag = {}, None
        for r, rows in parts:
            g, (_, gm) = ora[r]["grads"], ora[r]["frag"]
            for k in names:
                y = g[k][rows].reshape(g[k][rows].shape[0], -1)
                out[k] = y if k not in out else out[k] + y
            flag = gm[rows] if flag is None else (flag | gm[rows])
        return out, flag

    for label, Pn, parts in (
            ("scene", Ps, [("scene", slice(0, Ps))]),
            ("human", Ph, [("human", slice(0, Ph)), ("scene_human", slice(Ps, Ps + Ph))]),
            ("human_refined", Ph, [("human_refined", slice(0, Ph)), ("scene_human_refined", slice(Ps, Ps + Ph))])):
        views = plan.grads(label)
        y, flag = expect(parts)
        for k in names:
            compare(f"C4-{engine}/" + label, "d_" + k, views[k].cpu().numpy().reshape(Pn, -1), y[k], flag[:, None], kind="grad")


def _stack_in_one_tile(n, seed):
    g = torch.Generator().manual_seed(seed)
    pos = torch.stack([0.04 * (torch.rand(n, generator=g) - 0.5), 0.04 * (torch.rand(n, generator=g) - 0.5),
                       2.0 + 2.0 * torch.rand(n, generator=g)], 1)
    # a few exact depth ties (cloned Gaussians): the (depth, id) order must put the lower index first
    pos[n // 2: n // 2 + 8, 2] = pos[n // 3: n // 3 + 8, 2]
    return {"mean_3d": pos, "scale": 0.004 + 0.004 * torch.rand(n, 3, generator=g),
            "rotation": torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=1),
            # n <= 3000: faint splats, so pixels walk (almost) the whole list -- many staging batches and, in the
            # segmented composites, many segments; n = 20000: pixels saturate after a few hundred entries
            "opacity": (0.004 + 0.008 * torch.rand(n, 1, generator=g)) if n <= 3000 else (0.02 + 0.05 * torch.rand(n, 1, generator=g)),
            "rgb": torch.rand(n, 3, generator=g)}


@pytest.mark.parametrize("n", [600, 3000, 20000])
def test_long_list_sort_is_bit_exact(dev, n):
    """Per-tile depth-sorted id lists identical to the oracle's (tile culling off = reference list membership) for a
    tile of ~n entries: 600 -> the one-CTA class (512..2047), 3000 -> two 2048-entry chunks + merge_chunks_kernel,
    20000 -> ten chunks.  Includes bit-identical depths (index tie-break).  Then forward + backward on the same scene
    with the strict tolerance."""
    from exavatar_release_b200 import _lib as L
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    a = _stack_in_one_tile(n, seed=n)
    W, H = 64, 48
    st_c = kat_settings(W=W, H=H, f=60.0, bg=(0.1, 0.2, 0.3))
    st_g = settings_on(st_c, dev, rz.GaussianRasterizationSettings)
    oc, orad, od, oa, octx = O.forward(st_c, a["mean_3d"], a["opacity"], colors_precomp=a["rgb"], scales=a["scale"],
                                       rotations=a["rotation"])
    o_ids, o_ranges = octx.sorted_ids(), octx.ranges()
    lens = o_ranges[:, 1] - o_ranges[:, 0]
    assert lens.max() >= 0.9 * n, f"generator must stack the splats in one tile (max list {lens.max()})"
    ag = {k: v.to(dev) for k, v in a.items()}
    for flags in (L.B2R_FLAG_NO_TILE_CULL, 0):
        plan = FramePlan(n, W, H, 200_000, dev)
        sc = plan.scene(flags, st_g, ag, flags=flags)
        plan.forward(sc)
        torch.cuda.synchronize()
        assert plan.status()["overflow"] == 0
        ranges, ids, ncon, fT = ctx_arrays(plan.lib, plan, plan.P, plan.W, plan.H)
        if flags:
            assert plan.status()["num_dups"] == octx.num_dups
            for t in range(ranges.shape[0]):
                mine = ids[ranges[t, 0]:ranges[t, 1]]
                ref = o_ids[o_ranges[t, 0]:o_ranges[t, 1]]
                assert np.array_equal(mine, ref), f"tile {t} (n = {len(ref)}): sorted id list differs from the oracle"
        else:  # culled lists: ordered sub-sequences of the reference lists
            for t in range(ranges.shape[0]):
                mine = ids[ranges[t, 0]:ranges[t, 1]].tolist()
                it = iter(o_ids[o_ranges[t, 0]:o_ranges[t, 1]].tolist())
                assert all(m in it for m in mine), f"tile {t}: culled list is not an ordered subsequence"
        pm, gm = O.fragility(octx)
        case = f"stack{n}/" + ("nocull" if flags else "cull")
        assert np.array_equal(plan.radii.cpu().numpy(), orad)
        compare(case, "color", plan.color.cpu().numpy(), oc, pm[None], kind="image")
        contributor_report(case, last_contributor(ids, ranges, ncon, W, H), fT, _oracle_last(octx), octx.final_T(), pm,
                           max_frac=5e-3)
        gi = torch.randn(3, H, W, generator=torch.Generator().manual_seed(n + 1))
        flat, views = grad_bucket(n, dev)
        plan.backward(sc, gi.to(dev), views)
        torch.cuda.synchronize()
        og = O.backward(octx, gi.numpy())
        for k in ("means3D", "means2D", "opacities", "scales", "rotations", "colors"):
            y = og[k]
            compare(case, "d_" + k, views[k].cpu().numpy().reshape(y.shape), y, gm.reshape((-1,) + (1,) * (y.ndim - 1)),
                    kind="grad", max_flagged_viol=5e-3)
