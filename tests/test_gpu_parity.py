"""Parity of the sm_100a CUDA path against the CPU oracle, through the public autograd API and the C ABI (FramePlan).

Tolerance (north_star: "within 1e-4 rel fp32"): for every output tensor, max|x - y| <= 1e-4 * max|y| over all
elements whose discrete composite decisions (alpha < 1/255, T(1-a) < 1e-4, power > 0) are not on a threshold; the
oracle marks threshold cases itself (oracle.fragility) -- those must be rare and are held to a loose bound.  For scale:
the fp32 and fp64 builds of the oracle itself agree to ~1e-5 on this metric (test_oracle_autograd.py).
Discrete outputs (radii, per-tile sorted id lists) must be identical.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from util import kat_settings, pack, splat, workload_settings
from exavatar_release_b200.synthetic import WORKLOADS, make_assets, make_grad_image
from oracle import oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def RZ():
    from exavatar_release_b200 import rasterizer
    return rasterizer


def _check(name, x, y, bad=None, tol=TOL, max_bad_frac=0.02, loose=0.05):
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    assert x.shape == y.shape, name
    if y.size == 0:
        return
    ninf = np.abs(y).max()
    d = np.abs(x - y)
    if bad is None:
        bad = np.zeros(y.shape, bool)
    viol = d > tol * ninf
    # (1) every element beyond tolerance is explained by a composite decision sitting on its threshold ...
    unexplained = viol & ~bad
    worst = d[~bad].max() if (~bad).any() else 0.0
    assert not unexplained.any(), f"{name}: max|d|={worst:.3e} vs {tol}*|y|inf={tol * ninf:.3e} ({unexplained.sum()} elements)"
    # (2) ... such elements are rare (a large splat touches thousands of pixels, so MANY Gaussians are flagged in a
    # big scene, but a single flipped pixel rarely moves their gradient by 1e-4 of the tensor norm) ...
    assert viol.mean() <= max_bad_frac * 0.05, f"{name}: {viol.mean():.5f} of elements beyond tolerance"
    # (3) ... and bounded.
    if viol.any():
        assert d[viol].max() <= loose * max(ninf, 1e-30), f"{name}: threshold element off by {d[viol].max():.3e}"


def _run_pair(dev, wl_name, yaw=12.0, seed=0, with_da=False, bg=(0.2, 0.6, 0.9), mode=None):
    rz = RZ()
    wl = WORKLOADS[wl_name]
    assets = make_assets(wl_name, seed=seed)
    st_c = workload_settings(wl_name, yaw=yaw, bg=bg)
    st_g = workload_settings(wl_name, yaw=yaw, bg=bg, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    use_sh = wl.sh_degree > 0
    if use_sh:
        st_c, st_g = st_c._replace(sh_degree=wl.sh_degree), st_g._replace(sh_degree=wl.sh_degree)
    kw_o = dict(shs=assets["shs"]) if use_sh else dict(colors_precomp=assets["rgb"])
    oc, orad, od, oa, octx = O.forward(st_c, assets["mean_3d"], assets["opacity"], scales=assets["scale"],
                                       rotations=assets["rotation"], **kw_o)
    g = {k: v.to(dev).requires_grad_() for k, v in assets.items()}
    m2 = torch.zeros(g["mean_3d"].shape[0], 3, device=dev, requires_grad=True)
    rast = rz.GaussianRasterizer(st_g)
    color, radii, depth, alpha = rast(means3D=g["mean_3d"], means2D=m2, opacities=g["opacity"],
                                      shs=g["shs"] if use_sh else None, colors_precomp=None if use_sh else g["rgb"],
                                      scales=g["scale"], rotations=g["rotation"])
    pm, gm = O.fragility(octx)
    assert np.array_equal(radii.cpu().numpy(), orad), "radii must be identical"
    _check("color", color.detach().cpu().numpy(), oc, np.broadcast_to(pm, oc.shape))
    _check("depth", depth.detach().cpu().numpy(), od, pm[None])
    _check("alpha", alpha.detach().cpu().numpy(), oa, pm[None])
    gi = make_grad_image(wl_name, seed)
    loss = (color * gi.to(dev)).sum()
    gd = ga = None
    if with_da:
        gen = torch.Generator().manual_seed(77)
        gd = torch.randn(1, wl.height, wl.width, generator=gen)
        ga = torch.randn(1, wl.height, wl.width, generator=gen)
        loss = loss + (depth * gd.to(dev)).sum() + (alpha * ga.to(dev)).sum()
    loss.backward()
    og = O.backward(octx, gi.numpy(), None if gd is None else gd.numpy()[0], None if ga is None else ga.numpy()[0])
    row = lambda a: np.broadcast_to(gm.reshape((-1,) + (1,) * (a.ndim - 1)), a.shape)
    pairs = [("means3D", g["mean_3d"].grad), ("means2D", m2.grad), ("opacities", g["opacity"].grad),
             ("scales", g["scale"].grad), ("rotations", g["rotation"].grad)]
    pairs.append(("shs", g["shs"].grad) if use_sh else ("colors", g["rgb"].grad))
    for k, t in pairs:
        y = og[k]
        if np.abs(y).max() == 0:  # e.g. rotations of an all-isotropic avatar
            assert np.abs(t.cpu().numpy()).max() <= 1e-6
            continue
        _check("d_" + k, t.cpu().numpy().reshape(y.shape), y, row(y), max_bad_frac=0.2)
    assert torch.all(m2.grad[:, 2] == 0)
    return octx, (color, radii, depth, alpha)


@pytest.mark.parametrize("wl,yaw,da", [("T0", 12.0, False), ("T1", 12.0, True), ("T1", -30.0, False), ("T2", 12.0, True),
                                       ("C1", 12.0, False), ("T3", 12.0, True), ("T4", -20.0, False)])
def test_forward_backward_parity(dev, wl, yaw, da):
    _run_pair(dev, wl, yaw=yaw, with_da=da)


def test_full_size_c2_parity(dev):
    """BASELINE configs[1]: 512x512, 100k splats; the oracle needs ~1 s for it."""
    _run_pair(dev, "C2", yaw=5.0)


def _stage_buffers(dev, wl_name, no_cull):
    """Runs the C ABI directly and returns geometry / lists for stage-level comparison."""
    from exavatar_release_b200 import _lib as L
    from exavatar_release_b200.plan import FramePlan
    rz = RZ()
    wl = WORKLOADS[wl_name]
    assets = {k: v.to(dev) for k, v in make_assets(wl_name, seed=0).items()}
    st = workload_settings(wl_name, yaw=12.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    P = assets["mean_3d"].shape[0]
    plan = FramePlan(P, wl.width, wl.height, 4_000_000, dev)
    sc = plan.scene(0, st, assets, flags=L.B2R_FLAG_NO_TILE_CULL if no_cull else 0)
    plan.forward(sc)
    torch.cuda.synchronize()
    lib = plan.lib
    buf = plan.ctx_buf.cpu().numpy()
    base = plan.ctx_buf.data_ptr()
    tiles = ((wl.width + 15) // 16) * ((wl.height + 15) // 16)
    off = lambda fn: fn(C.byref(plan.ws), P, wl.width, wl.height) - base
    geom = np.frombuffer(buf[off(lib.b2r_ctx_geom):off(lib.b2r_ctx_geom) + P * 48].tobytes(), np.float32).reshape(P, 12)
    aux = np.frombuffer(buf[off(lib.b2r_ctx_aux):off(lib.b2r_ctx_aux) + P * 16].tobytes(), np.int32).reshape(P, 4)
    ranges = np.frombuffer(buf[off(lib.b2r_ctx_ranges):off(lib.b2r_ctx_ranges) + tiles * 8].tobytes(), np.uint32).reshape(tiles, 2)
    ids = plan.ids.cpu().numpy().view(np.uint32)
    return geom, aux, ranges, ids, plan.status(), plan


def test_stage_geometry_matches_oracle(dev):
    geom, aux, ranges, ids, status, _ = _stage_buffers(dev, "T1", no_cull=True)
    assets = make_assets("T1", seed=0)
    st = workload_settings("T1", yaw=12.0)
    _, orad, _, _, ctx = O.forward(st, assets["mean_3d"], assets["opacity"], colors_precomp=assets["rgb"],
                                   scales=assets["scale"], rotations=assets["rotation"])
    vis = orad > 0
    assert np.array_equal(aux[:, 2], orad)
    assert status["num_visible"] == int(vis.sum())
    assert np.allclose(geom[vis, 0:2], ctx.xy()[vis], rtol=0, atol=2e-4)
    assert np.allclose(geom[vis, 6], ctx.depth()[vis], rtol=1e-6)
    L2E = 1.4426950408889634
    co = ctx.conic_opacity()[vis]
    assert np.allclose(geom[vis, 2] / (-0.5 * L2E), co[:, 0], rtol=2e-5, atol=1e-7)
    assert np.allclose(geom[vis, 3] / (-L2E), co[:, 1], rtol=2e-5, atol=1e-6)
    assert np.allclose(geom[vis, 4] / (-0.5 * L2E), co[:, 2], rtol=2e-5, atol=1e-7)
    rect = ctx.rect()[vis]
    assert np.array_equal(aux[vis, 0] & 0xffff, rect[:, 0]) and np.array_equal(aux[vis, 0] >> 16, rect[:, 1])
    assert np.array_equal(aux[vis, 1] & 0xffff, rect[:, 2]) and np.array_equal(aux[vis, 1] >> 16, rect[:, 3])


def test_per_tile_sorted_lists_identical_without_culling(dev):
    geom, aux, ranges, ids, status, _ = _stage_buffers(dev, "T1", no_cull=True)
    assets = make_assets("T1", seed=0)
    st = workload_settings("T1", yaw=12.0)
    *_, ctx = O.forward(st, assets["mean_3d"], assets["opacity"], colors_precomp=assets["rgb"], scales=assets["scale"],
                        rotations=assets["rotation"])
    assert status["num_dups"] == ctx.num_dups
    o_ids, o_ranges = ctx.sorted_ids(), ctx.ranges()
    for t in range(ranges.shape[0]):
        mine = ids[ranges[t, 0]:ranges[t, 1]]
        ref = o_ids[o_ranges[t, 0]:o_ranges[t, 1]]
        assert np.array_equal(mine, ref), f"tile {t}"


def test_culled_lists_are_ordered_subsets(dev):
    geom, aux, ranges, ids, status, _ = _stage_buffers(dev, "T1", no_cull=False)
    assets = make_assets("T1", seed=0)
    st = workload_settings("T1", yaw=12.0)
    *_, ctx = O.forward(st, assets["mean_3d"], assets["opacity"], colors_precomp=assets["rgb"], scales=assets["scale"],
                        rotations=assets["rotation"])
    assert status["num_dups"] < ctx.num_dups  # the exact tile test removes pairs ...
    o_ids, o_ranges = ctx.sorted_ids(), ctx.ranges()
    for t in range(ranges.shape[0]):
        mine = ids[ranges[t, 0]:ranges[t, 1]].tolist()
        ref = o_ids[o_ranges[t, 0]:o_ranges[t, 1]].tolist()
        it = iter(ref)
        assert all(m in it for m in mine), f"tile {t}: culled list is not an ordered subsequence"  # ... and only removes


@pytest.mark.parametrize("n", [3000, 20000])
def test_very_long_tile_lists(dev, n):
    """n splats stacked on a 2x2-tile patch: lists of >= 2048 entries are sorted in 2048-entry chunks and merged by rank
    (binning.cu: sort_mixed_kernel + merge_chunks_kernel; 2 chunks for n = 3000, 10 for n = 20000), and both composites
    stage many batches.  Strict tolerance (tests/parity.py); bit-exact lists for these sizes are pinned in
    test_gpu_fullsize.py::test_long_list_sort_is_bit_exact."""
    from parity import compare
    rz = RZ()
    g = torch.Generator().manual_seed(n)
    pos = torch.stack([0.12 * (torch.rand(n, generator=g) - 0.5), 0.12 * (torch.rand(n, generator=g) - 0.5),
                       2.0 + 2.0 * torch.rand(n, generator=g)], 1)
    assets = {"mean_3d": pos, "scale": 0.01 + 0.02 * torch.rand(n, 3, generator=g),
              "rotation": torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=1),
              "opacity": 0.02 + 0.05 * torch.rand(n, 1, generator=g), "rgb": torch.rand(n, 3, generator=g)}
    st_c = kat_settings(W=64, H=48, f=60.0, bg=(0.1, 0.2, 0.3))
    st_g = kat_settings(W=64, H=48, f=60.0, bg=(0.1, 0.2, 0.3), device=dev, settings_cls=rz.GaussianRasterizationSettings)
    oc, orad, od, oa, octx = O.forward(st_c, assets["mean_3d"], assets["opacity"], colors_precomp=assets["rgb"],
                                       scales=assets["scale"], rotations=assets["rotation"])
    assert (octx.ranges()[:, 1] - octx.ranges()[:, 0]).max() > 0.5 * n
    gl = {k: v.to(dev).requires_grad_() for k, v in assets.items()}
    m2 = torch.zeros(n, 3, device=dev, requires_grad=True)
    color, radii, depth, alpha = rz.GaussianRasterizer(st_g)(means3D=gl["mean_3d"], means2D=m2, opacities=gl["opacity"],
                                                            colors_precomp=gl["rgb"], scales=gl["scale"],
                                                            rotations=gl["rotation"])
    assert np.array_equal(radii.cpu().numpy(), orad)
    pm, gm = O.fragility(octx)
    case = f"longlist{n}"
    compare(case, "color", color.detach().cpu().numpy(), oc, pm[None], kind="image")
    gi = torch.randn(3, 48, 64, generator=g)
    (color * gi.to(dev)).sum().backward()
    og = O.backward(octx, gi.numpy())
    for k, t in (("means3D", gl["mean_3d"].grad), ("colors", gl["rgb"].grad), ("opacities", gl["opacity"].grad),
                 ("scales", gl["scale"].grad), ("means2D", m2.grad)):
        y = og[k]
        compare(case, "d_" + k, t.cpu().numpy().reshape(y.shape), y, gm.reshape((-1,) + (1,) * (y.ndim - 1)),
                kind="grad", max_flagged_viol=5e-3)


def test_kats_on_gpu(dev):
    rz = RZ()
    st = kat_settings(device=dev, settings_cls=rz.GaussianRasterizationSettings, bg=(0.25, 0.5, 0.75))
    run = lambda sp: rz.GaussianRasterizer(st)(means2D=torch.zeros(len(sp), 3, device=dev),
                                               **{k: v for k, v in pack(sp, device=dev).items()})
    c, r, d, a = run([splat((0, 0, 2.0))])  # KAT 1/2
    assert r.tolist() == [6]
    assert float(a[0, 15, 15]) == pytest.approx(0.458149, rel=1e-5)
    assert float(d[0, 15, 15]) == pytest.approx(0.916299, rel=1e-5)
    assert float(c[0, 15, 15]) == pytest.approx(0.458149 + (1 - 0.458149) * 0.25, rel=1e-5)
    # KAT 4: three coincident opacity-1 splats centred on pixel (16,16): stop after the first, second not applied
    sp = [splat((0.03125, 0.03125, 2.0 + 0.1 * i), o=1.0, rgb=col) for i, col in enumerate([(1, 0, 0), (0, 1, 0), (0, 0, 1)])]
    c, r, d, a = run(sp)
    assert float(a[0, 16, 16]) == pytest.approx(0.99, rel=1e-6)
    assert float(c[1, 16, 16]) == pytest.approx(0.01 * 0.5, rel=1e-4)
    # KAT 6: near plane
    c, r, d, a = run([splat((0, 0, 0.2)), splat((0, 0, 0.2001))])
    assert r[0] == 0 and r[1] > 0
    rast = rz.GaussianRasterizer(st)
    assert rast.markVisible(torch.tensor([[0, 0, 0.2], [0, 0, 0.2001]], device=dev)).tolist() == [False, True]
    # KAT 5: equal depth -> lower index in front
    c, *_ = run([splat((0, 0, 2.0), o=0.9, rgb=(1, 0, 0)), splat((0, 0, 2.0), o=0.9, rgb=(0, 0, 1))])
    assert float(c[0, 15, 15]) > float(c[2, 15, 15])


def test_cov3d_precomp_path(dev):
    rz = RZ()
    assets = make_assets("T0", seed=2)
    P = assets["mean_3d"].shape[0]
    g = torch.Generator().manual_seed(5)
    A = torch.randn(P, 3, 3, generator=g) * 0.05
    S = A @ A.transpose(1, 2) + 1e-4 * torch.eye(3)
    cov = torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1)
    st_c = workload_settings("T0", yaw=7.0)
    st_g = workload_settings("T0", yaw=7.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    oc, orad, od, oa, octx = O.forward(st_c, assets["mean_3d"], assets["opacity"], colors_precomp=assets["rgb"], cov3D_precomp=cov)
    cg = cov.to(dev).requires_grad_()
    m3 = assets["mean_3d"].to(dev).requires_grad_()
    color, radii, depth, alpha = rz.GaussianRasterizer(st_g)(
        means3D=m3, means2D=torch.zeros(P, 3, device=dev), opacities=assets["opacity"].to(dev),
        colors_precomp=assets["rgb"].to(dev), cov3D_precomp=cg)
    assert np.array_equal(radii.cpu().numpy(), orad)
    gi = make_grad_image("T0", 2)
    (color * gi.to(dev)).sum().backward()
    og = O.backward(octx, gi.numpy())
    pm, gm = O.fragility(octx)
    _check("color", color.detach().cpu().numpy(), oc, np.broadcast_to(pm, oc.shape))
    _check("d_cov3D", cg.grad.cpu().numpy(), og["cov3D"], np.broadcast_to(gm[:, None], og["cov3D"].shape), max_bad_frac=0.2)
    _check("d_means3D", m3.grad.cpu().numpy(), og["means3D"], np.broadcast_to(gm[:, None], og["means3D"].shape), max_bad_frac=0.2)


@pytest.mark.parametrize("case", ["rgb", "sh", "cov", "depth_alpha_only", "noncontiguous", "odd_size"])
def test_compiled_binding_equals_python_route(dev, monkeypatch, case):
    """The C++ autograd Function (csrc_torch/b2r_torch.cpp) and the Python one (_RasterizeGaussians) are two hosts of the
    same kernels: identical forward outputs bit for bit, gradients equal up to the order of the backward's atomic sums,
    None exactly where the other route returns None.  "odd_size": 101x77 (T3), scalar output stores and cut-off tiles."""
    rz = RZ()
    assert rz._compiled_binding(), "the compiled binding (_b2r_torch.so) must be built: python -m exavatar_release_b200.build_ext"
    wl = {"sh": "T2", "odd_size": "T3"}.get(case, "T1")
    st = workload_settings(wl, yaw=9.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    if case == "sh":
        st = st._replace(sh_degree=3)
    if case == "noncontiguous":  # module.py:605-606 hands over transposed views
        st = st._replace(viewmatrix=st.viewmatrix.t().contiguous().t(), projmatrix=st.projmatrix.t().contiguous().t())
        assert not st.viewmatrix.is_contiguous()
    a0 = make_assets(wl, seed=3)
    P = a0["mean_3d"].shape[0]
    if case == "cov":
        g = torch.Generator().manual_seed(5)
        A = torch.randn(P, 3, 3, generator=g) * 0.05
        S = A @ A.transpose(1, 2) + 1e-4 * torch.eye(3)
        a0 = dict(a0, cov=torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1))
    gi = make_grad_image(wl, 4).to(dev)

    def run(compiled):
        monkeypatch.setattr(rz, "_COMPILED", rz._compiled_binding() if compiled else False)
        a = {k: v.to(dev).requires_grad_() for k, v in a0.items()}
        m2 = torch.zeros(P, 3, device=dev, requires_grad=True)
        kw = dict(means3D=a["mean_3d"], means2D=m2, opacities=a["opacity"])
        if case == "sh":
            kw.update(shs=a["shs"], scales=a["scale"], rotations=a["rotation"])
        elif case == "cov":
            kw.update(colors_precomp=a["rgb"], cov3D_precomp=a["cov"])
        else:
            kw.update(colors_precomp=a["rgb"], scales=a["scale"], rotations=a["rotation"])
        out = rz.GaussianRasterizer(st)(**kw)
        color, radii, depth, alpha = out
        if case == "depth_alpha_only":
            loss = (depth * gi[:1]).sum() + (alpha * gi[1:2]).sum()
        elif case in ("rgb", "odd_size"):
            loss = (color * gi).sum() + 0.3 * (depth * gi[:1]).sum()
        else:
            loss = (color * gi).sum()
        loss.backward()
        return [t.detach() for t in out], {k: v.grad for k, v in a.items()}, m2.grad

    o_c, g_c, m_c = run(True)
    o_p, g_p, m_p = run(False)
    for x, y in zip(o_c, o_p):
        assert torch.equal(x, y)
    close = lambda x, y: torch.allclose(x, y, rtol=1e-4, atol=1e-5 * float(y.abs().max()) + 1e-12)
    for k in g_p:
        assert (g_c[k] is None) == (g_p[k] is None), k
        if g_p[k] is not None:
            assert g_c[k].shape == g_p[k].shape and close(g_c[k], g_p[k]), k
    assert close(m_c, m_p)


def test_compiled_binding_handles_an_empty_call(dev):
    rz = RZ()
    assert rz._compiled_binding()
    st = workload_settings("T0", yaw=0.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    z = lambda *s: torch.zeros(*s, device=dev, requires_grad=True)
    m3, op = z(0, 3), z(0, 1)
    color, radii, depth, alpha = rz.GaussianRasterizer(st)(means3D=m3, means2D=z(0, 3), opacities=op, colors_precomp=z(0, 3),
                                                           scales=z(0, 3), rotations=z(0, 4))
    assert float(color.abs().max()) == 0.0 and radii.numel() == 0
    color.sum().backward()
    assert m3.grad.shape == (0, 3) and op.grad.shape == (0, 1)


def test_five_live_contexts_then_one_backward(dev):
    """ExAvatar renders five asset sets before the single loss.backward() (model.py:130-162, train.py:46)."""
    rz = RZ()
    st = workload_settings("T1", yaw=3.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    losses, leaves = [], []
    for s in range(5):
        a = {k: v.to(dev).requires_grad_() for k, v in make_assets("T1", seed=20 + s).items()}
        m2 = torch.zeros(a["mean_3d"].shape[0], 3, device=dev, requires_grad=True)
        img = rz.GaussianRasterizer(st)(means3D=a["mean_3d"], means2D=m2, opacities=a["opacity"], colors_precomp=a["rgb"],
                                        scales=a["scale"], rotations=a["rotation"])[0]
        losses.append((img * make_grad_image("T1", s).to(dev)).sum())
        leaves.append((a, m2))
    sum(losses).backward()
    for s, (a, m2) in enumerate(leaves):
        b = {k: v.detach().clone().requires_grad_() for k, v in a.items()}
        m2b = torch.zeros_like(m2, requires_grad=True)
        img = rz.GaussianRasterizer(st)(means3D=b["mean_3d"], means2D=m2b, opacities=b["opacity"], colors_precomp=b["rgb"],
                                        scales=b["scale"], rotations=b["rotation"])[0]
        (img * make_grad_image("T1", s).to(dev)).sum().backward()
        for k in a:
            assert torch.allclose(a[k].grad, b[k].grad, rtol=1e-4, atol=1e-4 * float(b[k].grad.abs().max())), (s, k)
        assert torch.allclose(m2.grad, m2b.grad, rtol=1e-4, atol=1e-4 * float(m2b.grad.abs().max()))


@pytest.mark.parametrize("route", ["compiled", "python"])
def test_forward_is_deterministic_and_capacity_modes_agree(dev, monkeypatch, route):
    rz = RZ()
    if route == "python":
        monkeypatch.setattr(rz, "_COMPILED", False)
    else:
        assert rz._compiled_binding(), "the compiled binding (_b2r_torch.so) must be built: python -m exavatar_release_b200.build_ext"
    st = workload_settings("T1", yaw=12.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=0).items()}
    P = a["mean_3d"].shape[0]

    def render():
        return rz.GaussianRasterizer(st)(means3D=a["mean_3d"], means2D=torch.zeros(P, 3, device=dev), opacities=a["opacity"],
                                         colors_precomp=a["rgb"], scales=a["scale"], rotations=a["rotation"])

    monkeypatch.setattr(rz, "CAPACITY_MODE", "exact")
    ref = render()
    again = render()
    for x, y in zip(ref, again):
        assert torch.equal(x, y)  # sort key (depth, id) makes the pipeline independent of atomic arrival order
    monkeypatch.setattr(rz, "CAPACITY_MODE", "speculative")
    spec = render()
    for x, y in zip(ref, spec):
        assert torch.equal(x, y)
    # a misprediction (capacity far too small) must be repaired transparently
    rz._state(dev).predicted[(P, st.image_width, st.image_height)] = 10
    if route == "compiled":
        rz._compiled_binding().set_predicted(dev.index, P, st.image_width, st.image_height, 10)
    monkeypatch.setattr(rz, "CAPACITY_HEADROOM", 1.0)
    small = render()
    for x, y in zip(ref, small):
        assert torch.equal(x, y)


def test_properties_at_full_size(dev):
    """Size-independent properties on BASELINE configs[1] (C2)."""
    rz = RZ()
    wl = WORKLOADS["C2"]
    a = {k: v.to(dev) for k, v in make_assets("C2", seed=1).items()}
    P = a["mean_3d"].shape[0]
    bg1, bg2 = (0.0, 0.0, 0.0), (1.0, 0.5, 0.25)

    def render(assets, bg, perm=None):
        st = workload_settings("C2", yaw=-9.0, bg=bg, device=dev, settings_cls=rz.GaussianRasterizationSettings)
        if perm is not None:
            assets = {k: v[perm] for k, v in assets.items()}
        return rz.GaussianRasterizer(st)(means3D=assets["mean_3d"], means2D=torch.zeros(P, 3, device=dev),
                                         opacities=assets["opacity"], colors_precomp=assets["rgb"], scales=assets["scale"],
                                         rotations=assets["rotation"])

    c1, r1, d1, a1 = render(a, bg1)
    c2, r2, d2, a2 = render(a, bg2)
    # background enters linearly through the final transmittance only: c2 - c1 = T * (bg2 - bg1), depth/alpha untouched
    T = (c2[0] - c1[0])
    assert torch.equal(d1, d2) and torch.equal(a1, a2) and torch.equal(r1, r2)
    assert torch.allclose(c2[1] - c1[1], 0.5 * T, atol=2e-6) and torch.allclose(c2[2] - c1[2], 0.25 * T, atol=2e-6)
    assert torch.allclose(T, 1 - a1[0], atol=2e-5)  # alpha = sum alpha_i T_i = 1 - T_final
    assert float(T.min()) >= 0 and float(a1.max()) <= 1 + 1e-5
    # permutation of the input order: radii permute; the image can only change where two splats share a view depth
    # bit for bit (index tie-break, App. A.2) -- a handful of pairs among 1e5 fp32 depths
    perm = torch.randperm(P, generator=torch.Generator().manual_seed(3)).to(dev)
    cp, rp, dp, ap = render(a, bg1, perm)
    assert torch.equal(rp, r1[perm])
    assert float((cp != c1).float().mean()) < 1e-3 and torch.allclose(cp, c1, atol=2e-2)
    assert torch.allclose(dp, d1, atol=0.2)
    # zero-opacity Gaussians are a no-op
    extra = {k: torch.cat([v, v[:1000]]) for k, v in a.items()}
    extra["opacity"][-1000:] = 0.0
    st = workload_settings("C2", yaw=-9.0, bg=bg1, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    ce = rz.GaussianRasterizer(st)(means3D=extra["mean_3d"], means2D=torch.zeros(P + 1000, 3, device=dev),
                                   opacities=extra["opacity"], colors_precomp=extra["rgb"], scales=extra["scale"],
                                   rotations=extra["rotation"])[0]
    assert torch.equal(ce, c1)


def test_accumulate_mode_sums_frames(dev):
    """B2R_BWD_ACCUMULATE: two frames summed in place == sum of two separate backward passes."""
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    rz = RZ()
    wl = WORKLOADS["T1"]
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=0).items()}
    P = a["mean_3d"].shape[0]
    plan = FramePlan(P, wl.width, wl.height, 1_000_000, dev)
    sts = [workload_settings("T1", yaw=y, device=dev, settings_cls=rz.GaussianRasterizationSettings) for y in (-10.0, 10.0)]
    gis = [make_grad_image("T1", s).to(dev) for s in (0, 1)]
    scenes = [plan.scene(i, sts[i], a) for i in range(2)]
    flat_acc, v_acc = grad_bucket(P, dev)
    sep = []
    for i in range(2):
        plan.forward(scenes[i])
        plan.backward(scenes[i], gis[i], v_acc, accumulate=(i > 0))
        flat_i, v_i = grad_bucket(P, dev)
        plan.backward(scenes[i], gis[i], v_i, accumulate=False)
        sep.append(flat_i)
    torch.cuda.synchronize()
    ref = sep[0] + sep[1]
    assert torch.allclose(flat_acc, ref, rtol=1e-4, atol=1e-5 * float(ref.abs().max()))
    assert plan.status()["overflow"] == 0


def test_split_entry_points_agree_with_the_one_call_forward(dev):
    """b2r_forward == count-only b2r_forward_project + b2r_forward_render == b2r_forward_project (with the capacity) +
    b2r_forward_render == ... + b2r_forward_bin + b2r_forward_composite(view = NULL); also with a clean-flagged ctx."""
    import ctypes as C
    from exavatar_release_b200 import _lib as L
    from exavatar_release_b200.plan import FramePlan
    rz = RZ()
    wl = WORKLOADS["T1"]
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=3).items()}
    P = a["mean_3d"].shape[0]
    st = workload_settings("T1", yaw=-5.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    plan = FramePlan(P, wl.width, wl.height, 1_000_000, dev)
    sc = plan.scene(0, st, a)
    lib, sp = plan.lib, torch.cuda.current_stream(dev).cuda_stream
    plan.forward(sc)
    torch.cuda.synchronize()
    ref = (plan.color.clone(), plan.depth.clone(), plan.alpha.clone(), plan.radii.clone())
    ref_ids = plan.ids.clone()

    def check(tag):
        torch.cuda.synchronize()
        assert plan.status()["overflow"] == 0, tag
        for x, y in zip((plan.color, plan.depth, plan.alpha, plan.radii), ref):
            assert torch.equal(x, y), tag
        n = plan.status()["num_dups"]
        assert torch.equal(plan.ids[:n], ref_ids[:n]), tag

    for flags in (0, L.B2R_FLAG_CTX_CLEAN):  # every sequence below leaves the counters clean again
        sc.flags = flags
        plan.color.zero_()
        ws0 = L.B2RWorkspace(plan.ctx_buf.data_ptr(), plan.ctx_bytes, None, 0, None, 0, None, 0, None, 0)
        L.check(lib.b2r_forward_project(C.byref(sc), C.byref(ws0), plan.radii.data_ptr(), sp), "project(count only)")
        L.check(lib.b2r_forward_render(C.byref(sc), C.byref(plan.ws), C.byref(plan.out), sp), "render")
        check(f"count-only project + render, flags {flags}")
        sc.flags = L.B2R_FLAG_CTX_CLEAN
        plan.color.zero_()
        L.check(lib.b2r_forward_project(C.byref(sc), C.byref(plan.ws), plan.radii.data_ptr(), sp), "project(capacity)")
        L.check(lib.b2r_forward_render(C.byref(sc), C.byref(plan.ws), C.byref(plan.out), sp), "render")
        check("project with capacity + render")
        plan.color.zero_()
        L.check(lib.b2r_forward_project(C.byref(sc), C.byref(plan.ws), plan.radii.data_ptr(), sp), "project(capacity)")
        L.check(lib.b2r_forward_bin(C.byref(sc), C.byref(plan.ws), sp), "bin")
        L.check(lib.b2r_forward_composite(C.byref(sc), C.byref(plan.ws), None, C.byref(plan.out), sp), "composite")
        check("project + bin + composite")
    sc.flags = 0


def test_cuda_graph_replay_matches_eager(dev):
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    rz = RZ()
    wl = WORKLOADS["T1"]
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=0).items()}
    P = a["mean_3d"].shape[0]
    plan = FramePlan(P, wl.width, wl.height, 1_000_000, dev)
    st = workload_settings("T1", yaw=4.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    gi = make_grad_image("T1", 0).to(dev)
    sc = plan.scene(0, st, a)
    flat, views = grad_bucket(P, dev)

    def body():
        plan.forward(sc)
        plan.backward(sc, gi, views)

    body()
    torch.cuda.synchronize()
    eager_img, eager_grad = plan.color.clone(), flat.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body()
    plan.color.zero_()
    flat.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(plan.color, eager_img)
    assert torch.allclose(flat, eager_grad, rtol=1e-4, atol=1e-5 * float(eager_grad.abs().max()))


def test_frame_lanes_match_serial_accumulation(dev):
    """FrameLanes (frames in flight on S streams, per-lane buckets, fixed-order sum) == one plan run serially; also
    inside a CUDA graph capture (the lanes fork from / join into the capturing stream)."""
    from exavatar_release_b200.plan import FrameLanes, FramePlan, grad_bucket
    rz = RZ()
    wl = WORKLOADS["T1"]
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=0).items()}
    P = a["mean_3d"].shape[0]
    yaws = (-15.0, -5.0, 0.0, 7.0, 14.0)
    sts = [workload_settings("T1", yaw=y, device=dev, settings_cls=rz.GaussianRasterizationSettings) for y in yaws]
    gis = [make_grad_image("T1", s).to(dev) for s in range(len(yaws))]
    plan = FramePlan(P, wl.width, wl.height, 1_000_000, dev)
    scenes = [plan.scene(i, sts[i], a) for i in range(len(yaws))]
    flat, views = grad_bucket(P, dev)
    for i, sc in enumerate(scenes):
        plan.forward(sc)
        plan.backward(sc, gis[i], views, accumulate=(i > 0))
    torch.cuda.synchronize()
    tol = dict(rtol=1e-4, atol=2e-6 * float(flat.abs().max()))
    for S in (1, 2, 3, 8):
        lanes = FrameLanes(S, P, wl.width, wl.height, 1_000_000, dev)
        lanes.step(scenes, gis)
        torch.cuda.synchronize()
        assert torch.allclose(lanes.bucket, flat, **tol), S
        assert lanes.status()["overflow"] == 0
    lanes = FrameLanes(3, P, wl.width, wl.height, 1_000_000, dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        lanes.step(scenes, gis)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        lanes.step(scenes, gis)
    lanes.bucket.zero_()
    lanes.lane_flat.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.allclose(lanes.bucket, flat, **tol)


def test_unused_outputs_get_no_materialised_gradients(dev):
    """A loss on depth alone (colour / alpha unused) == explicit zero colour gradient; a loss on colour alone takes the
    kernel variant without depth / alpha gradients (autograd hands the node None for unused outputs)."""
    rz = RZ()
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=0).items()}
    st = workload_settings("T1", yaw=3.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)
    P = a["mean_3d"].shape[0]

    def run(loss_fn):
        lv = {k: v.clone().requires_grad_() for k, v in a.items()}
        m2 = torch.zeros(P, 3, device=dev, requires_grad=True)
        out = rz.GaussianRasterizer(st)(means3D=lv["mean_3d"], means2D=m2, opacities=lv["opacity"],
                                        colors_precomp=lv["rgb"], scales=lv["scale"], rotations=lv["rotation"])
        loss_fn(out).backward()
        return lv, m2

    gd = make_grad_image("T1", 1).to(dev)[:1]
    lv1, m1 = run(lambda o: (o[2] * gd).sum())
    lv2, m2_ = run(lambda o: (o[2] * gd).sum() + (o[0] * 0.0).sum() + (o[3] * 0.0).sum())
    # the two runs differ only in the arrival order of the fp32 vector reductions
    close = lambda x, y: torch.allclose(x, y, rtol=1e-4, atol=1e-5 * float(y.abs().max()) + 1e-12)
    for k in lv1:
        assert close(lv1[k].grad, lv2[k].grad), k
    assert close(m1.grad, m2_.grad)
    assert float(lv1["mean_3d"].grad.abs().sum()) > 0
    assert float(lv1["rgb"].grad.abs().max()) == 0.0


@pytest.mark.parametrize("engine,wl_name", [("merged", "T1"), ("separate", "T1"), ("merged", "T3"), ("separate", "T3")],
                         ids=["merged", "separate", "T3-merged", "T3-separate"])
def test_five_render_plan_matches_the_reference_pattern(dev, engine, wl_name):
    """FiveRenderPlan (five concurrent renders, detached scene prefix via `first_row`) and MergedFivePlan (two merged
    projection / binning passes, five views; SURVEY 8f-3) == ExAvatar's pattern written
    with the public autograd API: renderer(scene), renderer(human, bg), renderer(cat(scene.detach(), human)), and the
    same two for the refined human (avatar/main/model.py:81-162), two frames accumulated; at 128x96 (T1) and at
    101x77 (T3: cut-off tiles, scalar stores, views pre-filled and composited over partial tiles)."""
    from exavatar_release_b200 import GaussianRenderer
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS, FiveRenderPlan, MergedFivePlan
    from exavatar_release_b200.renderer import render_settings
    from exavatar_release_b200.synthetic import make_population_assets
    rz = RZ()
    wl = WORKLOADS[wl_name]
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets(wl_name, seed=0, device=dev)
    Ps, Ph = scene["mean_3d"].shape[0], human["mean_3d"].shape[0]
    bg_w, bg_r = torch.ones(3, device=dev), torch.tensor([0.3, 0.7, 0.2], device=dev)
    yaws = (-8.0, 11.0)
    cams = [look_at_cam_param(y, (H, W), device=dev) for y in yaws]
    gcol = [{r: make_grad_image(wl_name, 10 * f + j).to(dev) for j, r in enumerate(RENDERS)} for f in range(len(yaws))]

    # reference pattern through the public API
    lv = {n: {k: v.clone().requires_grad_() for k, v in a.items()} for n, a in (("scene", scene), ("human", human), ("refined", refined))}
    R = GaussianRenderer()
    cat = lambda a, b: {k: torch.cat((a[k].detach(), b[k])) for k in a}
    loss = 0.0
    for f, cam in enumerate(cams):
        imgs = {"scene": R(lv["scene"], (H, W), cam)["img"], "human": R(lv["human"], (H, W), cam, bg_r)["img"],
                "scene_human": R(cat(lv["scene"], lv["human"]), (H, W), cam)["img"],
                "human_refined": R(lv["refined"], (H, W), cam, bg_r)["img"],
                "scene_human_refined": R(cat(lv["scene"], lv["refined"]), (H, W), cam)["img"]}
        loss = loss + sum((imgs[r] * gcol[f][r]).sum() for r in RENDERS)
    loss.backward()

    plan = (MergedFivePlan if engine == "merged" else FiveRenderPlan)(Ps, Ph, W, H, None, dev)
    plan.set_scene(scene)
    for f, cam in enumerate(cams):
        st_w = render_settings((H, W), cam, bg_w)
        st_r = render_settings((H, W), cam, bg_r)
        plan.frame(f, st_w, st_r, scene, human, refined, gcol[f], accumulate=(f > 0))
    torch.cuda.synchronize()
    assert not plan.overflowed()
    names = {"mean_3d": "means3D", "opacity": "opacities", "scale": "scales", "rotation": "rotations", "rgb": "colors"}
    plan.reduce()
    for which, leaves, P in zip(("scene", "human", "human_refined"), (lv["scene"], lv["human"], lv["refined"]), (Ps, Ph, Ph)):
        views = plan.grads(which)
        for k, n in names.items():
            ref = leaves[k].grad.reshape(P, -1)
            assert torch.allclose(views[n], ref, rtol=1e-4, atol=1e-5 * float(ref.abs().max()) + 1e-12), (k, P)
    assert float(lv["scene"]["mean_3d"].grad.abs().sum()) > 0 and float(lv["refined"]["rgb"].grad.abs().sum()) > 0


@pytest.mark.parametrize("use_graph,wl_name", [(False, "T1"), (True, "T1"), (False, "T3"), (True, "T3")],
                         ids=["False", "True", "T3-False", "T3-True"])
def test_training_frame_renderer_equals_five_renderer_calls(dev, use_graph, wl_name):
    """`TrainingFrameRenderer` (one autograd call, two merged passes) against the reference's five `GaussianRenderer`
    calls written with the drop-in rasteriser (avatar/main/model.py:117-162): images, masks, radii, and the gradients
    `loss.backward()` leaves in the three asset dicts and in the scene render's mean_2d; a render left out of the loss
    gets no backward launch (eager) or a zero dL/dimage (use_graph: the frame replays two captured CUDA graphs, three
    frames so that the third is a pure replay with a new camera).  At 128x96 (T1) and at 101x77 (T3)."""
    from exavatar_release_b200 import GaussianRenderer, TrainingFrameRenderer
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS
    from exavatar_release_b200.synthetic import make_population_assets
    wl = WORKLOADS[wl_name]
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets(wl_name, seed=0, device=dev)
    Ps, Ph = scene["mean_3d"].shape[0], human["mean_3d"].shape[0]
    bg_r = torch.tensor([0.3, 0.7, 0.2], device=dev)
    gcol = {r: make_grad_image(wl_name, 50 + j).to(dev) for j, r in enumerate(RENDERS)}
    gmask = make_grad_image(wl_name, 60).to(dev)[:1]
    used = ("scene", "human", "scene_human", "scene_human_refined")  # human_refined stays out of the loss
    mk = lambda: {n: {k: v.clone().requires_grad_() for k, v in a.items()} for n, a in
                  (("scene", scene), ("human", human), ("refined", refined))}
    frame = TrainingFrameRenderer(Ps, Ph, (H, W), dev, {"A": 2_000_000, "B": 2_000_000}, use_graph=use_graph,
                                  graph_depth_alpha=use_graph)
    for yaw in (-9.0, 6.0, 14.0):  # three frames through the same instance
        cam = look_at_cam_param(yaw, (H, W), device=dev)
        a = mk()
        R = GaussianRenderer()
        cat = lambda x, y: {k: torch.cat((x[k].detach(), y[k])) for k in x}
        ref = {"scene": R(a["scene"], (H, W), cam), "human": R(a["human"], (H, W), cam, bg_r),
               "scene_human": R(cat(a["scene"], a["human"]), (H, W), cam), "human_refined": R(a["refined"], (H, W), cam, bg_r),
               "scene_human_refined": R(cat(a["scene"], a["refined"]), (H, W), cam)}
        (sum((ref[r]["img"] * gcol[r]).sum() for r in used) + (ref["human"]["mask"] * gmask).sum()).backward()
        b = mk()
        out = frame(b["scene"], b["human"], b["refined"], cam, bg_r)
        (sum((out[r]["img"] * gcol[r]).sum() for r in used) + (out["human"]["mask"] * gmask).sum()).backward()
        torch.cuda.synchronize()
        assert not frame.overflowed()
        for r in RENDERS:
            assert torch.equal(out[r]["radius"], ref[r]["radius"]) and torch.equal(out[r]["is_vis"], ref[r]["is_vis"]), r
            assert torch.allclose(out[r]["img"], ref[r]["img"], atol=2e-6), r
            assert torch.allclose(out[r]["mask"], ref[r]["mask"], atol=2e-6) and torch.allclose(out[r]["depthmap"], ref[r]["depthmap"], atol=2e-5), r
        close = lambda x, y: torch.allclose(x, y, rtol=1e-4, atol=1e-5 * float(y.abs().max()) + 1e-12)
        for n in ("scene", "human", "refined"):
            for k in a[n]:
                if n == "refined" and False:
                    continue
                assert b[n][k].grad is not None and close(b[n][k].grad, a[n][k].grad), (n, k)
        assert close(out["scene"]["mean_2d"].grad, ref["scene"]["mean_2d"].grad)
        assert float(a["refined"]["rgb"].grad.abs().sum()) > 0 and float(a["scene"]["mean_3d"].grad.abs().sum()) > 0


@pytest.mark.parametrize("deg,M", [(1, 4), (2, 9), (1, 16)])
def test_sh_rows_of_any_width_are_staged_correctly(dev, deg, M):
    """K1 / K6 move SH rows through shared memory; (P,16,3) takes the 128-bit path, every other coefficient count the
    generic one.  GPU vs oracle for narrower rows, in write and in accumulate mode (two identical frames = 2x)."""
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    rz = RZ()
    wl = WORKLOADS["T2"]
    a = make_assets("T2", seed=0)
    shs = a["shs"][:, :M, :].contiguous()
    st_c = workload_settings("T2", yaw=5.0)._replace(sh_degree=deg)
    st_g = workload_settings("T2", yaw=5.0, device=dev, settings_cls=rz.GaussianRasterizationSettings)._replace(sh_degree=deg)
    oc, orad, _, _, octx = O.forward(st_c, a["mean_3d"], a["opacity"], shs=shs, scales=a["scale"], rotations=a["rotation"])
    gi = make_grad_image("T2", 0)
    og = O.backward(octx, gi.numpy())
    pm, gm = O.fragility(octx)
    P = shs.shape[0]
    assets = {k: v.to(dev) for k, v in a.items()}
    assets["shs"] = shs.to(dev)
    plan = FramePlan(P, wl.width, wl.height, 2_000_000, dev, sh_coeffs=M)
    sc = plan.scene(0, st_g, assets)
    flat, views = grad_bucket(P, dev, M)
    for rep in range(2):
        plan.forward(sc)
        plan.backward(sc, gi.to(dev), views, accumulate=(rep > 0))
        torch.cuda.synchronize()
        assert np.array_equal(plan.radii.cpu().numpy(), orad)
        _check("color", plan.color.cpu().numpy(), oc, np.broadcast_to(pm, oc.shape))
        y = og["shs"] * (rep + 1)
        row = np.broadcast_to(gm.reshape(-1, 1, 1), y.shape)
        _check("d_shs", views["shs"].cpu().numpy(), y, row, max_bad_frac=0.2)
        y3 = og["means3D"] * (rep + 1)
        _check("d_means3D", views["means3D"].cpu().numpy(), y3, np.broadcast_to(gm[:, None], y3.shape), max_bad_frac=0.2)
    if M > (deg + 1) ** 2:  # coefficients above the active degree receive exactly zero
        assert float(views["shs"][:, (deg + 1) ** 2:, :].abs().max()) == 0.0


def test_renderer_end_to_end_on_gpu(dev):
    from exavatar_release_b200 import GaussianRenderer
    from exavatar_release_b200.camera import look_at_cam_param
    a = {k: v.to(dev).requires_grad_() for k, v in make_assets("T1", seed=0).items() }
    out = GaussianRenderer()(a, (96, 128), look_at_cam_param(0.0, (96, 128), device=dev), torch.ones(3, device=dev))
    P = a["mean_3d"].shape[0]
    assert out["img"].shape == (3, 96, 128) and out["radius"].shape == (P,) and out["is_vis"].dtype == torch.bool
    out["img"].mean().backward()
    assert out["mean_2d"].grad.shape == (P, 3) and float(out["mean_2d"].grad.abs().sum()) > 0


def test_fused_densification_stats_match_reference_bookkeeping(dev):
    """SURVEY 8f-1: K6 updates xyz_grad_accum / track_cnt / radius_max exactly as module.py:155-157 + model.py:283-285."""
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    rz = RZ()
    wl = WORKLOADS["T1"]
    a = {k: v.to(dev) for k, v in make_assets("T1", seed=0).items()}
    P = a["mean_3d"].shape[0]
    plan = FramePlan(P, wl.width, wl.height, 1_000_000, dev)
    fused = {"grad_accum": torch.zeros(P, device=dev), "count": torch.zeros(P, device=dev),
             "radius_max": torch.zeros(P, device=dev)}
    ref_accum, ref_cnt, ref_rmax = torch.zeros(P, 1, device=dev), torch.zeros(P, 1, device=dev), torch.zeros(P, device=dev)
    for i, yaw in enumerate((-12.0, 0.0, 14.0)):
        st = workload_settings("T1", yaw=yaw, device=dev, settings_cls=rz.GaussianRasterizationSettings)
        sc = plan.scene(i, st, a)
        flat, views = grad_bucket(P, dev)
        plan.forward(sc)
        plan.backward(sc, make_grad_image("T1", i).to(dev), views, densify=fused)
        torch.cuda.synchronize()
        # the reference's own statements, on the tensors the rasteriser returned
        is_vis = plan.radii > 0
        ref_rmax[is_vis] = torch.maximum(ref_rmax[is_vis], plan.radii[is_vis].float())
        ref_accum[is_vis, :] += torch.norm(views["means2D"][is_vis, :2], dim=1, keepdim=True)
        ref_cnt[is_vis, :] += 1
    assert torch.equal(fused["count"], ref_cnt[:, 0]) and torch.equal(fused["radius_max"], ref_rmax)
    assert torch.allclose(fused["grad_accum"], ref_accum[:, 0], rtol=1e-5, atol=1e-6 * float(ref_accum.max()))
    assert float(fused["count"].max()) == 3.0 and float(fused["grad_accum"].max()) > 0
