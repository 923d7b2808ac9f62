"""The rasteriser at its shape boundaries, against the CPU oracle.

The kernels branch on shape in places the workload-shaped tests never reach:
  (a) list-length classes of the per-tile sort (`sort_mixed_kernel`: register rank sort up to 32 entries, warp sort
      with cached peer masks up to 256, warp sort up to 511, one-CTA sort up to 2047, 2048-entry chunks +
      `merge_chunks_kernel` from 2048 on, whose "all 2048 entries below" case needs 4096+), the composites' batches and
      512-entry checkpoint cuts, and runs of bit-identical depths (ExAvatar's clone densification copies `mean`
      exactly), down to a whole list at one depth, where every digit pass is skipped and only the tie fix-up orders it;
  (b) more than 1024 tiles in a class (second pass of `scan_units`, global-memory chunk table of the merge);
  (c) partial tiles and odd image sizes through the C ABI, with guard words around every output plane, the scalar
      store path forced by a misaligned colour pointer, and a segmented list in a partial tile;
  (d) the exact tile cull from the other side: every (tile, Gaussian) pair the GPU drops is empty, i.e. its alpha is
      below 1/255 at every pixel centre of the tile inside the image (evaluated in fp64);
  (e) the densification statistics of `MergedFivePlan` against ExAvatar's bookkeeping on the scene render.
The generator checks at the end need no GPU: they run the oracle alone and pin what the GPU tests claim to reach.
"""
import functools

import numpy as np
import pytest
import torch

from parity import TOL, compare, contributor_report, last_contributor
from util import ctx_arrays, kat_settings, settings_on, workload_settings
from exavatar_release_b200.synthetic import WORKLOADS, Workload, make_assets, make_grad_image, make_population_assets
from oracle import oracle as O

gpu = pytest.mark.gpu

TILE = 16
SEG = 512  # entries per checkpoint segment of the composites
ALPHA_MIN = 1.0 / 255.0
F = 100.0  # focal length (px) of the stacked-tile scenes
GRADS = ("means3D", "means2D", "opacities", "scales", "rotations", "colors")

# (a): one tile per list length, on both sides of every class boundary of the sort ...
LENGTHS = (1, 2, 31, 32, 33, 64, 65, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096, 4097,
           6145)
# ... plus whole lists at one depth in the register, warp, CTA and chunked classes
FLAT = (20, 100, 600, 2500)
FLAT_Z = 3.0
# runs of bit-identical depths inside otherwise random lists: tile length -> run length
RUNS = {33: 3, 257: 33, 1025: 3, 4097: 33}
CLASS_GRID = (8, 4)  # tiles across, down: 128x64 pixels

PARTIAL_SIZES = ((1, 1), (5, 3), (16, 1), (1, 40), (17, 17), (101, 77), (100, 68))  # (W, H)
STACK = 1200  # entries stacked in the bottom-right (partial) tile of each size in (c)
NAN_WORD = np.uint32(0xFFC0DEAD)  # guard / unwritten marker: a NaN no kernel computes


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


# ---------------------------------------------------------------------------------------------------------------------
# generators
# ---------------------------------------------------------------------------------------------------------------------

def _stacked_tiles(counts, gx, W, H, seed, flat_tiles=(), runs=None):
    """counts[t] splats whose 3-sigma rect is tile t alone: centres on pixel centres within 3 px of the tile centre,
    radius <= 3 px (f = 100, scale 0.004-0.012 m on the optical axis, z in [2, 4]), faint (opacity 0.0045-0.0145) so that pixels walk
    long lists.  Tiles in `flat_tiles` hold one depth; `runs` {tile: k}: k entries of the tile share one depth.  The
    input order is shuffled, so a tile's entries (and a run's) reach the scatter from many CTAs."""
    g = torch.Generator().manual_seed(seed)
    counts = torch.as_tensor(counts, dtype=torch.int64)
    tile = torch.repeat_interleave(torch.arange(len(counts)), counts)
    n = tile.numel()
    cx = (TILE * (tile % gx) + 8 + torch.randint(-3, 4, (n,), generator=g)).double()
    cy = (TILE * (tile // gx) + 8 + torch.randint(-3, 4, (n,), generator=g)).double()
    z = (2.0 + 2.0 * torch.rand(n, generator=g, dtype=torch.float64)).float().double()
    start = torch.cumsum(counts, 0) - counts
    for t in flat_tiles:
        z[start[t]:start[t] + counts[t]] = FLAT_Z
    for t, k in (runs or {}).items():
        z[start[t]:start[t] + k] = z[start[t]]
    # pixel = x f / z + W / 2 - 0.5 for the camera of kat_settings
    pos = torch.stack([(cx + 0.5 - W / 2) * z / F, (cy + 0.5 - H / 2) * z / F, z], 1).float()
    # off axis the projection stretches a Gaussian by sqrt(1 + tan^2) at most: scale it back so the radius stays <= 3 px
    shrink = torch.rsqrt(1.0 + ((cx + 0.5 - W / 2) / F) ** 2 + ((cy + 0.5 - H / 2) / F) ** 2).float()[:, None]
    assets = {"mean_3d": pos, "scale": (0.004 + 0.008 * torch.rand(n, 3, generator=g)) * shrink,
              "rotation": torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=1),
              "opacity": 0.0045 + 0.01 * torch.rand(n, 1, generator=g), "rgb": torch.rand(n, 3, generator=g)}
    perm = torch.randperm(n, generator=g)
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n)
    # ids of each run, in the shuffled input order
    run_ids = {t: inv[start[t]:start[t] + k].sort().values for t, k in (runs or {}).items()}
    flat_ids = {t: inv[start[t]:start[t] + counts[t]].sort().values for t in flat_tiles}
    return {k: v[perm].contiguous() for k, v in assets.items()}, run_ids, flat_ids


@functools.lru_cache(maxsize=None)
def _class_scene():
    """(a): 23 list lengths + 4 single-depth lists on an 8x4-tile image; tile t holds counts[t] entries."""
    gx, gy = CLASS_GRID
    counts = list(LENGTHS) + list(FLAT)
    counts += [0] * (gx * gy - len(counts))
    flat_tiles = tuple(range(len(LENGTHS), len(LENGTHS) + len(FLAT)))
    runs = {LENGTHS.index(n): k for n, k in RUNS.items()}
    assets, run_ids, flat_ids = _stacked_tiles(counts, gx, TILE * gx, TILE * gy, seed=7, flat_tiles=flat_tiles, runs=runs)
    return assets, TILE * gx, TILE * gy, np.array(counts), run_ids, flat_ids


@functools.lru_cache(maxsize=None)
def _wide_class_scene():
    """(b): 33 x 32 = 1056 tiles of 2049 entries each on 528x512 (2.16 M Gaussians)."""
    gx, gy = 33, 32
    counts = [2049] * (gx * gy)
    assets, _, _ = _stacked_tiles(counts, gx, TILE * gx, TILE * gy, seed=11)
    return assets, TILE * gx, TILE * gy, np.array(counts)


@functools.lru_cache(maxsize=None)
def _partial_scene(W, H):
    """(c): a T1-like scene (avatar + scene populations, the camera of yaw 0) at W x H, plus STACK faint splats
    centred inside the bottom-right tile's part of the image."""
    wl = Workload(f"{W}x{H}", H, W, 1000, 1000, 0, True)
    a = make_assets(wl, seed=W * 1000 + H)
    g = torch.Generator().manual_seed(W * 7 + H)
    f = 1.465 * H  # look_at_cam_param(0) is R = I, t = 0 with this focal length
    x0, y0 = TILE * ((W - 1) // TILE), TILE * ((H - 1) // TILE)
    n = STACK
    z = 2.0 + 2.0 * torch.rand(n, generator=g)
    cx = x0 - 0.5 + (W - x0) * torch.rand(n, generator=g)
    cy = y0 - 0.5 + (H - y0) * torch.rand(n, generator=g)
    stack = {"mean_3d": torch.stack([(cx + 0.5 - W / 2) * z / f, (cy + 0.5 - H / 2) * z / f, z], 1),
             "scale": 0.004 + 0.008 * torch.rand(n, 3, generator=g),
             "rotation": torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=1),
             "opacity": 0.0045 + 0.01 * torch.rand(n, 1, generator=g), "rgb": torch.rand(n, 3, generator=g)}
    assets = {k: torch.cat([a[k], stack[k]]).contiguous() for k in a}
    return assets, kat_settings(W=W, H=H, f=f, bg=(0.2, 0.6, 0.9))


def _oracle(st, a, variant="f32"):
    return O.forward(st, a["mean_3d"], a["opacity"], colors_precomp=a["rgb"], scales=a["scale"], rotations=a["rotation"],
                     variant=variant)


def _lens(ranges):
    return (ranges[:, 1].astype(np.int64) - ranges[:, 0].astype(np.int64))


def _tile_alpha_max(xy, co, tiles, W, H, chunk=4096):
    """fp64: for each (tile, Gaussian) pair the largest alpha = o exp(power) over the pixel centres of the tile inside
    the image (0 where power > 0: the composite skips those)."""
    gx = (W + TILE - 1) // TILE
    t, i = tiles
    out = np.empty(len(i))
    off = np.arange(TILE)
    for s in range(0, len(i), chunk):
        tt, ii = t[s:s + chunk], i[s:s + chunk]
        px = (tt % gx)[:, None] * TILE + off[None, :]
        py = (tt // gx)[:, None] * TILE + off[None, :]
        dx = (xy[ii, 0][:, None] - px)[:, None, :]  # (K, 1, 16x)
        dy = (xy[ii, 1][:, None] - py)[:, :, None]  # (K, 16y, 1)
        a, b, c, o = (co[ii, k][:, None, None] for k in range(4))
        power = -0.5 * (a * dx * dx + c * dy * dy) - b * dx * dy
        alpha = np.where(power > 0, 0.0, o * np.exp(np.minimum(power, 0.0)))
        inside = (px < W)[:, None, :] & (py < H)[:, :, None]
        out[s:s + chunk] = np.where(inside, alpha, 0.0).reshape(len(ii), -1).max(1)
    return out


def _pairs(ranges, ids):
    """(tile, id) of every list entry, as two int64 arrays."""
    lens = _lens(ranges)
    tile = np.repeat(np.arange(len(lens), dtype=np.int64), lens)
    first = np.repeat(ranges[:, 0].astype(np.int64), lens)
    pos = first + (np.arange(lens.sum(), dtype=np.int64) - np.repeat(np.cumsum(lens) - lens, lens))
    return tile, ids[pos].astype(np.int64)


def _assert_lists_equal(case, ranges, ids, o_ranges, o_ids):
    lens, o_lens = _lens(ranges), _lens(o_ranges)
    differ = np.flatnonzero(lens != o_lens)
    assert differ.size == 0, f"{case}: list lengths differ in tiles {differ[:8].tolist()}"
    for t in np.flatnonzero(o_lens):
        mine = ids[ranges[t, 0]:ranges[t, 1]]
        ref = o_ids[o_ranges[t, 0]:o_ranges[t, 1]]
        if not np.array_equal(mine, ref):
            k = int(np.flatnonzero(mine != ref)[0])
            raise AssertionError(f"{case}: tile {t} (n = {len(ref)}): sorted id list differs from the oracle's from "
                                 f"position {k} on (gpu {mine[k:k + 4].tolist()}, oracle {ref[k:k + 4].tolist()})")


# ---------------------------------------------------------------------------------------------------------------------
# (a), (b): sort classes, tie runs, segment cuts
# ---------------------------------------------------------------------------------------------------------------------

def _lists_and_parity(dev, case, assets, W, H, cap):
    """Tile culling off and on: num_dups, every per-tile list bit for bit, radii, colour / depth / alpha, the
    contributor report, and every gradient with depth and alpha gradients (the HAS_DA backward)."""
    from exavatar_release_b200 import _lib as L
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    st_c = kat_settings(W=W, H=H, f=F, bg=(0.1, 0.2, 0.3))
    st_g = settings_on(st_c, dev, rz.GaussianRasterizationSettings)
    oc, orad, od, oa, octx = _oracle(st_c, assets)
    pm, gm = O.fragility(octx)
    gen = torch.Generator().manual_seed(W * H)
    gi, gd, ga = torch.randn(3, H, W, generator=gen), torch.randn(1, H, W, generator=gen), torch.randn(1, H, W, generator=gen)
    og = O.backward(octx, gi.numpy(), gd.numpy()[0], ga.numpy()[0])
    o_ids, o_ranges = octx.sorted_ids(), octx.ranges()
    o_last = last_contributor(o_ids, o_ranges, octx.n_contrib(), W, H)
    # faint splats sit near alpha = 1/255 at some pixel of their tile, so the oracle flags nearly every Gaussian as
    # threshold-sensitive; flagged elements are held to the strict bound as well (measured: < 1e-6 * max|y|)
    strict = dict(loose=TOL)
    P = assets["mean_3d"].shape[0]
    ag = {k: v.to(dev) for k, v in assets.items()}
    for flags in (L.B2R_FLAG_NO_TILE_CULL, 0):
        tag = f"{case}/" + ("nocull" if flags else "cull")
        plan = FramePlan(P, W, H, cap, dev)
        sc = plan.scene(0, st_g, ag, flags=flags)
        plan.forward(sc)
        torch.cuda.synchronize()
        status = plan.status()
        assert status["overflow"] == 0, status
        # every pair of these scenes reaches alpha >= 1/255 in its tile (generator checks), so the cull keeps them all
        assert status["num_dups"] == octx.num_dups, tag
        ranges, ids, ncon, fT = ctx_arrays(plan.lib, plan, P, W, H)
        _assert_lists_equal(tag, ranges, ids, o_ranges, o_ids)
        assert np.array_equal(plan.radii.cpu().numpy(), orad), tag
        compare(tag, "color", plan.color.cpu().numpy(), oc, pm[None], kind="image", **strict)
        compare(tag, "depth", plan.depth.cpu().numpy(), od, pm[None], kind="image", **strict)
        compare(tag, "alpha", plan.alpha.cpu().numpy(), oa, pm[None], kind="image", **strict)
        contributor_report(tag, last_contributor(ids, ranges, ncon, W, H), fT, o_last, octx.final_T(), pm, max_frac=5e-3)
        flat, views = grad_bucket(P, dev)
        plan.backward(sc, gi.to(dev), views, g_depth=gd.to(dev), g_alpha=ga.to(dev))
        torch.cuda.synchronize()
        for k in GRADS:
            y = og[k]
            compare(tag, "d_" + k, views[k].cpu().numpy().reshape(y.shape), y, gm.reshape((-1,) + (1,) * (y.ndim - 1)),
                    kind="grad", **strict)
        del plan, flat, views
        torch.cuda.empty_cache()


@gpu
def test_list_length_classes_and_tie_runs(dev):
    """One tile per list length on both sides of every sort-class, batch and checkpoint-cut boundary (1 ... 6145),
    runs of 3 and 33 bit-identical depths, and whole lists at one depth in every sort class."""
    assets, W, H, counts, _, _ = _class_scene()
    _lists_and_parity(dev, "classes", assets, W, H, cap=int(counts.sum()) + 1024)


@gpu
def test_more_than_1024_tiles_in_the_chunked_class(dev):
    """1056 tiles of 2049 entries: the second pass of the tile scan's unit counts and the merge's chunk table in global
    memory (more than MERGE_TABLE = 1024 chunked tiles)."""
    assets, W, H, counts = _wide_class_scene()
    _lists_and_parity(dev, "wide2049", assets, W, H, cap=int(counts.sum()) + 1024)


# ---------------------------------------------------------------------------------------------------------------------
# (c): partial tiles through the C ABI, guard words around every output
# ---------------------------------------------------------------------------------------------------------------------

class _Guarded:
    """An output plane of `n` words inside a buffer filled with NAN_WORD: `guard` words before it (+ `shift`) and after."""

    def __init__(self, n, dev, guard=64, shift=0):
        self.n, self.lo = n, guard + shift
        self.buf = torch.full((self.lo + n + guard,), int(NAN_WORD.view(np.int32)), dtype=torch.int32, device=dev)

    def ptr(self):
        return self.buf.data_ptr() + 4 * self.lo

    def plane(self):
        return self.buf[self.lo:self.lo + self.n]

    def check(self, what):
        w = self.buf.cpu().numpy().view(np.uint32)
        guards = np.concatenate([w[:self.lo], w[self.lo + self.n:]])
        assert np.all(guards == NAN_WORD), f"{what}: a guard word was overwritten"
        unwritten = np.flatnonzero(w[self.lo:self.lo + self.n] == NAN_WORD)
        assert unwritten.size == 0, f"{what}: {unwritten.size} elements never written (first {unwritten[:4].tolist()})"


@gpu
@pytest.mark.parametrize("W,H", PARTIAL_SIZES, ids=[f"{w}x{h}" for w, h in PARTIAL_SIZES])
def test_partial_tiles_through_the_c_abi_with_guards(dev, W, H):
    """b2r_forward into output planes surrounded by guard words: every pixel written, no guard touched, outputs equal
    to the oracle's; again with the colour plane 4 bytes off 16-byte alignment (scalar stores on every width):
    bit-identical; then the backward (depth / alpha gradients on) against the oracle.  The bottom-right partial tile
    holds a list of more than 1100 entries: checkpoint records and segmented backward work in a partial tile."""
    from exavatar_release_b200 import _lib as L
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.plan import FramePlan, grad_bucket
    assets, st_c = _partial_scene(W, H)
    st_g = settings_on(st_c, dev, rz.GaussianRasterizationSettings)
    oc, orad, od, oa, octx = _oracle(st_c, assets)
    pm, gm = O.fragility(octx)
    P, N = assets["mean_3d"].shape[0], W * H
    plan = FramePlan(P, W, H, 200_000, dev)
    sc = plan.scene(0, st_g, {k: v.to(dev) for k, v in assets.items()})
    case = f"partial{W}x{H}"
    runs = []
    for shift in (0, 1):
        outs = [_Guarded(3 * N, dev, shift=shift), _Guarded(N, dev), _Guarded(N, dev), _Guarded(P, dev)]
        plan.out = L.B2RForwardOutputs(*(o.ptr() for o in outs))
        plan.forward(sc)
        torch.cuda.synchronize()
        assert plan.status()["overflow"] == 0
        for o, what in zip(outs, ("color", "depth", "alpha", "radii")):
            o.check(f"{case}/shift{shift}/{what}")
        runs.append([o.plane().clone() for o in outs])
    for x, y, what in zip(runs[0], runs[1], ("color", "depth", "alpha", "radii")):
        assert torch.equal(x, y), f"{case}: {what} differs between the vector and the scalar store path"
    color, depth, alpha, radii = runs[0]
    f32 = lambda t, *s: t.view(torch.float32).reshape(*s).cpu().numpy()
    assert np.array_equal(radii.cpu().numpy(), orad), case
    compare(case, "color", f32(color, 3, H, W), oc, pm[None], kind="image")
    compare(case, "depth", f32(depth, 1, H, W), od, pm[None], kind="image")
    compare(case, "alpha", f32(alpha, 1, H, W), oa, pm[None], kind="image")
    ranges, ids, ncon, fT = ctx_arrays(plan.lib, plan, P, W, H)
    contributor_report(case, last_contributor(ids, ranges, ncon, W, H), fT,
                       last_contributor(octx.sorted_ids(), octx.ranges(), octx.n_contrib(), W, H), octx.final_T(), pm,
                       max_frac=5e-3)
    gen = torch.Generator().manual_seed(N)
    gi, gd, ga = torch.randn(3, H, W, generator=gen), torch.randn(1, H, W, generator=gen), torch.randn(1, H, W, generator=gen)
    flat, views = grad_bucket(P, dev)
    plan.backward(sc, gi.to(dev), views, g_depth=gd.to(dev), g_alpha=ga.to(dev))
    torch.cuda.synchronize()
    og = O.backward(octx, gi.numpy(), gd.numpy()[0], ga.numpy()[0])
    for k in GRADS:
        y = og[k]
        compare(case, "d_" + k, views[k].cpu().numpy().reshape(y.shape), y, gm.reshape((-1,) + (1,) * (y.ndim - 1)),
                kind="grad", max_flagged_viol=5e-3)


# ---------------------------------------------------------------------------------------------------------------------
# (d): every pair the exact tile cull drops is empty
# ---------------------------------------------------------------------------------------------------------------------

def _assert_dropped_pairs_empty(case, ranges, ids, settings, assets, W, H):
    """ranges / ids: the GPU's culled lists.  Dropped pairs = the f32 oracle's unculled lists minus those, tile by
    tile; each must stay below alpha 1/255 at every pixel centre of its tile inside the image (fp64 oracle geometry)."""
    *_, o32 = _oracle(settings, assets)
    *_, o64 = _oracle(settings, assets, variant="f64")
    P = o32.P
    kt, ki = _pairs(ranges, ids)
    rt, ri = _pairs(o32.ranges(), o32.sorted_ids())
    kept, ref = kt * P + ki, rt * P + ri
    assert np.isin(kept, ref).all(), f"{case}: the culled lists hold a pair the oracle's 3-sigma lists do not"
    dropped = np.setdiff1d(ref, kept)
    amax = _tile_alpha_max(o64.xy(), o64.conic_opacity(), (dropped // P, dropped % P), W, H)
    worst = float(amax.max()) if amax.size else 0.0
    print(f"CULL {case}: {len(ref)} pairs in the 3-sigma lists, {len(kept)} kept, {len(dropped)} dropped; largest alpha "
          f"of a dropped pair {worst:.6g} (1/255 = {ALPHA_MIN:.6g})", flush=True)
    assert len(dropped) > 0, f"{case}: the cull dropped nothing; the test would not see a wrong drop"
    bad = np.flatnonzero(amax >= ALPHA_MIN)
    assert bad.size == 0, (f"{case}: {bad.size} dropped pairs reach alpha >= 1/255, e.g. (tile, id) = "
                           f"{[(int(dropped[j] // P), int(dropped[j] % P)) for j in bad[:4]]}")


@gpu
@pytest.mark.parametrize("wl_name", ["T1", "T3", "T4", "C2"])
def test_every_culled_pair_is_empty(dev, wl_name):
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.plan import FramePlan
    wl = WORKLOADS[wl_name]
    assets = make_assets(wl_name, seed=0)
    st_c = workload_settings(wl_name, yaw=5.0)
    P = assets["mean_3d"].shape[0]
    plan = FramePlan(P, wl.width, wl.height, 4_000_000, dev)
    sc = plan.scene(0, settings_on(st_c, dev, rz.GaussianRasterizationSettings), {k: v.to(dev) for k, v in assets.items()})
    plan.forward(sc)
    torch.cuda.synchronize()
    assert plan.status()["overflow"] == 0
    ranges, ids, _, _ = ctx_arrays(plan.lib, plan, P, wl.width, wl.height)
    _assert_dropped_pairs_empty(wl_name, ranges, ids, st_c, assets, wl.width, wl.height)


@gpu
def test_every_culled_pair_is_empty_in_both_merged_passes(dev):
    """Both projection + binning passes of a C4 MergedFivePlan frame: cat(scene, human) and cat(scene, refined)."""
    from exavatar_release_b200 import rasterizer as rz
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS, MergedFivePlan
    from exavatar_release_b200.renderer import render_settings
    wl = WORKLOADS["C4"]
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets("C4", seed=0)
    Ps, Ph = scene["mean_3d"].shape[0], human["mean_3d"].shape[0]
    cam = look_at_cam_param(-6.0, (H, W))
    st_c = render_settings((H, W), cam, torch.ones(3), O.OracleSettings)
    st_w = settings_on(st_c, dev, rz.GaussianRasterizationSettings)
    st_r = settings_on(render_settings((H, W), cam, torch.tensor([0.3, 0.7, 0.2]), O.OracleSettings), dev,
                       rz.GaussianRasterizationSettings)
    to = lambda d: {k: v.to(dev) for k, v in d.items()}
    plan = MergedFivePlan(Ps, Ph, W, H, None, dev)
    plan.set_scene(to(scene))
    plan.frame(0, st_w, st_r, to(scene), to(human), to(refined), {r: make_grad_image("C4", j).to(dev)
                                                                   for j, r in enumerate(RENDERS)}, accumulate=False)
    torch.cuda.synchronize()
    assert not plan.overflowed()
    for pk, other in (("A", human), ("B", refined)):
        ps = plan.passes[pk]
        ranges, ids, _, _ = ctx_arrays(plan.lib, ps, ps.P, W, H)
        cat = {k: torch.cat((scene[k], other[k])) for k in scene}
        _assert_dropped_pairs_empty(f"C4-merged/{pk}", ranges, ids, st_c, cat, W, H)


# ---------------------------------------------------------------------------------------------------------------------
# (e): densification statistics of the merged plan
# ---------------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("wl_name", ["T1", "T3"])
def test_merged_plan_densification_stats_match_reference_bookkeeping(dev, wl_name):
    """Three frames of MergedFivePlan.frame(densify=...) (pass A's scene rows, fed by the scratch its three views
    share) against module.py:155-157 + model.py:283-285 applied to the scene render of the reference pattern: its
    `radius` and the `mean_2d.grad` autograd returns.  The other four renders see the scene detached and do not reach
    the scene's mean_2d."""
    from exavatar_release_b200 import GaussianRenderer
    from exavatar_release_b200.camera import look_at_cam_param
    from exavatar_release_b200.plan import RENDERS, MergedFivePlan
    from exavatar_release_b200.renderer import render_settings
    wl = WORKLOADS[wl_name]
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets(wl_name, seed=0, device=dev)
    Ps, Ph = scene["mean_3d"].shape[0], human["mean_3d"].shape[0]
    bg_w, bg_r = torch.ones(3, device=dev), torch.tensor([0.3, 0.7, 0.2], device=dev)
    plan = MergedFivePlan(Ps, Ph, W, H, {"A": 2_000_000, "B": 2_000_000}, dev)
    plan.set_scene(scene)
    fused = {k: torch.zeros(Ps, device=dev) for k in ("grad_accum", "count", "radius_max")}
    ref_accum, ref_cnt, ref_rmax = torch.zeros(Ps, 1, device=dev), torch.zeros(Ps, 1, device=dev), torch.zeros(Ps, device=dev)
    R = GaussianRenderer()
    for f, yaw in enumerate((-12.0, 0.0, 14.0)):
        cam = look_at_cam_param(yaw, (H, W), device=dev)
        gcol = {r: make_grad_image(wl_name, 10 * f + j).to(dev) for j, r in enumerate(RENDERS)}
        plan.frame(f, render_settings((H, W), cam, bg_w), render_settings((H, W), cam, bg_r), scene, human, refined, gcol,
                   accumulate=(f > 0), densify=fused)
        lv = {k: v.clone().requires_grad_() for k, v in scene.items()}
        out = R(lv, (H, W), cam, bg_w)
        (out["img"] * gcol["scene"]).sum().backward()
        # the reference's own statements
        is_vis = out["radius"] > 0
        ref_rmax[is_vis] = torch.maximum(ref_rmax[is_vis], out["radius"][is_vis].float())
        ref_accum[is_vis, :] += torch.norm(out["mean_2d"].grad[is_vis, :2], dim=1, keepdim=True)
        ref_cnt[is_vis, :] += 1
    torch.cuda.synchronize()
    assert not plan.overflowed()
    assert torch.equal(fused["count"], ref_cnt[:, 0]) and torch.equal(fused["radius_max"], ref_rmax)
    assert torch.allclose(fused["grad_accum"], ref_accum[:, 0], rtol=1e-5, atol=1e-6 * float(ref_accum.max()))
    assert float(fused["count"].max()) == 3.0 and float(fused["grad_accum"].max()) > 0


# ---------------------------------------------------------------------------------------------------------------------
# generator checks (oracle only, no GPU): the scenes reach what the GPU tests above claim
# ---------------------------------------------------------------------------------------------------------------------

def _single_tile_rects(octx, W):
    gx = (W + TILE - 1) // TILE
    rect = octx.rect()
    vis = octx.tiles_touched() > 0
    assert vis.all(), "every Gaussian of a stacked-tile scene is visible"
    assert np.all(rect[:, 2] - rect[:, 0] == 1) and np.all(rect[:, 3] - rect[:, 1] == 1), "a rect spans several tiles"
    return rect[:, 1] * gx + rect[:, 0]


def _every_pair_is_kept(octx):
    """Every Gaussian reaches alpha > 1.05/255 at the pixel centre nearest its centre (inside its tile), so the exact
    tile cull must keep every pair and the culled lists equal the oracle's."""
    xy, co = octx.xy().astype(np.float64), octx.conic_opacity().astype(np.float64)
    d = xy - np.round(xy)
    power = -0.5 * (co[:, 0] * d[:, 0] ** 2 + co[:, 2] * d[:, 1] ** 2) - co[:, 1] * d[:, 0] * d[:, 1]
    alpha = co[:, 3] * np.exp(power)
    assert alpha.min() > 1.05 * ALPHA_MIN, alpha.min()


def test_class_scene_generator():
    assets, W, H, counts, run_ids, flat_ids = _class_scene()
    *_, octx = _oracle(kat_settings(W=W, H=H, f=F), assets)
    lens = _lens(octx.ranges())
    assert np.array_equal(lens, counts), "list lengths are not the targets"
    tile_of = _single_tile_rects(octx, W)
    depth = octx.depth()
    z = assets["mean_3d"][:, 2].numpy()
    for t, ids in list(run_ids.items()) + list(flat_ids.items()):
        ids = ids.numpy()
        assert np.all(tile_of[ids] == t)
        assert len(np.unique(depth[ids].view(np.uint32))) == 1 and len(np.unique(z[ids].view(np.uint32))) == 1, t
    assert sorted(len(v) for v in run_ids.values()) == sorted(RUNS.values())
    assert sorted(len(v) for v in flat_ids.values()) == sorted(FLAT)
    _every_pair_is_kept(octx)
    # every checkpoint cut is crossed: in every tile of more than SEG entries some pixel's last contributor lies in
    # the last segment (so its walk continues behind every earlier cut)
    ncon = octx.n_contrib().astype(np.int64)
    gx = W // TILE
    for t in np.flatnonzero(counts > SEG):
        tx, ty = t % gx, t // gx
        last = ncon[ty * TILE:(ty + 1) * TILE, tx * TILE:(tx + 1) * TILE].max()
        assert last > SEG * ((counts[t] - 1) // SEG), f"tile {t} (n = {counts[t]}): no pixel reaches the last segment"


def test_wide_class_generator():
    assets, W, H, counts = _wide_class_scene()
    *_, octx = _oracle(kat_settings(W=W, H=H, f=F), assets)
    lens = _lens(octx.ranges())
    assert np.array_equal(lens, counts)
    assert (lens >= 2048).sum() > 1024
    _single_tile_rects(octx, W)
    _every_pair_is_kept(octx)


@pytest.mark.parametrize("W,H", PARTIAL_SIZES, ids=[f"{w}x{h}" for w, h in PARTIAL_SIZES])
def test_partial_tile_generator(W, H):
    assets, st = _partial_scene(W, H)
    *_, octx = _oracle(st, assets)
    gx = (W + TILE - 1) // TILE
    last = ((H - 1) // TILE) * gx + (W - 1) // TILE
    assert W % TILE or H % TILE, "the bottom-right tile must be partial"
    assert _lens(octx.ranges())[last] > 2 * SEG, "the partial tile's list must span several checkpoint segments"
