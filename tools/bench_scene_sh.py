"""What colouring the scene Gaussians from SH inside the merged five-render frame saves per training frame.

  python tools/bench_scene_sh.py [--workload C4] [--frames 200] [--block 20] [--warmup 20] [--probe-frames 20]

ExAvatar colours its scene Gaussians from degree-3 SH on the caller's side every frame (`SceneGaussian.forward`,
module.py:253-272) and back-propagates through that PyTorch code.  This runs the five-render training frame through
`TrainingFrameRenderer`, eager and with `use_graph=True`, in two configurations:
  (a) caller-side: scene_gaussian_assets(in_kernel_sh=False) + autograd, TrainingFrameRenderer(scene_sh_coeffs=0);
  (b) in-kernel:   scene_gaussian_assets(in_kernel_sh=True), TrainingFrameRenderer(scene_sh_coeffs=16).
A training frame is: build the scene asset dict from the SceneGaussian parameters, the frame's forward, a loss over the
five images, backward to the parameters.  Times come from CUDA events around the forward (asset build included) and
the backward, after warm-up, over `--frames` frames per configuration; (a) and (b) alternate in blocks of `--block`
frames within the run, cycling through eight cameras.  It then prints the per-stage kernel times of
`MergedFivePlan.frame(serial=True, probe=...)` (in-library CUDA-event profiler, mean over `--probe-frames` frames) with
an rgb scene and with an SH scene: what the SH rows add to the projection (K1, in "bin") and to the backward
projection (K6) of both passes.  The GPU's name and power limit are printed with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exavatar_release_b200 import TrainingFrameRenderer  # noqa: E402
from exavatar_release_b200 import _lib as L  # noqa: E402
from exavatar_release_b200.camera import look_at_cam_param  # noqa: E402
from exavatar_release_b200.plan import RENDERS, MergedFivePlan  # noqa: E402
from exavatar_release_b200.rasterizer import GaussianRasterizationSettings  # noqa: E402
from exavatar_release_b200.renderer import render_settings, scene_gaussian_assets  # noqa: E402
from exavatar_release_b200.synthetic import WORKLOADS, make_grad_image, make_population_assets, make_scene_sh_params  # noqa: E402

SH_DEGREE = 3  # ExAvatar trains at max_sh_degree = 3 from iteration 3000 on (config.py:15-16)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="C4")
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--block", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--probe-frames", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene_sh: needs a CUDA device (there is no CPU measurement)")
    wl = WORKLOADS[args.workload]
    dev = torch.device("cuda:0")
    H, W = wl.height, wl.width
    _, human, refined = make_population_assets(args.workload, seed=0, device=dev)
    params = make_scene_sh_params(args.workload, seed=0, device=dev)
    params = {k: v.requires_grad_(True) for k, v in params.items()}
    leaves_h = {n: {k: v.clone().requires_grad_(True) for k, v in a.items()} for n, a in (("human", human), ("refined", refined))}
    Ps, Ph = params["mean"].shape[0], human["mean_3d"].shape[0]
    cams = [look_at_cam_param(-20.0 + 5.0 * i, (H, W), device=dev) for i in range(8)]
    bg_r = torch.tensor([0.3, 0.7, 0.2], device=dev)
    gimg = {r: make_grad_image(args.workload, 10 + j, device=dev) for j, r in enumerate(RENDERS)}
    name, power = gpu_info()
    print(f"GPU: {name}; power limit, max SM clock: {power}")
    print(f"workload {args.workload}: {Ps} scene Gaussians at SH degree {SH_DEGREE}, {Ph} human, {W}x{H}")

    caps = {"A": 8_000_000, "B": 8_000_000}
    configs = {}
    for graph in (False, True):
        for in_kernel in (False, True):
            fr = TrainingFrameRenderer(Ps, Ph, (H, W), dev, caps, use_graph=graph, scene_sh_coeffs=16 if in_kernel else 0)
            configs[("graph" if graph else "eager", "b_in_kernel" if in_kernel else "a_caller_side")] = (fr, in_kernel)

    def one_frame(fr, in_kernel, cam, ev):
        ev[0].record()
        sa = scene_gaussian_assets(params["mean"], params["opacity_logit"], params["log_scale"], params["rotation"],
                                   params["feature_dc"], params["feature_rest"], SH_DEGREE, cam, in_kernel_sh=in_kernel)
        out = fr(sa, leaves_h["human"], leaves_h["refined"], cam, bg_r)
        loss = sum((out[r]["img"] * gimg[r]).sum() for r in RENDERS)
        ev[1].record()
        loss.backward()
        ev[2].record()

    def zero_grads():
        for t in list(params.values()) + [v for a in leaves_h.values() for v in a.values()]:
            t.grad = None

    times = {k: [] for k in configs}
    for mode in ("eager", "graph"):
        keys = [k for k in configs if k[0] == mode]
        for k in keys:  # warm-up (graph mode: captures the graphs of every camera's key)
            fr, ik = configs[k]
            for i in range(args.warmup):
                one_frame(fr, ik, cams[i % len(cams)], [torch.cuda.Event(enable_timing=True) for _ in range(3)])
                zero_grads()
        torch.cuda.synchronize()
        done = 0
        while done < args.frames:
            n = min(args.block, args.frames - done)
            for k in keys:  # (a) and (b) alternate block by block
                fr, ik = configs[k]
                for i in range(n):
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                    one_frame(fr, ik, cams[(done + i) % len(cams)], ev)
                    zero_grads()
                    times[k].append(ev)
            done += n
        torch.cuda.synchronize()
        for k in configs:
            assert not configs[k][0].overflowed(), k

    results = {}
    print(f"\nmean per training frame over {args.frames} frames (ms), (a)/(b) alternated in blocks of {args.block}:")
    print(f"  {'mode':6s} {'config':14s} {'forward':>9s} {'backward':>9s} {'frame':>9s}")
    for k, evs in times.items():
        f = sum(e[0].elapsed_time(e[1]) for e in evs) / len(evs)
        b = sum(e[1].elapsed_time(e[2]) for e in evs) / len(evs)
        results["/".join(k)] = {"forward_ms": f, "backward_ms": b, "frame_ms": f + b, "frames": len(evs)}
        print(f"  {k[0]:6s} {k[1]:14s} {f:9.3f} {b:9.3f} {f + b:9.3f}")
    for mode in ("eager", "graph"):
        a, b = results[f"{mode}/a_caller_side"]["frame_ms"], results[f"{mode}/b_in_kernel"]["frame_ms"]
        print(f"  {mode}: in-kernel SH saves {a - b:.3f} ms per frame ({100 * (a - b) / a:.1f} %)")

    # per-stage kernel times, serial frame, rgb scene vs SH scene
    lib = L.load()
    nk = 9  # B2R_NUM_KERNELS
    names = [lib.b2r_kernel_name(i).decode() for i in range(nk)]
    ms, cnt = (C.c_double * nk)(), (C.c_uint64 * nk)()
    stages = {}
    for sh in (False, True):
        plan = MergedFivePlan(Ps, Ph, W, H, caps, dev, scene_sh_coeffs=16 if sh else 0)
        acc = {}

        def probe(label):
            torch.cuda.synchronize()
            lib.b2r_profile_read(ms, cnt, 1)
            d = acc.setdefault(label, [0.0] * nk)
            for i in range(nk):
                d[i] += ms[i]

        with torch.no_grad():
            for i in range(3 + args.probe_frames):
                cam = cams[i % len(cams)]
                sa = scene_gaussian_assets(params["mean"], params["opacity_logit"], params["log_scale"], params["rotation"],
                                           params["feature_dc"], params["feature_rest"], SH_DEGREE, cam, in_kernel_sh=sh)
                plan.set_scene(sa)
                st_w = render_settings((H, W), cam, torch.ones(3, device=dev), GaussianRasterizationSettings)
                st_r = st_w._replace(bg=bg_r)
                if sh:
                    st_w, st_r = st_w._replace(sh_degree=SH_DEGREE), st_r._replace(sh_degree=SH_DEGREE)
                measured = i >= 3
                if measured and i == 3:
                    torch.cuda.synchronize()
                    lib.b2r_profile_enable(1)
                    lib.b2r_profile_read(ms, cnt, 1)
                plan.frame(None, st_w, st_r, None, human, refined, gimg, accumulate=False, serial=True,
                           probe=probe if measured else None)
            torch.cuda.synchronize()
            lib.b2r_profile_enable(0)
        stages["sh" if sh else "rgb"] = {lab: [v / args.probe_frames for v in d] for lab, d in acc.items()}
    print(f"\nper-stage kernel times (us), serial frame, mean over {args.probe_frames} frames: rgb scene | SH scene (degree {SH_DEGREE})")
    for lab in stages["rgb"]:
        r, s = stages["rgb"][lab], stages["sh"][lab]
        parts = [f"{names[i]} {r[i] * 1e3:.1f} | {s[i] * 1e3:.1f}" for i in range(nk) if r[i] or s[i]]
        print(f"  {lab:28s} " + ", ".join(parts))
    tot = {k: sum(sum(v) for v in st.values()) for k, st in stages.items()}
    print(f"  all stages: rgb {tot['rgb'] * 1e3:.1f} us, SH {tot['sh'] * 1e3:.1f} us")
    print("RESULT " + json.dumps({"gpu": name, "power_limit_max_sm_clock": power, "workload": args.workload,
                                  "frames": results, "stage_ms": stages, "kernel_names": names}))


if __name__ == "__main__":
    main()
