"""Per-stage kernel times of one C4 training frame on MergedFivePlan (serial, in-library CUDA-event profiler).

  python tools/five_breakdown.py [--workload C4]
Runs `MergedFivePlan.frame` in serial mode and prints, after each stage (a pass's projection + binning, the forward /
backward composite of each view, a pass's backward projection), the kernels it ran and their microseconds.
"""
import argparse
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exavatar_release_b200 import _lib as L  # noqa: E402
from exavatar_release_b200 import plan as PL  # noqa: E402
from exavatar_release_b200.camera import look_at_cam_param  # noqa: E402
from exavatar_release_b200.renderer import render_settings  # noqa: E402
from exavatar_release_b200.synthetic import WORKLOADS, make_grad_image, make_population_assets  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="C4")
    a = ap.parse_args()
    wl = WORKLOADS[a.workload]
    dev = torch.device("cuda:0")
    lib = L.load()
    H, W = wl.height, wl.width
    scene, human, refined = make_population_assets(a.workload, seed=0, device=dev)
    cam = look_at_cam_param(-6.0, (H, W), device=dev)
    st_w = render_settings((H, W), cam, torch.ones(3, device=dev))
    st_r = render_settings((H, W), cam, torch.tensor([0.3, 0.7, 0.2], device=dev))
    g = {r: make_grad_image(a.workload, 10 + j, device=dev) for j, r in enumerate(PL.RENDERS)}
    plan = PL.MergedFivePlan(wl.n_scene, wl.n_avatar, W, H, None, dev)
    plan.set_scene(scene)
    for _ in range(3):
        plan.frame(0, st_w, st_r, scene, human, refined, g, accumulate=False, serial=True)
    torch.cuda.synchronize()
    print("dups", plan.dups())

    ms = (C.c_double * 9)()
    cnt = (C.c_uint64 * 9)()
    names = [lib.b2r_kernel_name(i).decode() for i in range(9)]

    def read(label):
        torch.cuda.synchronize()
        lib.b2r_profile_read(ms, cnt, 1)
        parts = [f"{names[i]} {ms[i] * 1e3:.1f}" for i in range(9) if cnt[i]]
        print(f"  {label:34s}", ", ".join(parts))

    lib.b2r_profile_enable(1)
    lib.b2r_profile_read(ms, cnt, 1)
    plan.frame(0, st_w, st_r, scene, human, refined, g, accumulate=False, serial=True, probe=read)
    lib.b2r_profile_enable(0)


if __name__ == "__main__":
    main()
