#!/usr/bin/env python
"""bench.py -- avatar train-step frames/s (forward + backward Gaussian rasterisation), BASELINE.json's metric.

Default workload: BASELINE.json configs[3] = **C4, the NeuMan-style training frame**: 167 k human + 130 k scene Gaussians
at 512x512, rendered the way ExAvatar trains (avatar/main/model.py:81-162): FIVE rasteriser calls per frame -- scene |
human (random bg) | cat(scene.detach(), human) | human_refined | cat(scene.detach(), human_refined) -- each forward +
backward.  One "step" = every rank runs F such training frames (default 8) and, when N > 1, ONE NCCL all-reduce of the
flat gradient bucket plus the small densification-statistics all-reduce (SURVEY.md section 8e).  `value` = training
frames/s of the whole job (a frame = 5 renders).  `--pattern single` (and every workload without both populations: C1,
C3, C5) times one render per frame instead, as round 1 did; the C2 single-render number stays in the line as
`single_render`.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4] [--pattern auto|five|single] [--frames F]
                  [--lanes S] [--impl b200|reference] [--dump-outputs DIR]

Legs (one JSON line, rank 0):
  value        device-resident: inputs in HBM, C ABI driven through the plan objects, the step captured in a CUDA graph
  e2e          the public plugin API (GaussianRenderer -> GaussianRasterizer autograd, L1 loss, backward) with pinned HOST
               buffers; host->device: the Gaussian parameter sets once per step + one target image per frame; device->host:
               the step's summed gradients + per-frame losses; the whole step in one CUDA graph (fixed-capacity mode)
  e2e_eager    same API with the UNMODIFIED reference call shape (GaussianRenderer.forward(assets, shape, cam, bg): camera
               matrices rebuilt per call, adaptive capacity, no graph) -- what a user who only swaps the import gets
  roofline     dominant kernel's algorithmic bytes / its live CUDA-event duration (in-library profiler, renders one at a
               time); per-kernel table
  strong_scaling (N > 1) BASELINE configs[3] literally: a global batch of 8 frames sharded over the ranks (rank r takes
               frames r::N), loss pre-divided by the global batch (train.py:43), same collectives
  cpu_baseline the CPU oracle (oracle/, kind "port") on the host cores, bounded sample of the same pattern (N = 1 only)
`--impl reference` times that CPU oracle on the same pattern through the same GaussianRenderer call (reference arm).

Timing: W >= 3 warm-up steps, then K timed steps in every GPU leg; L2 flushed (256 MiB memset) before every timed
step, outside the per-step CUDA event pairs; per-rank time = sum of per-step event durations; max over ranks.  Clocks:
NVML polled by a thread during the timed region.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from

from exavatar_release_b200.camera import look_at_cam_param  # noqa: E402
from exavatar_release_b200.synthetic import WORKLOADS, make_assets, make_grad_image, make_population_assets  # noqa: E402

METRIC = "avatar train-step frames/sec (fwd+bwd raster)"
UNIT = "frames/s"
FIVE = ("scene", "human", "scene_human", "human_refined", "scene_human_refined")
BG_RAND = (0.3, 0.7, 0.2)  # stands for model.py:72 `bg = torch.rand(3)` (fixed so runs are comparable)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=[k for k in WORKLOADS if k.startswith("C")])
    ap.add_argument("--pattern", default="auto", choices=["auto", "five", "single"],
                    help="five: ExAvatar's five renders per training frame (needs both populations); single: one render")
    ap.add_argument("--frames", type=int, default=8, help="frames per rank per step")
    ap.add_argument("--lanes", type=int, default=None,
                    help="frames in flight per rank (CUDA streams): default 4 (single pattern), 3 (five pattern)")
    ap.add_argument("--engine", default=os.environ.get("B2R_FIVE_ENGINE", "merged"), choices=["merged", "separate"],
                    help="five pattern: merged = two projection/binning passes shared by the five renders (SURVEY 8f-3); "
                         "separate = five independent renders on five streams (round-1 FiveRenderPlan)")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step in a CUDA graph")
    ap.add_argument("--no-graph-collectives", action="store_true", help="N > 1: issue the all-reduces after the graph replay")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-lanes", type=int, default=None, help="five pattern: frames in flight on the autograd path of the e2e legs")
    ap.add_argument("--no-eager", action="store_true", help="skip the e2e_eager leg")
    ap.add_argument("--no-single", action="store_true", help="five pattern: skip the extra C2 single-render key")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-upload", default="per-step", choices=["per-step", "per-frame"],
                    help="single pattern e2e: Gaussian set host->device once per step or once per frame")
    ap.add_argument("--trace-e2e", default=None, help="write a chrome trace (CUPTI via torch.profiler) of one e2e step here")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU budget of the cpu_baseline leg")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the timed step computed in its last step as DIR/<name>.npy (float32); the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    return ap.parse_args()


def frame_yaw(global_frame: int) -> float:
    return -20.0 + 40.0 * ((global_frame % 8) / 7.0)  # 8 distinct cameras, yaw +-20 deg (SURVEY section 8d, C4)


def resolve_pattern(args, wl) -> str:
    if getattr(args, "_lanes_user", None) is None:
        args._lanes_user = args.lanes
    can_five = wl.backward and wl.n_avatar > 0 and wl.n_scene > 0 and wl.sh_degree == 0
    if args.pattern == "five" and not can_five:
        raise SystemExit(f"bench.py: workload {wl.name} cannot run the five-render pattern")
    pattern = "five" if (args.pattern == "five" or (args.pattern == "auto" and can_five)) else "single"
    args.lanes = args._lanes_user if args._lanes_user is not None else (3 if pattern == "five" else 4)
    return pattern


def workload_label(wl, pattern) -> str:
    if pattern == "five":
        return (f"{wl.name} as ExAvatar trains it: five renders per frame (model.py:81-162: scene | human rand-bg | "
                f"cat(scene.detach(),human) | human_refined | cat(scene.detach(),human_refined)), fwd+bwd each")
    return wl.name


def config_dict(args, wl, pattern, extra=None):
    c = {"workload": workload_label(wl, pattern), "pattern": pattern, "frames_per_rank_per_step": args.frames,
         "renders_per_frame": 5 if pattern == "five" else 1, "P": wl.n_avatar + wl.n_scene,
         "P_scene": wl.n_scene, "P_human": wl.n_avatar, "image": f"{wl.width}x{wl.height}", "sh_degree": wl.sh_degree,
         "backward": wl.backward,
         "parallelism": f"frames sharded over {args.gpus} rank(s), one gradient all-reduce per step" if args.gpus > 1
         else "single GPU", "l2": "256 MiB L2 flush before every timed step (outside the event pairs)"}
    if extra:
        c.update(extra)
    return c


# ---------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the CPU oracle behind the reference-facing call
# ---------------------------------------------------------------------------------------------------------------
def cpu_frame_fn(wl_name, pattern, seed=0):
    """Returns (closure running one frame of the pattern on the CPU oracle through GaussianRenderer, threads used)."""
    from oracle import oracle as O
    from exavatar_release_b200.renderer import GaussianRenderer, render_settings

    wl = WORKLOADS[wl_name]
    O.set_num_threads(os.cpu_count() or 1)
    renderer = GaussianRenderer(rasterizer_cls=O.OracleRasterizer, settings_cls=O.OracleSettings)
    bg = torch.ones(3)
    shape = (wl.height, wl.width)

    if pattern == "five":
        scene, human, refined = make_population_assets(wl_name, seed=seed)
        gis = [make_grad_image(wl_name, 10 + j) for j in range(5)]
        bg_r = torch.tensor(BG_RAND)

        def frame(i):
            cam = look_at_cam_param(frame_yaw(i), shape)
            lv = {n: {k: v.clone().requires_grad_() for k, v in a.items()} for n, a in
                  (("scene", scene), ("human", human), ("refined", refined))}
            cat = lambda a, b: {k: torch.cat((a[k].detach(), b[k])) for k in a}  # model.py:117-125
            imgs = [renderer(lv["scene"], shape, cam)["img"], renderer(lv["human"], shape, cam, bg_r)["img"],
                    renderer(cat(lv["scene"], lv["human"]), shape, cam)["img"],
                    renderer(lv["refined"], shape, cam, bg_r)["img"],
                    renderer(cat(lv["scene"], lv["refined"]), shape, cam)["img"]]
            sum((im * g).sum() for im, g in zip(imgs, gis)).backward()
            return float(imgs[2].detach().sum())
    else:
        assets = make_assets(wl_name, seed=seed)
        gi = make_grad_image(wl_name, seed)
        use_sh = wl.sh_degree > 0

        def frame(i):
            cam = look_at_cam_param(frame_yaw(i), shape)
            leaves = {k: v.clone().requires_grad_(wl.backward) for k, v in assets.items()}
            if use_sh:  # C3: colours from SH inside the rasteriser
                st = render_settings(shape, cam, bg, O.OracleSettings)._replace(sh_degree=wl.sh_degree)
                m2 = torch.zeros(leaves["mean_3d"].shape[0], 3, requires_grad=wl.backward)
                img = O.OracleRasterizer(st)(means3D=leaves["mean_3d"], means2D=m2, opacities=leaves["opacity"],
                                             shs=leaves["shs"], scales=leaves["scale"], rotations=leaves["rotation"])[0]
            else:
                img = renderer(leaves, shape, cam, bg)["img"]
            if wl.backward:
                (img * gi).sum().backward()
            return float(img.detach().sum())

    # "all the host threads it can use": OpenMP scaling of the oracle saturates (atomics in the backward), so pick the
    # fastest thread count among a few candidates instead of blindly using every core
    ncpu = os.cpu_count() or 1
    best, best_t = ncpu, None
    for cand in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):
        O.set_num_threads(cand)
        t0 = time.perf_counter()
        frame(0)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = cand, dt
    O.set_num_threads(best)
    return frame, best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    pattern = resolve_pattern(args, wl)
    frame, threads = cpu_frame_fn(args.workload, pattern)
    # bounded sample: one training frame per step; the step count shrinks if a frame is slow so the arm ends in minutes
    t0 = time.perf_counter()
    frame(0)
    one = time.perf_counter() - t0
    warm = max(0, min(args.warmup, int(20.0 / max(one, 1e-3))))
    steps = max(1, min(args.steps, int(120.0 / max(one, 1e-3))))
    for i in range(warm):
        frame(i)
    t0 = time.perf_counter()
    for i in range(steps):
        frame(i)
    dt = time.perf_counter() - t0
    fps = steps / dt
    what = "5 renders fwd+bwd" if pattern == "five" else ("fwd+bwd" if wl.backward else "fwd")
    sample = f"1 frame of {wl.name} per step ({what}), {steps} timed steps, {threads} threads"
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, wl, pattern, {"frames_per_rank_per_step": 1,
                                                      "parallelism": f"{threads} host threads (OpenMP)", "l2": "n/a (CPU)"}),
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  The region lasts tens of milliseconds, far too
    short for `nvidia-smi -lms`, so a thread polls NVML directly (~1 kHz); nvidia-smi is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        import threading
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.window = "timed region"
        self._stop = threading.Event()
        self._thread = None
        self.proc, self.path = None, None
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            bits = {"hw_slowdown": getattr(N, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(N, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(N, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(N, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}

            def poll():
                while not self._stop.is_set():
                    try:
                        self.samples.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                        r = int(N.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        for name, bit in bits.items():
                            if r & bit:
                                self.reasons.add(name)
                    except Exception:
                        pass
                    time.sleep(0.001)

            self._thread = threading.Thread(target=poll, daemon=True)
            self._thread.start()
            return
        except Exception:
            self._thread = None
        exe = shutil.which("nvidia-smi")
        if exe is None:
            return
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        self.f = open(self.path, "w")
        self.proc = subprocess.Popen([exe, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                      "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
            if not self.samples:
                return None
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                    "samples": len(sm), "source": "nvml thread", "window": self.window}
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
        os.unlink(self.path)
        sm, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi -lms 20"}


# ---------------------------------------------------------------------------------------------------------------
# B200 arm: shared plumbing
# ---------------------------------------------------------------------------------------------------------------
class Env:
    """Process-wide state of the B200 arm: ranks, device, the loaded library, timing helpers."""

    def __init__(self, args):
        import torch.distributed as dist
        from exavatar_release_b200 import _lib as L
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.lib = L.load()
        self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        self.args = args

    def barrier(self):
        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()

    def timed(self, fn, steps):
        """K steps, each bracketed by CUDA events after an L2 flush; returns (ms summed, max over ranks; wall s; launches)."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        l0 = self.lib.b2r_launch_count()
        t0 = time.perf_counter()
        for s in range(steps):
            self.flush_buf.zero_()
            ev[s][0].record()
            fn()
            ev[s][1].record()
        self.barrier()
        wall = time.perf_counter() - t0
        ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item()), wall, self.lib.b2r_launch_count() - l0

    def capture(self, body):
        """Warm `body` on a side stream, then capture it into a CUDA graph; returns (graph, launches of this library)."""
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            body()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        l0 = self.lib.b2r_launch_count()
        with torch.cuda.graph(g):
            body()
        return g, self.lib.b2r_launch_count() - l0

    def profile_read(self, reset=True):
        ms_arr = (C.c_double * 9)()
        cnt_arr = (C.c_uint64 * 9)()
        self.lib.b2r_profile_read(ms_arr, cnt_arr, 1 if reset else 0)
        return {self.lib.b2r_kernel_name(i).decode(): {"ms_avg": (ms_arr[i] / cnt_arr[i]) if cnt_arr[i] else 0.0,
                                                       "launches": int(cnt_arr[i])} for i in range(9)}


def peaks_and_traffic(workload_key, dom):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload_key, {}).get(dom)
    except Exception:
        pass
    return peaks, traffic


def roofline_dict(per_kernel, algo, workload_key, extra):
    dom = max(("composite_fwd", "composite_bwd"), key=lambda k: per_kernel[k]["ms_avg"] * (1 if per_kernel[k]["launches"] else 0))
    peaks, traffic = peaks_and_traffic(workload_key, dom)
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ms = per_kernel[dom]["ms_avg"]
    ach = algo[dom] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    other = "composite_fwd" if dom == "composite_bwd" else "composite_bwd"
    oms = per_kernel[other]["ms_avg"]
    r = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
         "frac": ach / peak if peak else None, "traffic": traffic,
         "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s",
         "algorithmic_bytes_per_launch": algo[dom], "kernel_ms_avg": ms,
         "other_composite": {"kernel": other, "kernel_ms_avg": oms, "algorithmic_bytes_per_launch": algo[other],
                             "frac": (algo[other] / (oms * 1e-3) / 1e9 / peak) if oms > 0 and peak else None},
         "binding_bound": "instruction issue (ALU/SFU/shared memory), not HBM -- see DESIGN.md section 5",
         "per_kernel_ms": {k: round(v["ms_avg"], 5) for k, v in per_kernel.items() if v["launches"]},
         "per_kernel_launches": {k: v["launches"] for k, v in per_kernel.items() if v["launches"]}}
    r.update(extra)
    return r


def consumed_units(stt):
    """List entries staged per TILE by the composites, from the status block (units documented in b200raster.h)."""
    return stt["consumed_fwd"] / stt.get("consumed_fwd_div", 4.0), stt["consumed_bwd"] / stt.get("consumed_bwd_div", 4.0)


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much in all


def dump_outputs(out_dir, arrays):
    """Writes `arrays` (device tensors) as out_dir/<name>.npy in float32.  When they hold more than DUMP_BYTES, every
    array keeps the same share of its elements: a sorted sample of its flattened elements drawn with a fixed seed, so
    every run with the same arguments writes the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    keep = min(1.0, DUMP_BYTES / (4 * sum(v.numel() for v in arrays.values())))
    for name, v in arrays.items():
        a = v.detach().float().cpu()
        if keep < 1.0:
            a = a.reshape(-1)
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[: int(a.numel() * keep)]
            a = a[idx.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


# ---------------------------------------------------------------------------------------------------------------
# pattern "five": ExAvatar's training frame
# ---------------------------------------------------------------------------------------------------------------
def make_five_engine(kind, Ps, Ph, W, H, caps, dev):
    from exavatar_release_b200 import plan as PL
    if kind == "merged" and hasattr(PL, "MergedFivePlan"):
        return PL.MergedFivePlan(Ps, Ph, W, H, caps, dev), "merged"
    return PL.FiveRenderPlan(Ps, Ph, W, H, caps, dev), "separate"


def bench_five(env, args, wl, wl_key):
    from exavatar_release_b200 import rasterizer as RZ
    from exavatar_release_b200.renderer import GaussianRenderer, render_settings
    from exavatar_release_b200.sharding import shard_frames
    dev, lib, world, rank = env.dev, env.lib, env.world, env.rank
    F, K, Wm = args.frames, args.steps, max(args.warmup, 3)
    H, Wd = wl.height, wl.width
    N = H * Wd
    Ps, Ph = wl.n_scene, wl.n_avatar
    bg_w = torch.ones(3, device=dev)
    bg_r = torch.tensor(BG_RAND, device=dev)
    scene_a, human_a, refined_a = make_population_assets(wl_key, seed=0, device=dev)

    def cams_for(frames):
        cs = [look_at_cam_param(frame_yaw(f), (H, Wd), device=dev) for f in frames]
        return cs, [render_settings((H, Wd), c, bg_w) for c in cs], [render_settings((H, Wd), c, bg_r) for c in cs]

    weak_frames = [rank * F + f for f in range(F)]
    cams, st_w, st_r = cams_for(weak_frames)
    g5 = [{r: make_grad_image(wl_key, seed=10 * f + j, device=dev) for j, r in enumerate(FIVE)} for f in range(8)]

    # ---- capacities: one probing pass with generous room, then the real engines ----
    probe, _ = make_five_engine(args.engine, Ps, Ph, Wd, H, None, dev)
    probe.set_scene(scene_a)
    need = {}
    for f in range(len(cams)):
        probe.frame(("probe", f), st_w[f], st_r[f], scene_a, human_a, refined_a, g5[f % 8], accumulate=False)
        torch.cuda.synchronize(dev)
        for k, v in probe.dups().items():
            need[k] = max(need.get(k, 0), v)
    del probe
    torch.cuda.empty_cache()
    caps = {k: int(v * 1.1) + 4096 for k, v in need.items()}
    # S training frames in flight ("lanes"): frame f runs on engine f mod S, each engine on its own stream with its own
    # workspace, gradient bucket and densification statistics; the latency-bound head of one frame (project / scan /
    # scatter / sort) then overlaps the composites of another.  Buckets are summed in a fixed order: deterministic.
    S = max(1, min(args.lanes, F))
    engines, engine_kind = [], None
    for _ in range(S):
        e, engine_kind = make_five_engine(args.engine, Ps, Ph, Wd, H, caps, dev)
        engines.append(e)
    engine = engines[0]
    lane_streams = [torch.cuda.Stream(dev) for _ in range(S)]
    # densification statistics of the step: the two sums live at the tail of each engine's flat bucket (one sum all-reduce
    # covers gradients and statistics), the maximum is its own small tensor
    lane_stats = [dict(e.stats(), radius_max=torch.zeros(Ps, device=dev)) for e in engines]
    stats = lane_stats[0]  # xyz_grad_accum / track_cnt increments and radius_max of the step (after the lane fold)
    flat = engine.flat_bucket()  # ONE flat fp32 buffer: every per-Gaussian gradient of the three parameter sets + the sums

    def body_for(frame_ids, sts_w, sts_r, scale=None):
        gimgs = g5 if scale is None else [{r: g * scale for r, g in gf.items()} for gf in g5]

        def body():
            cur = torch.cuda.current_stream(dev)
            used = min(S, len(frame_ids))
            for s_ in range(used):
                st_ = lane_streams[s_]
                st_.wait_stream(cur)
                with torch.cuda.stream(st_):
                    e = engines[s_]
                    e.set_scene(scene_a)
                    e.zero_stats()
                    lane_stats[s_]["radius_max"].zero_()
                    for j, idx in enumerate(range(s_, len(frame_ids), S)):
                        f = frame_ids[idx]
                        e.frame(("f", f), sts_w[idx], sts_r[idx], scene_a, human_a, refined_a, gimgs[f % 8],
                                accumulate=(j > 0), densify=lane_stats[s_])
                    e.reduce()
            for s_ in range(used):
                cur.wait_stream(lane_streams[s_])
            for s_ in range(1, used):  # fold the lanes, fixed order (the statistics sums are part of the bucket)
                flat.add_(engines[s_].flat_bucket())
                torch.maximum(stats["radius_max"], lane_stats[s_]["radius_max"], out=stats["radius_max"])
        return body

    body = body_for(weak_frames, st_w, st_r)
    graph, launches_per_step = (None, 0)
    coll_in_graph = False
    if not args.no_graph:
        if world > 1 and not args.no_graph_collectives:
            # the collectives as nodes of the step graph: no host launch gap between the last kernel and the all-reduce
            try:
                for _ in range(2):  # NCCL warm-up outside the capture
                    env.dist.all_reduce(flat)
                    env.dist.all_reduce(lane_stats[0]["radius_max"], op=env.dist.ReduceOp.MAX)
                torch.cuda.synchronize(dev)

                def body_c():
                    body()
                    env.dist.all_reduce(flat)
                    env.dist.all_reduce(lane_stats[0]["radius_max"], op=env.dist.ReduceOp.MAX)
                graph, launches_per_step = env.capture(body_c)
                coll_in_graph = True
            except Exception as exc:
                print(f"bench.py: capturing the collectives failed ({type(exc).__name__}: {exc}); issuing them after the replay",
                      file=sys.stderr)
                torch.cuda.synchronize(dev)
                graph = None
        if graph is None:
            graph, launches_per_step = env.capture(body)

    def collectives():
        """SURVEY 8e: ONE sum all-reduce of the flat bucket (gradients + the xyz_grad_accum / track_cnt increments of
        module.py:155-157 at its tail) and one small max all-reduce (radius_max, model.py:283-285)."""
        env.dist.all_reduce(flat)
        env.dist.all_reduce(stats["radius_max"], op=env.dist.ReduceOp.MAX)

    def step():
        if graph is not None:
            graph.replay()
        else:
            body()
        if world > 1 and not coll_in_graph:
            collectives()

    for _ in range(Wm):
        step()
    clocks = ClockSampler(env.local) if rank == 0 else None
    ms_total, wall, launches_eager = env.timed(step, K)
    outputs = None
    if args.dump_outputs and rank == 0:
        # what the step hands its caller: the summed gradients of the three parameter sets, the densification
        # statistics (both after the lane fold) and the five renders of the step's last frame
        outputs = {f"grad_{s}_{k}": v for s in ("scene", "human", "human_refined") for k, v in engine.grads(s).items()}
        outputs.update({f"densify_{k}": v for k, v in stats.items()})
        for r in FIVE:
            outputs.update(zip((f"{r}_color", f"{r}_alpha", f"{r}_radii"), engines[(F - 1) % S].render_outputs(r)))
        outputs = {k: v.clone() for k, v in outputs.items()}
    if clocks is not None and len(clocks.samples) < 20:
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end and len(clocks.samples) < 40:
            step()
            torch.cuda.synchronize(dev)
        clocks.window = "timed region, then the same step replayed untimed until >= 20 NVML samples were taken"
    clk = clocks.stop() if clocks else None
    if any(e.overflowed() for e in engines):
        raise SystemExit("bench.py: duplicate capacity overflowed; results invalid")
    launches = launches_eager if graph is None else K * launches_per_step
    fps = world * F * K / (ms_total * 1e-3)

    # ---- collective cost alone (N > 1): the same reductions, timed without the renders ----
    coll = None
    if world > 1:
        for _ in range(3):
            collectives()
        ms_c, _, _ = env.timed(collectives, 10)
        coll = {"ms_per_step": ms_c / 10, "bucket_bytes": int(flat.numel() * 4), "in_step_graph": coll_in_graph,
                "what": "ncclAllReduce(sum) of the flat bucket (gradients + densification sums) + one small max all-reduce "
                        "(radius_max), timed alone"}

    # ---- per-kernel durations: the renders of one step, one at a time, in-library events ----
    lib.b2r_profile_enable(1)
    env.profile_read()
    prof_steps = min(K, 3)
    cons = []
    for s in range(prof_steps):
        env.flush_buf.zero_()
        engine.set_scene(scene_a)
        for j, f in enumerate(weak_frames):
            engine.frame(("f", f), st_w[j], st_r[j], scene_a, human_a, refined_a, g5[f % 8], accumulate=(j > 0),
                         densify=stats, serial=True)
            if s == 0:
                cons.append(engine.consumed())
    per_kernel = env.profile_read()
    lib.b2r_profile_enable(0)
    tiles = ((Wd + 15) // 16) * ((H + 15) // 16)
    # average over the composite launches of a frame (5 forward, 5 backward)
    Cf = sum(sum(c["fwd"]) for c in cons) / sum(len(c["fwd"]) for c in cons)
    Cb = sum(sum(c["bwd"]) for c in cons) / sum(len(c["bwd"]) for c in cons)
    algo = {"composite_fwd": 44.0 * Cf + 24.0 * N + 8.0 * tiles, "composite_bwd": 84.0 * Cb + 20.0 * N}
    frame_kernel_ms = sum(v["ms_avg"] * v["launches"] for v in per_kernel.values()) / (prof_steps * F)
    # per-view composite launches of one frame (merged engine): the five launches differ by an order of magnitude in work
    per_view = None
    if engine_kind == "merged":
        from exavatar_release_b200 import _lib as LL
        peak = float(peaks_and_traffic(wl_key, "composite_fwd")[0].get("hbm_gbs", 6650.0))
        lib.b2r_profile_enable(1)
        env.profile_read()
        per_view, last = {}, {"A": (0, 0), "B": (0, 0)}

        def probe(label):
            torch.cuda.synchronize(dev)
            pk_ms = env.profile_read()
            parts = label.split(":")
            if len(parts) != 3:
                return
            pk, name, which = parts
            st = engine.passes[pk].status()
            key = "consumed_fwd" if which == "fwd" else "consumed_bwd"
            div = LL.CONSUMED_FWD_DIV if which == "fwd" else LL.CONSUMED_BWD_DIV
            idx = 0 if which == "fwd" else 1
            c = (st[key] - last[pk][idx]) / div
            last[pk] = (st[key], last[pk][1]) if which == "fwd" else (last[pk][0], st[key])
            ms = pk_ms["composite_fwd" if which == "fwd" else "composite_bwd"]["ms_avg"]
            nbytes = (44.0 * c + 24.0 * N + 8.0 * tiles) if which == "fwd" else (84.0 * c + 20.0 * N)
            per_view.setdefault(name, {})[which] = {"ms": round(ms, 5), "consumed": c, "algorithmic_bytes": nbytes,
                                                     "frac": (nbytes / (ms * 1e-3) / 1e9 / peak) if ms > 0 else None}

        engine.set_scene(scene_a)
        engine.frame(("f", weak_frames[0]), st_w[0], st_r[0], scene_a, human_a, refined_a, g5[weak_frames[0] % 8],
                     accumulate=False, serial=True, probe=probe)
        torch.cuda.synchronize(dev)
        lib.b2r_profile_enable(0)
    roofline = roofline_dict(per_kernel, algo, wl_key + "/five", {
        "sum_kernel_ms_per_training_frame": frame_kernel_ms, "consumed_fwd_per_render": Cf, "consumed_bwd_per_render": Cb,
        "dups_needed": need, "per_view": per_view,
        "note": "per-launch averages over the five composite launches of a training frame; three of the five views skip "
                "the tiles no human Gaussian reaches (see per_view for each launch)"})

    # ---- strong scaling (configs[3] literally): global batch of 8 frames over the ranks ----
    strong = None
    if world > 1:
        G = 8
        mine = shard_frames(G, rank, world)
        cs, sw, sr = cams_for(mine)
        sbody = body_for(mine, sw, sr, scale=1.0 / G) if mine else (lambda: None)  # loss pre-divided (train.py:43)
        sgraph = None
        if mine and not args.no_graph:
            sgraph, _ = env.capture(sbody)

        def sstep():
            if sgraph is not None:
                sgraph.replay()
            else:
                sbody()
            collectives()

        for _ in range(3):
            sstep()
        ks = K
        ms_s, _, _ = env.timed(sstep, ks)
        strong = {"value": G * ks / (ms_s * 1e-3), "unit": UNIT, "global_batch": G, "frames_per_rank": len(mine),
                  "ms_per_step": ms_s / ks, "steps": ks,
                  "semantics": "rank r renders frames r::N of the 8-frame batch, dL/dimage pre-divided by 8 "
                               "(loss.mean(), train.py:43); gradient bucket + densify statistics all-reduced"}

    # ---- end to end through the public API with host buffers ----
    e2e, e2e_eager, e2e_merged = None, None, None
    if not args.no_e2e:
        caps_merged = caps if "A" in caps else {"A": int(need["scene_human"] * 1.1) + 4096,
                                                 "B": int(need["scene_human_refined"] * 1.1) + 4096}
        e2e, e2e_eager, e2e_merged = e2e_five(env, args, wl, wl_key, cams, st_w, st_r, scene_a, human_a, refined_a,
                                              max(caps.values()), caps_merged, collectives if world > 1 else None)

    extra = {"cuda_graph": graph is not None, "dup_capacity": caps, "engine": engine_kind, "lanes": S,
             "streams": engine.describe() + f"; {S} training frame(s) in flight"}
    return {"value": fps, "ms_per_step": ms_total / K, "clocks": clk, "launches": int(launches), "roofline": roofline,
            "e2e": e2e, "e2e_eager": e2e_eager, "e2e_merged": e2e_merged, "strong_scaling": strong, "collective": coll,
            "wall": wall, "config": extra, "warmup": Wm, "outputs": outputs}


def e2e_five(env, args, wl, wl_key, cams, st_w, st_r, scene_a, human_a, refined_a, cap, caps_merged, collectives):
    """ExAvatar's training frame through the PUBLIC API with pinned host buffers (see module docstring)."""
    from exavatar_release_b200 import rasterizer as RZ
    from exavatar_release_b200.renderer import GaussianRenderer
    dev, world = env.dev, env.world
    F, K = args.frames, args.steps
    H, Wd = wl.height, wl.width
    N = H * Wd
    bg_w = torch.ones(3, device=dev)
    bg_r = torch.tensor(BG_RAND, device=dev)
    sets = {"scene": scene_a, "human": human_a, "refined": refined_a}
    host = {n: {k: v.cpu().pin_memory() for k, v in a.items()} for n, a in sets.items()}
    host_grads = {n: {k: torch.empty_like(v).pin_memory() for k, v in a.items()} for n, a in host.items()}
    host_targets = [torch.rand(3, H, Wd).pin_memory() for _ in range(F)]
    host_loss = torch.empty(F).pin_memory()
    nbytes = lambda d: sum(v.numel() * 4 for a in d.values() for v in a.values())
    h2d = nbytes(host) + F * 3 * N * 4
    d2h = nbytes(host_grads) + F * 4
    renderer = GaussianRenderer()
    # frames in flight on the autograd path (each frame: five renders in sequence on its lane)
    # measured on C4 (e2e | e2e_merged): 4 lanes 960 | 1312, 6: 957 | 1228, 8: 997 | 1249 training frames/s
    S = max(1, min(args.e2e_lanes if args.e2e_lanes else 8, F))        # five-call legs (graph and eager)
    S_fused = max(1, min(args.e2e_lanes if args.e2e_lanes else 4, F))  # one fused call per frame keeps ~6 kernels in flight itself
    cat = lambda a, b: {k: torch.cat((a[k].detach(), b[k])) for k in a}  # model.py:117-125

    fused = []  # one TrainingFrameRenderer per lane (built lazily for the e2e_merged leg)

    def frame_loss_fused(lv, f, tgt, lane, wait_set):
        wait_set("human"); wait_set("refined")  # one call renders all five: it needs every set
        out = fused[lane](lv["scene"], lv["human"], lv["refined"], cams[f], bg_r, raster_settings=st_w[f],
                          raster_settings_human=st_r[f])
        imgs = [out[r]["img"] for r in FIVE]
        wait_set("target")
        return sum(torch.nn.functional.l1_loss(im, tgt) for im in imgs), imgs

    def frame_loss(lv, f, tgt, use_cached_settings, wait_set):
        kw_w = {"raster_settings": st_w[f]} if use_cached_settings else {}
        kw_r = {"raster_settings": st_r[f]} if use_cached_settings else {}
        shape = (H, Wd)
        imgs = [renderer(lv["scene"], shape, cams[f], **kw_w)["img"]]
        wait_set("human")
        imgs += [renderer(lv["human"], shape, cams[f], bg_r, **kw_r)["img"],
                 renderer(cat(lv["scene"], lv["human"]), shape, cams[f], **kw_w)["img"]]
        wait_set("refined")
        imgs += [renderer(lv["refined"], shape, cams[f], bg_r, **kw_r)["img"],
                 renderer(cat(lv["scene"], lv["refined"]), shape, cams[f], **kw_w)["img"]]
        wait_set("target")
        return sum(torch.nn.functional.l1_loss(im, tgt) for im in imgs), imgs

    keep_alive = []
    h2d_s, d2h_s = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    lane_s_all = [torch.cuda.Stream(dev) for _ in range(S)]

    def body(use_cached_settings=True, use_fused=False):
        cur = torch.cuda.current_stream(dev)
        S = S_fused if use_fused else len(lane_s_all)
        lane_s = lane_s_all[:S]
        for st_ in lane_s:
            st_.wait_stream(cur)
        d2h_s.wait_stream(cur)
        h2d_s.wait_stream(cur)
        with torch.cuda.stream(h2d_s):
            # scene first: the frames start on it while the two human sets are still on the wire (each render waits for
            # the sets it reads, below)
            params, ev_set = {}, {}
            tgts, ev_t = [None] * F, [None] * F

            def up_set(n):
                params[n] = {k: v.to(dev, non_blocking=True) for k, v in host[n].items()}
                ev_set[n] = torch.cuda.Event()
                ev_set[n].record(h2d_s)

            def up_tgt(f):
                tgts[f] = host_targets[f].to(dev, non_blocking=True)
                ev_t[f] = torch.cuda.Event()
                ev_t[f].record(h2d_s)

            for n in ("scene", "human", "refined"):
                up_set(n)
            for f in range(F):  # the losses come after the fifth render: the targets travel last
                up_tgt(f)
        keep_alive.append((params, tgts))
        leaves = []
        for st_ in lane_s:
            st_.wait_event(ev_set["scene"])
            with torch.cuda.stream(st_):  # views of the uploaded tensors: no kernel runs here
                leaves.append({n: {k: v.detach().requires_grad_() for k, v in a.items()} for n, a in params.items()})
        need = {}  # per lane: has this lane's stream waited for the set yet?
        losses = []
        for f in range(F):
            fs, lv = lane_s[f % S], leaves[f % S]
            with torch.cuda.stream(fs):
                wait_set = lambda n, fs=fs, lane=f % S, f=f: (fs.wait_event(ev_t[f]) if n == "target" else
                                                               need.setdefault((lane, n), fs.wait_event(ev_set[n]) or True))
                loss, imgs = (frame_loss_fused(lv, f, tgts[f], f % S, wait_set) if use_fused
                              else frame_loss(lv, f, tgts[f], use_cached_settings, wait_set))
                loss.backward()
                losses.append(loss.detach().reshape(1))
                keep_alive.append((imgs, loss))
        for st_ in lane_s:
            cur.wait_stream(st_)
        total = {n: {k: leaves[0][n][k].grad for k in host[n]} for n in host}
        for lv in leaves[1:]:
            if lv["scene"]["mean_3d"].grad is not None:
                total = {n: {k: total[n][k] + lv[n][k].grad for k in host[n]} for n in host}
        lvec = torch.cat(losses)
        keep_alive.append((leaves, total, lvec))
        done = torch.cuda.Event()
        done.record(cur)
        with torch.cuda.stream(d2h_s):
            d2h_s.wait_event(done)
            host_loss.copy_(lvec, non_blocking=True)
            for n in host:
                for k in host[n]:
                    host_grads[n][k].copy_(total[n][k], non_blocking=True)
        cur.wait_stream(d2h_s)
        cur.wait_stream(h2d_s)

    # ---- graph-captured step (fixed-capacity mode of the rasteriser: no polling) ----
    RZ.set_fixed_capacity(cap)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            body()
            torch.cuda.synchronize(dev)
            keep_alive.clear()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = None
    if not args.no_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                body()
        except Exception as exc:
            print(f"bench.py: e2e graph capture failed ({type(exc).__name__}: {exc}); timing the eager step", file=sys.stderr)
            graph = None
            torch.cuda.synchronize(dev)

    def step():
        if graph is not None:
            graph.replay()
        else:
            body()
            torch.cuda.synchronize(dev)
            keep_alive.clear()
        if collectives is not None:
            collectives()

    for _ in range(3):
        step()
    ke = K
    ms_e, _, _ = env.timed(step, ke)
    if args.trace_e2e and env.rank == 0:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize(dev)
        prof.export_chrome_trace(args.trace_e2e)
    if RZ.overflowed():
        raise SystemExit("bench.py: e2e leg overflowed its fixed duplicate capacity; results invalid")
    RZ.set_fixed_capacity(None)
    e2e = {"value": world * F * ke / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "upload": "per step: the three Gaussian parameter sets (scene, human, human_refined) + one target image per "
                     "frame up; the summed gradients of the three sets + per-frame losses down",
           "api": "5x GaussianRenderer.forward -> GaussianRasterizer (autograd) per frame, L1 loss on each image, one "
                  "backward per frame, pinned host buffers; " + ("whole step captured in a CUDA graph, copies on forked streams"
                                                                  if graph is not None else "eager, copies on side streams"),
           "steps": ke, "lanes": S}

    # ---- the same step through TrainingFrameRenderer: one autograd call per frame, two merged passes (SURVEY 8f-3) ----
    merged = None
    try:
        from exavatar_release_b200 import TrainingFrameRenderer
        for _ in range(S_fused):
            fused.append(TrainingFrameRenderer(wl.n_scene, wl.n_avatar, (H, Wd), dev, caps_merged))
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                body(use_fused=True)
                torch.cuda.synchronize(dev)
                keep_alive.clear()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        mgraph = None
        if not args.no_graph:
            mgraph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(mgraph):
                body(use_fused=True)

        def mstep():
            if mgraph is not None:
                mgraph.replay()
            else:
                body(use_fused=True)
                torch.cuda.synchronize(dev)
                keep_alive.clear()
            if collectives is not None:
                collectives()

        for _ in range(3):
            mstep()
        ms_m, _, _ = env.timed(mstep, ke)
        if any(fr.overflowed() for fr in fused):
            raise RuntimeError("fixed duplicate capacity overflowed")
        merged = {"value": world * F * ke / (ms_m * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                  "steps": ke, "lanes": S_fused,
                  "api": "TrainingFrameRenderer (exavatar_release_b200/fused.py): the five renders of model.py:117-162 as one "
                         "autograd call per frame (two merged projection+binning passes, five views), same losses, copies "
                         "and graph capture as `e2e`; needs the caller to replace model.py:117-162 (INTEGRATION.md)"}
        del mgraph
        fused.clear()
        keep_alive.clear()
        torch.cuda.empty_cache()
    except Exception as exc:  # an extra leg: report, do not fail the bench
        print(f"bench.py: e2e_merged leg failed ({type(exc).__name__}: {exc})", file=sys.stderr)
        torch.cuda.synchronize(dev)

    # ---- eager: the unmodified reference call shape, adaptive capacity, no graph ----
    eager = None
    if not args.no_eager:
        del graph
        keep_alive.clear()

        def eager_step():
            body(use_cached_settings=False)
            torch.cuda.synchronize(dev)
            keep_alive.clear()
            if collectives is not None:
                collectives()

        for _ in range(2):
            eager_step()
        kk = K
        t0 = time.perf_counter()
        ms_g, _, _ = env.timed(eager_step, kk)
        eager = {"value": world * F * kk / (ms_g * 1e-3), "unit": UNIT, "steps": kk,
                 "host_ms_per_render": ms_g / (kk * F * 5),
                 "api": "GaussianRenderer.forward(assets, img_shape, cam_param, bg) exactly as module.py:592 (camera matrices "
                        "rebuilt per call, no cached settings), adaptive duplicate capacity, no CUDA graph"}
    return e2e, eager, merged


# ---------------------------------------------------------------------------------------------------------------
# pattern "single": one render per frame (round-1 bench; C1 / C3 / C5 and the `single_render` key)
# ---------------------------------------------------------------------------------------------------------------
def bench_single(env, args, wl, wl_key, brief=False):
    from exavatar_release_b200 import rasterizer as RZ
    from exavatar_release_b200.plan import FrameLanes
    from exavatar_release_b200.renderer import GaussianRenderer, render_settings
    dev, lib, world, rank = env.dev, env.lib, env.world, env.rank
    dist = env.dist
    F, K, Wm = args.frames, args.steps, max(args.warmup, 3)
    P, H, Wd = wl.n_avatar + wl.n_scene, wl.height, wl.width
    N = H * Wd
    use_sh = wl.sh_degree > 0
    M = (wl.sh_degree + 1) ** 2 if use_sh else 0
    bg = torch.ones(3, device=dev)

    assets = make_assets(wl_key, seed=0, device=dev)
    gimgs = [make_grad_image(wl_key, seed=f, device=dev) for f in range(F)]
    cams = [look_at_cam_param(frame_yaw(rank * F + f), (H, Wd), device=dev) for f in range(F)]
    settings = []
    for c in cams:
        st = render_settings((H, Wd), c, bg)
        settings.append(st._replace(sh_degree=wl.sh_degree) if use_sh else st)

    def public_frame(f, leaves=None, grad=True):
        lv = leaves or {k: v.detach().requires_grad_(wl.backward and grad) for k, v in assets.items()}
        m2 = torch.zeros(P, 3, device=dev, requires_grad=wl.backward and grad)
        rast = RZ.GaussianRasterizer(settings[f])
        img = rast(means3D=lv["mean_3d"], means2D=m2, opacities=lv["opacity"], shs=lv["shs"] if use_sh else None,
                   colors_precomp=None if use_sh else lv["rgb"], scales=lv["scale"], rotations=lv["rotation"])[0]
        return img, lv, m2

    dups = []
    with torch.no_grad():
        for f in range(F):
            public_frame(f, grad=False)
            dups.append(RZ.last_duplicate_count(dev, P, Wd, H))
    cap = int(max(dups) * 1.1) + 4096

    S = max(1, min(args.lanes, F))
    lanes = FrameLanes(S, P, Wd, H, cap, dev, sh_coeffs=M)
    plan = lanes.plans[0]
    scenes = [lanes.scene(f, settings[f], assets) for f in range(F)]
    bucket, views = lanes.bucket, lanes.lane_views[0]

    def step_body():
        lanes.step(scenes, gimgs, backward=wl.backward)

    graph, launches_per_step = (None, 0)
    if not args.no_graph:
        graph, launches_per_step = env.capture(step_body)

    def step():
        if graph is not None:
            graph.replay()
        else:
            step_body()
        if world > 1 and wl.backward:
            dist.all_reduce(bucket)

    for _ in range(Wm):
        step()
    clocks = ClockSampler(env.local) if (rank == 0 and not brief) else None
    ms_total, wall, launches_eager = env.timed(step, K)
    outputs = None
    if args.dump_outputs and rank == 0 and not brief:
        last = lanes.plans[(F - 1) % S]  # frame f runs on lane f mod S
        outputs = {"color": last.color, "depth": last.depth, "alpha": last.alpha, "radii": last.radii}
        if wl.backward:  # the gradients summed over the step's frames
            outputs.update({f"grad_{k}": v for k, v in lanes.views.items()})
        outputs = {k: v.clone() for k, v in outputs.items()}
    if clocks is not None and len(clocks.samples) < 20:
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end and len(clocks.samples) < 40:
            for _ in range(4):
                step()
            torch.cuda.synchronize(dev)
        clocks.window = "timed region, then the same step replayed untimed until >= 20 NVML samples were taken"
    clk = clocks.stop() if clocks else None
    if lanes.status()["overflow"]:
        raise SystemExit("bench.py: duplicate capacity overflowed; results invalid")
    launches = launches_eager if graph is None else K * launches_per_step
    fps = world * F * K / (ms_total * 1e-3)
    # ---- per-kernel durations (same step, eager, in-library events) ----
    lib.b2r_profile_enable(1)
    env.profile_read()
    cons_f, cons_b, ndups = [], [], []
    prof_steps = min(K, 5)
    for s in range(prof_steps):
        env.flush_buf.zero_()
        for f in range(F):
            plan.forward(scenes[f])
            if wl.backward:
                plan.backward(scenes[f], gimgs[f], views, accumulate=(f > 0))
            if s == 0:
                stt = plan.status()
                cf, cb = consumed_units(stt)
                cons_f.append(cf); cons_b.append(cb); ndups.append(stt["num_dups"])
    per_kernel = env.profile_read()
    lib.b2r_profile_enable(0)
    tiles = ((Wd + 15) // 16) * ((H + 15) // 16)
    Cf = sum(cons_f) / len(cons_f)
    Cb = sum(cons_b) / len(cons_b) if wl.backward else 0.0
    algo = {"composite_fwd": 44.0 * Cf + 24.0 * N + 8.0 * tiles, "composite_bwd": 84.0 * Cb + 20.0 * N}
    frame_kernel_ms = sum(v["ms_avg"] * v["launches"] for v in per_kernel.values()) / (prof_steps * F)
    roofline = roofline_dict(per_kernel, algo, wl_key, {
        "sum_kernel_ms_per_frame": frame_kernel_ms, "consumed_fwd_per_frame": Cf, "consumed_bwd_per_frame": Cb,
        "dups_per_frame": sum(ndups) / len(ndups)})
    if brief:  # the extra key of the five-render line: throughput + the composites' own roofline numbers on this workload
        oc = roofline["other_composite"]
        comp = {roofline["kernel"]: {"kernel_ms_avg": roofline["kernel_ms_avg"], "frac": roofline["frac"],
                                     "algorithmic_bytes_per_launch": roofline["algorithmic_bytes_per_launch"]},
                oc["kernel"]: {"kernel_ms_avg": oc["kernel_ms_avg"], "frac": oc["frac"],
                               "algorithmic_bytes_per_launch": oc["algorithmic_bytes_per_launch"]}}
        return {"value": fps, "ms_per_step": ms_total / K, "workload": wl.name, "frames_per_rank_per_step": F, "lanes": S,
                "steps": K, "unit": UNIT, "roofline": {"composites": comp, "per_kernel_ms": roofline["per_kernel_ms"],
                                                        "peak": roofline["peak"], "traffic": roofline["traffic"]}}

    # ---- end to end through the public API with host buffers ----
    e2e = None
    e2e_eager = None
    if not args.no_e2e:
        host_assets = {k: v.cpu().pin_memory() for k, v in assets.items() if (k != "rgb" or not use_sh)}
        host_targets = [torch.rand(3, H, Wd).pin_memory() for _ in range(F)]
        host_grads = {k: torch.empty_like(v).pin_memory() for k, v in host_assets.items()}
        host_m2 = torch.empty(P, 3).pin_memory()
        host_loss = torch.empty(F).pin_memory()
        renderer = GaussianRenderer()
        h2d = F * (sum(v.numel() * 4 for v in host_assets.values()) + 3 * N * 4)
        d2h = F * ((sum(v.numel() * 4 for v in host_grads.values()) + P * 12 + 4) if wl.backward else 3 * N * 4)
        host_img = torch.empty(3, H, Wd).pin_memory()
        RZ.set_fixed_capacity(cap)
        h2d_s, d2h_s = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        lane_s_all = [torch.cuda.Stream(dev) for _ in range(S)] if S > 1 else None
        keep_alive = []  # nothing allocated inside the capture may be recycled across the forked streams

        def upload(f, cur):
            h2d_s.wait_stream(cur)
            with torch.cuda.stream(h2d_s):
                lv = {k: v.to(dev, non_blocking=True) for k, v in host_assets.items()}
                tgt = host_targets[f].to(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(h2d_s)
            keep_alive.append((lv, tgt))
            return lv, tgt, ev

        def e2e_frame(f, lv, tgt):
            lv = {k: v.requires_grad_(wl.backward) for k, v in lv.items()}
            if use_sh:
                img, _, m2 = public_frame(f, leaves=lv)
            else:
                o = renderer(lv, (H, Wd), cams[f], bg, raster_settings=settings[f])
                img, m2 = o["img"], o["mean_2d"]
            if wl.backward:
                loss = (img - tgt).abs().mean()
                loss.backward()
                outs = [(host_loss[f:f + 1], loss.detach().reshape(1)), (host_m2, m2.grad)]
                outs += [(host_grads[k], lv[k].grad) for k in host_grads]
            else:
                outs = [(host_img, img.detach())]
            keep_alive.append((lv, img, m2, outs))
            return outs

        def e2e_body_per_frame():
            cur = torch.cuda.current_stream(dev)
            if lane_s:
                for ls in lane_s:
                    ls.wait_stream(cur)
            d2h_s.wait_stream(cur)
            nxt = upload(0, cur)
            for f in range(F):
                lv, tgt, ev = nxt
                if f + 1 < F:
                    nxt = upload(f + 1, cur)
                fs = lane_s[f % S] if lane_s else cur  # frame f runs on lane f mod S
                fs.wait_event(ev)
                with torch.cuda.stream(fs):
                    outs = e2e_frame(f, lv, tgt)
                    done = torch.cuda.Event()
                    done.record(fs)
                with torch.cuda.stream(d2h_s):
                    d2h_s.wait_event(done)
                    for dst, src in outs:
                        dst.copy_(src, non_blocking=True)
            cur.wait_stream(d2h_s)  # the step ends when its last result is in host memory (joins the forked streams)
            cur.wait_stream(h2d_s)
            if lane_s:
                for ls in lane_s:
                    cur.wait_stream(ls)

        eager_call = [False]  # True: the unmodified reference call shape (no cached raster settings)

        def e2e_body_per_step():
            """One training step as ExAvatar runs it (train.py:35-57): the frames of the batch render the SAME parameter
            set, the loss gradients of all frames are summed into the parameters' .grad, the optimiser would read those.
            Host -> device: the parameter set once, one target image per frame.  Device -> host: the summed gradients
            and the per-frame losses."""
            cur = torch.cuda.current_stream(dev)
            streams = lane_s if lane_s else [cur]
            for st_ in (lane_s or []):
                st_.wait_stream(cur)
            d2h_s.wait_stream(cur)
            h2d_s.wait_stream(cur)
            with torch.cuda.stream(h2d_s):
                params = {k: v.to(dev, non_blocking=True) for k, v in host_assets.items()}
                ev_p = torch.cuda.Event()
                ev_p.record(h2d_s)
                tgts, ev_t = [], []
                for f in range(F):
                    tgts.append(host_targets[f].to(dev, non_blocking=True))
                    e = torch.cuda.Event()
                    e.record(h2d_s)
                    ev_t.append(e)
            keep_alive.append((params, tgts))
            leaves = []
            for st_ in streams:  # lane-private leaf views of the one uploaded parameter set
                st_.wait_event(ev_p)
                with torch.cuda.stream(st_):
                    leaves.append({k: v.detach().requires_grad_(wl.backward) for k, v in params.items()})
            losses = []
            for f in range(F):
                fs = streams[f % len(streams)]
                lv = leaves[f % len(streams)]
                with torch.cuda.stream(fs):
                    if use_sh:
                        img, _, m2 = public_frame(f, leaves=lv)
                    else:
                        kw = {} if eager_call[0] else {"raster_settings": settings[f]}
                        o = renderer(lv, (H, Wd), cams[f], bg, **kw)
                        img, m2 = o["img"], o["mean_2d"]
                    if wl.backward:
                        fs.wait_event(ev_t[f])  # the target image is only needed here: its upload overlaps the forward
                        loss = torch.nn.functional.l1_loss(img, tgts[f])
                        loss.backward()  # accumulates into this lane's leaves
                        losses.append(loss.detach().reshape(1))
                        keep_alive.append((img, m2, loss))
                    else:
                        done = torch.cuda.Event()
                        done.record(fs)
                        keep_alive.append((img, m2))
                        with torch.cuda.stream(d2h_s):
                            d2h_s.wait_event(done)
                            host_img.copy_(img.detach(), non_blocking=True)
            for st_ in (lane_s or []):
                cur.wait_stream(st_)
            if wl.backward:
                total = {k: leaves[0][k].grad for k in host_grads}
                for lv in leaves[1:]:
                    if lv[next(iter(host_grads))].grad is not None:
                        total = {k: total[k] + lv[k].grad for k in host_grads}
                lvec = torch.cat(losses)
                keep_alive.append((leaves, total, lvec))
                done = torch.cuda.Event()
                done.record(cur)
                with torch.cuda.stream(d2h_s):
                    d2h_s.wait_event(done)
                    host_loss.copy_(lvec, non_blocking=True)
                    for k in host_grads:
                        host_grads[k].copy_(total[k], non_blocking=True)
            cur.wait_stream(d2h_s)
            cur.wait_stream(h2d_s)

        per_step = args.e2e_upload == "per-step"
        e2e_body = e2e_body_per_step if per_step else e2e_body_per_frame
        if per_step:
            h2d = sum(v.numel() * 4 for v in host_assets.values()) + F * 3 * N * 4
            d2h = (sum(v.numel() * 4 for v in host_grads.values()) + F * 4) if wl.backward else F * 3 * N * 4

        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                e2e_body()
                torch.cuda.synchronize(dev)  # buffers cross streams: do not recycle them while a lane may still read
                keep_alive.clear()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        e2e_graph = None
        if not args.no_graph:
            try:
                e2e_graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(e2e_graph):
                    e2e_body()
            except Exception as exc:  # report, fall back to eager replay of the same body
                print(f"bench.py: e2e graph capture failed ({type(exc).__name__}: {exc}); timing the eager step", file=sys.stderr)
                e2e_graph = None
                torch.cuda.synchronize(dev)

        def e2e_step():
            if e2e_graph is not None:
                e2e_graph.replay()
            else:
                e2e_body()
                torch.cuda.synchronize(dev)
                keep_alive.clear()
            if world > 1 and wl.backward:
                dist.all_reduce(bucket)  # same collective as the device-resident leg

        for _ in range(3):
            e2e_step()
        ke = K
        ms_e, _, _ = env.timed(e2e_step, ke)
        if args.trace_e2e and rank == 0:  # after the timed region: one more step under the profiler
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                e2e_step()
                torch.cuda.synchronize(dev)
            prof.export_chrome_trace(args.trace_e2e)
        if RZ.overflowed():
            raise SystemExit("bench.py: e2e leg overflowed its fixed duplicate capacity; results invalid")
        RZ.set_fixed_capacity(None)
        e2e = {"value": world * F * ke / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "upload": args.e2e_upload + (": parameter set once per step + one target image per frame up; summed "
                                            "gradients + per-frame losses down" if per_step else
                                            ": every frame uploads the full Gaussian set + target and downloads its gradients"),
               "api": "GaussianRenderer.forward -> GaussianRasterizer (autograd) + L1 loss + backward, pinned host buffers; "
                      + ("whole step captured in a CUDA graph, copies on forked streams" if e2e_graph is not None
                         else "eager, copies on side streams"),
               "steps": ke}

        # ---- eager: the unmodified reference call shape, adaptive duplicate capacity, no graph ----
        if not args.no_eager and per_step and not use_sh:
            e2e_graph = None
            keep_alive.clear()
            eager_call[0] = True

            def eager_step():
                e2e_body()
                torch.cuda.synchronize(dev)
                keep_alive.clear()
                if world > 1 and wl.backward:
                    dist.all_reduce(bucket)

            for _ in range(2):
                eager_step()
            kk = K
            ms_g, _, _ = env.timed(eager_step, kk)
            eager_call[0] = False
            e2e_eager = {"value": world * F * kk / (ms_g * 1e-3), "unit": UNIT, "steps": kk,
                         "host_ms_per_render": ms_g / (kk * F), "lanes": S,
                         "api": "GaussianRenderer.forward(assets, img_shape, cam_param, bg) exactly as module.py:592 (camera "
                                "matrices rebuilt per call, no cached settings), adaptive duplicate capacity, no CUDA graph; "
                                "same copies as `e2e`"}

    return {"value": fps, "ms_per_step": ms_total / K, "clocks": clk, "launches": int(launches), "roofline": roofline,
            "e2e": e2e, "e2e_eager": e2e_eager, "e2e_merged": None, "strong_scaling": None, "collective": None, "wall": wall,
            "config": {"cuda_graph": graph is not None, "dup_capacity": cap, "lanes": S}, "warmup": Wm, "outputs": outputs}


def run_b200(args):
    env = Env(args)
    wl = WORKLOADS[args.workload]
    pattern = resolve_pattern(args, wl)
    res = bench_five(env, args, wl, args.workload) if pattern == "five" else bench_single(env, args, wl, args.workload)

    single = None
    if pattern == "five" and not args.no_single:  # continuity with round 1: BASELINE configs[1], one render per frame
        args.lanes = args._lanes_user if args._lanes_user is not None else 4
        single = bench_single(env, args, WORKLOADS["C2"], "C2", brief=True)

    cpu = None
    if env.rank == 0 and env.world == 1 and not args.no_cpu_baseline:  # reported at N = 1 only
        frame, threads = cpu_frame_fn(args.workload, pattern)
        frame(0)
        n, t0 = 0, time.perf_counter()
        while True:
            frame(n); n += 1
            if time.perf_counter() - t0 > args.cpu_seconds or n >= 64:
                break
        dt = time.perf_counter() - t0
        what = "training frame(s) (5 renders fwd+bwd each)" if pattern == "five" else "frame(s)"
        cpu = {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{n} {what} of {wl.name} on the CPU oracle (OpenMP, {threads} threads), {dt:.1f} s"}

    if env.rank == 0:
        cfg = config_dict(args, wl, pattern, res["config"])
        line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": env.world, "steps": args.steps,
                "warmup": res["warmup"], "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": res["clocks"],
                "e2e": res["e2e"], "gpu_launches": res["launches"], "roofline": res["roofline"], "cpu_baseline": cpu,
                "e2e_eager": res["e2e_eager"], "e2e_merged": res["e2e_merged"], "strong_scaling": res["strong_scaling"],
                "collective": res["collective"],
                "single_render": single, "wall_s_timed_region": res["wall"]}
        print(json.dumps(line), flush=True)
        if res["outputs"] is not None:
            dump_outputs(args.dump_outputs, res["outputs"])
    if env.world > 1:
        env.dist.destroy_process_group()
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs records the B200 arm's step; the reference arm writes none")
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
