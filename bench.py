#!/usr/bin/env python
"""bench.py -- the headline benchmark of the hot path (BASELINE.json).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload metric|cfg2|cfg3|cfg4] [--dump-outputs DIR]

metric   Msplats/s (= splat_count / frame time) and ms/frame, full frame = CSCalcDistances + radix sort + CSCalcViewData +
         draw/blend, sorted every frame (m_SortNthFrame = 1), the camera ORBITING the scene by a fixed step per frame (no two
         consecutive frames share an order, a tile-cost history or a row partition that is already perfect).
workload "metric" (default) is the one BASELINE.json's metric string names: bicycle-sized synthetic scene, 6,131,954 splats,
         Medium, @1920x1080.  At N=1 the line also carries, under "other_configs", the same measurement on configs[1]
         (1200x797, the north-star target / README config) and configs[2] (5,834,784 VeryHigh @1920x1080).
value    device-resident throughput (asset in HBM, render target stays in HBM), CUDA events on the library's stream.
e2e      the same frames through the public call with HOST buffers: per step the uniforms go host->device and the RGBA16F
         render target comes back into pinned host memory (double-buffered asynchronous read-back, all landed before the
         clock stops).
roofline the radix-sort digit pass (k_onesweep), the kernel BASELINE.json's metric names ("radix-sort GB/s vs HBM peak");
         `traffic` and every `*_dram_gbs_physical` come from the committed ncu --set full summary named in "ncu_source".
cpu_baseline / --impl reference: the CPU restatement of the reference's shaders (oracle/), all host cores -- the reference has
         no CPU implementation of this path (SURVEY.md 0 F1) and its C#/HLSL cannot run here, so kind = "port".
N > 1    the group path (include/gsplat_b200.h gs_group_*): key-range-sharded depth sort + one exchange of the order slabs
         (stores into the peers' order buffers over NVLink; NCCL all-gather if CUDA IPC is unavailable), row-range-sharded
         view-calc / binning / compositing + one NCCL exchange of the composited rows, all of it issued by the library
         itself.  Before the timed region EVERY rank renders the same frames on its own GPU alone and asserts that the
         group's draw order and render target are bit-identical.
--dump-outputs DIR  after the timed steps, the render target of the last timed step (what the caller of
         SortAndRenderSplats receives) goes to DIR/render_target.npy as float32 (h, w, 4).  Above 60 MB a fixed, seeded
         sample of its pixels goes instead: render_target_pixels.npy (k, 4) and render_target_pixel_index.npy (k,
         row-major pixel index, float64).  The scene and the camera path are seeded, so two builds run with the same
         arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SORT_BYTES_PER_PAIR_PASS = 16.0   # one digit pass: read key+payload, write key+payload
SORT_BYTES_PER_PAIR = 68.0        # SURVEY.md 8d: one histogram read + 4 passes
FRAME_BYTES_PER_SPLAT = {"Medium": 212.5, "VeryHigh": 408.0}   # SURVEY.md 8d

# name -> (splats, quality, width, height, vertical fov, generator seed, what BASELINE.json calls it)
WORKLOADS = {
    "metric": (6_131_954, "Medium", 1920, 1080, 39.09651, 0x5EED0002, "BASELINE.json metric: bicycle-sized 6.1M splats @1920x1080"),
    "cfg2": (6_131_954, "Medium", 1200, 797, 39.09651, 0x5EED0002, "BASELINE configs[1]: bicycle-sized 6.1M splats @1200x797 (README bench, north-star target)"),
    "cfg3": (5_834_784, "VeryHigh", 1920, 1080, 47.0, 0x5EED0003, "BASELINE configs[2]: garden-sized 5.8M splats @1920x1080, Very High"),
    "cfg4": (6_131_954, "Medium", 3840, 2160, 39.09651, 0x5EED0002, "BASELINE configs[3]: bicycle-sized 6.1M splats @3840x2160"),
}
# kept for the tools that import this module
N_SPLATS, WIDTH, HEIGHT, FOV, SEED = 6_131_954, 1200, 797, 39.09651, 0x5EED0002
ORBIT_STEP_DEG = 0.5
DUMP_BYTES = 60 * 10**6   # --dump-outputs writes less than 64 MB, .npy headers included
NCU_SOURCE = ROOT / "profiles" / "r02_kernels.json"   # written by tools/ncu_kernels_json.py from the committed ncu --set full capture

_assets = {}


def get_asset(n, quality, seed):
    import unitygaussiansplatting_b200 as g
    key = (n, quality, seed)
    if key not in _assets:
        _assets[key] = g.synthetic_asset(g.SCENE_CLUSTERED, n, seed, quality)
    return _assets[key]


def orbit_camera(k, width=None, height=None, fov=None):
    """Frame k of the benchmark's camera path: a circle of radius 6 around (0, 0.5, 0), ORBIT_STEP_DEG per frame, looking at
    the centre; frame 0 is the static camera of SURVEY.md 8d, (0, 0.5, -6) looking +z."""
    import unitygaussiansplatting_b200 as g
    a = np.radians(ORBIT_STEP_DEG * k)
    pos = np.array([-6.0 * np.sin(a), 0.5, -6.0 * np.cos(a)])
    return g.Camera(position=pos, rotation=g.look_rotation([np.sin(a), 0.0, np.cos(a)]), fieldOfView=FOV if fov is None else fov,
                    pixelWidth=WIDTH if width is None else width, pixelHeight=HEIGHT if height is None else height)


def make_scene(n=N_SPLATS, quality="Medium"):
    """(package, asset, frame-0 camera) of the cfg2 scene: what the tools and the full-size tests use."""
    import unitygaussiansplatting_b200 as g
    return g, get_asset(n, quality, SEED), orbit_camera(0)


def host_threads():
    """CPUs this process may really use: affinity mask capped by the cgroup quota.  torchrun exports OMP_NUM_THREADS=1 to its
    workers; the CPU arm must not inherit that."""
    t = len(os.sched_getaffinity(0))
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            t = min(t, max(1, -(-int(q) // int(p))))
    except Exception:
        pass
    return max(1, t)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_kernels():
    try:
        return json.loads(NCU_SOURCE.read_text())
    except Exception:
        return {}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.path = "/tmp/gs_clocks_%d.csv" % os.getpid()
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        return out


def cpu_frame(O, asset, fp, threads, width, height, prev_order=None):
    """One full frame of the CPU restatement; returns seconds per stage, the new order and the render target."""
    order = np.arange(asset.splatCount, dtype=np.uint32) if prev_order is None else prev_order.copy()
    t0 = time.perf_counter()
    keys = O.calc_distances(asset, fp, order, threads)
    t1 = time.perf_counter()
    O.sort_pairs(keys, order, threads)
    t2 = time.perf_counter()
    view = O.calc_view(asset, fp, threads)
    t3 = time.perf_counter()
    rt = O.render(view, order, width, height, 0, threads)
    t4 = time.perf_counter()
    return {"distances": t1 - t0, "sort": t2 - t1, "view": t3 - t2, "draw": t4 - t3, "total": t4 - t0}, order, rt


def dump_outputs(directory, rt):
    """--dump-outputs: the render target as float32, or a fixed, seeded sample of its pixels when it exceeds DUMP_BYTES."""
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    px = np.asarray(rt).reshape(-1, 4).astype(np.float32)
    if px.nbytes <= DUMP_BYTES:
        np.save(d / "render_target.npy", px.reshape(np.shape(rt)))
        return
    k = DUMP_BYTES // (px.itemsize * 4 + 8)
    idx = np.sort(np.random.default_rng(0).choice(px.shape[0], k, replace=False))
    np.save(d / "render_target_pixels.npy", px[idx])
    np.save(d / "render_target_pixel_index.npy", idx.astype(np.float64))


def workload_text(name, n, quality, w, h):
    return "%s: %d splats, %s, %dx%d, sort every frame, camera orbiting %.1f deg/frame" % (WORKLOADS[name][6], n, quality, w, h, ORBIT_STEP_DEG)


def run_reference(args):
    """--impl reference: the CPU restatement of the reference's shaders on all host cores (rank 0 only under torchrun)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    os.environ.pop("OMP_NUM_THREADS", None)   # torchrun's default of 1 is for its GPU workers, not for this arm
    threads = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(threads)
    from oracle import gs_oracle_py as O
    import unitygaussiansplatting_b200 as g
    n, quality, w, h, fov, seed, _ = WORKLOADS[args.workload]
    asset = get_asset(n, quality, seed)
    warm = max(0, min(args.warmup, 1))
    steps = args.steps
    order = None
    times = []
    for k in range(warm + steps):
        fp, _keep = g.make_frame_params(orbit_camera(k, w, h, fov))
        t, order, rt = cpu_frame(O, asset, fp, threads, w, h, order)
        if k >= warm:
            times.append(t)
    t = statistics.mean(x["total"] for x in times)
    val = n / t / 1e6
    line = {"impl": "reference", "metric": "splat throughput, full frame (sort + view-calc + draw)", "value": val, "unit": "Msplats/s",
            "n_gpus": args.gpus, "steps": len(times), "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(args.workload, n, quality, w, h)},
            "cpu_baseline": {"value": val, "unit": "Msplats/s", "cores": threads, "kind": "port",
                             "sample": "full frames of the whole workload; CPU restatement of the reference's "
                                       "HLSL -- the reference has no CPU path"},
            "e2e": {"value": val, "unit": "Msplats/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "stages_ms": {k: statistics.mean(x[k] for x in times) * 1e3 for k in times[0]}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rt)
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
def stage_report(n, quality, w, h, stages, pass_ms, peak, ms_step, nk):
    rep = dict(stages)
    rep["sort_pass_ms"] = pass_ms
    if stages.get("sort_ms"):
        rep["sort_gbs_68B"] = n * SORT_BYTES_PER_PAIR / (stages["sort_ms"] * 1e-3) / 1e9
        rep["sort_frac_of_peak"] = rep["sort_gbs_68B"] / peak
    per_splat_view = 88.25 if quality == "Medium" else 276.0
    per_splat_dist = 12.25 if quality == "Medium" else 20.0
    if stages.get("view_ms"):
        rep["view_gbs_algorithmic_%gB" % per_splat_view] = n * per_splat_view / (stages["view_ms"] * 1e-3) / 1e9
        rep["view_note"] = ("algorithmic bytes (SURVEY 8d) over the fused kernel's time: an EFFECTIVE rate -- the fused kernel skips colour/SH "
                            "of undrawable splats and never writes the 40-byte record; the physical figure is view_dram_gbs_physical")
    if stages.get("distances_ms"):
        rep["distances_gbs_algorithmic_%gB" % per_splat_dist] = n * per_splat_dist / (stages["distances_ms"] * 1e-3) / 1e9
    # physical DRAM traffic per launch from the committed ncu capture, over the time measured live in this run
    for stage, kern, launches in (("sort", "k_onesweep", 4), ("view", "k_calc_view", 1), ("distances", "k_calc_distances", 1), ("raster", "k_raster", 1)):
        k = nk.get(kern)
        if k and stages.get(stage + "_ms"):
            rep[stage + "_dram_gbs_physical"] = k["dram_bytes_per_launch"] * launches / (stages[stage + "_ms"] * 1e-3) / 1e9
    rep["frame_frac_of_hbm_roofline"] = (n * FRAME_BYTES_PER_SPLAT[quality] + w * h * 8) / (ms_step * 1e-3) / 1e9 / peak
    return rep


def measure_single(g, ctx, stream, torch, name, steps, warmup, want_e2e=True, keep_last=False):
    """One GPU, one workload: device-resident value, per-stage times, e2e through host buffers.  keep_last: also return
    the render target of the last timed step ("rt_last")."""
    n, quality, w, h, fov, seed, _ = WORKLOADS[name]
    asset = get_asset(n, quality, seed)
    r = g.GaussianSplatRenderer(asset, ctx)
    cams = [orbit_camera(k, w, h, fov) for k in range(warmup + steps)]
    fps = [r.frame_params(c) for c in cams]      # the app's camera path: uniforms built ahead, handed in (H2D) every frame
    with torch.cuda.stream(stream):
        rt_dev = torch.zeros((h, w, 4), dtype=torch.float16, device="cuda")
        for k in range(warmup):
            r.SortAndRenderSplats(cams[k], rt=rt_dev, fp=fps[k])
        torch.cuda.synchronize()
        launches0 = ctx.stage_times().kernel_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(warmup, warmup + steps):
            r.SortAndRenderSplats(cams[k], rt=rt_dev, fp=fps[k])
        e1.record(stream)
        torch.cuda.synchronize()
        ms_step = e0.elapsed_time(e1) / steps
        launches = ctx.stage_times().kernel_launches - launches0
        rt_last = rt_dev.cpu().numpy() if keep_last else None
        # per-stage device times (CUDA events inside the library, same stream), continuing the orbit
        ctx.set_timing(True)
        acc = {}
        reps = min(steps, 20)
        for k in range(reps):
            r.SortAndRenderSplats(cams[warmup + k], rt=rt_dev, fp=fps[warmup + k])
            st = ctx.stage_times()
            for f in ("distances_ms", "sort_ms", "view_ms", "bin_ms", "raster_ms"):
                acc.setdefault(f, []).append(getattr(st, f))
            acc.setdefault("p", []).append(list(st.sort_pass_ms))
            acc.setdefault("e", []).append(int(st.tile_entries))
        ctx.set_timing(False)
        stages = {k: statistics.median(v) for k, v in acc.items() if k not in ("p", "e")}
        pass_ms = [statistics.median(p[i] for p in acc["p"]) for i in range(4)]
        stages["tile_entries"] = int(statistics.median(acc["e"]))
        e2e_ms = None
        if want_e2e:
            pins = [torch.empty((h, w, 4), dtype=torch.float16, pin_memory=True) for _ in range(2)]
            host = [p.numpy() for p in pins]
            r.async_readback = True
            for k in range(warmup):
                r.SortAndRenderSplats(cams[k], rt=host[k & 1], fp=fps[k])
            ctx.sync()
            t0 = time.perf_counter()
            for k in range(warmup, warmup + steps):
                r.SortAndRenderSplats(cams[k], rt=host[k & 1], fp=fps[k])   # uniforms H2D as kernel arguments, image D2H enqueued
            ctx.sync()                                                      # every read-back has landed
            e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
            r.async_readback = False
    r.Dispose()
    return {"n": n, "quality": quality, "w": w, "h": h, "ms_step": ms_step, "launches": int(launches), "stages": stages, "pass_ms": pass_ms,
            "e2e_ms": e2e_ms, "rt_last": rt_last}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="metric", choices=sorted(WORKLOADS))
    ap.add_argument("--screen", default=None, help="WxH override of the workload's screen")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--baseline-partition", action="store_true", help="N > 1: round 1's interleaved bands + torch all-gather instead of the group path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's render target under DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.screen:
        w, h = (int(v) for v in args.screen.lower().split("x"))
        wl = list(WORKLOADS[args.workload]); wl[2], wl[3] = w, h
        WORKLOADS[args.workload] = tuple(wl)
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    os.environ.pop("OMP_NUM_THREADS", None)   # the synthetic-scene packer is host code: let it use the cores it may
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import unitygaussiansplatting_b200 as g
    from unitygaussiansplatting_b200 import multigpu as MG
    n, quality, W, H, fov, seed, _ = WORKLOADS[args.workload]
    stream = torch.cuda.Stream(priority=-1)   # high priority: the group path's helper stream (view-calc) runs at the lowest and only fills gaps
    ctx = g.GaussianSplatContext(local, stream.cuda_stream)
    dev = torch.device("cuda", local)
    peak, peak_src = peaks()
    nk = ncu_kernels()

    if world == 1:
        m = measure_single(g, ctx, stream, torch, args.workload, args.steps, args.warmup, keep_last=bool(args.dump_outputs))
        sampler = ClockSampler(local)
        # clocks: sampled over a second pass of the device-resident loop (the sampler's start-up would otherwise miss a 50 ms region)
        sampler.start()
        m2 = measure_single(g, ctx, stream, torch, args.workload, args.steps, args.warmup, want_e2e=False)
        clocks = sampler.stop()
        ms_step = min(m["ms_step"], m2["ms_step"])
        others = []
        if not args.no_other_configs and args.workload == "metric":
            for name in ("cfg2", "cfg3"):
                o = measure_single(g, ctx, stream, torch, name, min(args.steps, 30), args.warmup)
                others.append({"workload": workload_text(name, o["n"], o["quality"], o["w"], o["h"]), "ms_per_step": o["ms_step"],
                               "value": o["n"] / (o["ms_step"] * 1e-3) / 1e6, "unit": "Msplats/s", "fps": 1e3 / o["ms_step"],
                               "e2e_ms_per_step": o["e2e_ms"],
                               "stages": stage_report(o["n"], o["quality"], o["w"], o["h"], o["stages"], o["pass_ms"], peak, o["ms_step"], nk)})
        stages = stage_report(n, quality, W, H, m["stages"], m["pass_ms"], peak, ms_step, nk)
        sort_pass = statistics.mean(m["pass_ms"]) if any(m["pass_ms"]) else None
        roofline = None
        if sort_pass:
            ach = n * SORT_BYTES_PER_PAIR_PASS / (sort_pass * 1e-3) / 1e9
            k = nk.get("k_onesweep")
            roofline = {"kernel": "k_onesweep (one 8-bit digit pass of the radix sort, 4 launches per frame)", "bound": "hbm",
                        "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "traffic": k["dram_bytes_per_launch"] if k else None,
                        "traffic_source": ("%s (%s)" % (NCU_SOURCE.relative_to(ROOT), k.get("capture", "")) if k else None),
                        "algorithmic_bytes_per_launch": n * SORT_BYTES_PER_PAIR_PASS, "launch_ms": sort_pass, "peak_source": peak_src}
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import gs_oracle_py as O
            threads = host_threads()
            fp, _keep = g.make_frame_params(orbit_camera(0, W, H, fov))
            ct, _, _ = cpu_frame(O, get_asset(n, quality, seed), fp, threads, W, H)
            cpu = {"value": n / ct["total"] / 1e6, "unit": "Msplats/s", "cores": threads, "kind": "port",
                   "sample": "one full frame of the same workload (%.1f s): distances %.0f ms, sort %.0f ms, view %.0f ms, draw %.0f ms"
                             % (ct["total"], ct["distances"] * 1e3, ct["sort"] * 1e3, ct["view"] * 1e3, ct["draw"] * 1e3)}
        line = {
            "metric": "splat throughput, full frame (sort + view-calc + draw)", "value": n / (ms_step * 1e-3) / 1e6,
            "unit": "Msplats/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(args.workload, n, quality, W, H), "parallelism": "single GPU",
                       "l2": "inputs (296 MB asset + draw records + sort buffers) exceed the 126 MB L2 and the camera moves every step; no explicit flush",
                       "blend": "fp16 ROP emulation (reference-exact)"},
            "fps": 1e3 / ms_step, "published_reference": {"fps": 147, "ms": 6.8, "hardware": "RTX 3080 Ti @1200x797, readme.md:84"},
            "clocks": clocks, "gpu_launches": m["launches"],
            "e2e": {"value": n / (m["e2e_ms"] * 1e-3) / 1e6, "unit": "Msplats/s", "ms_per_step": m["e2e_ms"],
                    "h2d_bytes_per_step": 344, "d2h_bytes_per_step": W * H * 8},
            "roofline": roofline, "stages": stages, "ncu_source": str(NCU_SOURCE.relative_to(ROOT)) if nk else None,
            "other_configs": others, "cpu_baseline": cpu,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, m["rt_last"])
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------------------------------------------- N > 1
    asset = get_asset(n, quality, seed)
    total = args.warmup + args.steps

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        rt_dev = torch.zeros((H, W, 4), dtype=torch.float16, device=dev)
        cams = [orbit_camera(k, W, H, fov) for k in range(total)]
        if args.baseline_partition:
            r = g.GaussianSplatRenderer(asset, ctx)
            part = MG.BandPartition(H, world, rank)
            gathered = MG.alloc_gather(part, W, dev)
            fps = [r.frame_params(c) for c in cams]

            def step_device(k, out=rt_dev):
                MG.render_partitioned(r, cams[k], part, gathered, out)
            parallelism = "round-1 baseline: replicated sort + view-calc, interleaved 64-pixel bands x%d, one torch all-gather" % world
            verified = None
        else:
            grp = MG.GaussianSplatGroup.join(asset, ctx, rank, world, MG.share_unique_id_torch(rank))
            fps = [g.make_frame_params(c)[0] for c in cams]

            def step_device(k, out=rt_dev):
                grp.SortAndRenderSplats(cams[k], rts=[out], fp=fps[k])
            parallelism = ("group x%d: key-range-sharded sort + order exchange (NVLink peer stores, NCCL fallback), row-range-sharded "
                           "view-calc/bin/composite + NCCL row exchange (gs_group_frame)" % world)
            # ---- the NCCL path against this GPU alone, outside the timed region: order and pixels bit-equal, 3 orbit frames ----
            ctx1 = g.GaussianSplatContext(local)
            r1 = g.GaussianSplatRenderer(asset, ctx1)
            rt1 = torch.zeros((H, W, 4), dtype=torch.float16, device=dev)
            for k in range(3):
                step_device(k)
                grp.sync()
                r1.SortAndRenderSplats(cams[k], rt=rt1)
                ctx1.sync()
                same_order = bool(np.array_equal(grp.readback_order(0), r1.readback_order()))
                same_rt = bool(torch.equal(rt_dev.view(torch.int16), rt1.view(torch.int16)))
                if not (same_order and same_rt):
                    raise SystemExit("rank %d frame %d: group path differs from the single-GPU frame (order equal: %s, image equal: %s)"
                                     % (rank, k, same_order, same_rt))
            r1.Dispose(); ctx1.close()
            del rt1
            verified = "every rank: draw order and RGBA16F target of 3 orbit frames bit-equal to the same frames rendered on that GPU alone"
            # restart the sequence so that the timed frames follow a coherent history
        for k in range(args.warmup):
            step_device(k)
        barrier()
        lib_launch0 = ctx.stage_times().kernel_launches
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for k in range(args.warmup, total):
            step_device(k)
        e1.record(stream)
        barrier()
        ms_total = e0.elapsed_time(e1)
        rt_last = rt_dev.cpu().numpy() if args.dump_outputs and rank == 0 else None
        clocks = sampler.stop() if rank == 0 else None
        launches = ctx.stage_times().kernel_launches - lib_launch0
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / args.steps

        # per-stage device times on every rank (events inside the library); the slowest rank per stage names the limiter
        stage_names = ("distances_ms", "slab_sort_ms", "order_exchange_ms", "view_ms", "bin_ms", "raster_ms", "image_exchange_ms", "total_ms")
        mine = None
        if not args.baseline_partition:
            ctx.set_timing(True)
            acc = {s: [] for s in stage_names}
            for k in range(min(args.steps, 20)):
                step_device(args.warmup + k)
                st = grp.stats()
                for s in stage_names:
                    acc[s].append(getattr(st, s))
            ctx.set_timing(False)
            mine = torch.tensor([statistics.median(acc[s]) for s in stage_names], device=dev)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            st = grp.stats()
            bounds = list(st.row_bounds[: world + 1])
            slabs = list(st.slab_counts[:world])

        # e2e: rank 0 hands in pinned host images (the display GPU's read-back), two in rotation, filled asynchronously: frame
        # k's copy overlaps frame k+1's kernels and all copies have landed before the clock stops; the other ranks keep the
        # frame on the device.  (GS_BENCH_SYNC_E2E=1: one image, every frame blocks until it has landed.)
        pinned = torch.empty((H, W, 4), dtype=torch.float16, pin_memory=True)
        pinned2 = torch.empty((H, W, 4), dtype=torch.float16, pin_memory=True)
        host_rts = (pinned.numpy(), pinned2.numpy())
        async_e2e = (not args.baseline_partition) and os.environ.get("GS_BENCH_SYNC_E2E", "0") != "1"
        if async_e2e and rank == 0:
            grp.async_readback = True

        def step_e2e(k):
            if args.baseline_partition:
                step_device(k)
                if rank == 0:
                    pinned.copy_(rt_dev, non_blocking=True)
                stream.synchronize()
            else:
                step_device(k, host_rts[k & 1 if async_e2e else 0] if rank == 0 else rt_dev)   # host image: D2H enqueued (or awaited) inside gs_group_frame
        for k in range(args.warmup):
            step_e2e(k)
        if not args.baseline_partition:
            grp.sync()
        barrier()
        t0 = time.perf_counter()
        for k in range(args.warmup, total):
            step_e2e(k)
        if not args.baseline_partition:
            grp.sync()                       # every read-back has landed
        torch.cuda.synchronize()
        tt = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item()) / args.steps

    if rank != 0:
        dist.destroy_process_group()
        return
    stages = None
    roofline = None
    if mine is not None:
        per_rank = [[float(v) for v in r_.tolist()] for r_ in allr]
        worst = {s: max(pr[i] for pr in per_rank) for i, s in enumerate(stage_names)}
        crit = {k: v for k, v in worst.items() if k not in ("total_ms", "view_ms")}
        limiter = max(crit, key=crit.get)
        stages = {"max_over_ranks_ms": worst, "rank0_ms": dict(zip(stage_names, per_rank[0])), "limiter": limiter,
                  "note": "view-calc runs beside distances + slab sort on a second stream; the other stages are serial on the context stream",
                  "row_bounds_16px": bounds, "slab_splats": slabs}
        if worst["slab_sort_ms"] > 0:
            pairs = max(slabs)
            ach = pairs * SORT_BYTES_PER_PAIR / (worst["slab_sort_ms"] * 1e-3) / 1e9
            roofline = {"kernel": "slab sort of the largest slab: compaction + 4 x k_onesweep over %d pairs (one GPU's share)" % pairs,
                        "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                        "algorithmic_bytes_per_launch": pairs * SORT_BYTES_PER_PAIR, "launch_ms": worst["slab_sort_ms"], "peak_source": peak_src}
    line = {
        "metric": "splat throughput, full frame (sort + view-calc + draw)", "value": n / (ms_step * 1e-3) / 1e6,
        "unit": "Msplats/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args.workload, n, quality, W, H), "parallelism": parallelism,
                   "l2": "inputs exceed the 126 MB L2 and the camera moves every step; no explicit flush",
                   "blend": "fp16 ROP emulation (reference-exact)"},
        "fps": 1e3 / ms_step, "clocks": clocks, "gpu_launches": int(launches), "verified": verified,
        "e2e": {"value": n / (e2e_ms * 1e-3) / 1e6, "unit": "Msplats/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": 344 * world,
                "d2h_bytes_per_step": W * H * 8},
        "roofline": roofline, "stages": stages, "cpu_baseline": None,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rt_last)
    print(json.dumps(line))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
