#!/usr/bin/env python3
"""bench.py -- headline benchmark of the raytrace path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config 2] [--extra auto|none|3,5,4] [--dump-outputs DIR]

One "step" = one pass of the hot path over one frame of the BASELINE.json config-2 workload (6x6 tessellated-sphere grid
+ floor = 101 090 triangles, 1920x1080, 1 light, primary + shadow + 1 diffuse bounce, 1 sample/pixel): every pixel-sample
("ray" in the reference's own accounting, raytrace.c:545) traced and shaded into three 16-bit planes.

  value      Mrays/s with scene, acceleration lists and framebuffer already resident in HBM, device-timed with CUDA
             events on the launch stream, L2 flushed before every timed step, max over ranks.
  e2e        the same metric through the reference-facing call RaytraceAll (C-ABI, HOST buffers in and out): upload +
             repack + trace + read-back all inside the timed region.  N > 1: ONE process (rank 0) calls
             RaytraceAll(all devices) -- the analogue of the reference's multi-device tile loop, raytrace.c:507-556 -- on the N
             GPUs of the run (every GPU pulls 1/N of the scene over PCIe and fans it out over NVLink); the other ranks wait
             at a CPU-side barrier.
  parity_ok  N > 1: the frame assembled from the ranks' bands (device-timed path) AND the planes RaytraceAll(all devices)
             returned are bit-equal to a 1-GPU render of the same frame made in the same run; N = 1: the production
             pipeline's planes are bit-equal to the independent one-thread-per-pixel kernel's.
  roofline   algorithmic bytes (SURVEY.md section 8d formula, event counts from the counting build of the kernel, which
             tests/ pin to an instrumented copy of the reference) per launch / kernel time, against the measured HBM copy
             bandwidth in MEASURED_PEAKS.json; `issue` = the issue-slot x lane roof the kernel really sits under (ncu).
  configs    the same measurement on BASELINE.json's other GPU configs: 3 (1 M-triangle terrain, 3840x2160) at every N,
             5 (64-frame sweep, scene resident, device-built lists, frames dealt to the ranks), 4 (10 M triangles, 7680x4320)
             at N = 8.
  cpu_baseline  the reference's own C build of the kernel (oracle/_ref, "reference") or the C port ("port") on the host
             cores, on a bounded sample of rows of the same frame; plus RaytraceAll(0, ...) as shipped (1 thread).

--dump-outputs DIR writes the three 16-bit planes the timed path produced in its last timed step as DIR/r.npy, g.npy, b.npy
(float32, [rows, width]), so that two builds can be compared output for output: the workload is synthetic and seeded, the same
arguments give the same inputs.  A frame larger than DUMP_LIMIT_BYTES in float32 keeps every k-th row; the rows kept go to
DIR/rows.npy.

N > 1 (launched by torchrun, one process per GPU): the frame is cut into row bands dealt round-robin to the ranks, the
scene is replicated, and the planes are assembled by peer stores over NVLink (the path's only exchange step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_FALLBACK_GBS = 6650.0     # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
ROW_STEP = 4                  # CPU arms: every 4th row of the WHOLE frame (a quarter of the work, sky and geometry in proportion)
DUMP_LIMIT_BYTES = 64_000_000  # --dump-outputs: all files together


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--variant", type=int, default=-1)
    ap.add_argument("--band-rows", type=int, default=16)
    ap.add_argument("--extra", default="auto", help="other configs measured into `configs`: auto (3, 5; 4 at 8 GPUs), none, or a list")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the planes of the last timed step of the headline config to DIR/{r,g,b}.npy (float32)")
    return ap.parse_args()


def config_keys(cfg, sc, cam):
    """`config` of the JSON line: identical for both arms and for every N (the driver compares it)."""
    return {"workload": cfg["name"], "triangles": int(sc.triangle_count), "width": int(cam.width), "height": int(cam.height),
            "samples": int(cfg["samples"]), "ray_unit": "pixel-sample (raytrace.c:545)",
            "l2": "GPU arm: flushed before every timed step (256 MiB memset)",
            "partition": "GPU arm: row bands dealt round-robin over the GPUs of the run, scene replicated, frame assembled over NVLink"}


def build_workload(cfg_id, builders="host"):
    """builders: "host" = the product's host builders (list-for-list the reference's, tests/test_builders.py); "reference" = the
    reference's own SetCamera / CameraTriangleList::New / SceneTriangleList::New from oracle/_ref (the CPU arm: the product's shared
    library is never loaded in that process); "none" = scene and camera only (lists and grid are then built on the device)."""
    from opencl_render_b200 import api, scenes
    cfg = scenes.CONFIGS[cfg_id]
    sc = cfg["make"]()
    m = sc.meta["camera"]
    if builders == "reference":
        import ref
        tl, lr, tb, psi = ref.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], cfg["width"], cfg["height"])
        cam = api.CameraSetup(cfg["width"], cfg["height"], np.asarray(m["eye"], np.float32), tl, lr, tb, psi)
        lists = api.CameraLists(*ref.camera_lists(cam, sc))
        sc.box_min, sc.grid_start, sc.grid_list = ref.scene_grid(sc)
        sc.axes_div = 256
        return cfg, sc.normalise(), cam, lists
    cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], cfg["width"], cfg["height"])
    lists = None
    if builders == "host":
        lists = api.camera_triangle_list(cam, sc)
        api.scene_triangle_list(sc, 256)
    return cfg, sc, cam, lists


def algorithmic_bytes(cnt: dict, rays: int) -> float:
    """SURVEY.md section 8d: B = 8*[primary ray] + 68*C_prim + 8*K_cells + 68*C_grid + 212*H + 44*O + 12 per pixel-sample, counted
    in the reference layout; totals per launch."""
    grid_candidates = cnt["gridCandidates"] + cnt.get("mailboxSkips", 0)     # the reference tests these again in every cell
    return (8.0 * rays + 68.0 * cnt["primCandidates"] + 8.0 * cnt["cells"] + 68.0 * grid_candidates + 212.0 * cnt["shadedHits"] +
            44.0 * cnt["occluderLookups"] + 12.0 * rays)


def dump_outputs(out_dir, planes):
    """--dump-outputs: the uint16 planes (r, g, b) as float32 .npy files, every k-th row when the whole frame exceeds the limit."""
    h, w = planes[0].shape
    step = 1
    while 3 * len(range(0, h, step)) * w * 4 > DUMP_LIMIT_BYTES:
        step += 1
    rows = np.arange(0, h, step)
    os.makedirs(out_dir, exist_ok=True)
    for name, plane in zip("rgb", planes):
        np.save(os.path.join(out_dir, f"{name}.npy"), plane[rows].astype(np.float32))
    if step > 1:
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.index = index
        self.source = "nvidia-smi"
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        if self._run_nvml():
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.1)

    def _run_nvml(self) -> bool:
        """The same counters nvidia-smi prints, read through NVML directly: a query takes well under a millisecond, so a timed region
        of ~100 ms yields dozens of samples instead of one.  False when NVML is not usable (then nvidia-smi is polled)."""
        try:
            import pynvml
            pynvml.nvmlInit()
            index = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:      # CUDA's device index -> NVML's
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    index = int(ids[index])
            dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(dev, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(dev, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetCurrentClocksEventReasons(dev)
        except Exception:
            return False
        bits = {"hw_slowdown": pynvml.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": pynvml.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": pynvml.nvmlClocksEventReasonSwPowerCap}
        self.source = "nvml"
        while not self._stop.is_set():
            try:
                self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(dev, pynvml.NVML_CLOCK_SM)))
                r = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(dev))
                for n, b in bits.items():
                    if r & b:
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.002)
        return True

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "source": self.source}



def _cpu_renderer(cfg_id):
    """The reference's own CPU implementation of the path: oracle/_ref (the unmodified kernel compiled as C, driven over all host
    cores; lists from the reference's own builders) when that build travelled, else the C port with the product's host builders."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    cores = os.cpu_count() or 1
    try:
        import ref
        if ref.LIB.is_file() or ref.available():
            ref.load()
            # camera, camera lists and grid from the reference's OWN SetCamera / builders (outside the timed region; its scene-grid
            # builder is single-threaded: ~10 s for config 2).  Beyond 200 k triangles it needs minutes (SURVEY.md 6.2); there -- or
            # with OCLR_BENCH_REF_BUILDERS=0 -- the product's host builders stand in, proven list-for-list identical by tests/
            own = os.environ.get("OCLR_BENCH_REF_BUILDERS", "1") != "0"
            if own:
                from opencl_render_b200 import scenes
                own = scenes.CONFIGS[cfg_id]["make"]().triangle_count <= 200_000
            cfg, sc, cam, lists = build_workload(cfg_id, "reference" if own else "host")
            fn = lambda: ref.render(cam, lists, sc, cfg["samples"], threads=cores, row_step=ROW_STEP)
            return cfg, sc, cam, lists, fn, "reference", cores, ("the reference's own SetCamera / CameraTriangleList::New / SceneTriangleList::New (oracle/_ref)"
                                                              if own else "product host builders (== the reference's list for list, tests/test_builders.py)")
    except Exception as e:
        print(f"[bench] reference build unavailable ({type(e).__name__}: {e}); using the C port", file=sys.stderr)
    import port
    cfg, sc, cam, lists = build_workload(cfg_id, "host")
    fn = lambda: port.render(cam, lists, sc, cfg["samples"], threads=cores, row_step=ROW_STEP)
    return cfg, sc, cam, lists, fn, "port", cores, "product host builders"


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on all host cores, a bounded sample (every 4th row of the
    whole frame) of the same frame per step.  Rank 0 alone runs it."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg, sc, cam, lists, render, kind, cores, lists_by = _cpu_renderer(args.config)
    h, w = cam.height, cam.width
    n_rows = len(range(0, h, ROW_STEP))
    for _ in range(args.warmup):
        render()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        render()
    dt = time.perf_counter() - t0
    rays = n_rows * w * cfg["samples"]
    value = rays * args.steps / dt / 1e6
    sample = f"every {ROW_STEP}th row of all {h} ({rays} pixel-samples) per step"
    try:                                            # (evidence for the reader of the line: which shared libraries of this repo the process mapped)
        mapped = sorted({l.split("/")[-1].strip() for l in open("/proc/self/maps") if "/oracle/" in l or "libopencl_render_b200" in l})
    except OSError:
        mapped = None
    print(json.dumps({
        "impl": "reference", "repo_libraries_mapped": mapped, "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_keys(cfg, sc, cam), "sampling": sample, "acceleration_lists": lists_by,
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


class Run:
    """Process-wide state of the B200 arm."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the library has no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.device = torch.device("cuda", self.local)
        self.cpu_group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)
            # CPU-side barrier for the phases in which ONE process drives all GPUs (RaytraceAll(all devices)): an NCCL barrier would
            # park a spinning kernel on every waiting rank's GPU -- the very GPUs rank 0 is rendering on
            self.cpu_group = dist.new_group(backend="gloo")
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def cpu_barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier(group=self.cpu_group)

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]


def measure_config(run: Run, cfg_id: int, steps: int, warmup: int, primary: bool, device_built: bool = False, want_e2e: bool = True):
    """One config through the band-partitioned device-timed path (+ parity, e2e, roofline).  Returns (dict for the JSON line, extras)."""
    import torch
    from opencl_render_b200 import api, dist as odist
    args, world, rank, local = run.args, run.world, run.rank, run.local
    cfg, sc, cam, lists = build_workload(cfg_id, "none" if device_built else "host")
    h, w, S = cam.height, cam.width, cfg["samples"]
    rays_frame = h * w * S
    ds = api.DeviceScene(sc, local)                       # (no grid given: SceneTriangleList::New runs on the device)
    fr = api.DeviceFrame(ds, cam, lists)                  # (no lists given: CameraTriangleList::New runs on the device)
    part = odist.BandPartition(h, w, rank, world, args.band_rows)
    gather, gather_kind = odist.plane_exchange(fr, part, run.device) if world > 1 else (None, None)
    stream = torch.cuda.current_stream().cuda_stream

    def step(ev=None):
        run.flush.zero_()                                    # L2 flush (256 MiB > 126 MB L2), outside the timed events
        if ev is not None:
            ev[0].record()
        launches = part.render(fr, S, args.variant, stream)
        if ev is not None:
            ev[2].record()                                   # trace done, exchange not yet: "gather excluded" figure
        out = None
        if gather is not None:
            out = gather.run()
            launches += gather.launches
        if ev is not None:
            ev[1].record()
        return launches, out

    for _ in range(max(warmup, 3)):
        step()
    run.barrier()
    events = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(steps)]
    launches, assembled = 0, None
    with ClockSampler(local) as clocks:
        for k in range(steps):
            n, assembled = step(events[k])
            launches += n
        torch.cuda.synchronize()
    run.barrier()
    if primary and args.dump_outputs and rank == 0:      # before anything below renders into the frame again
        dump_outputs(args.dump_outputs, assembled.cpu().numpy().view(np.uint16) if world > 1 else fr.read())
    ms_total, ms_render = run.max_over_ranks([sum(a.elapsed_time(b) for a, b, _ in events), sum(a.elapsed_time(c) for a, _, c in events)])
    ms_step = ms_total / steps
    res = {"workload": cfg["name"], "triangles": int(sc.triangle_count), "width": w, "height": h, "samples": S,
           "value": rays_frame / ms_step / 1e3, "unit": "Mrays/s", "ms_per_step": ms_step, "steps": steps,
           "acceleration_lists": "built on the device (cam_builder.cuh / grid_builder.cuh)" if device_built else "host builders",
           "gather": {"kind": gather_kind, "ms_per_step": (ms_total - ms_render) / steps,
                      "value_without_gather": rays_frame / (ms_render / steps) / 1e3},
           # HBM held by the wavefront path state of this rank's launch domain (ring depth follows the scene's materials, DESIGN.md section 3)
           "path_state": {"bytes": fr.state_bytes, "bytes_per_path": fr.state_bytes / max(((part.owned_rows + 7) // 8 * 8) * w, 1)}}

    # ---- parity inside the run: 1-GPU render of the same frame on rank 0 (N > 1) / the independent per-pixel kernel (N = 1) ----------
    planes_1gpu = None
    parity = {}
    if world > 1:
        got = assembled.cpu().numpy().view(np.uint16) if rank == 0 else None
        run.barrier()                                        # every rank's pushes have landed and been read before rank 0 re-renders
        if rank == 0:
            fr.render(S, variant=args.variant)
            planes_1gpu = fr.read()
            parity["assembled_vs_1gpu"] = bool(all(np.array_equal(got[c], planes_1gpu[c]) for c in range(3)))
    elif rank == 0:
        fr.render(S, variant=args.variant)
        planes_1gpu = fr.read()
        fr.render(S, variant=api.KERNEL_SIMPLE)
        simple = fr.read()
        parity["pipeline_vs_per_pixel_kernel"] = bool(all(np.array_equal(simple[c], planes_1gpu[c]) for c in range(3)))

    # ---- roofline of the dominant kernel, wf_pipe_kernel (rank 0's share of the frame) ------------------------------------------
    roof = None
    if rank == 0:
        _, _, cnt = part.render_counted(fr, S, 0)      # event counts in the reference's accounting: the per-pixel kernel
        frame_ms, trace_ms = [], []
        for _ in range(5):
            run.flush.zero_()
            frame_ms.append(part.render_timed(fr, S, args.variant))
            trace_ms.append(fr.last_trace_ms)
        ms_frame, ms_trace = float(np.mean(frame_ms)), float(np.mean(trace_ms))
        n_trace = max(fr.last_trace_launches, 1)
        rays_rank = part.owned_rows * w * S
        algo_frame = algorithmic_bytes(cnt, rays_rank)
        # the grid-walk share of the formula is what the trace kernel is responsible for: 8 B per cell looked at, 68 B per
        # candidate tested (reference layout), plus its own ray fetch (36 B) and hit store (16 B) per grid ray
        algo_trace = 8.0 * cnt["cells"] + 68.0 * cnt["gridCandidates"] + 52.0 * cnt["gridRays"]
        peak, which = hbm_peak()
        achieved = (algo_trace / n_trace) / (ms_trace / n_trace * 1e-3) / 1e9
        roof = {"kernel": "wf_pipe_kernel (+ wf_setup_kernel)", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": which, "launches_per_step": n_trace, "avg_launch_ms": ms_trace / n_trace,
                "algorithmic_bytes_per_launch": algo_trace / n_trace,
                "note": "working set is L2-resident (DRAM traffic << algorithmic bytes); the kernel is issue-bound: see `issue`",
                "whole_step": {"ms": ms_frame, "algorithmic_bytes": algo_frame, "achieved_gbs": algo_frame / (ms_frame * 1e-3) / 1e9,
                               "frac": algo_frame / (ms_frame * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_ray": algo_frame / rays_rank},
                "per_ray_events": {k: v / rays_rank for k, v in cnt.items() if v},
                # comparable with other tracers (SURVEY 8d): ring segments and grid traversals per second, rank 0's share
                "rates": {"segments_per_s": cnt["segments"] / (ms_frame * 1e-3), "traversals_per_s": cnt["gridRays"] / (ms_frame * 1e-3),
                          "triangle_tests_per_s_reference_accounting": (cnt["primCandidates"] + cnt["gridCandidates"]) / (ms_frame * 1e-3)}}
        # DRAM traffic and the issue-slot / lane roof cannot be measured outside a profiler: they come from the committed ncu capture
        # of this kernel on this workload (profiles/), single GPU, and are printed only where they apply (N = 1) with their origin
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if world == 1 and os.path.isfile(prof):
            try:
                t = json.load(open(prof)).get(cfg["name"])
                if t:
                    roof["traffic"] = t["dram_bytes_per_launch"]
                    roof["traffic_source"] = t.get("source")
                    roof["traffic_commit"] = t.get("commit")
                    if "issue" in t:
                        roof["issue"] = t["issue"]
            except Exception:
                pass
        res["roofline"] = roof

    # ---- end to end through the drop-in call (host buffers), made by ONE plain host process like the plugin -------------------------
    if want_e2e and lists is not None and os.environ.get("OCLR_BENCH_NO_E2E") != "1":     # (profiling runs skip the probe process)
        run.cpu_barrier()                                     # nothing but the probe process touches the GPUs from here to the next barrier
        if rank == 0:
            e2e_calls = max(5, min(steps, 10))
            try:
                import hashlib
                r = subprocess.run([sys.executable, "-m", "opencl_render_b200.e2e_probe", str(cfg_id), str(world), str(e2e_calls)], cwd=ROOT,
                                   capture_output=True, text=True, timeout=300)
                lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
                if r.returncode != 0 or not lines:
                    raise RuntimeError(f"rc {r.returncode}: {r.stderr[-600:]}")
                pr = json.loads(lines[-1])
                call = (f"RaytraceAll(all devices) on {world} GPUs from one host process (C-ABI, host buffers; 1/{world} of the scene per GPU over PCIe, "
                        "NVLink fan-out)") if world > 1 else "RaytraceAll (C-ABI, host buffers) from a plain host process"
                res["e2e"] = {"value": pr["rays"] / pr["ms_per_call"] / 1e3, "unit": "Mrays/s", "ms_per_call": pr["ms_per_call"],
                              "ms_median": pr["ms_median"], "spread": pr["spread"], "h2d_bytes_per_step": pr["h2d_bytes"],
                              "h2d_bytes_per_step_per_gpu": pr["h2d_bytes"] // world, "d2h_bytes_per_step": pr["d2h_bytes"],
                              "steps": pr["calls"], "host_arrays": pr["host_arrays"], "call": call}
                want_sha = None
                if planes_1gpu is not None:
                    hsh = hashlib.sha256()
                    for pl in planes_1gpu:
                        hsh.update(np.ascontiguousarray(pl).tobytes())
                    want_sha = hsh.hexdigest()
                    parity["raytrace_all_vs_1gpu"] = pr["sha256"] == want_sha
                if "pageable" in pr:         # the same call the way the plugin makes it: plain new[] arrays (render.cpp:1086-1134)
                    pg = pr["pageable"]
                    res["e2e"]["value_pageable_host_arrays"] = pg["rays"] / pg["ms_per_call"] / 1e3
                    res["e2e"]["pageable"] = {"ms_per_call": pg["ms_per_call"], "ms_median": pg["ms_median"], "spread": pg["spread"],
                                              "steps": pg["calls"]}
                    if want_sha is not None:
                        parity["raytrace_all_pageable_vs_1gpu"] = pg["sha256"] == want_sha
            except Exception as e:
                res["e2e"] = {"value": None, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                              "error": f"{type(e).__name__}: {e}"}
                print(f"[bench] e2e probe failed: {type(e).__name__}: {e}", file=sys.stderr)
        run.cpu_barrier()
    if rank == 0:
        res["parity"] = parity
        res["parity_ok"] = bool(parity) and all(parity.values())
    extras = {"launches": launches, "clocks": clocks.summary(), "cfg": cfg, "sc": sc, "cam": cam, "lists": lists}
    del gather
    fr.close()
    ds.close()
    torch.cuda.empty_cache()
    return res, extras


def measure_sweep(run: Run, cfg_id: int = 5):
    """Config 5: the 64-frame camera sweep over the 1 M-triangle scene with mirror chains to the reference's maximum bounce depth.
    Scene uploaded ONCE (grid built on the device), per-frame camera lists built on the device, whole frames dealt round-robin to
    the ranks (independent frames: no exchange).  Wall clock around all of a rank's frames, max over ranks."""
    import torch
    from opencl_render_b200 import api, scenes
    world, rank, local = run.world, run.rank, run.local
    cfg = scenes.CONFIGS[cfg_id]
    sc = cfg["make"]()
    cams = scenes.sweep_cameras(sc, cfg["frames"])
    w, h, S = cfg["width"], cfg["height"], cfg["samples"]
    ds = api.DeviceScene(sc, local)
    mine = list(range(rank, len(cams), world))

    def render(k, variant=-1):
        m = cams[k]
        cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], w, h)
        fr = api.DeviceFrame(ds, cam, None)
        fr.render(S, variant=variant)
        return fr

    render(mine[0]).close()                                  # warm-up (allocations, first-use set-up)
    run.barrier()
    t0 = time.perf_counter()
    launches = 0
    for k in mine:
        fr = render(k)
        launches += fr.last_launches
        fr.close()
    torch.cuda.synchronize()
    dt = run.max_over_ranks([time.perf_counter() - t0])[0]
    res = {"workload": cfg["name"], "triangles": int(sc.triangle_count), "width": w, "height": h, "samples": S, "frames": len(cams),
           "value": len(cams) * w * h * S / dt / 1e6, "unit": "Mrays/s", "frames_per_s": len(cams) / dt, "ms_per_frame_per_gpu": dt / len(mine) * 1e3,
           "partition": "whole frames dealt round-robin to the ranks, scene resident, camera lists built on the device per frame",
           "timed": "wall clock around a rank's frames incl. the per-frame list build, max over ranks", "gpu_launches_rank0": launches}
    if rank == 0:
        a = render(0)
        pa = a.read()
        a.close()
        b = render(0, api.KERNEL_SIMPLE)
        pb, flags = b.read(), b.undefined_flags()
        b.close()
        ok = flags == 0
        res["parity"] = {"pipeline_vs_per_pixel_kernel_frame0": bool(all(np.array_equal(pa[c][ok], pb[c][ok]) for c in range(3)))}
        res["parity_ok"] = all(res["parity"].values())
    ds.close()
    torch.cuda.empty_cache()
    return res


def run_b200(args):
    # stdout carries ONE JSON line: everything libraries print there (NCCL's version banner, ...) is sent to stderr instead
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    run = Run(args)
    world, rank = run.world, run.rank
    main, ex = measure_config(run, args.config, args.steps, args.warmup, primary=True)
    cfg, sc, cam, lists = ex["cfg"], ex["sc"], ex["cam"], ex["lists"]
    cpu = cpu_baseline(args.config, cfg, sc, cam, lists) if (rank == 0 and world == 1) else None

    extra = args.extra
    ids = []
    if extra == "auto":
        ids = [c for c in (3, 5) if c != args.config] + ([4] if world == 8 and args.config != 4 else [])
    elif extra != "none":
        ids = [int(x) for x in extra.split(",") if x.strip()]
    configs = {}
    for cid in ids:
        try:
            if cid == 5:
                configs[str(cid)] = measure_sweep(run, cid)
            else:
                configs[str(cid)] = measure_config(run, cid, max(3, min(args.steps, 5)), 3, primary=False, device_built=(cid == 4),
                                                   want_e2e=(cid != 4))[0]
        except Exception as e:                                 # an extra config must not cost the headline line
            configs[str(cid)] = {"error": f"{type(e).__name__}: {e}"}
            print(f"[bench] config {cid} failed: {type(e).__name__}: {e}", file=sys.stderr)
            try:
                run.barrier()
            except Exception:
                pass

    if rank == 0:
        e2e = main.get("e2e") or {"value": None, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        line = {
            "metric": "Mrays/s", "value": main["value"], "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_keys(cfg, sc, cam),
            "run": {"band_rows": args.band_rows, "kernel_variant": args.variant, "frame_assembly": main["gather"]["kind"],
                    "path_state": main.get("path_state")},
            "e2e": e2e, "gpu_launches": ex["launches"], "clocks": ex["clocks"], "roofline": main.get("roofline"),
            "gather": dict(main["gather"], included_in_value=world > 1),
            "parity_ok": main.get("parity_ok"), "parity": main.get("parity"),
            "configs": configs,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    if world > 1:
        run.dist.barrier()
        run.dist.destroy_process_group()


def cpu_baseline(cfg_id, cfg, sc, cam, lists):
    """Bounded sample of the same workload on the host: the reference kernel on all cores over every 4th row, and the reference as
    shipped -- RaytraceAll(0, ...), "Local CPU single thread" (raytrace.c:604-655) -- once over the whole frame."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    cores = os.cpu_count() or 1
    h, w = cam.height, cam.width
    n_rows = len(range(0, h, ROW_STEP))
    kind = "port"
    fn = single = None
    try:
        import ref
        if ref.LIB.is_file():
            ref.load()
            kind = "reference"
            fn = lambda: ref.render(cam, lists, sc, cfg["samples"], threads=cores, row_step=ROW_STEP)
            single = lambda: ref.raytrace_all(cam, lists, sc, cfg["samples"])
    except Exception:
        fn = None
    if fn is None:
        import port
        kind = "port"
        fn = lambda: port.render(cam, lists, sc, cfg["samples"], threads=cores, row_step=ROW_STEP)
    fn()
    reps = 0
    t0 = time.perf_counter()
    while True:
        fn()
        reps += 1
        if time.perf_counter() - t0 > 10.0 or reps >= 20:
            break
    dt = time.perf_counter() - t0
    rays = n_rows * w * cfg["samples"] * reps
    out = {"value": rays / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": kind,
           "sample": f"every {ROW_STEP}th row of all {h}, {reps} passes, {dt:.1f} s"}
    if single is not None and h * w * cfg["samples"] <= 4_000_000:      # (~10 s for a 2 M-ray frame)
        t0 = time.perf_counter()
        single()
        dt1 = time.perf_counter() - t0
        out["single_thread"] = {"value": h * w * cfg["samples"] / dt1 / 1e6, "unit": "Mrays/s", "cores": 1,
                                "call": "the reference's RaytraceAll(0, ...) as shipped, whole frame once", "seconds": dt1}
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
