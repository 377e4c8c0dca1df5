#!/usr/bin/env python3
"""The walk grid (rt_types.h: runs of coincident split planes collapsed where their lists agree) per config: its extents and non-empty
cells against the reference grid's, the walk iterations per traced ray of the counting trace kernel (wf_pipe_kernel<COUNT>, which walks
the same grid as production), and the device time of a frame and of its trace stage (L2 flushed before every render, median of --reps).

    python scripts/walk_grid_probe.py [--reps 10] [--configs 2,3,5] [--out FILE.json]

Run it on two builds to compare them: the extents are 256 on every axis on a build without the walk grid."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--configs", default="2,3,5")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from opencl_render_b200 import api, scenes

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # 256 MiB > the 126 MB L2
    info = gpu_info()
    print(f"GPU: {info}", flush=True)
    result = {"gpu": info, "reps": args.reps, "configs": {}}
    for cid in [int(c) for c in args.configs.split(",")]:
        cfg = scenes.CONFIGS[cid]
        sc = cfg["make"]()
        W, H, S = cfg["width"], cfg["height"], cfg["samples"]
        ds = api.DeviceScene(sc, 0)                       # grid built on the device
        m = scenes.sweep_cameras(sc, cfg["frames"])[0] if cid == 5 else sc.meta["camera"]
        fr = api.DeviceFrame(ds, api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], W, H))
        ext = ds.debug_read(11).view(np.uint32).tolist() if len(ds.debug_read(11)) else [sc.axes_div] * 3
        ref_cells = ds.debug_read(3).size // 8
        walk_cells = ds.debug_read(8).size // 8 if len(ds.debug_read(11)) else 0
        cnt = fr.render(S, variant=api.KERNEL_PIPE, count=True)[2]
        frame, trace = [], []
        for i in range(args.reps + 2):
            flush.zero_()
            torch.cuda.synchronize()
            t = fr.render(S)[0]
            if i >= 2:
                frame.append(t)
                trace.append(fr.last_trace_ms)
        rays = max(cnt["gridRays"], 1)
        r = {"workload": cfg["name"], "walk_extents": ext, "reference_nonempty_cells": ref_cells,
             "walk_nonempty_cells": walk_cells or ref_cells,
             "per_traced_ray": {k: cnt[k] / rays for k in ("walkLaneIters", "cells", "cellsNonEmpty", "coarseSteps", "bricksLoaded", "gridCandidates")},
             "traced_rays": cnt["gridRays"], "walk_warp_iters": cnt["walkWarpIters"],
             "frame_ms": float(np.median(frame)), "frame_ms_range": [float(min(frame)), float(max(frame))],
             "trace_ms": float(np.median(trace)), "trace_ms_range": [float(min(trace)), float(max(trace))]}
        result["configs"][str(cid)] = r
        p = r["per_traced_ray"]
        print(f"cfg{cid} {cfg['name']}: walk extents {ext}, non-empty cells {r['walk_nonempty_cells']} (reference {ref_cells}); "
              f"per traced ray: walk iterations {p['walkLaneIters']:.1f}, cells {p['cells']:.1f}, occupied {p['cellsNonEmpty']:.2f}, "
              f"brick steps {p['coarseSteps']:.1f}, tests {p['gridCandidates']:.2f}; frame {r['frame_ms']:.3f} ms, trace {r['trace_ms']:.3f} ms",
              flush=True)
        fr.close()
        ds.close()
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
