#!/usr/bin/env python3
"""Device-timed rates of the ray queries (DeviceScene.intersect / transmittance) on BASELINE configs, next to the frame's own
trace-stage rate from the same process.

    python scripts/query_probe.py [--configs 2,3] [--reps 20] [--out FILE.json]

Ray sets per config (scene and camera of the config, image 1920x1080):
  eye            one primary ray through every pixel centre, rows in order
  bounce_tiles   from every primary hit a cosine-free random direction on the side the eye ray came from, the hit triangle excluded,
                 in the frame's tile order (16x8-pixel CTA tiles of 8x4-pixel warp tiles, rt_wavefront.cuh)
  bounce_shuffled the same rays in a random order
  shadow         from every primary hit to the config's first light (finite maxD for a positional light), hit triangle excluded
Rates are rays / device time (CUDA events around one call on device-memory torch tensors, median of --reps after 3 warm-ups); L2 is
flushed before every timed call by a 256 MiB memset.  The frame's trace-stage rate is gridRays of a counting render over traceMs of a
timed render of the config's own frame (its resolution and samples).
"""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def tile_order(w, h):
    """Pixel indices in the logic kernel's order: CTA tiles of 16x8 pixels, inside them four warps of 8x4 pixels."""
    y, x = np.mgrid[0:h, 0:w]
    cta = (y // 8) * ((w + 15) // 16) + x // 16
    warp = ((y % 8) // 4) * 2 + (x % 16) // 8
    lane = (y % 4) * 8 + x % 8
    return np.lexsort((lane.ravel(), warp.ravel(), cta.ravel()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="2,3")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from opencl_render_b200 import api, scenes

    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    info = {"gpu": gpu_info(), "l2": "flushed before every timed call (256 MiB memset)", "reps": args.reps, "configs": {}}
    print("GPU (name, power limit, max SM clock):", info["gpu"], flush=True)

    def timed(fn, rays):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = float(np.median(ms))
        return {"rays": int(rays), "ms_median": med, "ms_min": float(min(ms)), "ms_max": float(max(ms)), "mrays_per_s": rays / med / 1e3}

    for cid in [int(c) for c in args.configs.split(",")]:
        cfg = scenes.CONFIGS[cid]
        sc = cfg["make"]()
        m = sc.meta["camera"]
        ds = api.DeviceScene(sc)   # grid built on the device
        res = {"workload": cfg["name"], "triangles": int(sc.triangle_count)}
        # the frame's own trace-stage rate
        fcam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], cfg["width"], cfg["height"])
        fr = api.DeviceFrame(ds, fcam)
        _, _, cnt = fr.render(cfg["samples"], count=True)
        trace_ms = []
        for _ in range(5):
            fr.render(cfg["samples"])
            trace_ms.append(fr.last_trace_ms)
        res["frame"] = {"width": cfg["width"], "height": cfg["height"], "samples": cfg["samples"], "gridRays": cnt["gridRays"],
                        "traceMs_median": float(np.median(trace_ms)),
                        "mrays_per_s": cnt["gridRays"] / float(np.median(trace_ms)) / 1e3}
        fr.close()
        # ray sets at 1920x1080
        W, H = 1920, 1080
        cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], W, H)
        y, x = np.mgrid[0:H, 0:W]
        d = (cam.eye_to_top_left[:3] + (x.ravel() + 0.5)[:, None] * cam.left_to_right[:3] + (y.ravel() + 0.5)[:, None] * cam.top_to_bottom[:3])
        eo = np.zeros((W * H, 4), np.float32)
        eo[:, :3] = cam.eye[:3]
        ed = np.zeros((W * H, 4), np.float32)
        ed[:, :3] = d
        ed[:, 3] = np.inf
        ids, t, _, _ = ds.intersect(eo, ed)
        hit = ids != api.NO_TRIANGLE
        p = eo[:, :3] + t[:, None] * ed[:, :3]
        tri = sc.tri_idx[np.where(hit, ids, 0), :3]
        a, b, c = (sc.vertex[tri[:, k], :3] for k in range(3))
        n = np.cross(b - a, c - a)
        n *= np.where((n * ed[:, :3]).sum(1) > 0, -1.0, 1.0)[:, None]
        rng = np.random.default_rng(cid)
        r = rng.normal(size=(W * H, 3)).astype(np.float32)
        r *= np.where((r * n).sum(1) < 0, -1.0, 1.0)[:, None]
        order = tile_order(W, H)
        sel = order[hit[order]]
        bo = np.zeros((len(sel), 4), np.float32)
        bo[:, :3] = p[sel]
        bd = np.zeros((len(sel), 4), np.float32)
        bd[:, :3] = r[sel]
        bd[:, 3] = np.inf
        bex = ids[sel].astype(np.uint32)
        shuf = rng.permutation(len(sel))
        light = sc.light_pos[0, :3].astype(np.float64) if int(sc.light_type[0]) not in (3, 4, 5, 6) else None
        so = bo.copy()
        sd = np.zeros_like(bd)
        if light is not None:
            to = light - p[sel]
            dist = np.linalg.norm(to, axis=1)
            sd[:, :3] = to / dist[:, None]
            sd[:, 3] = dist
        else:
            sd[:, :3] = -sc.light_dir[0, :3]
            sd[:, 3] = np.inf
        sets = {"eye": (eo, ed, None), "bounce_tiles": (bo, bd, bex), "bounce_shuffled": (bo[shuf], bd[shuf], bex[shuf]),
                "shadow": (so, sd, bex)}
        res["sets"] = {}
        for name, (o4, d4, ex) in sets.items():
            to4, td4 = torch.from_numpy(np.ascontiguousarray(o4)).to(dev), torch.from_numpy(np.ascontiguousarray(d4)).to(dev)
            tex = torch.from_numpy(ex.view(np.int32)).to(dev) if ex is not None else None
            *_, qc = ds.intersect(to4, td4, exclude=tex, count=True)
            row = {"closest_hit": timed(lambda: ds.intersect(to4, td4, exclude=tex), len(o4)),
                   "transmittance": timed(lambda: ds.transmittance(to4, td4, exclude=tex), len(o4)),
                   "traced": int(qc["gridRays"])}
            row["closest_hit_vs_frame"] = row["closest_hit"]["mrays_per_s"] / res["frame"]["mrays_per_s"]
            res["sets"][name] = row
            print(f"config {cid} {name:16s} rays {len(o4):8d}  closest hit {row['closest_hit']['mrays_per_s']:8.1f} Mrays/s "
                  f"({row['closest_hit']['ms_median']:.3f} ms, {row['closest_hit_vs_frame']:.2f}x frame)  transmittance "
                  f"{row['transmittance']['mrays_per_s']:8.1f} Mrays/s ({row['transmittance']['ms_median']:.3f} ms)", flush=True)
        print(f"config {cid} frame trace stage: {res['frame']['gridRays']} grid rays in {res['frame']['traceMs_median']:.3f} ms = "
              f"{res['frame']['mrays_per_s']:.1f} Mrays/s", flush=True)
        info["configs"][str(cid)] = res
        ds.close()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(info, indent=1))


if __name__ == "__main__":
    main()
