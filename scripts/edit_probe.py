#!/usr/bin/env python3
"""What an edit of a resident scene saves: "edit -> first finished frame" against "destroy + create scene + frame -> first finished
frame" on config 2 (spheres, 101k triangles) at 1920x1080, one sample, in one process.

    python scripts/edit_probe.py [--reps 5] [--out FILE.json]

Edits, each towards the same target scene as its rebuild (timed from the edit call to the end of the next render, planes read back;
before every timed edit the scene is put back to the base scene and a frame is rendered there, outside the clock):
  light move        DeviceScene.update(lights=True): the one light moved and recoloured
  material swap     DeviceScene.update(materials=True): the atlas inverted (same tables)
  camera move       DeviceFrame.set_camera(camera): the eye moved; lists built on the device
  geometry (host)   DeviceScene.update(geometry=True): the spheres' vertices moved (y += 0.3 sin x), the floor left flat, numpy
                    arrays, grid built on the device at 256 cells per axis
  geometry (torch)  DeviceScene.update_geometry on CUDA torch tensors of the same arrays (read in place)
  geometry, floor tilted (host)  the same deformation applied to every vertex: the 22.5 x 22.5 floor no longer lies in one layer of
                    grid cells, so the grid of the target mesh is far larger than the base mesh's
The rebuild is DeviceScene(host arrays, grid built on the device) + DeviceFrame(device-built lists) + the same render and read.
"frame" is one more render and read of the target scene on the rebuilt frame: the part of both times that no edit can skip.
Both sides synchronise the device before the clock starts; medians of --reps after one warm-up.  For the geometry rows the base scene
is the same mesh with its vertices not moved.
"""
import argparse
import dataclasses
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from opencl_render_b200 import api, scenes

    dev = torch.device("cuda", 0)
    cfg = scenes.CONFIGS[2]
    sc = cfg["make"]().normalise()
    W, H = cfg["width"], cfg["height"]
    m = sc.meta["camera"]
    cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], W, H)
    eye2 = np.asarray(m["eye"], np.float64) + np.array([1.5, 0.5, 0.0])
    cam2 = api.set_camera(eye2, m["look_at"], m["up"], m["fov"], W, H)
    lit = dataclasses.replace(sc, light_pos=sc.light_pos + np.float32(1.0), light_colour=(sc.light_colour * np.float32(0.8)).astype(np.float32))
    mat = dataclasses.replace(sc, textures=(255 - sc.textures).astype(np.uint8))
    wave = (np.float32(0.3) * np.sin(sc.vertex[:, 0])).astype(np.float32)
    moved_v = sc.vertex.copy()
    moved_v[:, 1] += np.where(sc.vertex[:, 1] > 0, wave, np.float32(0))   # (the floor is the plane y = 0)
    tilted_v = sc.vertex.copy()
    tilted_v[:, 1] += wave
    geo = dataclasses.replace(sc, vertex=moved_v, axes_div=api.AXES_DIVISION, box_min=None, grid_start=None, grid_list=None)
    tilted = dataclasses.replace(geo, vertex=tilted_v)
    tgeo = [torch.from_numpy(a).to(dev) for a in (moved_v, sc.tri_idx, sc.tri_mat, sc.tri_uv, sc.tri_normal)]
    tbase = [torch.from_numpy(sc.vertex).to(dev)] + tgeo[1:]
    info = {"gpu (name, power limit, max SM clock)": gpu_info(), "config": cfg["name"], "width": W, "height": H, "samples": 1,
            "reps": args.reps, "unit": "ms, median", "edits": {}}
    print("GPU:", info["gpu (name, power limit, max SM clock)"], flush=True)

    def finish(fr):
        fr.render(1)
        fr.read()

    def rebuild(s, c):
        ds = api.DeviceScene(s, 0)
        fr = api.DeviceFrame(ds, c)
        finish(fr)
        return ds, fr

    def timed(fn, setup=None):
        out = []
        for k in range(args.reps + 1):
            if setup:
                setup()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(dev)
            if k:
                out.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(out))

    base = dataclasses.replace(sc, box_min=None, grid_start=None, grid_list=None)
    ds, fr = rebuild(base, cam)
    state = {"ds": ds, "fr": fr}

    def full(target, c):
        def run():
            state["fr"].close()
            state["ds"].close()
            state["ds"], state["fr"] = rebuild(target, c)
        return run

    def edit(to_target, to_base):
        def run():
            to_target()
            finish(state["fr"])

        def setup():   # back at the base scene, one frame rendered there (not timed)
            to_base()
            finish(state["fr"])
        return run, setup

    edits = {
        "light move": (edit(lambda: state["ds"].update(lit, lights=True), lambda: state["ds"].update(sc, lights=True)), full(lit, cam)),
        "material swap": (edit(lambda: state["ds"].update(mat, materials=True), lambda: state["ds"].update(sc, materials=True)), full(mat, cam)),
        "camera move": (edit(lambda: state["fr"].set_camera(cam2), lambda: state["fr"].set_camera(cam)), full(base, cam2)),
        "geometry (host)": (edit(lambda: state["ds"].update(geo, geometry=True), lambda: state["ds"].update(base, geometry=True)), full(geo, cam)),
        "geometry (torch)": (edit(lambda: state["ds"].update_geometry(*tgeo, axes_div=api.AXES_DIVISION),
                                  lambda: state["ds"].update_geometry(*tbase, axes_div=api.AXES_DIVISION)), full(geo, cam)),
        "geometry, floor tilted (host)": (edit(lambda: state["ds"].update(tilted, geometry=True), lambda: state["ds"].update(base, geometry=True)),
                                          full(tilted, cam)),
    }
    for name, ((e, setup), f) in edits.items():
        state["fr"].close()
        state["ds"].close()
        state["ds"], state["fr"] = rebuild(base, cam)
        te = timed(e, setup)
        tf = timed(f)
        tr = timed(lambda: finish(state["fr"]))
        info["edits"][name] = {"edit_ms": round(te, 2), "rebuild_ms": round(tf, 2), "frame_ms": round(tr, 2), "saved": round(1 - te / tf, 3)}
        print(f"{name:30s} edit -> frame {te:8.2f} ms   destroy + create -> frame {tf:8.2f} ms   frame alone {tr:8.2f} ms", flush=True)
    state["fr"].close()
    state["ds"].close()
    if args.out:
        Path(args.out).write_text(json.dumps(info, indent=1) + "\n")


if __name__ == "__main__":
    main()
