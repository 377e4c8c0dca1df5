#!/usr/bin/env python3
"""Device-timed rates of radiance queries (DeviceScene.radiance / oclr_scene_radiance) next to the frame's own rate, in the same process.

    python scripts/radiance_probe.py [--reps 20] [--out FILE.json]

Workloads:
  config 2, eye_tiles      one ray through every pixel centre of the 1920x1080 camera, S = 1, in the frame's tile order (16x8-pixel CTA
                           tiles of 8x4-pixel warp tiles, rt_wavefront.cuh)
  config 2, eye_shuffled   the same rays in a random order
  config 2 / 3, equirect   a 3840x1920 panorama around the config's eye (render.py --projection equirect), S = 1
  frame                    the config's own frame at 1920x1080, S = 1 (DeviceFrame.render), for comparison
Rates are paths / stats.deviceMs of one call on device-memory torch tensors (median of --reps after 2 warm-ups); L2 is flushed before
every timed call by a 256 MiB memset.
"""
import argparse
import ctypes as C
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


def tile_order(w, h):
    y, x = np.mgrid[0:h, 0:w]
    cta = (y // 8) * ((w + 15) // 16) + x // 16
    warp = ((y % 8) // 4) * 2 + (x % 16) // 8
    lane = (y % 4) * 8 + x % 8
    return np.lexsort((lane.ravel(), warp.ravel(), cta.ravel()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from opencl_render_b200 import _lib, api, render, scenes

    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = _lib.load()
    info = {"gpu": gpu_info(), "l2": "flushed before every timed call (256 MiB memset)", "reps": args.reps, "unit": "Mpaths/s", "configs": {}}
    print("GPU (name, power limit, max SM clock):", info["gpu"], flush=True)

    def timed_radiance(ds, cam, o4, d4):
        to, td = torch.from_numpy(np.ascontiguousarray(o4)).to(dev), torch.from_numpy(np.ascontiguousarray(d4)).to(dev)
        out = torch.empty((len(o4), 4), dtype=torch.float32, device=dev)
        c = cam.c()
        stream = torch.cuda.current_stream(dev).cuda_stream

        def call():
            st = _lib.RenderStats()
            if not lib.oclr_scene_radiance(ds.handle, C.byref(c), len(o4), C.c_void_p(to.data_ptr()), C.c_void_p(td.data_ptr()), None, 0, 1,
                                           C.c_void_p(out.data_ptr()), None, api.QUERY_DEVICE_MEMORY, 0, C.c_void_p(stream), C.byref(st)):
                raise api.OclrError(_lib.last_error())
            return st.deviceMs
        return timed(call, len(o4))

    def timed(call, paths):
        for _ in range(2):
            call()
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            torch.cuda.synchronize(dev)
            ms.append(call())
        med = float(np.median(ms))
        return {"paths": int(paths), "ms_median": med, "ms_min": float(min(ms)), "ms_max": float(max(ms)), "mpaths_per_s": paths / med / 1e3}

    for cid in (2, 3):
        cfg = scenes.CONFIGS[cid]
        sc = cfg["make"]()
        m = sc.meta["camera"]
        ds = api.DeviceScene(sc)
        W, H = 1920, 1080
        cam = api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], W, H)
        res = {"workload": cfg["name"], "triangles": int(sc.triangle_count), "sets": {}}
        fr = api.DeviceFrame(ds, cam)
        res["frame"] = timed(lambda: fr.render(1)[0], W * H)
        fr.close()
        print(f"config {cid} frame 1920x1080 S=1: {res['frame']['mpaths_per_s']:8.1f} Mpaths/s ({res['frame']['ms_median']:.3f} ms)", flush=True)
        sets = {}
        if cid == 2:
            y, x = np.mgrid[0:H, 0:W]
            d = cam.eye_to_top_left[:3] + (x.ravel() + 0.5)[:, None] * cam.left_to_right[:3] + (y.ravel() + 0.5)[:, None] * cam.top_to_bottom[:3]
            o4 = np.zeros((W * H, 4), np.float32)
            o4[:, :3] = cam.eye[:3]
            d4 = np.zeros((W * H, 4), np.float32)
            d4[:, :3] = d
            d4[:, 3] = np.inf
            order = tile_order(W, H)
            shuf = np.random.default_rng(2).permutation(W * H)
            sets["eye_tiles"] = (o4[order], d4[order])
            sets["eye_shuffled"] = (o4[shuf], d4[shuf])
        PW, PH = 3840, 1920
        dirs = render.equirect_directions(render.equirect_basis(m["eye"], m["look_at"], m["up"]), PW, PH)
        po = np.zeros((PW * PH, 4), np.float32)
        po[:, :3] = cam.eye[:3]
        pd = np.zeros((PW * PH, 4), np.float32)
        pd[:, :3] = dirs
        pd[:, 3] = np.inf
        sets["equirect_3840x1920"] = (po, pd)
        for name, (o4, d4) in sets.items():
            row = timed_radiance(ds, cam, o4, d4)
            row["vs_frame"] = row["mpaths_per_s"] / res["frame"]["mpaths_per_s"]
            res["sets"][name] = row
            print(f"config {cid} {name:20s} paths {len(o4):8d}  {row['mpaths_per_s']:8.1f} Mpaths/s ({row['ms_median']:.3f} ms, "
                  f"{row['vs_frame']:.2f}x frame)", flush=True)
        info["configs"][str(cid)] = res
        ds.close()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(info, indent=1))


if __name__ == "__main__":
    main()
