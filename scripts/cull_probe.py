#!/usr/bin/env python3
"""The hidden-side light cull (oclr_set_option "cull_hidden_lights") A/B on configs 2, 3 and 5 in one process: the same frames rendered
alternately with the cull off and on, device time per frame (stats.deviceMs, L2 flushed before every render) and trace-stage time
(stats.traceMs), planes compared.  Config 5: 8 of its 64 sweep cameras (every 8th), camera lists built on the device, summed per pass.

    python scripts/cull_probe.py [--reps 10] [--configs 2,3,5] [--out FILE.json]

"spread" is (max - min) / median over the passes of one setting: the run-to-run noise of the same build in the same process."""
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


def stats(v):
    v = np.asarray(v, np.float64)
    med = float(np.median(v))
    return {"median": med, "min": float(v.min()), "max": float(v.max()), "spread": float((v.max() - v.min()) / med)}


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
        if cid == 5:
            cams = scenes.sweep_cameras(sc, cfg["frames"])[::8]
        else:
            cams = [sc.meta["camera"]]
        cams = [api.set_camera(m["eye"], m["look_at"], m["up"], m["fov"], W, H) for m in cams]
        fr = api.DeviceFrame(ds, cams[0])                 # camera lists built on the device

        def one_pass(on):
            api.set_option("cull_hidden_lights", on)
            ms = tms = 0.0
            planes = []
            for cam in cams:
                if len(cams) > 1:
                    fr.set_camera(cam)
                flush.zero_()
                torch.cuda.synchronize()
                t, _, _ = fr.render(S)
                ms += t
                tms += fr.last_trace_ms
                planes.append(fr.read())
            return ms, tms, fr.last_trace_launches, planes

        for on in (0, 1, 0, 1):                          # warm-up: allocations, first launches
            one_pass(on)
        frame = {0: [], 1: []}
        trace = {0: [], 1: []}
        launches = {}
        equal = True
        for _ in range(args.reps):
            got = {}
            for on in (0, 1):
                ms, tms, launches[on], got[on] = one_pass(on)
                frame[on].append(ms)
                trace[on].append(tms)
            equal &= all(np.array_equal(a[c], b[c]) for a, b in zip(got[0], got[1]) for c in range(3))
        api.set_option("cull_hidden_lights", 1)
        r = {"workload": cfg["name"], "frames_per_pass": len(cams), "equal_planes": bool(equal),
             "off": {"frame_ms": stats(frame[0]), "trace_ms": stats(trace[0]), "trace_launches_last_frame": launches[0]},
             "on": {"frame_ms": stats(frame[1]), "trace_ms": stats(trace[1]), "trace_launches_last_frame": launches[1]}}
        r["frame_gain"] = r["off"]["frame_ms"]["median"] / r["on"]["frame_ms"]["median"] - 1.0
        r["trace_gain"] = r["off"]["trace_ms"]["median"] / r["on"]["trace_ms"]["median"] - 1.0
        result["configs"][str(cid)] = r
        for on in (0, 1):
            f, t = r["on" if on else "off"]["frame_ms"], r["on" if on else "off"]["trace_ms"]
            print(f"cfg{cid} {cfg['name']} ({len(cams)} frame{'s' if len(cams) > 1 else ''}/pass) cull {'on ' if on else 'off'}: "
                  f"frame {f['median']:.3f} ms [{f['min']:.3f}, {f['max']:.3f}] spread {100 * f['spread']:.1f} %, "
                  f"trace {t['median']:.3f} ms spread {100 * t['spread']:.1f} %", flush=True)
        print(f"cfg{cid}: frame {100 * r['frame_gain']:+.1f} %, trace {100 * r['trace_gain']:+.1f} % faster with the cull; planes equal: {equal}",
              flush=True)
        fr.close()
        ds.close()
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
