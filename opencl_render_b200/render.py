"""Standalone render harness: what the Cinema4D dialog + `parseAndRender` do around the raytrace path (source/render.cpp:174-186,
240-276, 300-365, 1009-1400), for a Linux shell.

    python -m opencl_render_b200.render SCENE --out img.png [--size 1024x768] [--samples 100] [--device 1] ...

SCENE is a Wavefront OBJ or a PLY file (loader.py) or the name of a built-in synthetic scene (`config1` .. `config4`, scenes.py).
Defaults are the dialog's: 1024x768, 100 samples per pixel (render.cpp:176-182); `--device` is the dialog's processor combo index
(`--list-devices` prints it; index 0 is the reference's CPU entry and is refused -- this library has no CPU path).

The scene is uploaded once; camera lists and -- unless `--host-builders` -- the 256^3 grid are built on the device.  Samples are
rendered in passes of `--pass-samples`; after every pass the dialog's three lines are printed (progress, estimated time left,
rendering time) and, with `--preview`, the picture so far is written.  `--checkpoint FILE` saves the planes and the number of
finished samples after every pass and resumes from the file when it exists.

`--projection equirect` renders a 360 x 180 degree panorama around the eye instead (what Cinema4D's spherical camera renders): one
radiance query per pixel (DeviceScene.radiance), in chunks of rows, with `--samples` samples per pixel.  The panorama is level: `--up`
is its pole, and longitude 0 looks towards the look-at point (projected onto the horizon).  The options of the pass loop (`--pass-samples`,
`--preview`, `--checkpoint`, `--float-accum`) belong to the pinhole path and are refused with it."""
from __future__ import annotations

import argparse
import sys
import time
from pathlib import Path

import numpy as np

from . import api, scenes


def _vec(text: str, n: int = 3):
    v = [float(x) for x in text.split(",")]
    if len(v) != n:
        raise argparse.ArgumentTypeError(f"expected {n} comma-separated numbers, got {text!r}")
    return v


def _light(text: str) -> dict:
    """type:px,py,pz:dx,dy,dz[:r,g,b[:radius[:half]]]   (type = the C4D light type number, raytrace_opencl.h:1-12)"""
    f = text.split(":")
    if len(f) < 3:
        raise argparse.ArgumentTypeError("light = type:px,py,pz:dx,dy,dz[:r,g,b[:radius[:half]]]")
    e = dict(type=int(f[0]), pos=_vec(f[1]), dir=_vec(f[2]))
    if len(f) > 3:
        e["colour"] = _vec(f[3])
    if len(f) > 4:
        e["radius"] = float(f[4])
    if len(f) > 5:
        e["half"] = float(f[5])
    return e


def _time_str(seconds: float) -> str:
    """GetTimeStr (render.cpp:280-297): d/h/m/s, the two most significant units."""
    s = int(seconds)
    if s >= 86400:
        return f"{s // 86400}d {s % 86400 // 3600}h"
    if s >= 3600:
        return f"{s // 3600}h {s % 3600 // 60}m"
    if s >= 60:
        return f"{s // 60}m {s % 60}s"
    return f"{s}s"


def equirect_basis(eye, look_at, up):
    """Orthonormal (right, up, forward) in float32 for a level panorama: up = unit(--up) is the pole, forward = the view direction with its
    component along the pole removed, right = up x forward (the pinhole camera's left-to-right direction, builders.cpp set_camera)."""
    f32 = lambda v: np.asarray(v, np.float32)[:3]
    norm = lambda v: np.float32(np.sqrt(np.float32((v * v).sum())))
    pole = f32(up) / norm(f32(up))
    view = f32(look_at) - f32(eye)
    horizontal = view - np.float32((view * pole).sum()) * pole
    if not norm(horizontal) > np.float32(1e-6) * norm(view):
        raise ValueError("the view direction is parallel to --up: the panorama has no horizontal reference direction")
    forward = horizontal / norm(horizontal)
    right = np.cross(pole, forward).astype(np.float32)
    return right / norm(right), pole, forward


def equirect_directions(basis, width: int, height: int, rows=None):
    """Directions of rows [rows[0], rows[1]) of a width x height equirectangular panorama, float32 [n*W,3] row-major.  Pixel (x, y) has
    longitude phi = 2 pi (x + 0.5) / W - pi and latitude theta = pi / 2 - pi (y + 0.5) / H; its direction is
    cos(theta) sin(phi) right + sin(theta) up + cos(theta) cos(phi) forward.  The angle tables cover the whole image, so a chunk's
    directions are bit for bit those of the whole panorama."""
    right, up, forward = (np.asarray(v, np.float32) for v in basis)
    y0, y1 = rows if rows is not None else (0, height)
    x = np.arange(width, dtype=np.float32)
    y = np.arange(height, dtype=np.float32)
    phi = np.float32(2 * np.pi) * (x + np.float32(0.5)) / np.float32(width) - np.float32(np.pi)
    theta = np.float32(np.pi / 2) - np.float32(np.pi) * (y + np.float32(0.5)) / np.float32(height)
    ct, st = np.cos(theta)[y0:y1, None, None], np.sin(theta)[y0:y1, None, None]
    cp, sp = np.cos(phi)[None, :, None], np.sin(phi)[None, :, None]
    d = ct * sp * right + st * up + ct * cp * forward
    return np.ascontiguousarray(d.reshape(-1, 3), np.float32)


def planes_from_mean(rgb, width: int, rows: int):
    """(int)(mean * 65535) clamped to 16 bits -- the frame's float-accumulation conversion -- as three uint16 [rows,W] planes."""
    v = np.nan_to_num(np.asarray(rgb, np.float32) * np.float32(65535), nan=0.0, posinf=0.0, neginf=0.0)
    v = np.clip(np.trunc(v), 0, 65535).astype(np.uint16)
    return tuple(np.ascontiguousarray(v[:, c].reshape(rows, width)) for c in range(3))


def render_equirect(ds: api.DeviceScene, cam: api.CameraSetup, basis, width: int, height: int, samples: int, say=lambda *x: None):
    """The panorama's planes (r, g, b) uint16 [H,W]; sample s of pixel p = y * W + x is seeded p * samples + s + 1."""
    planes = tuple(np.zeros((height, width), np.uint16) for _ in range(3))
    chunk = max(1, api.RADIANCE_BATCH // width)
    t0 = time.monotonic()
    eye = np.asarray(cam.eye[:3], np.float32)
    for y0 in range(0, height, chunk):
        y1 = min(height, y0 + chunk)
        d = equirect_directions(basis, width, height, (y0, y1))
        o = np.broadcast_to(eye, d.shape)
        rgb, _ = ds.radiance(o, d, samples=samples, index_base=y0 * width, camera=cam)
        for p, q in zip(planes, planes_from_mean(rgb, width, y1 - y0)):
            p[y0:y1] = q
        el = time.monotonic() - t0
        say(f"Rendering Progress {100 * y1 / height:.1f} %   Estimated Time Left {_time_str(el / y1 * (height - y1))}   "
            f"Rendering Time {_time_str(el)}")
    return planes


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m opencl_render_b200.render", description=__doc__.split("\n\n")[0])
    ap.add_argument("scene", nargs="?", help="OBJ / PLY file or config1..config4")
    ap.add_argument("--out", default="img.png", help=".png / .ppm (16 bit) or .bmp (8 bit); the reference writes img.bmp")
    ap.add_argument("--size", default="1024x768")
    ap.add_argument("--samples", type=int, default=100)
    ap.add_argument("--pass-samples", type=int, default=0, help="samples per pass (0: about 20 passes)")
    ap.add_argument("--device", type=int, default=1, help="computation type: 1 = first CUDA device")
    ap.add_argument("--list-devices", action="store_true")
    ap.add_argument("--eye", type=_vec)
    ap.add_argument("--look-at", type=_vec)
    ap.add_argument("--up", type=_vec, default=[0.0, 1.0, 0.0])
    ap.add_argument("--fov", type=float, help="horizontal field of view in radians")
    ap.add_argument("--light", type=_light, action="append")
    ap.add_argument("--float-accum", action="store_true", help="fp32 accumulation instead of the reference's per-sample truncation")
    ap.add_argument("--host-builders", action="store_true", help="build the grid and the camera lists on the host")
    ap.add_argument("--preview", action="store_true", help="write --out after every pass")
    ap.add_argument("--checkpoint", help="file the job state is saved to after every pass / resumed from")
    ap.add_argument("--bmp-reference-cast", action="store_true", help="BMP bytes = low byte, like writebmp3s (writebmp.cpp:136-141)")
    ap.add_argument("--projection", choices=["pinhole", "equirect"], default="pinhole",
                    help="pinhole: the camera's own image; equirect: a 360 x 180 degree panorama around --eye")
    ap.add_argument("--quiet", action="store_true")
    a = ap.parse_args(argv)
    say = (lambda *x: None) if a.quiet else (lambda *x: print(*x, file=sys.stderr, flush=True))
    if a.projection == "equirect":
        for flag, given in (("--checkpoint", a.checkpoint), ("--float-accum", a.float_accum), ("--pass-samples", a.pass_samples),
                            ("--preview", a.preview)):
            if given:
                ap.error(f"{flag} belongs to the pinhole pass loop and is not supported with --projection equirect")

    names = api.computation_types()
    if a.list_devices:
        for i, n in enumerate(names):
            print(f"{i}: {n}")
        return 0
    if not a.scene:
        ap.error("scene missing")
    if a.device <= 0 or a.device >= len(names) or "all" in names[a.device]:
        ap.error(f"--device must name one CUDA device (1..{max(1, len([n for n in names[1:] if 'all' not in n]))}); "
                 "0 is the reference's CPU entry, which this library does not implement")
    w, h = (int(x) for x in a.size.lower().split("x"))
    t_prepare = time.monotonic()

    if a.scene.lower().startswith("config") and not Path(a.scene).exists():
        cfg = scenes.CONFIGS[int(a.scene[6:])]
        sc = cfg["make"]()
        cm = dict(sc.meta["camera"])
    else:
        from . import loader
        eye = a.eye or [0.0, 1.0, -5.0]
        sc = loader.load_scene(a.scene, eye=eye, lights=a.light)
        cm = dict(eye=eye, look_at=[0.0, 0.0, 0.0], up=a.up, fov=0.9)
    if a.eye:
        cm["eye"] = a.eye
    if a.look_at:
        cm["look_at"] = a.look_at
    if a.fov:
        cm["fov"] = a.fov
    cm["up"] = a.up if a.up else cm.get("up", [0, 1, 0])
    cam = api.set_camera(cm["eye"], cm["look_at"], cm["up"], cm["fov"], w, h)
    lists = None
    if a.host_builders:
        if a.projection == "pinhole":   # (a panorama reads no camera lists)
            lists = api.camera_triangle_list(cam, sc)
        api.scene_triangle_list(sc, api.AXES_DIVISION)
    ds = api.DeviceScene(sc, a.device - 1)
    if a.projection == "equirect":
        say(f"{sc.name}: {sc.triangle_count} triangles, {sc.material_count} materials, {sc.light_count} lights on {names[a.device]}; "
            f"scene & device prepare time {_time_str(time.monotonic() - t_prepare)} ({time.monotonic() - t_prepare:.2f} s)")
        t0 = time.monotonic()
        img = render_equirect(ds, cam, equirect_basis(cm["eye"], cm["look_at"], cm["up"]), w, h, a.samples, say)
        el = time.monotonic() - t0
        api.write_image(a.out, img, bmp_reference_cast=a.bmp_reference_cast)
        say(f"{a.out}: {w}x{h} equirect, {a.samples} samples; {w * h * a.samples / max(el, 1e-9) / 1e6:.1f} Mpaths/s over {el:.2f} s")
        ds.close()
        return 0
    fr = api.DeviceFrame(ds, cam, lists)
    if a.float_accum:
        fr.set_accumulation(api.ACCUMULATE_FLOAT)
    say(f"{sc.name}: {sc.triangle_count} triangles, {sc.material_count} materials, {sc.light_count} lights on {names[a.device]}; "
        f"scene & device prepare time {_time_str(time.monotonic() - t_prepare)} ({time.monotonic() - t_prepare:.2f} s)")

    S = a.samples
    done = 0
    ck = Path(a.checkpoint) if a.checkpoint else None
    if ck and ck.exists():
        z = np.load(ck)
        if (int(z["samples"]), int(z["width"]), int(z["height"]), bool(z["float"])) != (S, w, h, bool(a.float_accum)):
            ap.error(f"{ck} belongs to a different job")
        done = int(z["done"])
        fr.write((z["r"], z["g"], z["b"]))
        if a.float_accum:
            fr.write_accum(z["acc"])
        say(f"resumed from {ck}: {done} of {S} samples")
    step = a.pass_samples or max(1, S // 20)
    t0 = time.monotonic()
    first = done
    while done < S:
        n = min(step, S - done)
        fr.render(S, samples=(done, done + n))
        done += n
        p = done / S
        el = time.monotonic() - t0
        left = el / max(done - first, 1) * (S - done)
        say(f"Rendering Progress {100 * p:.1f} %   Estimated Time Left {_time_str(left)}   Rendering Time {_time_str(el)}")
        if ck:
            img = fr.read()
            extra = dict(acc=fr.read_accum()) if a.float_accum else {}
            tmp = ck.with_suffix(ck.suffix + ".tmp.npz")
            np.savez(tmp, r=img[0], g=img[1], b=img[2], done=done, samples=S, width=w, height=h, float=bool(a.float_accum), **extra)
            tmp.replace(ck)
        if a.preview and done < S:
            api.write_image(a.out, fr.read(), bmp_reference_cast=a.bmp_reference_cast)
    el = time.monotonic() - t0
    img = fr.read()
    api.write_image(a.out, img, bmp_reference_cast=a.bmp_reference_cast)
    rays = w * h * (S - first)
    say(f"{a.out}: {w}x{h}, {S} samples; {rays / max(el, 1e-9) / 1e6:.1f} Mrays/s over {el:.2f} s (pixel-samples, raytrace.c:545)")
    fr.close()
    ds.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
