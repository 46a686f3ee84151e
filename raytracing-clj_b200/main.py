"""Entry points shaped like the reference's: `clojure -M:main [spp] [depth]`
(src/raytracing.clj:95-177) and `clojure -M:realm` (src/realm/raytracing.clj:259-358).

    python -m raytracing_clj_b200.main main [spp] [depth]     -> scene.ppm
    python -m raytracing_clj_b200.main main [spp] [depth] --every N
                                                              -> scene.ppm, rewritten every N samples
    python -m raytracing_clj_b200.main main [spp] [depth] --every N --tolerance ABS,REL
                                                              -> the same with adaptive sampling, and
                                                                 scene-samples.png (samples per pixel)
    python -m raytracing_clj_b200.main main ... --gpu-png     -> the same files, the PNGs compressed on the GPU
    python -m raytracing_clj_b200.main main [spp] [depth] --frames N [--gpu-png]
                                                              -> scene-0000.png ... scene-{N-1}.png, a turntable
    python -m raytracing_clj_b200.main realm                  -> scene-realm.ppm
    python -m raytracing_clj_b200.main i                      -> scene-i.ppm

Each renders the reference's literal scene and camera through the C ABI on the GPU and writes
the P3 file the reference writes.  `(time ...)` is mirrored by printing the elapsed time.

With --every N the image is rendered in passes of N samples (rounded up to the render's pass unit) and
scene.ppm / scene.png are replaced after each pass, so that an open viewer shows the image refine; the
last files are byte for byte those of a run without --every.

With --tolerance ABS,REL the passes trace only the pixels whose noise estimate is still above
ABS + REL * |pixel mean| (adaptive sampling, DESIGN.md section 4.10; every pixel gets at least two pass
units), and the run ends once no pixel is left.  scene-samples.png shows the samples each pixel received
(white: spp).

With --gpu-png scene.png (and scene-samples.png) are written by the device PNG writer from the render's 8-bit
image (DESIGN.md section 4.11): the same pixels, compressed, and only the compressed bytes leave the GPU.  Without
it every file is the one the host writer produces.

With --frames N the camera circles the scene: look_from turns about the vertical axis through look_at in N steps of
360/N degrees, frame 0 being the reference's camera, and all N frames are rendered as one camera sequence
(rtclj_render_frames, DESIGN.md section 4.12).  Each frame is written as a PNG only; frame 0 has the pixels of
scene.png from a run without --frames."""
from __future__ import annotations

import os
import sys
import time

import numpy as np

from . import _abi, camera, render, scenes


def _replace(path: str, data: bytes) -> None:
    """Writes `path` through a temporary file and a rename: a viewer never reads half a file."""
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(data)
    os.replace(tmp, path)


def samples_image(samples: np.ndarray, spp: int) -> np.ndarray:
    """The sample-count map as a grey 8-bit image: black 0, white spp samples per pixel."""
    v = np.rint(samples.astype(np.float64) * (255.0 / spp)).clip(0, 255).astype(np.uint8)
    return np.repeat(v[:, :, None], 3, axis=2)


def main_variant(spp: int = 100, depth: int = 50, out: str = "scene.ppm", seed: int = 1, every: int = 0,
                 tolerance=None, gpu_png: bool = False):
    print("config:", {"samples-per-px": spp, "max-depth": depth})
    t0 = time.perf_counter()
    png_device = 0 if gpu_png else None  # the render's device (devices default to [0])
    if tolerance is not None and every <= 0:
        every = max(1, spp // 10)
    if every > 0:
        png = out[:-4] + ".png" if out.endswith(".ppm") else out + ".png"
        cam = camera.main_camera()
        with render.Progressive(scenes.main_hittables(), cam, spp, depth, seed=seed, flags=_abi.FLAGS_MAIN,
                                tolerance=tolerance) as p:
            n = -(-every // p.pass_unit) * p.pass_unit
            segments = traced = 0
            active = cam.width * cam.height
            while p.samples_done < spp and active > 0:
                _, rgb8, st = p.step(min(n, spp - p.samples_done), want_linear=False)
                segments += st["segments"]
                traced += st["samples"]
                if p.adaptive:
                    samples, _, active = p.noise()
                if p.samples_done < spp and active > 0:  # the last image goes out below, as without --every
                    _replace(out, render.encode_ppm(rgb8))
                    _replace(png, render.encode_png(rgb8, png_device))
                left = f", {active} pixels active" if p.adaptive else ""
                print(f"{p.samples_done}/{spp} samples per pixel{left}: {out} ({1e3 * (time.perf_counter() - t0):.0f} ms)")
            if p.adaptive:
                grey = out[:-4] + "-samples.png" if out.endswith(".ppm") else out + "-samples.png"
                render.write_png(grey, samples_image(samples, spp), png_device)
                full = spp * cam.width * cam.height
                print(f"samples traced: {traced} of {full} ({100.0 * traced / full:.1f} %); sample counts in {grey}")
        st["segments"] = segments
    else:
        _, rgb8, st = render.render(scenes.main_hittables(), camera.main_camera(), spp, depth, seed=seed,
                                    flags=_abi.FLAGS_MAIN, want_linear=False)
    render.write_ppm(out, rgb8)
    png = out[:-4] + ".png" if out.endswith(".ppm") else out + ".png"
    if gpu_png:
        render.write_png(png, rgb8, png_device)
    else:
        render.ppm_to_png(out, png)  # (ppm->png "scene.ppm" "scene.png"), raytracing.clj:176
    print(f'"Elapsed time: {1e3 * (time.perf_counter() - t0):.3f} msecs"  ({st["segments"]} ray segments)')
    return st


def frames_variant(spp: int = 100, depth: int = 50, n_frames: int = 60, out: str = "scene", seed: int = 1,
                   gpu_png: bool = False):
    print("config:", {"samples-per-px": spp, "max-depth": depth, "frames": n_frames})
    t0 = time.perf_counter()
    _, rgb8, st = render.render_frames(scenes.main_hittables(), camera.turntable_cameras(n_frames), spp, depth,
                                       seed=seed, flags=_abi.FLAGS_MAIN, want_linear=False)
    t1 = time.perf_counter()
    for k in range(n_frames):
        render.write_png(f"{out}-{k:04d}.png", rgb8[k], 0 if gpu_png else None)
    print(f'"Elapsed time: {1e3 * (time.perf_counter() - t0):.3f} msecs"  (render {1e3 * (t1 - t0):.3f} ms, '
          f'{st["segments"]} ray segments, {out}-0000.png .. {out}-{n_frames - 1:04d}.png)')
    return st


def realm_variant(out: str = "scene-realm.ppm", seed: int = 1):
    t0 = time.perf_counter()
    _, rgb8, st = render.render(scenes.realm_hittables(), camera.realm_camera(), 100, 50, seed=seed,
                                flags=_abi.FLAGS_REALM, want_linear=False)
    print(f'"Elapsed time: {1e3 * (time.perf_counter() - t0):.3f} msecs"')  # realm times the loop only
    render.write_ppm(out, rgb8)
    return st


def i_variant(out: str = "scene-i.ppm", seed: int = 1):
    _, rgb8, st = render.render(scenes.i_hittables(), camera.i_camera(), 100, 50, seed=seed,
                                flags=_abi.FLAGS_I, want_linear=False)
    render.write_ppm(out, rgb8)
    return st


def _cli(argv):
    which = argv[0] if argv else "main"
    if which == "main":
        every, tolerance = 0, None
        gpu_png = "--gpu-png" in argv
        argv = [a for a in argv if a != "--gpu-png"]
        if "--frames" in argv:
            i = argv.index("--frames")
            if i + 1 >= len(argv) or not argv[i + 1].isdigit() or int(argv[i + 1]) <= 0:
                raise SystemExit("--frames needs a positive number of frames")
            n_frames = int(argv[i + 1])
            argv = argv[:i] + argv[i + 2:]
            frames_variant(int(argv[1]) if len(argv) > 1 else 100, int(argv[2]) if len(argv) > 2 else 50, n_frames,
                           gpu_png=gpu_png)
            return
        if "--tolerance" in argv:
            i = argv.index("--tolerance")
            try:
                tolerance = tuple(float(x) for x in argv[i + 1].split(","))
            except (IndexError, ValueError):
                tolerance = ()
            if len(tolerance) != 2 or min(tolerance) < 0:
                raise SystemExit("--tolerance needs ABS,REL: two numbers >= 0")
            argv = argv[:i] + argv[i + 2:]
        if "--every" in argv:
            i = argv.index("--every")
            if i + 1 >= len(argv) or int(argv[i + 1]) <= 0:
                raise SystemExit("--every needs a positive number of samples")
            every = int(argv[i + 1])
            argv = argv[:i] + argv[i + 2:]
        main_variant(int(argv[1]) if len(argv) > 1 else 100, int(argv[2]) if len(argv) > 2 else 50, every=every,
                     tolerance=tolerance, gpu_png=gpu_png)
    elif which == "realm":
        realm_variant()
    elif which == "i":
        i_variant()
    else:
        raise SystemExit(__doc__)


if __name__ == "__main__":
    _cli(sys.argv[1:])
