"""Entry points shaped like the reference's: `clojure -M:main [spp] [depth]`
(src/raytracing.clj:95-177) and `clojure -M:realm` (src/realm/raytracing.clj:259-358).

    python -m raytracing_clj_b200.main main [spp] [depth]     -> scene.ppm
    python -m raytracing_clj_b200.main main [spp] [depth] --every N
                                                              -> scene.ppm, rewritten every N samples
    python -m raytracing_clj_b200.main realm                  -> scene-realm.ppm
    python -m raytracing_clj_b200.main i                      -> scene-i.ppm

Each renders the reference's literal scene and camera through the C ABI on the GPU and writes
the P3 file the reference writes.  `(time ...)` is mirrored by printing the elapsed time.

With --every N the image is rendered in passes of N samples (rounded up to the render's pass unit) and
scene.ppm / scene.png are replaced after each pass, so that an open viewer shows the image refine; the
last files are byte for byte those of a run without --every."""
from __future__ import annotations

import os
import sys
import time

from . import _abi, camera, render, scenes


def _replace(path: str, data: bytes) -> None:
    """Writes `path` through a temporary file and a rename: a viewer never reads half a file."""
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(data)
    os.replace(tmp, path)


def main_variant(spp: int = 100, depth: int = 50, out: str = "scene.ppm", seed: int = 1, every: int = 0):
    print("config:", {"samples-per-px": spp, "max-depth": depth})
    t0 = time.perf_counter()
    if every > 0:
        png = out[:-4] + ".png" if out.endswith(".ppm") else out + ".png"
        with render.Progressive(scenes.main_hittables(), camera.main_camera(), spp, depth, seed=seed,
                                flags=_abi.FLAGS_MAIN) as p:
            n = -(-every // p.pass_unit) * p.pass_unit
            segments = 0
            while p.samples_done < spp:
                _, rgb8, st = p.step(min(n, spp - p.samples_done), want_linear=False)
                segments += st["segments"]
                if p.samples_done < spp:  # the last image goes out below, as without --every
                    _replace(out, render.encode_ppm(rgb8))
                    _replace(png, render.encode_png(rgb8))
                print(f"{p.samples_done}/{spp} samples per pixel: {out} ({1e3 * (time.perf_counter() - t0):.0f} ms)")
        st["segments"] = segments
    else:
        _, rgb8, st = render.render(scenes.main_hittables(), camera.main_camera(), spp, depth, seed=seed,
                                    flags=_abi.FLAGS_MAIN, want_linear=False)
    render.write_ppm(out, rgb8)
    render.ppm_to_png(out, out[:-4] + ".png" if out.endswith(".ppm") else out + ".png")  # (ppm->png "scene.ppm" "scene.png"), raytracing.clj:176
    print(f'"Elapsed time: {1e3 * (time.perf_counter() - t0):.3f} msecs"  ({st["segments"]} ray segments)')
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
        every = 0
        if "--every" in argv:
            i = argv.index("--every")
            if i + 1 >= len(argv) or int(argv[i + 1]) <= 0:
                raise SystemExit("--every needs a positive number of samples")
            every = int(argv[i + 1])
            argv = argv[:i] + argv[i + 2:]
        main_variant(int(argv[1]) if len(argv) > 1 else 100, int(argv[2]) if len(argv) > 2 else 50, every=every)
    elif which == "realm":
        realm_variant()
    elif which == "i":
        i_variant()
    else:
        raise SystemExit(__doc__)


if __name__ == "__main__":
    _cli(sys.argv[1:])
