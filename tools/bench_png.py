"""Measures the device PNG writer (rtclj_ctx_encode_png, DESIGN.md section 4.11) on one GPU.

For each input -- the cover render (c3's scene) at 1920x1080 100 spp, the config-4 image (raytracing-i) at
3840x2160, main's default scene (400x225, 100 spp) and a raytracing-i render at 7680x4320 (99.5 MB of filtered
stream, more than the 126 MB L2 holds together with F, the staging slots and the output) -- it reports:
  - the device time of rtclj_ctx_encode_png on a device-resident image: CUDA events around warm calls, median
    (the call synchronises, so a call is all its kernels plus the length read-back);
  - the kernels' own times from torch.profiler in a separate pass (filter, deflate, place);
  - bytes of the device PNG, of the host writer's stored PNG, and of zlib -1 / -6 on the same filtered stream with
    their host times;
  - end to end: rtclj_render_multi_png against rtclj_render_multi + the host encode_png, on 1 and 2 devices.
The card's name and power limit are read in the same run.  Prints one JSON line; --out writes it to a file.
Usage: python tools/bench_png.py [--reps N] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import png_model as M  # noqa: E402
import raytracing_clj_b200 as R  # noqa: E402
from raytracing_clj_b200 import _abi, render  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def inputs():
    S, CAM = R.scenes, R.camera
    return [
        ("cover_1920x1080_100spp", S.cover_hittables(7), CAM.main_camera(1920, 1080, **S.COVER_CAMERA), 100, 50, _abi.FLAGS_MAIN),
        ("c4_raytracing_i_3840x2160_100spp", S.i_hittables(), CAM.i_camera(3840), 100, 50, _abi.FLAGS_I),
        ("main_default_400x225_100spp", S.main_hittables(), CAM.main_camera(), 100, 50, _abi.FLAGS_MAIN),
        ("raytracing_i_7680x4320_4spp", S.i_hittables(), CAM.i_camera(7680), 4, 50, _abi.FLAGS_I),
    ]


def host_ms(fn, reps=3):
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        dt = 1e3 * (time.perf_counter() - t0)
        best = dt if best is None else min(best, dt)
    return out, best


def ndevices():
    n = torch.cuda.device_count()
    return n


def run(name, world, cam, spp, depth, flags, reps):
    H, W = cam.height, cam.width
    _, rgb, _ = render.render(world, cam, spp, depth, flags=flags, want_linear=False)
    ctx = render.Context(0)
    stream = torch.cuda.current_stream().cuda_stream
    d_img = torch.from_numpy(rgb).cuda()
    cap = ctx.encode_png(d_img.data_ptr(), W, H)
    d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda:0")
    for _ in range(3):
        n = ctx.encode_png(d_img.data_ptr(), W, H, d_out.data_ptr(), cap, stream)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = []
    for _ in range(reps):
        ev[0].record()
        ctx.encode_png(d_img.data_ptr(), W, H, d_out.data_ptr(), cap, stream)
        ev[1].record()
        ev[1].synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    dev_png = bytes(d_out[:n].cpu().numpy())
    model_equal = dev_png == M.encode(rgb)
    # kernel times in a pass of their own
    kern = {}
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            ctx.encode_png(d_img.data_ptr(), W, H, d_out.data_ptr(), cap, stream)
    for e in prof.key_averages():
        if "png_" in e.key:
            k = e.key.split("(")[0].split("::")[-1]
            kern[k] = round(e.device_time_total / 1e3 / e.count, 4) if hasattr(e, "device_time_total") else None
    ctx.close()
    F, _ = M.filter_rows(rgb)
    Fb = F.tobytes()
    host_png, host_png_ms = host_ms(lambda: render.encode_png(rgb))
    z1, z1_ms = host_ms(lambda: zlib.compress(Fb, 1))
    z6, z6_ms = host_ms(lambda: zlib.compress(Fb, 6))
    e2e = {}
    for nd in (1, 2):
        if ndevices() < nd:
            e2e[f"{nd}_devices"] = "not measured: one GPU"
            continue
        devs = list(range(nd))
        render.render_png(world, cam, spp, depth, flags=flags, devices=devs)  # warm
        (png, _), t_png = host_ms(lambda: render.render_png(world, cam, spp, depth, flags=flags, devices=devs))

        def host_path():
            _, img, _ = render.render(world, cam, spp, depth, flags=flags, devices=devs, want_linear=False)
            return render.encode_png(img)
        _, t_host = host_ms(host_path)
        e2e[f"{nd}_devices"] = {"render_multi_png_ms": round(t_png, 3), "render_multi_plus_host_encode_png_ms": round(t_host, 3),
                                "png_bytes": len(png)}
    algorithmic = rgb.nbytes + 2 * len(Fb) + 2 * n  # image in; F out and in; segments out and in (place); file out
    med = float(np.median(ms))
    return {
        "input": name, "width": W, "height": H, "filtered_bytes": len(Fb),
        "encode_ms_median": round(med, 4), "encode_ms_min": round(min(ms), 4), "reps": reps,
        "kernel_ms": kern,
        "device_png_bytes": n, "device_equals_model": model_equal,
        "host_stored_png_bytes": len(host_png), "host_stored_png_ms": round(host_png_ms, 3),
        "zlib1_bytes": len(z1), "zlib1_ms": round(z1_ms, 3), "zlib6_bytes": len(z6), "zlib6_ms": round(z6_ms, 3),
        "algorithmic_bytes": algorithmic, "algorithmic_GBps": round(algorithmic / (med * 1e-3) / 1e9, 1),
        "end_to_end": e2e,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    res = {"card": card(), "results": [run(*x, a.reps) for x in inputs()]}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
