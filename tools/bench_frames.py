"""Measures camera sequences (rtclj_ctx_render_frames, DESIGN.md section 4.12) against a loop of single renders.

For each case -- main's default scene at 400x225 on a 60-frame turntable at 100 and 16 spp, config 2 (1920x1080,
100 spp) on 8 frames, the cover scene at 1920x1080 x 16 spp on 8 frames and config 4 (raytracing-i, 3840x2160,
100 spp) on 4 frames -- it times, device-resident on GPU 0 with a host clock around each call plus a synchronise:
  - `loop`: one rtclj_ctx_render per camera into the frame's slice of the output;
  - `frames`: one rtclj_ctx_render_frames on the same cameras;
alternated run by run, and reports the medians, the spread (min / max) of each and the ratio of the medians.  The
images of the timed runs are compared bit for bit.  With more than one GPU it also times rtclj_render_frames on all
devices against a loop of rtclj_render_multi (host buffers); otherwise that is reported as not measured.  The card's
name and power limit are read in the same run.  Prints one JSON line; --out writes it to a file.
Usage: python tools/bench_frames.py [--reps N] [--out PATH]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import raytracing_clj_b200 as R  # noqa: E402
from raytracing_clj_b200 import _abi, render  # noqa: E402

S, CAM = R.scenes, R.camera


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def turntable(n, make, look_from, look_at, **kw):
    return [make(look_from=CAM.turntable_look_from(k, n, look_from, look_at), look_at=look_at, **kw) for k in range(n)]


def cases():
    main = (-2.0, 2.0, 1.0), (0.0, 0.0, -1.0)
    cover = dict(S.COVER_CAMERA)
    cover_at = cover.pop("look_from"), cover.pop("look_at")
    i4 = [CAM.i_camera(3840)] + [CAM.main_camera(3840, 2160, look_from=CAM.turntable_look_from(k, 4), defocus_angle=0.0)
                                 for k in range(1, 4)]
    return [
        ("main_400x225_100spp_60frames", S.main_hittables(), turntable(60, CAM.main_camera, *main), 100, 50, _abi.FLAGS_MAIN),
        ("main_400x225_16spp_60frames", S.main_hittables(), turntable(60, CAM.main_camera, *main), 16, 50, _abi.FLAGS_MAIN),
        ("c2_main_1920x1080_100spp_8frames", S.main_hittables(), turntable(8, CAM.main_camera, *main, width=1920), 100, 50,
         _abi.FLAGS_MAIN),
        ("cover_1920x1080_16spp_8frames", S.cover_hittables(7),
         turntable(8, CAM.main_camera, *cover_at, width=1920, height=1080, **cover), 16, 50, _abi.FLAGS_MAIN),
        ("c4_raytracing_i_3840x2160_100spp_4frames", S.i_hittables(), i4, 100, 50, _abi.FLAGS_I),
    ]


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def device_case(name, world, cams, spp, depth, flags, reps):
    ctx = render.Context(0)
    ctx.set_scene(world)
    k, H, W = len(cams), cams[0].height, cams[0].width
    stream = torch.cuda.current_stream().cuda_stream
    outs = {m: (torch.zeros((k, H, W, 3), dtype=torch.float64, device="cuda:0"),
                torch.zeros((k, H, W, 3), dtype=torch.uint8, device="cuda:0")) for m in ("loop", "frames")}

    def loop():
        lin, rgb = outs["loop"]
        for f, cam in enumerate(cams):
            ctx.render(cam, spp, depth, flags=flags, d_out_linear=lin[f].data_ptr(), d_out_rgb8=rgb[f].data_ptr(),
                       stream=stream)
        torch.cuda.synchronize()

    def frames():
        lin, rgb = outs["frames"]
        ctx.render_frames(cams, spp, depth, flags=flags, d_out_linear=lin.data_ptr(), d_out_rgb8=rgb.data_ptr(),
                          stream=stream)
        torch.cuda.synchronize()

    times = {"loop": [], "frames": []}
    loop(), frames()  # warm-up: module load, buffer growth
    for r in range(reps):
        for m, fn in (("loop", loop), ("frames", frames)) if r % 2 == 0 else (("frames", frames), ("loop", loop)):
            t0 = time.perf_counter()
            fn()
            times[m].append(1e3 * (time.perf_counter() - t0))
    same = bool(torch.equal(outs["loop"][0].view(torch.int64), outs["frames"][0].view(torch.int64)) and
                torch.equal(outs["loop"][1], outs["frames"][1]))
    ctx.close()
    lo, fr = spread(times["loop"]), spread(times["frames"])
    return {"case": name, "frames": k, "size": [W, H], "spp": spp, "loop_ms": lo, "frames_ms": fr,
            "speedup_of_medians": lo["median"] / fr["median"], "identical_images": same}


def host_case(name, world, cams, spp, depth, flags, reps, devices):
    k, H, W = len(cams), cams[0].height, cams[0].width
    lin_l, rgb_l = np.zeros((k, H, W, 3)), np.zeros((k, H, W, 3), dtype=np.uint8)
    lin_f, rgb_f = np.zeros((k, H, W, 3)), np.zeros((k, H, W, 3), dtype=np.uint8)

    def loop():
        for f, cam in enumerate(cams):
            render.render(world, cam, spp, depth, flags=flags, devices=devices, out_linear=lin_l[f], out_rgb8=rgb_l[f])

    def frames():
        lin, rgb, _ = render.render_frames(world, cams, spp, depth, flags=flags, devices=devices)
        lin_f[:], rgb_f[:] = lin, rgb

    times = {"loop": [], "frames": []}
    loop(), frames()
    for r in range(reps):
        for m, fn in (("loop", loop), ("frames", frames)) if r % 2 == 0 else (("frames", frames), ("loop", loop)):
            t0 = time.perf_counter()
            fn()
            times[m].append(1e3 * (time.perf_counter() - t0))
    lo, fr = spread(times["loop"]), spread(times["frames"])
    return {"case": name, "devices": list(devices), "loop_ms": lo, "frames_ms": fr,
            "speedup_of_medians": lo["median"] / fr["median"],
            "identical_images": bool(np.array_equal(lin_l.view(np.uint64), lin_f.view(np.uint64)) and np.array_equal(rgb_l, rgb_f))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    n = C.c_int()
    _abi.check(_abi.lib().rtclj_device_count(C.byref(n)))
    result = {"card": card(), "gpus": n.value, "device_resident_gpu0": [], "host_buffers_all_gpus": "not measured (one GPU)"}
    for c in cases():
        result["device_resident_gpu0"].append(device_case(*c, args.reps))
        print(json.dumps(result["device_resident_gpu0"][-1]), file=sys.stderr)
    if n.value > 1:
        devs = list(range(n.value))
        result["host_buffers_all_gpus"] = [host_case(*c, args.reps, devs) for c in cases()[:2]]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
