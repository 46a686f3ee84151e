"""Measures adaptive accumulations over frames (rtclj_ctx_accum_begin_frames, DESIGN.md section 4.15) on one GPU,
device-resident: ONE sequence accumulation against K single-camera accumulations run back to back on the same context,
with the same passes (spp/10 rounded up to the pass unit, as the CLI), each run until no pixel is active.
  main:  the CLI's 60-frame turntable of the default scene at 400x225, target 500, depth 50, tolerance (0.004, 0.04).
  cover: the cover scene at 1920x1080 on an 8-frame turntable about its look_at, target 500, depth 50, same tolerance.
Recorded per case: the time of each pass and in total (host wall clock around each step and a device synchronise, as
tools/bench_adaptive.py; the singles' pass p is the sum of their p-th passes), the samples traced (the library's
counters), the pixels live at each pass, and whether every frame's linear and 8-bit images and sample counts are
identical.  Both variants are warmed up once and then alternated --reps times; medians are reported.  The card's name
and power limit are read in the same run.  Prints one JSON line and writes it to --out.
Usage: python tools/bench_adaptive_frames.py [--reps N] [--out profiles/r3_bench_adaptive_frames.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import raytracing_clj_b200 as R  # noqa: E402
from raytracing_clj_b200 import _abi, render  # noqa: E402

S, CAM = R.scenes, R.camera
TOL, SPP, DEPTH, SEED = (0.004, 0.04), 500, 50, 1


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def cases():
    cover = dict(S.COVER_CAMERA)
    look_from, look_at = cover.pop("look_from"), cover.pop("look_at")
    return [("main_turntable_60x400x225", S.main_hittables(), CAM.turntable_cameras(60)),
            ("cover_turntable_8x1920x1080", S.cover_hittables(7),
             [CAM.main_camera(1920, 1080, look_from=CAM.turntable_look_from(k, 8, look_from, look_at), look_at=look_at,
                              **cover) for k in range(8)])]


class Images:
    def __init__(self, cam, k):
        self.lin = torch.zeros((k, cam.height, cam.width, 3), dtype=torch.float64, device="cuda:0")
        self.rgb = torch.zeros((k, cam.height, cam.width, 3), dtype=torch.uint8, device="cuda:0")
        self.samples = torch.zeros((k, cam.height, cam.width), dtype=torch.int32, device="cuda:0")
        self.stream = torch.cuda.current_stream().cuda_stream


def accumulate(ctx, cams, img, f0=None):
    """One accumulation until no pixel is active: all cameras (f0 None) or camera f0 into frame f0 of `img`.
    Returns per pass [(live pixels before it, ms, samples traced)]."""
    one = f0 is not None
    kw = dict(seed=SEED, flags=_abi.FLAGS_MAIN, stream=img.stream, tolerance=TOL)
    unit = ctx.accum_begin(cams[f0], SPP, DEPTH, **kw) if one else ctx.accum_begin_frames(cams, SPP, DEPTH, **kw)
    n = -(-(SPP // 10) // unit) * unit
    k = f0 or 0
    lin, rgb, smp = (t[k] if one else t for t in (img.lin, img.rgb, img.samples))
    active, done, log = cams[0].width * cams[0].height * (1 if one else len(cams)), 0, []
    while done < SPP and active > 0:
        t0 = time.perf_counter()
        done = ctx.accum_step(min(n, SPP - done), d_out_linear=lin.data_ptr(), d_out_rgb8=rgb.data_ptr(),
                              stream=img.stream)
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        traced = ctx.stats(img.stream)["samples"]
        log.append((active, ms, traced))
        active = ctx.accum_noise(smp.data_ptr(), stream=img.stream)
    return log


def singles(ctx, cams, img):
    """K single-camera accumulations back to back; per pass p the sums over the frames that ran a p-th pass."""
    out = []
    for f in range(len(cams)):
        for p, (a, ms, t) in enumerate(accumulate(ctx, cams, img, f)):
            if p == len(out):
                out.append([0, 0.0, 0])
            out[p][0] += a
            out[p][1] += ms
            out[p][2] += t
    return [tuple(x) for x in out]


def run_case(name, world, cams, reps):
    ctx = render.Context(0)
    ctx.set_scene(world)
    seq, one = Images(cams[0], len(cams)), Images(cams[0], len(cams))
    accumulate(ctx, cams, seq)  # warm-up of both shapes
    singles(ctx, cams, one)
    seq_runs, one_runs = [], []
    for _ in range(reps):  # alternated
        seq_runs.append(accumulate(ctx, cams, seq))
        one_runs.append(singles(ctx, cams, one))
    same = bool(torch.equal(seq.lin.view(torch.int64), one.lin.view(torch.int64)) and torch.equal(seq.rgb, one.rgb)
                and torch.equal(seq.samples, one.samples))
    ctx.close()
    med = lambda xs: sorted(xs)[len(xs) // 2]  # noqa: E731
    total = lambda log: sum(ms for _, ms, _ in log)  # noqa: E731

    def summary(runs):
        log = sorted(runs, key=total)[len(runs) // 2]  # the per-pass figures of the median run
        return {"total_ms": [total(r) for r in runs], "median_total_ms": med([total(r) for r in runs]),
                "samples_traced": sum(t for _, _, t in runs[0]), "passes": len(runs[0]),
                "per_pass": [{"live_pixels": a, "ms": ms, "samples": t,
                              "ns_per_sample": 1e6 * ms / t if t else None} for a, ms, t in log]}

    s, o = summary(seq_runs), summary(one_runs)
    pixels = len(cams) * cams[0].width * cams[0].height
    return {"case": name, "frames": len(cams), "size": [cams[0].width, cams[0].height], "target_spp": SPP,
            "tolerance": list(TOL), "sequence": s, "singles": o,
            "samples_pct_of_uniform": 100.0 * s["samples_traced"] / (SPP * pixels),
            "speedup": o["median_total_ms"] / s["median_total_ms"], "images_identical": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_adaptive_frames.json"))
    args = ap.parse_args()
    line = {"card": card(), "reps": args.reps, "cases": [run_case(*c, args.reps) for c in cases()]}
    text = json.dumps(line)
    print(text, flush=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
