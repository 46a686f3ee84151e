"""Measures adaptive sampling (rtclj_ctx_accum_begin_adaptive, DESIGN.md section 4.10) on one GPU, device-resident.
  overhead: the bench frame (c3: cover scene 1920x1080, target 500, depth 50) in passes of 4 pass units with
            min_samples = spp, so that no pixel stops: the listed kernels plus the adaptive fold and compaction
            against the plain accumulation of the same passes, alternated in one run.
  benefit:  cover scene and config 2 (5 spheres) at 1920x1080, target 500, passes of 4 pass units until no pixel
            is active, for three tolerances: time and samples traced; RMSE and 99th-percentile absolute error of
            the linear image against a uniform 4000-spp render with ANOTHER seed (independent samples); the same
            errors for a uniform render of the same total samples (equal work, rounded to whole samples per pixel).
  late passes: per-pass time against the pixels the pass traced.
Times are host wall clock around each step and a device synchronise, as tools/bench_progressive.py.  The card's name
and power limit are read in the same run.  Prints one JSON line and writes it to --out.
Usage: python tools/bench_adaptive.py [--reps N] [--out profiles/r3_bench_adaptive.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import workloads  # noqa: E402
from raytracing_clj_b200 import render  # noqa: E402

TOLERANCES = [(0.004, 0.04), (0.002, 0.02), (0.001, 0.01)]
REF_SPP, REF_SEED, SEED = 4000, 977, 1


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


class Images:
    def __init__(self, cam):
        self.lin = torch.zeros((cam.height, cam.width, 3), dtype=torch.float64, device="cuda:0")
        self.rgb = torch.zeros((cam.height, cam.width, 3), dtype=torch.uint8, device="cuda:0")
        self.stream = torch.cuda.current_stream().cuda_stream

    def ptrs(self):
        return dict(d_out_linear=self.lin.data_ptr(), d_out_rgb8=self.rgb.data_ptr(), stream=self.stream)


def passes_of(unit, spp):
    n = 4 * unit
    return [min(n, spp - d) for d in range(0, spp, n)]


def accumulate(ctx, cam, spp, depth, flags, img, tolerance=None, least=0, until_done=False):
    """One accumulation; returns (per-pass [(traced pixels, ms)], total ms, samples traced)."""
    unit = ctx.accum_begin(cam, spp, depth, seed=SEED, flags=flags, stream=img.stream, tolerance=tolerance,
                           min_samples=least)
    active, log, traced = cam.width * cam.height, [], 0
    for n in passes_of(unit, spp):
        t0 = time.perf_counter()
        ctx.accum_step(n, **img.ptrs())
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        log.append((active, ms))
        traced += active * n
        if tolerance is not None:
            active = ctx.accum_noise(stream=img.stream)
            if until_done and active == 0:
                break
    return log, sum(ms for _, ms in log), traced


def overhead(wl, reps):
    world, cam = wl["world"](), wl["cam"]()
    spp, depth, flags = wl["spp"], wl["depth"], wl["flags"]
    plain, adapt = render.Context(0), render.Context(0)
    plain.set_scene(world)
    adapt.set_scene(world)
    a, b = Images(cam), Images(cam)
    accumulate(plain, cam, spp, depth, flags, a)  # warm-up
    accumulate(adapt, cam, spp, depth, flags, b, (0.0, 0.0), spp)
    p_ms, a_ms = [], []
    for _ in range(reps):  # alternated
        p_ms.append(accumulate(plain, cam, spp, depth, flags, a)[1])
        a_ms.append(accumulate(adapt, cam, spp, depth, flags, b, (0.0, 0.0), spp)[1])
    same = bool(torch.equal(a.lin.view(torch.int64), b.lin.view(torch.int64)) and torch.equal(a.rgb, b.rgb))
    plain.close(), adapt.close()
    med = lambda xs: sorted(xs)[len(xs) // 2]  # noqa: E731
    return {"workload": wl["name"], "passes": passes_of(render.pass_unit(cam.width, cam.height, spp, depth, flags), spp),
            "plain_ms": p_ms, "adaptive_min_samples_spp_ms": a_ms, "plain_median_ms": med(p_ms),
            "adaptive_median_ms": med(a_ms), "overhead_pct": 100.0 * (med(a_ms) / med(p_ms) - 1.0),
            "plain_spread_pct": 100.0 * (max(p_ms) - min(p_ms)) / med(p_ms),
            "adaptive_spread_pct": 100.0 * (max(a_ms) - min(a_ms)) / med(a_ms),
            "images_identical": same}


def errors(lin, ref):
    e = np.abs(lin - ref)
    return {"rmse": float(np.sqrt(np.mean(e * e))), "p99_abs": float(np.percentile(e, 99))}


def benefit(label, world, cam, spp, depth, flags):
    ctx = render.Context(0)
    ctx.set_scene(world)
    img = Images(cam)
    t0 = time.perf_counter()
    ctx.render(cam, REF_SPP, depth, seed=REF_SEED, flags=flags, **img.ptrs())
    torch.cuda.synchronize()
    ref_ms = 1e3 * (time.perf_counter() - t0)
    ref = img.lin.cpu().numpy().copy()
    pixels = cam.width * cam.height
    rows = []
    uni_log, uni_ms, _ = accumulate(ctx, cam, spp, depth, flags, img)
    rows.append({"mode": f"uniform {spp}", "ms": uni_ms, "samples": spp * pixels, **errors(img.lin.cpu().numpy(), ref)})
    for tol in TOLERANCES:
        accumulate(ctx, cam, spp, depth, flags, img, tol, 0, until_done=True)  # warm-up of this shape
        log, ms, traced = accumulate(ctx, cam, spp, depth, flags, img, tol, 0, until_done=True)
        samples = torch.zeros((cam.height, cam.width), dtype=torch.int32, device="cuda:0")
        ctx.accum_noise(samples.data_ptr(), stream=img.stream)
        counts = samples.cpu().numpy()
        adaptive = errors(img.lin.cpu().numpy(), ref)
        eq_spp = max(1, int(round(traced / pixels)))
        t1 = time.perf_counter()
        ctx.render(cam, eq_spp, depth, seed=SEED, flags=flags, **img.ptrs())
        torch.cuda.synchronize()
        eq_ms = 1e3 * (time.perf_counter() - t1)
        rows.append({"mode": f"adaptive abs={tol[0]} rel={tol[1]}", "ms": ms, "samples": traced,
                     "samples_pct_of_uniform": 100.0 * traced / (spp * pixels), **adaptive,
                     "passes": len(log), "per_pass": [{"traced_pixels": a, "ms": m} for a, m in log],
                     "sample_count_percentiles": {str(q): float(np.percentile(counts, q)) for q in (1, 10, 50, 90, 99)},
                     "equal_work": {"spp": eq_spp, "ms": eq_ms, **errors(img.lin.cpu().numpy(), ref)}})
    ctx.close()
    return {"case": label, "size": [cam.width, cam.height], "target_spp": spp,
            "reference": {"spp": REF_SPP, "seed": REF_SEED, "ms": ref_ms}, "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_adaptive.json"))
    args = ap.parse_args()
    wls = workloads()
    c3, c2 = wls["c3"], wls["c2"]
    line = {"card": card(), "reps": args.reps,
            "overhead": overhead(c3, args.reps),
            "benefit": [benefit("cover", c3["world"](), c3["cam"](), 500, c3["depth"], c3["flags"]),
                        benefit("config2_5_spheres", c2["world"](), c2["cam"](), 500, c2["depth"], c2["flags"])]}
    text = json.dumps(line)
    print(text, flush=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
