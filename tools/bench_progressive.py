"""Measures progressive rendering (rtclj_ctx_accum_*, DESIGN.md section 4.9) against the one-shot render of
the same image on one GPU, device-resident:
  c3 (cover scene 1920x1080, 500 spp, depth 50) in 20 passes of 25 samples, chunked (samples_per_unit 25) and in
  strict order; c4 (raytracing-i, 3840x2160, 100 spp, strict by default) in 10 passes of 10.
Times are host wall clock around each launch and a device synchronise, so that the per-pass overhead (launches,
finalize, the sync a viewer needs before it reads the image) is in them; the one-shot time is measured the same
way.  Also: the accumulator and per-sample-buffer bytes the passes need, the device memory the accumulating context
allocates in its first accumulation, whether the last image equals the one-shot image bit for bit, and the card's name and
power limit, read in the same run.  Prints one JSON line.  Usage: python tools/bench_progressive.py [--reps N]"""
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

STRICT_BUF_BYTES = 2 << 30  # kAccumSampleBufBytes in rtclj_abi.cu


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def run_case(label, wl, spu, passes, reps):
    world, cam = wl["world"](), wl["cam"]()
    spp, depth, flags = wl["spp"], wl["depth"], wl["flags"]
    assert sum(passes) == spp
    H, W = cam.height, cam.width
    lin = torch.zeros((H, W, 3), dtype=torch.float64, device="cuda:0")
    rgb = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda:0")
    out = dict(d_out_linear=lin.data_ptr(), d_out_rgb8=rgb.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    one, acc = render.Context(0), render.Context(0)
    one.set_scene(world)
    acc.set_scene(world)

    def oneshot():
        t0 = time.perf_counter()
        one.render(cam, spp, depth, flags=flags, samples_per_unit=spu, **out)
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0)

    def progressive():
        free0 = torch.cuda.mem_get_info(0)[0]
        unit = acc.accum_begin(cam, spp, depth, flags=flags, samples_per_unit=spu, stream=out["stream"])
        ms, low = [], free0
        for n in passes:
            t0 = time.perf_counter()
            acc.accum_step(n, **out)
            torch.cuda.synchronize()
            ms.append(1e3 * (time.perf_counter() - t0))
            low = min(low, torch.cuda.mem_get_info(0)[0])
        return unit, ms, free0 - low

    oneshot()  # warm-up: modules, work buffers
    ref = (lin.cpu().numpy().copy(), rgb.cpu().numpy().copy())
    growth = progressive()[2]  # the accumulating context allocates its buffers in this first run
    one_ms, prog = [], []
    for _ in range(reps):  # alternated
        one_ms.append(oneshot())
        prog.append(progressive())
    unit = prog[-1][0]
    equal = bool(np.array_equal(lin.cpu().numpy().view(np.uint64), ref[0].view(np.uint64)) and
                 np.array_equal(rgb.cpu().numpy(), ref[1]))
    sums = [sum(p[1]) for p in prog]
    pixels = W * H
    strict = unit == 1
    general_strict = strict and not (depth == 1 or flags & 16)  # primary-ray renders: the seeded kernel, no buffer
    per = STRICT_BUF_BYTES // (pixels * 32)
    one.close(), acc.close()
    return {
        "case": label, "workload": wl["name"], "samples_per_unit": spu, "pass_unit": unit, "passes": list(passes),
        "oneshot_ms": sorted(one_ms)[len(one_ms) // 2], "oneshot_ms_all": one_ms,
        "passes_sum_ms": sorted(sums)[len(sums) // 2], "passes_sum_ms_all": sums,
        "pass_ms_median_run": prog[sorted(range(len(sums)), key=lambda i: sums[i])[len(sums) // 2]][1],
        "overhead_ms_per_pass": (sorted(sums)[len(sums) // 2] - sorted(one_ms)[len(one_ms) // 2]) / len(passes),
        "accumulator_bytes": pixels * 24,
        "sample_buf_bytes_peak": min(per, max(passes)) * pixels * 32 if general_strict else 0,
        "device_memory_growth_bytes": growth,
        "final_image_equals_oneshot": equal,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    wls = workloads()
    line = {"card": card(), "reps": args.reps, "cases": [
        run_case("c3_chunked_25x20", wls["c3"], 25, [25] * 20, args.reps),
        run_case("c3_strict_25x20", wls["c3"], 500, [25] * 20, args.reps),
        run_case("c4_strict_10x10", wls["c4"], 0, [10] * 10, args.reps),
    ]}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
