"""Measures the denoiser (rtclj_ctx_denoise, DESIGN.md section 4.13) on one GPU.
  filter:   CUDA events around 20 warm calls (median) of the default filter, device-resident, at 1920x1080, 3840x2160 and
            7680x4320; the inputs are a 16-spp cover render and its guide, tiled to the size.  Achieved bytes/s against
            the data-sheet HBM bandwidth, from the bytes each level must move (its float32 or f64 inputs once, its output
            once).  A separate torch.profiler pass splits the time per level.
  quality:  the cover scene and config 2 at 1920x1080, 4, 16 and 64 spp: render, guide and filter ms; RMSE and p99
            absolute error of the raw and denoised linear images against a 4000-spp render with ANOTHER seed, over the
            whole image, at guide edges and on the glass spheres (pixels whose first hit is a dielectric); the raw spp
            that reaches the denoised RMSE and its time.
  sweep:    levels x sigma_color x sigma_guide (and guide samples) on both scenes at 16 spp; the defaults are checked on
            main's default scene (400x225, 8 spp against 1024 spp with another seed) as a held-out case.
Times of renders are host wall clock around the call and a device synchronise.  The card's name and power limit are read
in the same run.  Prints one JSON line and writes it to --out.
Usage: python tools/bench_denoise.py [--out profiles/r3_bench_denoise.json] [--quick]"""
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

import raytracing_clj_b200 as R  # noqa: E402
from raytracing_clj_b200 import _abi, render  # noqa: E402

HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU
REF_SPP, REF_SEED, SEED = 4000, 977, 1
LEVELS, SC, SG, GS = render.DENOISE_LEVELS, render.DENOISE_SIGMA_COLOR, render.DENOISE_SIGMA_GUIDE, render.DENOISE_GUIDE_SAMPLES


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def scenes():
    S, CAM = R.scenes, R.camera
    return {"cover": (S.cover_hittables(7), lambda w, h: CAM.main_camera(w, h, **S.COVER_CAMERA)),
            "config2_5_spheres": (S.main_hittables(), lambda w, h: CAM.main_camera(w, h))}


def level_bytes(levels, npix):
    """Bytes each level must move: level 0 reads the f64 colour and guide and writes float4 colour and guide; a middle
    level reads float4 colour and guide and writes float4 colour; the last writes the f64 and 8-bit images instead."""
    out = []
    for i in range(levels):
        rd = 48 if i == 0 else 32
        wr = (27 if i == levels - 1 else 16) + (16 if i == 0 and levels > 1 else 0)
        out.append((rd + wr) * npix)
    return out


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def filter_time(ctx, reps=20):
    world, camf = scenes()["cover"]
    cam = camf(1920, 1080)
    lin0, _, _ = render.render(world, cam, 16, 50, seed=SEED, want_rgb8=False)
    gd0, _, _ = render.render(world, cam, GS, 1, seed=SEED, flags=_abi.FLAGS_I, want_rgb8=False)
    rows = []
    for W, H in ((1920, 1080), (3840, 2160), (7680, 4320)):
        ty, tx = H // 1080, W // 1920
        lin = torch.from_numpy(np.tile(lin0, (ty, tx, 1))).cuda()
        gd = torch.from_numpy(np.tile(gd0, (ty, tx, 1))).cuda()
        out = torch.empty_like(lin)
        rgb = torch.empty(lin.shape, dtype=torch.uint8, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        call = lambda: ctx.denoise(lin.data_ptr(), gd.data_ptr(), W, H, d_out_linear=out.data_ptr(),  # noqa: E731
                                   d_out_rgb8=rgb.data_ptr(), stream=s)
        for _ in range(3):
            call()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            call()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        med = sorted(ms)[len(ms) // 2]
        nb = sum(level_bytes(LEVELS, W * H))
        # per level, in a separate profiled pass
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                call()
            torch.cuda.synchronize()
        evs = sorted([e for e in prof.events() if "denoise_level_kernel" in e.name and e.device_type.name == "CUDA"],
                     key=lambda e: e.time_range.start)
        per = [[] for _ in range(LEVELS)]
        for k, e in enumerate(evs):
            per[k % LEVELS].append(e.time_range.elapsed_us() / 1e3)
        per_ms = [sorted(p)[len(p) // 2] if p else None for p in per]
        lb = level_bytes(LEVELS, W * H)
        rows.append({"size": [W, H], "levels": LEVELS, "ms": ms, "median_ms": med, "bytes": nb,
                     "achieved_TBps": nb / (med * 1e-3) / 1e12, "hbm_bound_ms": nb / (HBM_TBPS * 1e12) * 1e3,
                     "share_of_hbm_bound": (nb / (HBM_TBPS * 1e12) * 1e3) / med,
                     "per_level_ms": per_ms,
                     "per_level_TBps": [b / (m * 1e-3) / 1e12 if m else None for b, m in zip(lb, per_ms)]})
        del lin, gd, out, rgb
        torch.cuda.empty_cache()
    return rows


def errors(lin, ref, mask=None):
    e = np.abs(lin - ref)
    if mask is not None:
        e = e[mask]
    return {"rmse": float(np.sqrt(np.mean(e * e))), "p99_abs": float(np.percentile(e, 99))}


def edge_mask(guide, thr=0.05):
    d = np.zeros(guide.shape[:2], bool)
    dx = np.abs(np.diff(guide, axis=1)).max(axis=2) > thr
    dy = np.abs(np.diff(guide, axis=0)).max(axis=2) > thr
    d[:, 1:] |= dx
    d[:, :-1] |= dx
    d[1:] |= dy
    d[:-1] |= dy
    return d


def glass_mask(world, cam):
    """Pixels whose first hit is a dielectric: the guide changes when the dielectrics are removed."""
    soa = R.scenes.to_soa(world)
    keep = soa[2] != _abi.DIELECTRIC
    without = tuple(np.ascontiguousarray(a[keep]) for a in soa)
    a, _, _ = render.render(world, cam, 1, 1, seed=SEED, flags=_abi.FLAGS_I, want_rgb8=False)
    b, _, _ = render.render(without, cam, 1, 1, seed=SEED, flags=_abi.FLAGS_I, want_rgb8=False)
    return np.any(a != b, axis=2)


def render_ms(world, cam, spp, depth, seed, flags):
    out = {}

    def go():
        out["lin"] = render.render(world, cam, spp, depth, seed=seed, flags=flags, want_rgb8=False)[0]
    render.render(world, cam, min(spp, 4), depth, seed=seed, flags=flags, want_rgb8=False)  # warm this shape
    ms = timed(go)
    return out["lin"], ms


def quality(name, world, camf, ladder, spps):
    cam = camf(1920, 1080)
    ref, ref_ms = render_ms(world, cam, REF_SPP, 50, REF_SEED, _abi.FLAGS_MAIN)
    guide, guide_ms = render_ms(world, cam, GS, 1, SEED, _abi.FLAGS_I)
    edges, glass = edge_mask(guide), glass_mask(world, cam)
    raw = {}
    for s in ladder:
        lin, ms = render_ms(world, cam, s, 50, SEED, _abi.FLAGS_MAIN)
        raw[s] = (ms, errors(lin, ref)["rmse"])
    rows = []
    for spp in spps:
        lin, ms = render_ms(world, cam, spp, 50, SEED, _abi.FLAGS_MAIN)
        render.denoise(lin, guide)
        dn = {}
        f_ms = timed(lambda: dn.setdefault("lin", render.denoise(lin, guide)[0]))
        d_err = errors(dn["lin"], ref)
        match = next((s for s in ladder if raw[s][1] <= d_err["rmse"]), None)
        rows.append({"spp": spp, "render_ms": ms, "guide_ms": guide_ms, "filter_host_call_ms": f_ms,
                     "raw": {**errors(lin, ref), "edges": errors(lin, ref, edges), "glass": errors(lin, ref, glass)},
                     "denoised": {**d_err, "edges": errors(dn["lin"], ref, edges), "glass": errors(dn["lin"], ref, glass)},
                     "raw_spp_matching_denoised_rmse": match, "its_render_ms": raw[match][0] if match else None})
    return {"case": name, "size": [1920, 1080], "reference": {"spp": REF_SPP, "seed": REF_SEED, "ms": ref_ms},
            "guide_samples": GS, "edge_pixels": int(edges.sum()), "glass_pixels": int(glass.sum()),
            "raw_ladder": {str(s): {"ms": raw[s][0], "rmse": raw[s][1]} for s in ladder}, "rows": rows}


def sweep(name, world, camf, spp=16):
    cam = camf(1920, 1080)
    ref, _ = render_ms(world, cam, REF_SPP, 50, REF_SEED, _abi.FLAGS_MAIN)
    lin, _ = render_ms(world, cam, spp, 50, SEED, _abi.FLAGS_MAIN)
    guides = {g: render_ms(world, cam, g, 1, SEED, _abi.FLAGS_I)[0] for g in (1, 4, 16)}
    rows = []
    for L in (3, 4, 5, 6):
        for sc in (0.25, 0.5, 1.0, 2.0, 4.0):
            for sg in (0.05, 0.1, 0.2, 0.4):
                out, _ = render.denoise(lin, guides[GS], levels=L, sigma_color=sc, sigma_guide=sg)
                rows.append({"levels": L, "sigma_color": sc, "sigma_guide": sg, "guide_samples": GS, **errors(out, ref)})
    for g, gd in guides.items():
        out, _ = render.denoise(lin, gd)
        rows.append({"levels": LEVELS, "sigma_color": SC, "sigma_guide": SG, "guide_samples": g, **errors(out, ref)})
    best = min(rows, key=lambda r: r["rmse"])
    return {"case": name, "spp": spp, "raw": errors(lin, ref), "best": best, "rows": rows}


def held_out():
    S, CAM = R.scenes, R.camera
    world, cam = S.main_hittables(), CAM.main_camera()
    ref, _ = render_ms(world, cam, 1024, 50, 2, _abi.FLAGS_MAIN)
    out = {}
    for spp in (8, 32):
        lin, _ = render_ms(world, cam, spp, 50, SEED, _abi.FLAGS_MAIN)
        out[f"raw_{spp}"] = errors(lin, ref)
    dn, _, _ = render.render_denoised(world, cam, 8, 50, seed=SEED)
    out["denoised_8"] = errors(dn, ref)
    out["ratio_denoised8_over_raw32"] = out["denoised_8"]["rmse"] / out["raw_32"]["rmse"]
    return {"case": "main default scene 400x225, reference 1024 spp seed 2", **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_denoise.json"))
    ap.add_argument("--quick", action="store_true", help="skip the sweep")
    args = ap.parse_args()
    ctx = render.Context(0)
    line = {"card": card(), "defaults": {"levels": LEVELS, "sigma_color": SC, "sigma_guide": SG, "guide_samples": GS},
            "hbm_datasheet_TBps": HBM_TBPS, "filter": filter_time(ctx)}
    ctx.close()
    sc = scenes()
    ladder = [4, 8, 16, 32, 64, 128, 256, 512, 1024]
    line["quality"] = [quality(n, w, c, ladder, (4, 16, 64)) for n, (w, c) in sc.items()]
    line["held_out"] = held_out()
    if not args.quick:
        line["sweep"] = [sweep(n, w, c) for n, (w, c) in sc.items()]
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
