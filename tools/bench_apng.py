"""Measures the animated PNG writer (rtclj_ctx_encode_apng, DESIGN.md section 4.14) on one GPU.

  - Encode alone, on real renders of main's scene on its turntable at 400x225 x 60 frames, 1920x1080 x 16 and
    3840x2160 x 8, device-resident: one rtclj_ctx_encode_apng call against K rtclj_ctx_encode_png calls (one per
    frame).  Both synchronise (each returns a length read back from the device), so a call's wall time is all of its
    work; the two are alternated, and the medians are reported with min and max.
  - End to end, main's 60-frame turntable at the CLI's 100 spp / depth 50: rtclj_render_frames_apng against what the
    CLI's --frames --gpu-png does (rtclj_render_frames, then rtclj_encode_png_gpu per frame), alternated.
  - File sizes: the APNG against the K device PNGs and against Pillow's APNG writer (zlib level 6) of the same frames.
The card's name and power limit are read in the same run.  Prints one JSON line; --out writes it to a file.
Usage: python tools/bench_apng.py [--reps N] [--e2e-reps N] [--out PATH]"""
import argparse
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

import apng_model as A  # noqa: E402
import raytracing_clj_b200 as R  # noqa: E402
from raytracing_clj_b200 import _abi, render  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def stats(ms):
    return {"median": round(float(np.median(ms)), 4), "min": round(min(ms), 4), "max": round(max(ms), 4)}


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t0)


def pillow_apng(frames):
    ims = [Image.fromarray(f) for f in frames]
    buf = io.BytesIO()
    ims[0].save(buf, format="PNG", save_all=True, append_images=ims[1:], duration=1000 / 30, loop=0, compress_level=6)
    return buf.getvalue()


def encode_alone(width, K, spp, reps):
    cams = R.camera.turntable_cameras(K, width)
    _, rgb, _ = render.render_frames(R.scenes.main_hittables(), cams, spp, 50, seed=1, want_linear=False)
    _, H, W, _ = rgb.shape
    ctx = render.Context(0)
    stream = torch.cuda.current_stream().cuda_stream
    d_in = torch.from_numpy(rgb).cuda()
    cap = ctx.encode_apng(d_in.data_ptr(), W, H, K)
    d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda:0")
    png_cap = ctx.encode_png(d_in.data_ptr(), W, H)
    d_png = torch.zeros(png_cap, dtype=torch.uint8, device="cuda:0")
    frame = W * H * 3

    def apng():
        return ctx.encode_apng(d_in.data_ptr(), W, H, K, d_out.data_ptr(), cap, stream=stream)

    def pngs():
        return [ctx.encode_png(d_in.data_ptr() + k * frame, W, H, d_png.data_ptr(), png_cap, stream) for k in range(K)]
    for _ in range(3):
        n, lens = apng(), pngs()
    t_apng, t_pngs = [], []
    for _ in range(reps):
        torch.cuda.synchronize()
        t_apng.append(timed(apng)[1])
        torch.cuda.synchronize()
        t_pngs.append(timed(pngs)[1])
    data = bytes(d_out[:n].cpu().numpy())
    ctx.close()
    return {
        "frames": K, "width": W, "height": H, "spp": spp, "reps": reps,
        "apng_ms": stats(t_apng), "k_png_ms": stats(t_pngs),
        "speedup_median": round(float(np.median(t_pngs)) / float(np.median(t_apng)), 3),
        "apng_bytes": n, "k_png_bytes": int(sum(lens)), "pillow_apng_level6_bytes": len(pillow_apng(rgb)),
        "device_equals_model": data == A.encode(rgb) if K * W * H <= 1920 * 1080 * 16 else "not checked here",
    }


def end_to_end(reps, spp=100, depth=50, K=60):
    world, cams = R.scenes.main_hittables(), R.camera.turntable_cameras(K)

    def apng():
        return render.render_frames_apng(world, cams, spp, depth, seed=1)

    def cli_today():
        _, rgb, _ = render.render_frames(world, cams, spp, depth, seed=1, want_linear=False)
        return [render.encode_png(rgb[k], device=0) for k in range(K)]
    data, pngs = apng(), cli_today()
    t_apng, t_cli = [], []
    for _ in range(reps):
        t_apng.append(timed(apng)[1])
        t_cli.append(timed(cli_today)[1])
    frames = np.stack([np.array(Image.open(io.BytesIO(p)).convert("RGB")) for p in pngs])
    return {
        "frames": K, "width": cams[0].width, "height": cams[0].height, "spp": spp, "depth": depth, "reps": reps,
        "render_frames_apng_ms": stats(t_apng), "render_frames_plus_k_encode_png_gpu_ms": stats(t_cli),
        "speedup_median": round(float(np.median(t_cli)) / float(np.median(t_apng)), 3),
        "apng_bytes": len(data), "k_png_bytes": sum(len(p) for p in pngs),
        "pillow_apng_level6_bytes": len(pillow_apng(frames)),
        "apng_equals_encoding_the_rendered_frames": data == render.encode_apng(frames),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--e2e-reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    res = {"card": card(),
           "encode_alone": [encode_alone(w, k, spp, a.reps) for w, k, spp in ((400, 60, 100), (1920, 16, 8), (3840, 8, 4))],
           "end_to_end": end_to_end(a.e2e_reps)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
