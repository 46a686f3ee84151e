#!/usr/bin/env python
"""bench.py -- the headline measurement (BASELINE.json): rays/sec on the RTIOW cover scene.

A "ray" is one ray SEGMENT = one closest-hit search over all N spheres (SURVEY.md 8d),
counted by a device counter.  A "step" is one full render of the workload.  The headline
workload (no --workload flag, or --workload c3) is BASELINE.json config 3, the configuration the
metric is quoted on: cover scene (generator seed 7 -> 484 spheres), 1920x1080, 500 spp, depth 50,
`main` semantics (Schlick, defocus 0.6 deg), render seed 1.  --workload c1|c2|c4|c5 emit the same
JSON line for the other BASELINE.json configs (parity configurations, not the headline).
With N GPUs the image rows are interleaved over the ranks (tiles of 1 row, tile t -> rank t % N;
no collective on the data path), so the total work is fixed: strong scaling.

  value     whole-job segments/s with the scene resident on the device and the image left
            in HBM (device-resident C-ABI call on torch's current stream, CUDA events,
            per-step max over ranks)
  e2e       the same metric through the host-buffer C-ABI call rtclj_render: scene arrays
            copied H2D, image (linear f64 + rgb8) copied D2H into PINNED host memory every step
  e2e_single_process  (N > 1) the same again, but ONE process (rank 0) drives all N GPUs through
            rtclj_render_multi -- what a JVM host does (src/raytracing.clj:157-171) -- while
            the other ranks idle
  strict_order  value measured with samples_per_unit = spp: the reference's sequential sum
            per pixel (src/raytracing.clj:142-155), the mode the Clojure binding uses
  roofline  FP32 (CUDA-core) roofline of the render kernel: algorithmic flops = segments *
            (17*N + 5) (SURVEY.md 8d) / the kernel's CUDA-event time
  cpu_baseline  the CPU oracle (C restatement of the reference, NOT the JVM) timed on this
            box's host cores on a bounded row sample of the same workload

`--impl reference` times only the CPU restatement (the reference is Clojure; no JVM exists
in this image, so oracle/_ref cannot be built -- see DESIGN.md).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHARD_ROWS = 1
FLOP_PER_TEST, FLOP_PER_SEGMENT = 17, 5  # SURVEY.md 8d
DUMP_BYTES = 64 * 10 ** 6        # --dump-outputs writes at most this much
DUMP_SAMPLE_PIXELS = 1 << 20     # pixels kept when the whole image does not fit in DUMP_BYTES


def workloads():
    import raytracing_clj_b200 as R
    from raytracing_clj_b200 import _abi
    S, CAM = R.scenes, R.camera
    return {
        "c3": dict(name="rtiow_cover_seed7_1920x1080_500spp_depth50", world=lambda: S.cover_hittables(7),
                   cam=lambda: CAM.main_camera(1920, 1080, **S.COVER_CAMERA), spp=500, depth=50, flags=_abi.FLAGS_MAIN),
        "c1": dict(name="default_scene_main_400x225_100spp_depth50", world=S.main_hittables,
                   cam=lambda: CAM.main_camera(), spp=100, depth=50, flags=_abi.FLAGS_MAIN),
        "c2": dict(name="material_scene_1920x1080_100spp_depth50", world=S.main_hittables,
                   cam=lambda: CAM.main_camera(1920), spp=100, depth=50, flags=_abi.FLAGS_MAIN),
        "c4": dict(name="primary_ray_raytracing_i_3840x2160_100spp", world=S.i_hittables,
                   cam=lambda: CAM.i_camera(3840), spp=100, depth=50, flags=_abi.FLAGS_I),
        "c5": dict(name="field_10k_spheres_3840x2160_256spp_depth50", world=lambda: S.field_hittables(7),
                   cam=lambda: CAM.main_camera(3840, 2160, **S.FIELD_CAMERA), spp=256, depth=50, flags=_abi.FLAGS_MAIN),
    }


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        # median over the busiest half of the samples (the sampler also sees the idle gaps)
        busy = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_rate(wl, world, cam, threads=None, seconds_hint=8.0):
    """rays/s of the CPU oracle on a bounded sample: `threads` evenly spaced rows of the
    workload at a reduced spp (the rate does not depend on spp)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    import raytracing_clj_b200 as R
    threads = threads or min(os.cpu_count() or 1, 64)
    H = cam.height
    step = max(1, H // threads)
    begin = step // 2
    nrows = len(range(begin, H, step))
    soa = R.scenes.to_soa(world)
    oflags = wl["flags"] & 0xffff
    # calibrate spp for ~seconds_hint of work per thread
    t0 = time.perf_counter()
    _, _, st = O.render(soa, cam, 4, wl["depth"], seed=1, flags=oflags,
                        threads=threads, rows=(begin, H), row_step=step, want_rgb8=False)
    dt = time.perf_counter() - t0
    spp = int(max(8, min(wl["spp"], 4 * seconds_hint / max(dt, 1e-3))))
    t0 = time.perf_counter()
    _, _, st = O.render(soa, cam, spp, wl["depth"], seed=1, flags=oflags,
                        threads=threads, rows=(begin, H), row_step=step, want_rgb8=False)
    dt = time.perf_counter() - t0
    sample = f"{nrows} evenly spaced rows x {cam.width} px x {spp} spp of the workload ({st.segments} segments)"
    return st.segments / dt, min(threads, nrows), sample, dt


def config_of(wl, world, cam, world_size):
    """The SAME keys in both arms (the driver compares them)."""
    return {"workload": wl["name"], "n_spheres": len(world), "image": f"{cam.width}x{cam.height}", "spp": wl["spp"],
            "max_depth": wl["depth"], "scene_seed": 7, "render_seed": 1,
            "parallelism": f"rows interleaved over {world_size} GPU(s), tiles of {SHARD_ROWS} rows"}


def dump_outputs(dirname, lin, rgb8, world_size, rank):
    """Writes what the timed call left in its device buffers, so that two builds can be compared output for
    output: linear.npy (float64 radiance) and rgb8.npy (the 8-bit image as float32), both [H, W, 3].  An image
    larger than DUMP_BYTES is cut to a fixed, seeded sample of DUMP_SAMPLE_PIXELS pixels: then both are
    [pixels, 3] and pixel_index.npy holds the row-major index (y * W + x) of each pixel."""
    import numpy as np
    import torch.distributed as dist
    if world_size > 1:  # each rank wrote only its own rows of zero-initialised full-size buffers
        lin, rgb8 = lin.clone(), rgb8.clone()
        dist.all_reduce(lin)
        dist.all_reduce(rgb8)
    if rank != 0:
        return
    lin = lin.cpu().numpy()
    rgb8 = rgb8.cpu().numpy().astype(np.float32)
    out = {"linear": lin, "rgb8": rgb8}
    if lin.nbytes + rgb8.nbytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(lin.shape[0] * lin.shape[1], DUMP_SAMPLE_PIXELS, replace=False))
        out = {"linear": lin.reshape(-1, 3)[idx], "rgb8": rgb8.reshape(-1, 3)[idx], "pixel_index": idx.astype(np.float64)}
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    world, cam = wl["world"](), wl["cam"]()
    rates, sample, cores = [], "", 0
    for i in range(args.warmup + args.steps):
        rate, cores, sample, dt = cpu_oracle_rate(wl, world, cam, seconds_hint=6.0)
        if i >= args.warmup:
            rates.append((rate, dt))
    value = sum(r for r, _ in rates) / len(rates)
    line = {
        "impl": "reference", "metric": "rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(d for _, d in rates) / len(rates),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(wl, world, cam, world_size),
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "CPU restatement of the reference (oracle/rt_oracle.c); the JVM reference is not runnable here"},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="BASELINE.json config; c3 is the headline, the others are reported the same way")
    ap.add_argument("--kernel", default=None, choices=["lane", "lane2", "wave", "split"],
                    help="small-scene kernel to time (A/B); default: the library's choice")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip strict_order / e2e_single_process")
    ap.add_argument("--spp", type=int, default=None, help="override the workload's spp (invalid as a bench value)")
    ap.add_argument("--spu", type=int, default=0, help="samples per work unit for the timed steps (tuning; 0 = the library's choice)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the images the last timed step computed to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    wl = workloads()[args.workload]
    if args.spp:
        wl["spp"] = args.spp
        wl["name"] += f"_OVERRIDE_spp{args.spp}"
    if args.impl == "reference":
        return run_reference(args, wl)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpu_group = None
    if world_size > 1:
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")  # host-side barriers: an NCCL barrier parks a spinning kernel on the GPU

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    import raytracing_clj_b200 as R
    from raytracing_clj_b200 import _abi, render
    world, cam = wl["world"](), wl["cam"]()
    n = len(world)
    W, H, spp, depth = cam.width, cam.height, wl["spp"], wl["depth"]
    shard = (rank, world_size, SHARD_ROWS) if world_size > 1 else None
    flags = wl["flags"]
    if args.kernel:
        flags |= {"lane": _abi.F_LANE_KERNEL, "lane2": _abi.F_LANE2_KERNEL, "wave": _abi.F_WAVE_KERNEL, "split": _abi.F_SPLIT_KERNEL}[args.kernel]
    lib = _abi.lib()

    # arithmetic peaks of this GPU (pure-FMA kernels), before the timed region
    pk = [C.c_double(), C.c_double(), C.c_double()]
    sms = C.c_int32()
    _abi.check(lib.rtclj_calibrate_peaks(local_rank, C.byref(pk[0]), C.byref(pk[1]), C.byref(pk[2]), C.byref(sms)))

    ctx = render.Context(local_rank)
    ctx.set_scene(world)
    out_lin = torch.zeros((H, W, 3), dtype=torch.float64, device=dev)
    out_rgb = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def timed_device_steps(nsteps, samples_per_unit=0):
        def step():
            ctx.render(cam, spp, depth, seed=1, flags=flags, shard=shard, samples_per_unit=samples_per_unit,
                       d_out_linear=out_lin.data_ptr(), d_out_rgb8=out_rgb.data_ptr(), stream=stream)
        for _ in range(max(3, args.warmup) if samples_per_unit == args.spu else 1):
            step()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsteps)]
        k_ms, seg, spu = [], 0, 0
        for s0, s1 in evs:
            flush.zero_()  # L2 flush between timed iterations (not timed)
            s0.record()
            step()
            s1.record()
            st = ctx.stats(stream)  # synchronises the stream; reads the device counters
            k_ms.append(st["kernel_ms"])
            seg, spu = st["segments"], st["samples_per_unit"]
        barrier()
        step_ms = torch.tensor([a.elapsed_time(b) for a, b in evs], dtype=torch.float64, device=dev)
        segs = torch.tensor([float(seg)], dtype=torch.float64, device=dev)
        if world_size > 1:
            dist.all_reduce(step_ms, op=dist.ReduceOp.MAX)  # per step, the slowest rank
            dist.all_reduce(segs, op=dist.ReduceOp.SUM)
        return float(step_ms.sum().item()), float(segs.item()), k_ms, seg, spu

    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    total_ms, segs_per_step, kernel_ms, seg_local, spu_used = timed_device_steps(args.steps, samples_per_unit=args.spu)
    clocks = sampler.stop() if rank == 0 else None
    value = segs_per_step * args.steps / (total_ms * 1e-3)
    if args.dump_outputs:  # now: the strict-order and e2e legs below render into the same buffers
        dump_outputs(args.dump_outputs, out_lin, out_rgb, world_size, rank)

    # ---- the reference's strict summation order (one sequential sum per pixel), same timing rules
    strict = None
    if not args.no_extras:
        s_ms, s_segs, s_k, _, s_spu = timed_device_steps(max(1, min(args.steps, 2)), samples_per_unit=spp)
        strict = {"value": s_segs * max(1, min(args.steps, 2)) / (s_ms * 1e-3), "unit": "rays/s",
                  "samples_per_unit": s_spu, "ms_per_step": s_ms / max(1, min(args.steps, 2)),
                  "note": "samples_per_unit = spp: the reference's sequential sum per pixel (raytracing.clj:142-155); per-sample colours are buffered in HBM (32 B each) and added in sample order by finalize_kernel"}

    # ---- e2e: host buffers through rtclj_render, H2D + D2H (into pinned host memory) inside the timed region
    soa = R.scenes.to_soa(world)
    # one name per user and job: the ranks of a job share MASTER_PORT, other jobs (and users) on the host do not
    shm_path = f"/dev/shm/rtclj_bench_{os.getuid()}_{os.environ.get('MASTER_PORT') or os.getpid()}"
    lin_bytes, rgb_bytes = H * W * 3 * 8, H * W * 3
    if rank == 0:
        with open(shm_path, "wb") as f:
            f.truncate(lin_bytes + rgb_bytes)
    barrier()
    whole = np.memmap(shm_path, dtype=np.uint8, mode="r+", shape=(lin_bytes + rgb_bytes,))  # ONE mapping, shared by the ranks
    host_lin = whole[:lin_bytes].view(np.float64).reshape(H, W, 3)
    host_rgb = whole[lin_bytes:].reshape(H, W, 3)
    whole[:] = 0  # touch the pages, then pin the mapping once (outside the timed region)
    pinned = lib.rtclj_host_register(C.c_void_p(whole.ctypes.data), lin_bytes + rgb_bytes) == 0
    if not pinned:
        print("bench: rtclj_host_register failed (%s): e2e goes through the library's staging copy"
              % lib.rtclj_last_error().decode(), file=sys.stderr)

    def e2e_step():
        return render.render(soa, cam, spp, depth, seed=1, flags=flags, shard=shard,
                             devices=[local_rank], out_linear=host_lin, out_rgb8=host_rgb)[2]

    def time_wall(fn, steps, only_rank0=False):
        times = []
        for _ in range(steps):
            barrier()
            t0 = time.perf_counter()
            if not only_rank0 or rank == 0:
                fn()
            if only_rank0:
                # the idle ranks must leave their GPUs FREE while rank 0 drives them: wait on the host (gloo);
                # an NCCL barrier would keep a spinning kernel resident on every idle rank's device
                torch.cuda.synchronize()
                dist.barrier(group=cpu_group)
            else:
                barrier()
            times.append(time.perf_counter() - t0)
        t = torch.tensor(times, dtype=torch.float64, device=dev)
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.sum().item())

    e2e_step()
    e2e_steps = max(1, min(args.steps, 3))
    e2e_s = time_wall(e2e_step, e2e_steps)
    e2e_value = segs_per_step * e2e_steps / e2e_s
    checksum = int(np.asarray(host_rgb[::97, ::89]).sum()) if rank == 0 else 0
    h2d = sum(a.nbytes for a in soa) * world_size

    # ---- one process drives all N GPUs (rtclj_render_multi); the other ranks only take part in the barriers
    single = None
    if world_size > 1 and not args.no_extras:
        def multi_step():
            return render.render(soa, cam, spp, depth, seed=1, flags=flags, devices=list(range(world_size)),
                                 out_linear=host_lin, out_rgb8=host_rgb)[2]
        if rank == 0:
            multi_step()
        m_s = time_wall(multi_step, e2e_steps, only_rank0=True)
        single = {"value": segs_per_step * e2e_steps / m_s, "unit": "rays/s", "ms_per_step": 1e3 * m_s / e2e_steps,
                  "rgb8_checksum": int(np.asarray(host_rgb[::97, ::89]).sum()) if rank == 0 else 0,
                  "note": "rank 0 alone calls rtclj_render_multi over all GPUs (one worker thread per device)"}
    barrier()
    if pinned:
        lib.rtclj_host_unregister(C.c_void_p(whole.ctypes.data))
    if rank == 0:
        try:
            os.unlink(shm_path)
        except OSError:
            pass

    if rank != 0:
        if world_size > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    sm_max = float(peaks.get("sm_max_mhz") or 1965.0)
    peak_nominal = sms.value * 128 * 2 * sm_max * 1e6 / 1e12
    k_ms = sum(kernel_ms) / len(kernel_ms)
    achieved = seg_local * (FLOP_PER_TEST * n + FLOP_PER_SEGMENT) / (k_ms * 1e-3) / 1e12
    # DRAM bytes per launch: ncu cannot run inside a timed bench, so this figure is STATIC -- read from the
    # committed ncu --set full capture of this same workload (tools/ncu_traffic.py wrote it)
    traffic, traffic_source = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("workload") == wl["name"] and world_size == 1 and not args.kernel:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            traffic_source = "static: profiles/r2_traffic.json (ncu --set full of this workload and build)"
    except Exception:
        pass
    small_kernel = "render_kernel<false> (shared-memory table, TMA)" if n > 512 else (args.kernel or "library default")
    roofline = {
        "bound": "fp32", "achieved": achieved, "peak": peak_nominal, "unit": "TFLOP/s", "frac": achieved / peak_nominal,
        "traffic": traffic, "traffic_source": traffic_source, "kernel": small_kernel, "kernel_ms": k_ms,
        "peak_source": f"{sms.value} SMs x 128 lanes x 2 flop x {sm_max:.0f} MHz (sm_max_mhz of MEASURED_PEAKS.json"
                       f"{'' if peaks else ' MISSING: fallback 1965'}); the path is CUDA-core fp32, not HBM or tensor",
        "peak_calibrated": {"ffma": pk[0].value, "ffma2": pk[1].value, "dfma_fp64": pk[2].value, "unit": "TFLOP/s"},
        "frac_of_calibrated_ffma2": achieved / pk[1].value if pk[1].value else None,
        "algorithmic_flops": f"segments x ({FLOP_PER_TEST}*N + {FLOP_PER_SEGMENT}), N={n}",
    }
    cpu = None
    if world_size == 1 and not args.no_cpu_baseline:
        rate, cores, sample, _ = cpu_oracle_rate(wl, world, cam)
        # the reference itself renders on a pool of TWO threads (raytracing.clj:157): report that too
        rate2, cores2, sample2, _ = cpu_oracle_rate(wl, world, cam, threads=2, seconds_hint=4.0)
        cpu = {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample,
               "reference_pool_size_2": {"value": rate2, "unit": "rays/s", "cores": cores2, "sample": sample2}}
    config = config_of(wl, world, cam, world_size)
    line = {
        "metric": "rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world_size, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32 cull + f64 exact hit/shade", "data": "synthetic",
        "config": config,
        "workload_stats": {"samples_per_step": W * H * spp, "segments_per_step": segs_per_step,
                           "samples_per_sec": W * H * spp * args.steps / (total_ms * 1e-3),
                           "samples_per_unit": spu_used, "rgb8_checksum": checksum,
                           "l2": "flushed between timed steps (256 MiB write); the sphere table lives on chip"},
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": lin_bytes + rgb_bytes, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                "host_buffers": "pinned (rtclj_host_register)" if pinned else "pageable (staged inside the library)"},
        "e2e_single_process": single, "strict_order": strict,
        "gpu_launches": 2 * args.steps * world_size,  # render kernel + finalize_kernel per step per rank
        "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if world_size > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
