#!/usr/bin/env python3
"""bench.py -- Msamples/s of the per-sample render loop (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C2] [--dump-outputs DIR]

A "step" is one Tracer::render call over one frame of the workload.  The metric is Msamples/s
(GEODESIC): the default workload is the lensed one -- at N = 1 BASELINE configs[2] (C3: scene.json.gz +
the strong-lens mass, 3840x2160 at 64 spp, 530.8 Msamples); at N > 1 (torchrun, one rank per GPU)
BASELINE configs[4]'s frame (C5: the same scene at 7680x4320) STRONG-scaled at 64 spp: the frame's 16
passes are split across the ranks and the slices are summed with ONE NCCL reduce inside the step (the
full 1024-spp C5 frame is 33 974 Msamples -- over a minute per step on one GPU -- so the sweep renders
the frame at C3's spp; `--workload C5` runs the full thing).  `--workload` picks any other config;
C1-C4 are weak-scaled at N > 1 (every rank renders its own pass slice of the same frame size).
Rank 0 prints ONE JSON line.  `--impl reference` times the reference algorithm's CPU restatement
(oracle/, kind "port": the Rust crate cannot be built here) on a bounded sample of the same frame.
`--dump-outputs DIR` writes the frame of the last timed step (see dump_outputs) so that two builds can be
compared output for output: with the same arguments every run renders the same sample sets of the same scene.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (scene, width, height, passes, subsample, lens (x, y, z, r_s) or None)
    "C1": ("cornell", 512, 512, 4, 2, None),
    "C2": ("cornell2", 1920, 1080, 64, 2, None),
    "C3": ("scene", 3840, 2160, 16, 2, (1.362, 1.577, 6.114, 0.2)),
    "C4-cloud": ("cloud", 1920, 1080, 64, 2, None),
    "C4-volume": ("volume", 1920, 1080, 64, 2, None),
    # strong scaling: the 1024 spp of ONE frame are split across the ranks (BASELINE configs[4])
    "C5": ("scene", 7680, 4320, 256, 2, (1.362, 1.577, 6.114, 0.2)),
}
WORKLOADS["C5-128"] = ("scene", 7680, 4320, 32, 2, (1.362, 1.577, 6.114, 0.2))   # the C5 frame at 128 spp
WORKLOADS["C5-64"] = ("scene", 7680, 4320, 16, 2, (1.362, 1.577, 6.114, 0.2))    # ... at C3's 64 spp: the default at N > 1
WORKLOADS["C4-cloud-lens"] = ("cloud", 1920, 1080, 64, 2, (2.4 - 6 * 0.1705, 2.7 - 6 * 0.1908, 12.0 - 6 * 0.9667, 0.2))  # SURVEY 8d: C4 with the L1 mass
STRONG = {"C5", "C5-128", "C5-64"}
METRIC = "Msamples/s"
SCENE_DIR = os.path.join(ROOT, "tests", "golden", "scenes")
FLOPS_RECT, FLOPS_SPHERE = 35, 25      # SURVEY 8d per-test algorithmic flops
PRIMS = {"cornell": (18, 0), "cornell2": (18, 0), "scene": (0, 5), "volume": (0, 4), "cloud": (0, 4)}


def describe(name, world=1):
    scene, w, h, passes, sub, lens = WORKLOADS[name]
    spp = passes * max(sub, 1) ** 2
    text = f"{name}: {scene}.json.gz {w}x{h} at {spp} spp ({passes} passes x Subpixel({sub}))" + (f" + lens r_s={lens[3]}" if lens else "")
    if world > 1 and name in STRONG:
        text += f"; the {spp} spp are split across {world} ranks ({spp // world} spp each), one NCCL reduce per step"
    elif world > 1:
        text += f"; each of {world} ranks renders its own {spp}-spp pass slice, one NCCL reduce per step"
    return {"workload": text, "scene": scene, "width": w, "height": h, "spp": spp}


def make_config(name, world):
    """the `config` object of the JSON line: identical in both arms (the driver compares them)"""
    return {"workload": describe(name, world)["workload"], "seed": 0,
            "l2": "GPU arm: 256 MiB device memset between timed steps (L2 flush)"}


def default_workload(world):
    return "C3" if world == 1 else "C5-64"


DUMP_BYTES = 60_000_000      # the .npy headers stay within 64 MB as well


def dump_outputs(out_dir, frame):
    """Writes the RGBA32F frame a caller of the timed path receives (running sums, (h, w, 4)) as out_dir/frame.npy.
    A frame above DUMP_BYTES is written as a fixed sample of its pixels instead: frame.npy (k, 4) holds the pixels
    whose flat indices (y * w + x, ascending, float64) are in frame_pixels.npy; the sample depends only on the frame
    size (seed 0), so runs with the same arguments write the same pixels."""
    os.makedirs(out_dir, exist_ok=True)
    frame = np.ascontiguousarray(frame, np.float32)
    h, w, c = frame.shape
    if frame.nbytes <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "frame.npy"), frame)
        return
    k = DUMP_BYTES // (c * 4 + 8)                   # values + a float64 index per sampled pixel
    pixels = np.sort(np.random.default_rng(0).choice(h * w, k, replace=False))
    np.save(os.path.join(out_dir, "frame.npy"), frame.reshape(h * w, c)[pixels])
    np.save(os.path.join(out_dir, "frame_pixels.npy"), pixels.astype(np.float64))


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons with NVML during the timed region"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.mhz, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.mhz.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report it instead of inventing clocks
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        self.stop_flag = True
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.mhz)) if self.mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def load_oracle_scene(name):
    import oracle_ffi as O
    scene, w, h, passes, sub, lens = WORKLOADS[name]
    osc = O.OracleScene.load(os.path.join(SCENE_DIR, scene + ".json.gz"))
    cam = osc.find_by_tag("camera")
    osc.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    if lens:
        osc.set_lenses(np.array([lens], np.float32))
    return O, osc, cam


def cpu_sample(name, passes):
    """the reference algorithm (CPU restatement, all host threads) on `passes` passes of the frame.  Frames above
    1080p are sampled at 1920x1080 with the same camera, lensed ones (~1 Msample/s on 16 threads) at 960x540:
    throughput per sample does not depend on the resolution, and the CPU leg has to stay within seconds per step"""
    O, osc, cam = load_oracle_scene(name)
    scene, w, h, _, sub, lens = WORKLOADS[name]
    if lens:
        w, h = 960, 540
    elif w * h > 1920 * 1080:
        w, h = 1920, 1080
    cores = os.cpu_count() or 1
    cfg = O.make_config(samples=passes, subsample=sub)
    t0 = time.perf_counter()
    img, n, _ = osc.render(cam, cfg, w, h, seed=0, n_threads=cores)
    dt = time.perf_counter() - t0
    return w * h * n / dt / 1e6, cores, n, dt, (w, h), img


def run_reference(args, json_out):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores"""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    name = args.workload or default_workload(world)
    d = describe(name, world)
    passes = 1  # bounded sample: 1 pass x Subpixel(2) = 4 spp of the (sub-sampled) frame per step
    for _ in range(args.warmup):
        cpu_sample(name, passes)
    t = 0.0
    for _ in range(args.steps):
        v, cores, n, dt, (sw, sh), img = cpu_sample(name, passes)
        t += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, img)
    value = sw * sh * n * args.steps / t / 1e6
    sample = f"{n} spp of the frame at {sw}x{sh} per step (the full step is {d['spp']} spp at {d['width']}x{d['height']})"
    json_out.write(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
        "scaling": "strong" if name in STRONG else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(name, world),
        "cpu_baseline": {"value": value, "unit": METRIC, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference algorithm restated in C++ (oracle/, g++ -O3 -march=x86-64-v3), all host threads, rank 0 only; "
                "the Rust crate cannot be built here",
    }) + "\n")
    json_out.flush()


def algorithmic_flops(st, scene_name, n_lens):
    """SURVEY 8d accounting of the work counters of one render call"""
    n_rect, n_sph = PRIMS[scene_name]
    fl_scan = n_rect * FLOPS_RECT + n_sph * FLOPS_SPHERE
    fl_step = 136 * n_lens + 78 if n_lens else 0
    return st["scans"] * fl_scan + st["rk4_steps"] * fl_step, fl_scan, fl_step


def stepper_roofline(engine, torch, peak_tflops, n_rays=1 << 24, n_steps=256):
    """SURVEY 8d stepper micro-benchmark: rays past M point masses, fixed RK4 step count"""
    out = {}
    rng = np.random.default_rng(1234)
    b = rng.uniform(2.6, 40.0, n_rays)
    phi = rng.uniform(0, 2 * np.pi, n_rays)
    xv = np.zeros((n_rays, 6), np.float32)
    xv[:, 0], xv[:, 1], xv[:, 2], xv[:, 5] = b * np.cos(phi), b * np.sin(phi), 20.0, -1.0
    for m in (1, 4, 16):
        lenses = np.zeros((m, 4), np.float32)
        lenses[:, :3] = rng.uniform(-3, 3, (m, 3))
        lenses[0, :3] = 0
        lenses[:, 3] = 1.0 / m
        d_xv = torch.from_numpy(xv).cuda()
        engine.geodesic_integrate(lenses, d_xv, 16)  # warm-up
        torch.cuda.synchronize()
        best = None
        for _ in range(3):
            d_xv.copy_(torch.from_numpy(xv))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            engine.geodesic_integrate(lenses, d_xv, n_steps)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        flops = float(n_rays) * n_steps * (136 * m + 78)   # F_step(M), SURVEY 8d
        tf = flops / (best * 1e-3) / 1e12
        out[f"M{m}"] = {"tflops": tf, "frac": tf / peak_tflops, "ms": best, "steps_per_s": n_rays * n_steps / (best * 1e-3)}
    return out


def main():
    # stdout carries exactly ONE JSON line: anything a library prints on fd 1 meanwhile (NCCL's version
    # banner under NCCL_DEBUG=VERSION, ...) is sent to stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: C3 on one GPU, C5-64 (the C5 frame at 64 spp, strong-scaled) on several")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / stepper roofline / other scenes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step to DIR/frame.npy (a fixed pixel sample above 60 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args, json_out)

    import torch
    import torch.distributed as dist

    import bendy_tracer_b200 as bt

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))

    # `--gpus N` without torchrun: ONE process drives N GPUs through the multi-device engine of the C ABI
    # (bt_engine_create_multi: the pass split and the peer-memory reduce happen inside bt_render)
    in_process = world == 1 and args.gpus > 1
    n_gpus = args.gpus if in_process else world
    name = args.workload or default_workload(n_gpus)
    scene_name, w, h, passes, sub, lens = WORKLOADS[name]
    d = describe(name, n_gpus)
    scene = bt.Scene.load(os.path.join(SCENE_DIR, scene_name + ".json.gz"))
    cam = scene.find_by_tag("camera")
    scene.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
    if lens:
        scene.set_lenses(np.array([lens], np.float32))
    engine = bt.Engine(devices=list(range(args.gpus))) if in_process else bt.Engine.default(local)
    tracer = bt.Tracer(bt.Config(chunks_x=8, chunks_y=4), engine=engine, seed=0)
    strong = name in STRONG
    if strong and not in_process:
        if passes % world:
            raise SystemExit(f"{name}: {passes} passes do not split across {world} ranks")
        passes //= world                      # this rank's share of the frame's passes
    if in_process and not strong:
        passes *= n_gpus                      # weak scaling: every device renders a full pass slice; the engine splits the call
    rc = bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(sub))
    frame = bt.Buffer(w, h, device=dev)       # this rank's slice of the frame
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    reduce_evs = []

    def step(i, timed=False):
        frame.clear()
        # rank r renders global passes [r*passes, (r+1)*passes) of step i's frame
        tracer.render(scene, cam, rc, frame, sample_base=(i * world + rank) * passes, sync=False)
        if world > 1:
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            dist.reduce(frame.data, dst=0, op=dist.ReduceOp.SUM)   # ONE framebuffer reduce over NVLink
            r1.record()
            if timed:
                reduce_evs.append((r0, r1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = engine.launch_count
    evs = []
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xff)                 # L2 flush between timed steps (outside the event pairs)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(args.warmup + i, timed=True)
        e1.record()
        evs.append((e0, e1))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = engine.launch_count - launches0
    clocks = sampler.summary()
    ms = sum(a.elapsed_time(b) for a, b in evs)
    reduce_ms = sum(a.elapsed_time(b) for a, b in reduce_evs) / max(len(reduce_evs), 1)
    if world > 1:
        t = torch.tensor([ms, reduce_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, reduce_ms = float(t[0].item()), float(t[1].item())
    samples_per_step = w * h * d["spp"] * (1 if strong else n_gpus)
    value = samples_per_step * args.steps / (ms * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:     # before the e2e steps below reuse `frame`
        dump_outputs(args.dump_outputs, frame.data.cpu().numpy())

    # ---- e2e: the same step with HOST buffers at N ranks -------------------------------------------
    # N = 1: the blocking C-ABI call with a pinned host frame (bt_render, BT_MEM_HOST: upload, kernels and download
    # inside the call, pipelined in row bands).  N > 1: rank 0 uploads the caller's pinned host frame (the running
    # sums), every rank renders its pass slice on its GPU, ONE NCCL reduce adds the slices onto rank 0's frame, rank 0
    # downloads it.  Wall clock between barriers around each step, max over ranks.
    n_e2e = args.steps
    host = dhost = None
    if rank == 0:
        host = torch.zeros((h, w, 4), dtype=torch.float32).pin_memory()
        host[..., 3] = 1.0
    if world == 1:
        hb = bt.Buffer(w, h)
        hb.data = host.numpy()

        def e2e_step(i):
            tracer.render(scene, cam, rc, hb, sample_base=i * passes)   # blocking bt_render, BT_MEM_HOST
            return float(hb.data[0, 0, 0])                              # the result is in host memory when the call returns
    else:
        dhost = bt.Buffer(w, h, device=dev) if rank == 0 else None

        def e2e_step(i):
            frame.clear()
            if rank == 0:
                dhost.data.copy_(host, non_blocking=True)               # H2D: the caller's running sums
            tracer.render(scene, cam, rc, frame, sample_base=(i * world + rank) * passes, sync=False)
            dist.reduce(frame.data, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                dhost.data[..., :3] += frame.data[..., :3]              # Buffer::write_color: rgb += value, alpha untouched
                host.copy_(dhost.data, non_blocking=True)               # D2H: the summed frame
                torch.cuda.synchronize()
                return float(host[0, 0, 0])
            torch.cuda.synchronize()
            return 0.0
    for i in range(2):
        e2e_step(i)
    te = 0.0
    for i in range(n_e2e):
        if rank == 0:
            host[..., :3] = 0.0                # a fresh frame (host-side work of the caller: not timed)
        flush.fill_(i & 0xff)
        barrier()
        t0 = time.perf_counter()
        e2e_step(2 + i)
        barrier()
        te += time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([te], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        te = float(t.item())
    del host, dhost

    info = scene.info()
    exact = scene_name in ("cloud", "volume")     # bt_scene_set_precision AUTO: exact for volumetric scenes, fast otherwise
    pool_w = int(os.environ.get("BT_POOL_W", "-1"))
    result = {
        "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": make_config(name, n_gpus),
        "gpu_launches": launches, "clocks": clocks, "wall_s": t_wall,
        "e2e": {"value": samples_per_step * n_e2e / te / 1e6, "unit": METRIC,
                "h2d_bytes_per_step": w * h * 16, "d2h_bytes_per_step": w * h * 16, "steps": n_e2e,
                "note": ("blocking bt_render with a pinned host RGBA32F frame (upload, kernels and download inside the call; the frame "
                         "is pipelined in row bands over two streams); wall clock around each call" if world == 1 else
                         f"rank 0 uploads the pinned host frame, {world} ranks render their pass slices, one NCCL reduce onto rank 0, "
                         "rank 0 downloads the summed frame; wall clock between barriers, max over ranks")},
        "notes": {"timing": "CUDA events per step on torch's current stream (the launch stream), summed; max over ranks",
                  "arithmetic": "exact flavour (IEEE operation sequence of the reference)" if exact else
                                "fast flavour (f32; FMA contraction, MUFU rcp / sqrt / rsqrt within ~1 ulp; tested <= 1e-4 MAE on surface scenes)",
                  "stepper": "MUFU.RSQ (default; endpoints <= 1e-4 relative vs the f64 oracle)" if lens else None,
                  "kernel": "pool_w=%s (env BT_POOL_W; -1: engine default)" % pool_w,
                  "primitives": info["n_primitives"], "lenses": info["n_lenses"],
                  "process_model": ("one process, %d GPUs through bt_engine_create_multi (pass slices + peer-memory reduce inside bt_render)" % n_gpus
                                    if in_process else "one process per GPU (torch.distributed / NCCL)" if world > 1 else "one process, one GPU")},
    }
    if world > 1:
        result["reduce_ms"] = reduce_ms
        result["notes"]["reduce"] = ("CUDA events around dist.reduce (NCCL, %d B per rank): max over ranks of the per-step mean; it includes "
                                     "waiting for the slowest rank's render" % (w * h * 16))

    if rank == 0 and not args.no_extras:
        # ---- roofline of the dominant kernel (render kernel) + the geodesic stepper ----
        peak = engine.fp32_peak_tflops(8192)
        nominal = 148 * 128 * 2 * (clocks["sm_max_mhz"] or 1965) * 1e6 / 1e12
        result["fp32_peak"] = {"measured_fma_tflops": peak, "nominal_tflops_at_max_clock": nominal,
                               "how": "bt_fp32_peak: 8 independent FFMA chains/thread, 8 CTAs/SM, CUDA events"}
        result["stepper_roofline"] = stepper_roofline(engine, torch, peak)
        # exact work counters of the first timed step (deterministic paths): an instrumented copy of
        # the kernel, run outside the timed region.  Counters per path do not depend on the frame size: frames
        # above 4K are counted on their 3840x2160 version and scaled.
        cw, ch = (w, h) if w * h <= 3840 * 2160 else (3840, 2160)
        st = tracer.render_stats(scene, cam, rc, cw, ch, sample_base=args.warmup * world * passes)
        scale = (w * h) / (cw * ch) * (world if strong and not in_process else 1)     # the whole frame's work, all ranks
        st = {k_: v * scale for k_, v in st.items()}
        flops, fl_scan, fl_step = algorithmic_flops(st, scene_name, 1 if lens else 0)
        step_s = ms / args.steps * 1e-3
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(name)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak, hbm_src = (json.load(open(peaks_path))["hbm_gbs"], "measured") if os.path.exists(peaks_path) else (6650.0, "fallback")
        result["roofline"] = {
            "bound": "fp32", "kernel": "render kernel (render_pool_kernel / render_kernel)", "unit": "TFLOP/s", "peak": peak * n_gpus,
            "achieved": flops / step_s / 1e12, "frac": flops / step_s / 1e12 / (peak * n_gpus), "traffic": traffic,
            "work": {**st, "segments_per_path": st["events"] / max(st["paths"], 1),
                     "flops_per_scan": fl_scan, "flops_per_rk4_step": fl_step},
            "note": "CUDA-core FP32 issue bound (no dense contraction on this path: neither the hbm nor the tensor "
                    "roofline binds); achieved = algorithmic flops of the work EXECUTED (SURVEY 8d: a scan = every "
                    "primitive of the reference's try_hit loop, 35 flops per rect test -- a cuboid is six -- and 25 per "
                    "sphere test; 136M+78 per RK4 step; chords skipped by the free-distance test, shading, RNG and ray "
                    "generation count as 0) / CUDA-event step time; peak = live FMA-chain measurement x GPUs",
            "hbm": {"algorithmic_bytes_per_launch": w * h * 32, "achieved_gbs": w * h * 32 / step_s / 1e9,
                    "peak_gbs": hbm_peak, "peak_source": hbm_src},
        }
        try:
            result["pool"] = tracer.render_pool_stats(scene, cam, bt.RenderConfig.with_samples_subsample(1, bt.Subsample(sub)), min(w, 1920), min(h, 1080))
        except bt.BendyError:
            result["pool"] = None
    if rank == 0 and not args.no_extras and n_gpus == 1:
        # ---- the other shipped scenes / the synthetic lens (1 warm-up + 2 timed steps each) ----
        scenes = {}
        for other in ("C1", "C2", "C3", "C4-cloud", "C4-volume", "C4-cloud-lens"):
            if other == name:
                continue
            sn, ow, oh, op, osub, olens = WORKLOADS[other]
            osc = bt.Scene.load(os.path.join(SCENE_DIR, sn + ".json.gz"))
            ocam = osc.find_by_tag("camera")
            osc.set_camera_aspect(ocam, float(np.float32(ow) / np.float32(oh)))
            if olens:
                osc.set_lenses(np.array([olens], np.float32))
            obuf = bt.Buffer(ow, oh, device=dev)
            orc = bt.RenderConfig.with_samples_subsample(op, bt.Subsample(osub))
            tracer.render(osc, ocam, orc, obuf)
            best = None
            for i in range(2):
                obuf.clear()
                flush.fill_(i)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                tracer.render(osc, ocam, orc, obuf, sample_base=(i + 1) * op, sync=False)
                e1.record()
                torch.cuda.synchronize()
                t_ms = e0.elapsed_time(e1)
                best = t_ms if best is None else min(best, t_ms)
            # work counters from one pass (per-path averages are stable), scaled to the timed call
            ost = tracer.render_stats(osc, ocam, bt.RenderConfig.with_samples_subsample(1, bt.Subsample(osub)), ow, oh, sample_base=op)
            oflops, _, _ = algorithmic_flops(ost, sn, 1 if olens else 0)
            scale = ow * oh * describe(other)["spp"] / max(ost["paths"], 1)
            tf = oflops * scale / (best * 1e-3) / 1e12
            scenes[other] = {"workload": describe(other)["workload"], "ms": best,
                             "Msamples_per_s": ow * oh * describe(other)["spp"] / best / 1e3,
                             "segments_per_path": ost["events"] / max(ost["paths"], 1),
                             "scans_per_path": ost["scans"] / max(ost["paths"], 1),
                             "rk4_steps_per_path": ost["rk4_steps"] / max(ost["paths"], 1),
                             "fp32_tflops": tf, "fp32_frac": tf / peak}
            del obuf
        # ---- synthetic many-primitive scene: the BVH path (global-memory nodes, shared-memory stack) ----
        import json as _json
        from common import synthetic_scene
        syn = bt.Scene.from_json(_json.dumps(synthetic_scene(20000, 6000, 1000, seed=1, extent=14.0)))
        scam = syn.find_by_tag("camera")
        sw, sh, sp = 1920, 1080, 4
        syn.set_camera_aspect(scam, float(np.float32(sw) / np.float32(sh)))
        sbuf = bt.Buffer(sw, sh, device=dev)
        src = bt.RenderConfig.with_samples_subsample(sp, bt.Subsample(2))
        tracer.render(syn, scam, src, sbuf)
        best = None
        for i in range(2):
            sbuf.clear()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tracer.render(syn, scam, src, sbuf, sample_base=(i + 1) * sp, sync=False)
            e1.record()
            torch.cuda.synchronize()
            best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        sinfo = syn.info()
        scenes["S-bvh"] = {"workload": f"synthetic scene, {sinfo['n_primitives']} flattened primitives, {sinfo['n_bvh_nodes']} BVH nodes, "
                                       f"{sw}x{sh} at {sp * 4} spp", "ms": best, "Msamples_per_s": sw * sh * sp * 4 / best / 1e3}
        result["scenes"] = scenes
    if rank == 0 and not args.no_extras:
        # ---- CPU baseline: the reference algorithm's restatement on this box's host cores (rank 0, bounded sample) ----
        v, cores, n, dt, (sw, sh), _ = cpu_sample(name, 4 if not lens else 1)
        result["cpu_baseline"] = {"value": v, "unit": METRIC, "cores": cores, "kind": "port",
                                  "sample": f"{n} spp of the frame at {sw}x{sh} ({dt:.1f} s wall on {cores} threads)"}
    if rank == 0:
        json_out.write(json.dumps(result) + "\n")
        json_out.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
