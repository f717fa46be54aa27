#!/usr/bin/env python3
"""What the environment map costs (DESIGN.md "Environment map"), measured with CUDA events on one GPU.

    python tools/bench_environment.py [--baseline-lib OTHER/libbendy_b200.so] [--rounds 6] [--out profiles]
                                      [--image lensed_star_field.png]

1. Cost of a map: bench.py's C3 frame (scene.json.gz + the strong-lens mass, 3840 x 2160 at 64 spp) with a 2048 x 1024
   procedural star-field map against the same frame without one, alternating step by step.
2. No map, no regression (with --baseline-lib, a build of the parent commit): the C3 frame and the C2 frame (cornell2,
   1920 x 1080 at 256 spp: the one-path-per-lane kernel) rendered by both libraries, alternating step by step in this one
   process, each build repeated --rounds times so that the difference can be read against the run-to-run spread.  The
   frames of the two builds are compared bit for bit.

Each timed step is one bt_render_async call bracketed by CUDA events, after a 256 MiB memset that flushes the 126 MB L2;
every configuration is warmed up first.  The GPU's name and power limit are read in the same run.  Writes
r3_environment.json and r3_environment.md to --out.  --image also renders the lensed star field through the CLI
(bendy_b200_cli --environment sky.pfm) to a PNG.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCENE_DIR = os.path.join(ROOT, "tests", "golden", "scenes")
LENS = (1.362, 1.577, 6.114, 0.2)
WORKLOADS = {"C3": ("scene", 3840, 2160, 16, 2, LENS), "C2": ("cornell2", 1920, 1080, 64, 2, None)}


def star_field(w=2048, h=1024, seed=0):
    """equirectangular RGB: a faint band of light along a tilted great circle and ~40 000 stars of a steep
    brightness distribution, one texel each, with a spread of colours"""
    rng = np.random.default_rng(seed)
    r, c = np.meshgrid((np.arange(h) + 0.5) / h, (np.arange(w) + 0.5) / w, indexing="ij")
    theta, phi = (0.5 - r) * np.pi, (c - 0.5) * 2 * np.pi
    d = np.stack([np.cos(theta) * np.sin(phi), np.sin(theta), -np.cos(theta) * np.cos(phi)], -1)
    axis = np.array([0.3, 0.9, 0.3]) / np.linalg.norm([0.3, 0.9, 0.3])
    band = np.exp(-((d @ axis) / 0.18) ** 2)
    env = (0.04 + 0.5 * band)[..., None] * np.array([0.55, 0.6, 0.9])
    n = 40_000
    rows, cols = rng.integers(0, h, n), rng.integers(0, w, n)
    mag = np.minimum(2.0 * rng.pareto(1.6, n) + 0.5, 40.0)
    tint = rng.uniform(0.6, 1.0, (n, 3))
    env[rows, cols] += mag[:, None] * tint
    return env.astype(np.float32)


class Build:
    """one build of libbendy_b200.so driven through its C ABI (two builds can live in one process)"""

    def __init__(self, path, device=0):
        from bendy_tracer_b200 import _ffi
        self.ffi = _ffi
        self.L = C.CDLL(path)
        for name, (res, args) in _ffi.SIGNATURES.items():
            if hasattr(self.L, name):
                fn = getattr(self.L, name)
                fn.restype, fn.argtypes = res, args
        self.engine = C.c_void_p()
        self.check(self.L.bt_engine_create(device, C.byref(self.engine)))
        self.cfg = _ffi.BtConfig()
        self.L.bt_config_default(C.byref(self.cfg))
        self.cfg.chunks_x, self.cfg.chunks_y = 8, 4

    def check(self, code):
        if code != 0:
            raise RuntimeError(f"{code}: {self.L.bt_last_error().decode()}")

    def scene(self, workload, env=None):
        name, w, h, passes, sub, lens = WORKLOADS[workload]
        data = open(os.path.join(SCENE_DIR, name + ".json.gz"), "rb").read()
        sc, cam = C.c_void_p(), C.c_uint64()
        self.check(self.L.bt_scene_create_json(None, data, len(data), C.byref(sc)))
        self.check(self.L.bt_scene_find_by_tag(sc, b"camera", C.byref(cam)))
        self.check(self.L.bt_scene_set_camera_aspect(sc, cam.value, float(np.float32(w) / np.float32(h))))
        if lens:
            xyzr = np.array([lens], np.float32)
            self.check(self.L.bt_scene_set_lenses(sc, xyzr.ctypes.data, 1, None))
        if env is not None:
            self.check(self.L.bt_scene_set_environment(sc, env.ctypes.data, env.shape[1], env.shape[0]))
        rc = self.ffi.BtRenderConfig()
        self.L.bt_render_config_default(C.byref(rc))
        rc.samples, rc.subsample = passes, sub
        return sc, cam.value, rc

    def render(self, scene, frame, stream, sample_base=0):
        sc, cam, rc = scene
        h, w = frame.shape[:2]
        n, st = C.c_uint64(0), C.c_int32(0)
        self.check(self.L.bt_render_async(self.engine, sc, cam, C.byref(self.cfg), C.byref(rc), 0, sample_base, frame.data_ptr(),
                                          w, h, C.byref(n), C.byref(st), C.c_void_p(stream)))


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        info.update(nvidia_smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # report, do not invent
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def time_alternating(arms, rounds, warmup=1):
    """arms: {label: (build, scene, frame)}.  Each round times one step of every arm in turn.  -> {label: [ms, ...]}"""
    import torch
    stream = torch.cuda.current_stream(0).cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    for _ in range(warmup):
        for build, scene, frame in arms.values():
            frame.zero_()
            build.render(scene, frame, stream)
    torch.cuda.synchronize()
    out = {k: [] for k in arms}
    for i in range(rounds):
        order = list(arms) if i % 2 == 0 else list(arms)[::-1]
        for k in order:
            build, scene, frame = arms[k]
            frame.zero_()
            flush.fill_(i & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            build.render(scene, frame, stream)
            e1.record()
            e1.synchronize()
            out[k].append(e0.elapsed_time(e1))
    return out


def stats(ms, samples):
    ms = np.array(ms)
    rate = samples / (ms * 1e-3) / 1e6
    return {"ms": ms.round(3).tolist(), "ms_median": float(np.median(ms)), "msamples_per_s_median": float(np.median(rate)),
            "msamples_per_s_min": float(rate.min()), "msamples_per_s_max": float(rate.max()),
            "spread_pct": float((ms.max() - ms.min()) / np.median(ms) * 100)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="libbendy_b200.so of the build to compare the no-map frames with")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--image", default=None, help="also render the lensed star field with the CLI to this PNG")
    args = ap.parse_args()

    import torch

    import bendy_tracer_b200  # noqa: F401  (the build of this tree)
    from bendy_tracer_b200 import _ffi
    info = gpu_info()
    print(json.dumps(info), flush=True)
    new = Build(_ffi.LIB_PATH)
    env = star_field()
    res = {"gpu": info, "rounds": args.rounds, "l2": "a 256 MiB memset (L2 flush)", "map": "2048 x 1024 star field (32 MiB of float4 texels)"}

    def frame(workload):
        _, w, h, _, _, _ = WORKLOADS[workload]
        return torch.zeros((h, w, 4), dtype=torch.float32, device="cuda:0")

    def samples(workload):
        _, w, h, passes, sub, _ = WORKLOADS[workload]
        return w * h * passes * sub * sub

    # ---- 1. cost of a map (C3)
    arms = {"C3 no map": (new, new.scene("C3"), frame("C3")), "C3 + map": (new, new.scene("C3", env), frame("C3"))}
    t = time_alternating(arms, args.rounds)
    res["map_cost"] = {k: stats(v, samples("C3")) for k, v in t.items()}
    cost = np.median(t["C3 + map"]) / np.median(t["C3 no map"]) - 1
    res["map_cost"]["cost_pct"] = float(cost * 100)
    a, b = (arms[k][2][..., :3].mean().item() / 64 for k in arms)
    res["map_cost"]["mean_pixel"] = {"no map": a, "map": b}
    print(json.dumps(res["map_cost"]), flush=True)
    del arms

    # ---- 2. no map, no regression: the parent build against this one
    if args.baseline_lib:
        base = Build(args.baseline_lib)
        res["baseline_lib"] = os.path.relpath(args.baseline_lib, ROOT)
        res["no_map"] = {}
        for wl in ("C3", "C2"):
            arms = {"parent": (base, base.scene(wl), frame(wl)), "this": (new, new.scene(wl), frame(wl))}
            t = time_alternating(arms, args.rounds)
            r = {k: stats(v, samples(wl)) for k, v in t.items()}
            r["delta_pct"] = float((np.median(t["parent"]) / np.median(t["this"]) - 1) * 100)   # > 0: this build is faster
            r["frames_bit_identical"] = bool(torch.equal(arms["parent"][2], arms["this"][2]))
            res["no_map"][wl] = r
            print(wl, json.dumps(r), flush=True)
            del arms

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r3_environment.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(args.out, "r3_environment.md"), "w") as f:
        f.write(report(res))

    if args.image:
        render_image(env, args.image)


def report(res):
    g = res["gpu"]
    lines = ["# Environment map: cost and no-map regression check", "",
             f"Measured on {g.get('nvidia_smi_name', g['name'])}, power limit {g.get('power_limit')}, max SM clock "
             f"{g.get('max_sm_clock', '?')}, with `tools/bench_environment.py` (CUDA events, {res['l2']} before every timed step, "
             f"one warm-up step per configuration, {res['rounds']} timed steps per configuration, configurations alternating "
             "step by step in one process).", "",
             f"## Cost of a map: C3 (3840 x 2160, 64 spp, lensed) with a {res['map']}", "",
             "| configuration | median ms / step | Msamples/s (median) | min .. max | spread |", "|---|---|---|---|---|"]
    mc = res["map_cost"]
    for k in ("C3 no map", "C3 + map"):
        s = mc[k]
        lines.append(f"| {k} | {s['ms_median']:.1f} | {s['msamples_per_s_median']:.1f} | {s['msamples_per_s_min']:.1f} .. "
                     f"{s['msamples_per_s_max']:.1f} | {s['spread_pct']:.1f} % |")
    lines += ["", f"Cost of the map: **{mc['cost_pct']:+.2f} %** step time (median against median).", ""]
    if "no_map" in res:
        lines += ["## No map, no regression: parent build against this one", "",
                  "| workload | build | median ms / step | Msamples/s (median) | min .. max | spread |", "|---|---|---|---|---|---|"]
        for wl, r in res["no_map"].items():
            for k in ("parent", "this"):
                s = r[k]
                lines.append(f"| {wl} | {k} | {s['ms_median']:.2f} | {s['msamples_per_s_median']:.1f} | {s['msamples_per_s_min']:.1f} .. "
                             f"{s['msamples_per_s_max']:.1f} | {s['spread_pct']:.1f} % |")
        lines.append("")
        for wl, r in res["no_map"].items():
            lines.append(f"- {wl}: this build {r['delta_pct']:+.2f} % against the parent (positive: faster); frames bit-identical: "
                         f"{r['frames_bit_identical']}.")
        lines.append("")
    return "\n".join(lines)


def write_pfm(path, rgb):
    h, w, _ = rgb.shape
    with open(path, "wb") as f:
        f.write(f"PF\n{w} {h}\n-1.0\n".encode() + np.ascontiguousarray(rgb[::-1], "<f4").tobytes())


def render_image(env, png):
    """the CLI: scene.json.gz, the C3 mass, the star field as a PFM map"""
    cli = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")
    with tempfile.TemporaryDirectory() as tmp:
        pfm = os.path.join(tmp, "sky.pfm")
        write_pfm(pfm, env)
        cmd = [cli, "--output", "full", "--width", "960", "--height", "540", "--samples", "256", "--scene",
               os.path.join(SCENE_DIR, "scene.json.gz"), "--lens", ",".join(str(x) for x in LENS), "--environment", pfm,
               "--screenshot", png]
        subprocess.run(cmd, check=True)
    print("wrote", png)


if __name__ == "__main__":
    main()
