#!/usr/bin/env python3
"""What an equirectangular panorama (DESIGN.md §3.6) renders at, measured with CUDA events on one GPU.

    python tools/bench_panorama.py [--baseline-lib OTHER/libbendy_b200.so] [--rounds 6] [--out profiles]
                                   [--image panorama.png]

1. Rate: the panorama of bench.py's C3 scene (scene.json.gz + the strong-lens mass) at 4096 x 2048 and 64 spp (16 passes
   at subsample 2), without and with a 2048 x 1024 star-field map, alternating step by step with bench.py's C3 frame
   (3840 x 2160 at 64 spp, perspective) in the same process.
2. No regression (with --baseline-lib, a build of the parent commit): the perspective C3 and C2 frames rendered by both
   libraries, alternating step by step, the frames compared bit for bit -- as tools/bench_environment.py does.

Timing, L2 flush, warm-up and the GPU's name / power limit / clock come from tools/bench_environment.py (imported).  Writes
r3_panorama.json to --out.  --image renders the lensed star field as a 1024 x 512 panorama through the CLI
(bendy_b200_cli --projection equirectangular --environment sky.pfm) to a PNG.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

import bench_environment as BE

ROOT = BE.ROOT
BE.WORKLOADS["P3"] = ("scene", 4096, 2048, 16, 2, BE.LENS)


def panorama(build, env=None):
    sc, cam, rc = build.scene("P3", env)
    build.check(build.L.bt_scene_set_camera_projection(sc, cam, 1))    # BT_PROJECTION_EQUIRECTANGULAR
    return sc, cam, rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="libbendy_b200.so of the build to compare the perspective frames with")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--image", default=None, help="also render the lensed star-field panorama with the CLI to this PNG")
    args = ap.parse_args()

    import torch

    from bendy_tracer_b200 import _ffi
    info = BE.gpu_info()
    print(json.dumps(info), flush=True)
    new = BE.Build(_ffi.LIB_PATH)
    env = BE.star_field()
    res = {"gpu": info, "rounds": args.rounds, "l2": "a 256 MiB memset (L2 flush)", "map": "2048 x 1024 star field"}

    def frame(workload):
        _, w, h, _, _, _ = BE.WORKLOADS[workload]
        return torch.zeros((h, w, 4), dtype=torch.float32, device="cuda:0")

    def samples(workload):
        _, w, h, passes, sub, _ = BE.WORKLOADS[workload]
        return w * h * passes * sub * sub

    # ---- 1. the panorama's rate, next to the perspective C3 frame
    arms = {"C3 perspective": (new, new.scene("C3"), frame("C3")), "panorama": (new, panorama(new), frame("P3")),
            "panorama + map": (new, panorama(new, env), frame("P3"))}
    t = BE.time_alternating(arms, args.rounds)
    res["rate"] = {k: BE.stats(v, samples("C3" if k.startswith("C3") else "P3")) for k, v in t.items()}
    print(json.dumps(res["rate"]), flush=True)
    del arms

    # ---- 2. perspective frames: the parent build against this one
    if args.baseline_lib:
        base = BE.Build(args.baseline_lib)
        res["baseline_lib"] = os.path.relpath(args.baseline_lib, ROOT)
        res["perspective"] = {}
        for wl in ("C3", "C2"):
            arms = {"parent": (base, base.scene(wl), frame(wl)), "this": (new, new.scene(wl), frame(wl))}
            t = BE.time_alternating(arms, args.rounds)
            r = {k: BE.stats(v, samples(wl)) for k, v in t.items()}
            r["delta_pct"] = float((np.median(t["parent"]) / np.median(t["this"]) - 1) * 100)   # > 0: this build is faster
            r["frames_bit_identical"] = bool(torch.equal(arms["parent"][2], arms["this"][2]))
            res["perspective"][wl] = r
            print(wl, json.dumps(r), flush=True)
            del arms

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r3_panorama.json"), "w") as f:
        json.dump(res, f, indent=1)

    if args.image:
        render_image(env, args.image)


def render_image(env, png):
    """the CLI: scene.json.gz, the C3 mass, the star field as a PFM map, a 1024 x 512 panorama at 64 spp"""
    cli = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")
    with tempfile.TemporaryDirectory() as tmp:
        pfm = os.path.join(tmp, "sky.pfm")
        BE.write_pfm(pfm, env)
        cmd = [cli, "--output", "full", "--width", "1024", "--height", "512", "--samples", "64", "--scene",
               os.path.join(BE.SCENE_DIR, "scene.json.gz"), "--lens", ",".join(str(x) for x in BE.LENS), "--environment", pfm,
               "--projection", "equirectangular", "--screenshot", png]
        subprocess.run(cmd, check=True)
    print("wrote", png)


if __name__ == "__main__":
    sys.exit(main())
