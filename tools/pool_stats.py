"""Scheduling counters of the pooled kernel (bt_render_pool_stats) + work counters of the same call.

    python tools/pool_stats.py [workload] [passes] [knob=value ...]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bendy_tracer_b200 as bt  # noqa: E402
from bench import SCENE_DIR, WORKLOADS  # noqa: E402

full = "--full" in sys.argv
sys.argv = [a for a in sys.argv if a != "--full"]
name = sys.argv[1] if len(sys.argv) > 1 else "C3"
passes = int(sys.argv[2]) if len(sys.argv) > 2 else 2
knobs = dict(kv.split("=") for kv in sys.argv[3:])
scene_name, w, h, _, sub, lens = WORKLOADS[name]
if not full:
    w, h = min(w, 1920), min(h, 1080)
scene = bt.Scene.load(os.path.join(SCENE_DIR, scene_name + ".json.gz"))
cam = scene.find_by_tag("camera")
scene.set_camera_aspect(cam, float(np.float32(w) / np.float32(h)))
if lens:
    scene.set_lenses(np.array([lens], np.float32))
eng = bt.Engine.default(0)
eng.set_tuning(pool_w=3)
eng.set_tuning(**{k: int(v) for k, v in knobs.items()})
tr = bt.Tracer(bt.Config(), engine=eng, seed=0)
rc = bt.RenderConfig.with_samples_subsample(passes, bt.Subsample(sub))
ps = tr.render_pool_stats(scene, cam, rc, w, h)
st = tr.render_stats(scene, cam, rc, w, h)
paths = st["paths"]
print(f"{name} at {w}x{h}, {passes * max(sub, 1) ** 2} spp, knobs {knobs}")
print("work per path:", {k: round(v / paths, 2) for k, v in st.items()})
print("pool:", {k: (round(v, 2) if isinstance(v, float) else v) for k, v in ps.items()})
print(f"per path: step iterations x32 / rk4 steps = {ps['step_iterations'] * 32 / max(st['rk4_steps'], 1):.3f}, "
      f"refill rounds per step iteration = {ps['refill_rounds'] / max(ps['step_iterations'], 1):.3f}, "
      f"step iterations per STEP entry = {ps['step_iterations'] / max(ps['step_entries'], 1):.1f}")
n_ref = ps["refresh_lanes_grid"] + ps["refresh_lanes_outside"]
print(f"free-distance refreshes: STEP iterations with one {ps['refresh_iterations'] / max(ps['step_iterations'], 1):.3f}, "
      f"with lanes inside and outside the box {ps['refresh_mixed_iterations'] / max(ps['refresh_iterations'], 1):.3f} of those, "
      f"lanes per such iteration {n_ref / max(ps['refresh_iterations'], 1):.2f}, outside the box {ps['refresh_lanes_outside'] / max(n_ref, 1):.3f} of the lanes, "
      f"per RK4 step {n_ref / max(st['rk4_steps'], 1):.3f}")
