"""CPU-side tests of the host logic and the C-ABI boundary (no compute calls: there is no GPU here)."""
import ctypes as C
import gzip
import json
import os
import re
import sys

import numpy as np
import pytest

import bendy_tracer_b200 as bt
import oracle_ffi as O
from bendy_tracer_b200 import _ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = ["cornell", "cornell2", "scene", "volume", "cloud"]


def test_library_exports_every_header_symbol():
    header = open(os.path.join(ROOT, "include", "bendy_b200.h")).read()
    declared = set(re.findall(r"\b(bt_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = C.CDLL(_ffi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in include/bendy_b200.h but not exported"
    assert declared == set(_ffi.SIGNATURES), declared ^ set(_ffi.SIGNATURES)


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry point fails loudly (BT_ERR_CUDA), nothing renders."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(bt.BendyError) as e:
        bt.Engine(0)
    assert e.value.code == _ffi.ERR_CUDA and "no CPU fallback" in e.value.message
    scene = bt.Scene.load(O.scene_path("cornell"))
    with pytest.raises(bt.BendyError):
        bt.Tracer().render(scene, 0, bt.RenderConfig.with_samples(1), bt.Buffer(8, 8))


def test_product_never_touches_the_oracle():
    """the engine sources and the package must not include, link or import anything under oracle/"""
    pkg = os.path.join(ROOT, "bendy_tracer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "bendy_oracle" not in text and "oracle_ffi" not in text and "oracle/" not in text, f


@pytest.mark.parametrize("name", SCENES)
def test_scene_round_trip(name):
    """serde wire format: load -> to_json -> identical JSON value (src/main.rs:93-102, 299-313)"""
    path = O.scene_path(name)
    scene = bt.Scene.load(path)
    original = json.load(gzip.open(path))
    assert json.loads(scene.to_json()) == original
    again = bt.Scene.from_json(scene.to_json())
    assert again.to_json() == scene.to_json()
    info = scene.info()
    n_obj = len(original["objects"]["collection"])
    assert info["n_objects"] == n_obj and info["n_data"] == len(original["data"]["collection"])
    expect_prims = {"cornell": 18, "cornell2": 18, "scene": 5, "volume": 4, "cloud": 4}[name]
    assert info["n_primitives"] == expect_prims and info["n_lights"] == 1
    assert info["n_volumes"] == (1 if name in ("volume", "cloud") else 0)
    assert info["root_material"] == original["root_material"]
    assert scene.find_by_tag("camera") == 0 and scene.find_by_tag("no such tag") is None


UPSTREAM_DIR = os.path.join(ROOT, "tests", "golden", "scenes_upstream")


@pytest.mark.parametrize("name", SCENES)
def test_upstream_scene_bytes(name):
    """the reference's shipped files, byte for byte (hash-ordered keys, the reference's own gzip stream; SHA256SUMS holds the
    hashes of the reference's files): they load, round-trip to the same JSON value, and flatten to exactly what the
    re-serialised copy flattens to"""
    import hashlib
    path = os.path.join(UPSTREAM_DIR, name + ".json.gz")
    sums = dict(reversed(l.split()) for l in open(os.path.join(UPSTREAM_DIR, "SHA256SUMS")))
    raw = open(path, "rb").read()
    assert hashlib.sha256(raw).hexdigest() == sums[name + ".json.gz"]
    up, ours = bt.Scene(raw), bt.Scene.load(O.scene_path(name))
    original = json.loads(gzip.decompress(raw))
    assert list(original["objects"]["collection"]) != sorted(original["objects"]["collection"], key=int) or name != "cornell"
    assert json.loads(up.to_json()) == original
    assert up.to_json() == ours.to_json()                       # canonical (ascending ObjectRef) order either way
    assert up.info() == ours.info()
    assert up.find_by_tag("camera") == ours.find_by_tag("camera") == 0


def test_scene_plain_json_and_gzip(tmp_path):
    text = gzip.open(O.scene_path("scene")).read()
    a, b = bt.Scene(text), bt.Scene.load(O.scene_path("scene"))
    assert a.to_json() == b.to_json()
    a.save(tmp_path / "s.json.gz")
    a.save(tmp_path / "s.json")
    assert bt.Scene.load(tmp_path / "s.json.gz").to_json() == bt.Scene.load(tmp_path / "s.json").to_json() == a.to_json()


def test_scene_lens_extension_round_trip():
    scene = json.load(gzip.open(O.scene_path("scene")))
    scene["lenses"] = [[1.362, 1.577, 6.114, 0.2], [0.0, 0.0, 0.0, 0.0]]
    s = bt.Scene.from_json(json.dumps(scene))
    assert s.info()["n_lenses"] == 1                    # r_s = 0 masses are dropped (exact flat limit)
    assert json.loads(s.to_json())["lenses"] == [[1.362, 1.577, 6.114, 0.2], [0.0, 0.0, 0.0, 0.0]]
    s.set_lenses(np.zeros((0, 4), np.float32))
    assert s.info()["n_lenses"] == 0 and "lenses" not in json.loads(s.to_json())


def test_scene_parse_errors():
    good = json.load(gzip.open(O.scene_path("cornell")))
    for mutate, code in [
        (lambda s: s.pop("root_material"), _ffi.ERR_PARSE),                               # missing field
        (lambda s: s["objects"]["collection"]["1"].__setitem__("inner", {"Torus": {}}), _ffi.ERR_PARSE),
        (lambda s: s["objects"]["collection"]["1"]["transform"].__setitem__("transform_world", [1.0] * 11), _ffi.ERR_PARSE),
        (lambda s: s.__setitem__("root_material", 99), _ffi.ERR_SCENE),                    # invalid data ref
        (lambda s: s["objects"]["collection"]["1"]["inner"]["Rect"].__setitem__("material", 99), _ffi.ERR_SCENE),
    ]:
        bad = json.loads(json.dumps(good))
        mutate(bad)
        with pytest.raises(bt.BendyError) as e:
            bt.Scene.from_json(json.dumps(bad))
        assert e.value.code == code, e.value
    with pytest.raises(bt.BendyError) as e:
        bt.Scene(b"{ not json")
    assert e.value.code == _ffi.ERR_PARSE
    with pytest.raises(bt.BendyError) as e:
        bt.Scene(b"\x1f\x8b\x08\x00garbage")
    assert e.value.code == _ffi.ERR_PARSE
    vol = json.load(gzip.open(O.scene_path("volume")))
    vol["data"]["collection"]["5"]["inner"]["Volume"]["DensityMap"]["buffer"][3] = -0.5   # gen_bool(p < 0) panics
    with pytest.raises(bt.ScenePanic):
        bt.Scene.from_json(json.dumps(vol))
    vol = json.load(gzip.open(O.scene_path("volume")))
    vol["objects"]["collection"]["2"]["inner"]["Sphere"]["volume"] = 4                     # a material, not a volume
    with pytest.raises(bt.ScenePanic, match="expected volume data"):
        bt.Scene.from_json(json.dumps(vol))


def test_apply_transform_propagates_to_children():
    """Object::apply_transform + UpdateQueue::commit (object/mod.rs:200-223, scene/mod.rs:204-213)"""
    scene = json.load(gzip.open(O.scene_path("scene")))
    objs = scene["objects"]["collection"]
    objs["4"]["children"] = [5]                                        # glass sphere -> parent of the metal sphere
    s = bt.Scene.from_json(json.dumps(scene))
    shift = [1, 0, 0, 0, 1, 0, 0, 0, 1, 0.5, 1.0, -2.0]
    s.apply_transform(4, shift)
    out = json.loads(s.to_json())["objects"]["collection"]
    assert out["4"]["transform"]["transform_world"][9:] == [0.0, 1.0, -2.0]
    assert out["4"]["transform"]["transform_local"] == out["4"]["transform"]["transform_world"]
    child = out["5"]["transform"]
    assert child["transform_parent"] == out["4"]["transform"]["transform_world"]
    # world = parent * local: the child's local (2.5, 0, -2.5) is now relative to the parent at (0, 1, -2)
    assert np.allclose(child["transform_world"][9:], [2.5, 1.0, -4.5])
    assert child["transform_local"] == objs["5"]["transform"]["transform_local"]
    with pytest.raises(bt.ScenePanic, match="invalid object ref"):
        s.apply_transform(42, shift)


def test_box_shaped_cuboids_are_recognised():
    """Cuboid::new boxes under a rigid transform flatten to one BOX record each (one slab test instead
    of six rect tests); a cuboid whose faces no longer form a box keeps its six rect tests."""
    doc = O.read_scene_json(O.scene_path("cornell"))
    sc = bt.Scene.from_json(json.dumps(doc))
    assert sc.info()["n_boxes"] == 2 and sc.info()["n_primitives"] == 18
    sc.set_accel("linear_faces")
    assert sc.info()["n_boxes"] == 0
    sc.set_accel("bvh")
    assert sc.info()["n_boxes"] == 0
    cub = [o for o in doc["objects"]["collection"].values() if "Cuboid" in o["inner"]]
    assert len(cub) == 2
    cub[0]["inner"]["Cuboid"]["faces"][0][1]["half_width"] *= 0.5      # a face that no longer spans the box
    assert bt.Scene.from_json(json.dumps(doc)).info()["n_boxes"] == 1
    m = cub[1]["transform"]["transform_world"]
    m[3] += 0.3 * m[0]; m[4] += 0.3 * m[1]; m[5] += 0.3 * m[2]          # shear: y axis leans along x
    cub[1]["transform"]["transform_local"] = list(m)
    assert bt.Scene.from_json(json.dumps(doc)).info()["n_boxes"] == 0


def test_cuboid_light_flattens():
    """A LIGHT Cuboid is one light object (its six faces become sub-records behind the object lights)
    and the oracle samples it (Cuboid::random_point / pdf, cuboid.rs:48-81)."""
    from common import cornell_with_cuboid_light, oracle_render
    doc = cornell_with_cuboid_light(True)
    sc = bt.Scene.from_json(json.dumps(doc))
    info = sc.info()
    assert info["n_lights"] == 2 and info["n_primitives"] == 18 and info["n_boxes"] == 2
    assert json.loads(sc.to_json())["objects"]["collection"]["8"]["flags"]["bits"] == 1
    osc = O.OracleScene(doc)
    img, n, _ = oracle_render(osc, 0, 32, 32, 2, 0, 0, seed=1)
    base, _, _ = oracle_render(O.OracleScene.load(O.scene_path("cornell")), 0, 32, 32, 2, 0, 0, seed=1)
    assert np.isfinite(img).all() and img[..., :3].sum() > 1.5 * base[..., :3].sum()


def test_precision_and_accel_arguments():
    s = bt.Scene.load(O.scene_path("cloud"))
    for mode in ("auto", "fast", "exact"):
        s.set_precision(mode)
    assert _ffi.lib.bt_scene_set_precision(s.handle, 3) == _ffi.ERR_INVALID_ARG
    assert _ffi.lib.bt_scene_set_accel(s.handle, 4) == _ffi.ERR_INVALID_ARG
    assert _ffi.lib.bt_scene_set_accel(s.handle, 3) == _ffi.OK


def test_camera_aspect_update():
    s = bt.Scene.load(O.scene_path("cornell"))
    s.set_camera_aspect(0, 1.7777778)
    assert json.loads(s.to_json())["objects"]["collection"]["0"]["inner"]["Camera"]["aspect_ratio"] == 1.7777778
    with pytest.raises(bt.ScenePanic):
        s.set_camera_aspect(1, 1.0)                                    # object 1 is a Rect
    with pytest.raises(bt.ScenePanic):
        s.set_camera_aspect(99, 1.0)


def test_api_mirror_defaults():
    c = bt.Config()
    assert (c.max_bounces, c.max_volume_bounces, c.clip_min, c.clip_max, c.volume_step, c.chunks_x, c.chunks_y,
            c.output) == (8, 32, 0.01, 1000.0, 0.1, 4, 2, bt.Output.Full)                  # Config::DEFAULT, mod.rs:29-38
    r = bt.RenderConfig()
    assert r.samples == 64 and r.subsample == bt.Subsample.none() and r.output is None     # RenderConfig::DEFAULT
    assert bt.RenderConfig.with_samples(3).samples == 3
    rc = bt.RenderConfig.with_samples_subsample(2, bt.Subsample.subpixel(3))
    assert rc.subsample.subpixel_count() == 9 and abs(rc.subsample.subpixel_size() - 1 / 3) < 1e-7
    offs = list(bt.Subsample.subpixel(2))
    assert offs == [(0.0, 0.0), (0.5, 0.0), (0.0, 0.5), (0.5, 0.5)]                        # i fastest (mod.rs:96-101)
    assert list(bt.Subsample.none()) == [(0.0, 0.0)] and bt.Subsample.none().subpixel_count() == 1
    cc, cr = _ffi.BtConfig(), _ffi.BtRenderConfig()
    _ffi.lib.bt_config_default(C.byref(cc))
    _ffi.lib.bt_render_config_default(C.byref(cr))
    assert (cc.max_bounces, cc.max_volume_bounces, cc.chunks_x, cc.chunks_y, cc.output) == (8, 32, 4, 2, 0)
    assert abs(cc.clip_min - 0.01) < 1e-9 and cc.clip_max == 1000.0 and abs(cc.volume_step - 0.1) < 1e-8
    assert cr.samples == 64 and cr.subsample == 0 and not (cr.has_output or cr.has_max_bounces or cr.has_volume_step)
    lc = _ffi.BtLensConfig()
    _ffi.lib.bt_lens_config_default(C.byref(lc))
    d = bt.LensConfig()
    assert (lc.max_steps, lc.flags) == (d.max_steps, 0) and abs(lc.kappa - d.kappa) < 1e-9


def test_buffer_mirror():
    b = bt.Buffer(6, 4, bt.ColorSpace.SRgb)
    assert b.dimensions() == (6, 4) and b.samples() == 0 and b.width() == 6 and b.height() == 4
    assert (b.into_buffer()[..., :3] == 0).all() and (b.into_buffer()[..., 3] == 1).all()     # BLACK_ALPHA_ONE
    assert abs(b.pixel_width() - 2 / 6) < 1e-7 and abs(b.pixel_height() - 0.5) < 1e-7
    b.data[..., 0] = 5
    b._samples = 3
    b.clear()
    assert (b.data[..., :3] == 0).all() and (b.data[..., 3] == 1).all() and b.samples() == 0
    b.resize(3, 2)
    assert b.dimensions() == (3, 2) and b.maybe_preview() is None and b.take_preview() is None


@pytest.mark.parametrize("w,h,cx,cy", [(512, 512, 8, 4), (1920, 1080, 8, 4), (100, 70, 8, 4), (7, 3, 4, 2), (5, 5, 8, 8)])
def test_buffer_chunks(w, h, cx, cy):
    """Buffer::chunks / Chunks::next (buffer.rs:102-115, 293-326): the tiles partition the image, in
    row-major order, ceil-div sized with the last row / column clipped"""
    buf = bt.Buffer(w, h)
    tiles = list(buf.chunks(cx, cy))
    cover = np.zeros((h, w), np.int32)
    cw, ch = -(-w // cx), -(-h // cy)
    for i, (x0, y0, x1, y1) in enumerate(tiles):
        assert 0 <= x0 < x1 <= w and 0 <= y0 < y1 <= h and x1 - x0 <= cw and y1 - y0 <= ch
        assert x0 % cw == 0 and y0 % ch == 0
        cover[y0:y1, x0:x1] += 1
    assert (cover == 1).all()
    assert tiles == sorted(tiles, key=lambda t: (t[1], t[0]))
    assert len(tiles) == -(-w // cw) * -(-h // ch)
    if (w, h, cx, cy) == (512, 512, 8, 4):
        assert tiles[0] == (0, 0, 64, 128) and len(tiles) == 32           # SURVEY 8a row 1: C1 tiles are 64 x 128


def test_shard_passes_partition():
    for samples in (1, 7, 64, 1024):
        for world in (1, 2, 3, 4, 8):
            cuts = [bt.shard_passes(samples, world, r) for r in range(world)]
            assert cuts[0][0] == 0 and cuts[-1][1] == samples
            assert all(cuts[i][1] == cuts[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in cuts]
            assert max(sizes) - min(sizes) <= 1


def test_cli_builtin_scene_and_flags(tmp_path):
    """the headless CLI (csrc/cli.cpp): --output is required (clap), and with no scene file it builds the
    Cornell box of main.rs:108-213 -- which is exactly what the reference shipped as cornell2.json.gz"""
    import subprocess
    cli = os.path.join(ROOT, "bendy_tracer_b200", "csrc", "bendy_b200_cli")
    r = subprocess.run([cli, "--width", "8"], capture_output=True, text=True)
    assert r.returncode != 0 and "--output" in r.stderr
    out = tmp_path / "builtin.json"
    r = subprocess.run([cli, "--output", "full", "--width", "100", "--height", "100", "--samples", "0",
                        "--scene", str(tmp_path / "missing.json"), "--save-scene", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert json.load(open(out)) == json.load(gzip.open(O.scene_path("cornell2")))
    r = subprocess.run([cli, "--output", "normal", "--width", "300", "--height", "200", "--samples", "0",
                        "--scene", O.scene_path("scene"), "--save-scene", str(out)], capture_output=True, text=True)
    assert r.returncode == 0 and "loaded scene" in r.stderr
    assert json.load(open(out))["objects"]["collection"]["0"]["inner"]["Camera"]["aspect_ratio"] == 1.5   # w / h


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` (the reference algorithm on the host cores): one JSON line with the
    contract's keys; under torchrun only rank 0 prints, the other ranks exit 0 without work.  `--dump-outputs`
    writes the frame of the last timed step: the oracle's image of that step."""
    import subprocess
    import sys
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--workload", "C1", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, check=True, env={**os.environ, "RANK": "0"}).stdout
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == d["unit"] == "Msamples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "C1" in d["config"]["workload"]
    osc = O.OracleScene.load(O.scene_path("cornell"))
    osc.set_camera_aspect(0, 1.0)
    ref, _, _ = osc.render(0, O.make_config(samples=1, subsample=2), 512, 512, seed=0)
    assert sorted(os.listdir(tmp_path)) == ["frame.npy"]
    assert np.array_equal(np.load(tmp_path / "frame.npy"), ref)
    os.remove(tmp_path / "frame.npy")
    other = subprocess.run(cmd, capture_output=True, text=True, check=True, env={**os.environ, "RANK": "1"})
    assert other.stdout.strip() == "" and os.listdir(tmp_path) == []


def test_bench_dump_outputs_samples_large_frames(tmp_path, monkeypatch):
    """a frame above bench.DUMP_BYTES is dumped as the same seeded pixel sample on every run, with its flat indices"""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 24)
    frame = np.random.default_rng(2).random((30, 40, 4), dtype=np.float32)
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, frame)
        assert sorted(os.listdir(tmp_path / run)) == ["frame.npy", "frame_pixels.npy"]
    values, pixels = np.load(tmp_path / "a" / "frame.npy"), np.load(tmp_path / "a" / "frame_pixels.npy")
    assert values.shape == (100, 4) and values.dtype == np.float32 and pixels.dtype == np.float64
    assert (np.diff(pixels) > 0).all() and pixels[-1] < 30 * 40
    assert np.array_equal(values, frame.reshape(-1, 4)[pixels.astype(np.int64)])
    assert np.array_equal(np.load(tmp_path / "b" / "frame_pixels.npy"), pixels)
    assert np.array_equal(np.load(tmp_path / "b" / "frame.npy"), values)
    bench.dump_outputs(tmp_path / "small", frame[:5, :5])
    assert np.array_equal(np.load(tmp_path / "small" / "frame.npy"), frame[:5, :5])


def test_rust_sys_crate_matches_header():
    """bendy-b200-sys/src/lib.rs declares every function of include/bendy_b200.h with the same arity and pointer
    shape, every #[repr(C)] struct with the header's fields in the header's order, and every enum constant with its
    value; build.rs compiles the same translation units as csrc/Makefile; the generated file is not stale."""
    import re
    import subprocess
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_rust_sys as G
    opaque, structs, consts, funcs = G.parse_header()
    rs = open(os.path.join(ROOT, "bendy-b200-sys", "src", "lib.rs")).read()
    assert subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_rust_sys.py"), "--check"]).returncode == 0, "lib.rs is stale"
    assert len(funcs) >= 30 and {"bt_config", "bt_render_config", "bt_lens_config", "bt_segment", "bt_scene_info"} <= set(structs)
    for name, ret, params in funcs:
        m = re.search(r"pub fn %s\((.*?)\)( -> ([^;]+))?;" % name, rs)
        assert m, f"{name} missing from lib.rs"
        args = [a for a in m.group(1).split(", ") if a]
        assert len(args) == len(params), name
        for (pname, ctype), a in zip(params, args):
            rname, rtype = a.split(": ")
            assert rname.replace("r#", "") == pname
            assert rtype.count("*") == ctype.count("*"), (name, pname)
            if "*" in ctype:
                assert rtype.startswith("*const") == ctype.startswith("const"), (name, pname)
        assert (m.group(3) is None) == (ret == "void"), name
    for name, fields in structs.items():
        body = re.search(r"pub struct %s \{(.*?)\n\}" % name, rs, flags=re.S).group(1)
        got = re.findall(r"pub (\w+): ([^,]+),", body)
        assert [f for f, _ in got] == [f for f, _, _ in fields], name
        for (f, ctype, arr), (_, rtype) in zip(fields, got):
            assert rtype == (f"[{G.SCALARS[ctype]}; {arr}]" if arr else G.SCALARS[ctype]), (name, f)
    for name, value in consts:
        assert re.search(r"pub const %s: c_int = %d;" % (name, value), rs), name
    for name in opaque:
        assert f"pub struct {name} {{" in rs
    # the ctypes binding and the Rust crate describe the same ABI: every header function is bound by both
    from bendy_tracer_b200 import _ffi
    assert {n for n, _, _ in funcs} == set(_ffi.SIGNATURES)
    build_rs = open(os.path.join(ROOT, "bendy-b200-sys", "build.rs")).read()
    for unit in ("engine.cu", "kernels.cu", "scene.cpp", "-DBT_EXACT_SCAN", "compute_100a"):
        assert unit in build_rs


def test_reference_patch_is_well_formed():
    """patches/bendy_tracer_b200.patch (the change a maintainer applies to the reference crate) only touches the render
    boundary, calls entry points that the header declares, and fills every field of the two config structs"""
    import re
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_rust_sys as G
    _, structs, _, funcs = G.parse_header()
    patch = open(os.path.join(ROOT, "patches", "bendy_tracer_b200.patch")).read()
    files = re.findall(r"^\+\+\+ b/(\S+)", patch, flags=re.M)
    assert files == ["Cargo.toml", "src/scene/object/mod.rs", "src/tracer/buffer.rs", "src/tracer/mod.rs"]
    added = "\n".join(l[1:] for l in patch.splitlines() if l.startswith("+") and not l.startswith("+++"))
    declared = {n for n, _, _ in funcs}
    used = set(re.findall(r"sys::(bt_\w+)\(", added))
    assert used and used <= declared, used - declared
    assert {"bt_engine_create_multi", "bt_scene_create_json", "bt_render", "bt_engine_destroy", "bt_scene_destroy"} <= used
    for struct in ("bt_config", "bt_render_config"):
        body = re.search(r"sys::%s \{(.*?)\n        \};" % struct, added, flags=re.S).group(1)
        assert re.findall(r"^ {12}(\w+):", body, flags=re.M) == [f for f, _, _ in structs[struct]], struct
    # the hunks are consistent on their own (what `patch -p1` checks before it reads the reference's files; inside a
    # checkout of the reference, `patch -p1 --dry-run -i patches/bendy_tracer_b200.patch` checks the rest): every body
    # has the line counts of its header, and a file's hunks are in order, disjoint, and start where the net growth of
    # the hunks before them puts them
    lines = patch.splitlines()
    i = n_hunks = 0
    while i < len(lines):
        if lines[i].startswith("--- "):
            assert lines[i + 1].startswith("+++ "), lines[i]
            i, old_end, growth = i + 2, 0, 0
            continue
        m = re.fullmatch(r"@@ -(\d+)(?:,(\d+))? \+(\d+)(?:,(\d+))? @@.*", lines[i])
        assert m, f"line {i + 1}: {lines[i]!r}"
        old_start, n_old, new_start, n_new = (int(g) if g is not None else 1 for g in m.groups())
        assert old_start > old_end and new_start == old_start + growth, lines[i]
        old_end, growth, n_hunks = old_start + n_old - 1, growth + n_new - n_old, n_hunks + 1
        i += 1
        while n_old or n_new:
            tag = lines[i][:1] if i < len(lines) else "end of file"
            assert tag in (" ", "-", "+") and (n_old > 0 or tag == "+") and (n_new > 0 or tag == "-"), \
                f"line {i + 1}: the hunk body does not match its header"
            n_old -= tag != "+"
            n_new -= tag != "-"
            i += 1
    assert n_hunks == 7


def test_json_nesting_limit_is_an_error_not_a_crash():
    """serde_json stops at 128 nested arrays / objects with an error; so does the loader (a scene file is untrusted input:
    100 000 '[' must not overflow the host stack)"""
    for text in ("[" * 100000, "{\"a\":" * 5000 + "1" + "}" * 5000, "[" * 129 + "]" * 129):
        with pytest.raises(bt.BendyError) as e:
            bt.Scene.from_json(text)
        assert e.value.code == _ffi.ERR_PARSE
    ok = "[" * 100 + "]" * 100          # within the limit: parses (and is then rejected as a scene, not as JSON)
    with pytest.raises(bt.BendyError) as e:
        bt.Scene.from_json(ok)
    assert "recursion" not in str(e.value)


def test_bvh_build_survives_skewed_and_coincident_primitives():
    """200 spheres on one spot and a geometric cluster that makes every SAH split lopsided: the builder falls back to
    median splits near its depth budget instead of rejecting the scene (flattening happens at load: no GPU needed)"""
    from common import skewed_scene
    doc = skewed_scene()
    sc = bt.Scene.from_json(json.dumps(doc))
    sc.set_accel("bvh")
    info = sc.info()
    assert info["n_primitives"] == 402 and info["n_bvh_nodes"] > 3


def _check_bvh(sc, max_depth=11, types=None):
    """structural invariants of the 4-wide BVH (bt_scene_copy_bvh): every primitive in exactly one leaf, every child box
    holds what is below it (conservatively padded), empty slots last, children stored behind their parent, depth and
    stack demand within what the traversal kernels allocate"""
    b = sc.bvh()
    nodes, refs, order, bounds = b["nodes"], b["refs"], b["order"], b["bounds"]
    n, n_prims = len(nodes), len(order)
    assert n > 0 and sorted(order.tolist()) == list(range(n_prims))
    LEAF, EMPTY = 0x80000000, 0xFFFFFFFE
    seen = np.zeros(n_prims, np.int32)
    visited = np.zeros(n, np.int32)
    deepest = 0

    def walk(node, depth):
        nonlocal deepest
        deepest = max(deepest, depth)
        visited[node] += 1
        lo = np.full(3, np.inf, np.float32)
        hi = np.full(3, -np.inf, np.float32)
        empty_seen = False
        for c in range(4):
            r = int(refs[node, c])
            if r == EMPTY:
                empty_seen = True
                continue
            assert not empty_seen, "an empty slot before a child"
            box_lo, box_hi = nodes[node, 0:6:2, c], nodes[node, 1:6:2, c]
            if r & LEAF:
                first, count, kind = r & 0xFFFFFF, (r >> 24) & 0x1F, (r >> 29) & 3
                assert 1 <= count <= 31 and first + count <= n_prims
                prims = order[first:first + count]
                if types is not None:         # the leaf's kind: 1 = all spheres, 2 = no sphere, 0 = mixed
                    sph = int(types[prims].sum())
                    assert kind == (1 if sph == count else 2 if sph == 0 else 0), (kind, sph, count)
                seen[first:first + count] += 1
                c_lo, c_hi = bounds[prims, :3].min(0), bounds[prims, 3:].max(0)
            else:
                assert node < r < n, "children are stored behind their parent (refit sweeps backwards)"
                c_lo, c_hi = walk(r, depth + 1)
            assert (box_lo <= c_lo).all() and (box_hi >= c_hi).all(), (node, c)
            pad = 2e-4 * np.maximum(1, np.maximum(np.abs(box_lo), np.abs(box_hi))) + 1e-6     # (the builder pads by 1e-4 of that)
            if not (node == 0 and r & LEAF):      # (the leaf of scene-spanning primitives carries the whole scene's box)
                assert (c_lo - box_lo <= pad).all() and (box_hi - c_hi <= pad).all(), "the box is the padded union, no looser"
            lo, hi = np.minimum(lo, c_lo), np.maximum(hi, c_hi)
        assert refs[node, 0] != EMPTY
        return lo, hi

    sys.setrecursionlimit(10000)
    walk(0, 1)
    assert (seen == 1).all() and (visited == 1).all()
    assert deepest <= max_depth and 3 * deepest <= 40       # BVH_STACK (layout.h): 3 pushes per level
    return deepest


def test_bvh4_structure_and_refit():
    from common import skewed_scene, synthetic_scene
    def record_types(doc):          # 1 per sphere record, 0 per rect / cuboid-face record, in canonical (ascending ObjectRef) order
        out = []
        for key in sorted(doc["objects"]["collection"], key=int):
            inner = doc["objects"]["collection"][key]["inner"]
            kind = inner if isinstance(inner, str) else next(iter(inner))
            out += {"Sphere": [1], "Rect": [0], "Cuboid": [0] * 6}.get(kind, [])
        return np.array(out, np.int32)

    for doc in (synthetic_scene(300, 100, 20, seed=4), synthetic_scene(3000, 500, 100, seed=5, extent=6.0), skewed_scene(), skewed_scene(120, 60, 0.3)):
        sc = bt.Scene.from_json(json.dumps(doc))
        sc.set_accel("bvh")
        types = record_types(doc)
        assert len(types) == sc.info()["n_primitives"]
        _check_bvh(sc, types=types)
    # a shipped scene forced onto the BVH (a scene-spanning ground sphere goes to its own leaf beside the tree)
    sc = bt.Scene.load(O.scene_path("scene"))
    sc.set_accel("bvh")
    _check_bvh(sc)
    # refit after transform edits: same topology, boxes follow the primitives
    doc = synthetic_scene(3000, 500, 100, seed=5, extent=6.0)
    sc = bt.Scene.from_json(json.dumps(doc))
    before = sc.bvh()
    objs = json.loads(sc.to_json())["objects"]["collection"]
    moved = [int(k) for k in list(objs)[10:400:7]]
    for ref in moved:
        t = list(objs[str(ref)]["transform"]["transform_world"])
        t[9] += 0.37
        t[11] -= 0.21
        sc.apply_transform(ref, t)
    sc.commit()
    after = sc.bvh()
    assert np.array_equal(before["refs"], after["refs"]) and np.array_equal(before["order"], after["order"])
    assert not np.array_equal(before["bounds"], after["bounds"]) and not np.array_equal(before["nodes"], after["nodes"])
    _check_bvh(sc)
    fresh = bt.Scene.from_json(sc.to_json())
    assert np.array_equal(np.sort(fresh.bvh()["bounds"], axis=0), np.sort(after["bounds"], axis=0))
