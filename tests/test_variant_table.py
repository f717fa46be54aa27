"""Which compiled kernel variant serves a call (bendy_tracer_b200/csrc/variants.h), over the whole request space (CPU only).

tests/variant_table.cpp wraps the table and its selection in a C ABI; it is built with the host compiler on first use into a
cache directory keyed by the sources' contents (the tree may be read-only).
"""
import ctypes as C
import hashlib
import itertools
import os
import subprocess
import tempfile

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "bendy_tracer_b200", "csrc")
SOURCES = [os.path.join(HERE, "variant_table.cpp"), os.path.join(CSRC, "variants.h"), os.path.join(CSRC, "layout.h")]
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")   # vector_types.h
CXXFLAGS = ["-O1", "-std=c++17", "-Wall", "-fPIC", "-shared", f"-I{CSRC}", f"-I{CUDA_INCLUDE}"]

CT_SPHERES, CT_RECTS, CT_VOLUMES, CT_METAL, CT_GLASS, CT_AOV, CT_CUBOID_LIGHT, CT_ALL = 1, 2, 4, 8, 16, 32, 64, 127
V_LANE, V_LANE_STATS, V_POOL, V_POOL_STATS, V_POOL_BVH, V_TRACE = 1, 2, 4, 8, 16, 32
FAMILIES = (V_LANE, V_LANE_STATS, V_POOL, V_POOL_STATS, V_POOL_BVH, V_TRACE)
RENDER, WORK_COUNTERS, POOL_COUNTERS, TRACE = range(4)
POOL_MAX_BOUNCES, POOL_MAX_OBJECTS = 254, 126


@pytest.fixture(scope="module")
def vt():
    key = hashlib.sha256(b"".join(open(p, "rb").read() for p in SOURCES) + " ".join(CXXFLAGS).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"bendy_variant_table_{os.getuid()}")
    path = os.path.join(out_dir, f"libvariant_table_{key}.so")
    if not os.path.exists(path):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CXX", "g++"), *CXXFLAGS, "-o", tmp, SOURCES[0]], check=True)
        os.replace(tmp, path)
    L = C.CDLL(path)
    L.vt_row.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int)]
    L.vt_select.argtypes = [C.c_uint32, C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                            C.c_int, C.c_int, C.POINTER(C.c_int)]
    return L


def rows(vt, exact_flavour):
    """[(LENS, EXACT, NL, BVH, C, families compiled in the flavour)]"""
    out = []
    for i in range(vt.vt_count()):
        r = (C.c_int * 6)()
        vt.vt_row(i, exact_flavour, r)
        out.append(tuple(r))
    return out


def select(vt, content, output=0, n_lens=0, lens_exact=0, bvh=False, mode=RENDER, pool_w=0, max_bounces=8, n_prims=10,
           exact_flavour=False):
    """(family, row index or None)"""
    fam = C.c_int()
    row = vt.vt_select(content, output, n_lens, lens_exact, 5 if bvh else 0, pool_w, max_bounces, n_prims, mode,
                       int(exact_flavour), C.byref(fam))
    return fam.value, (None if row < 0 else row)


def requests():
    """every content mask, output, lens table, stepper, accelerator, mode, pool size and limit, in both flavours"""
    limits = ((8, 10), (POOL_MAX_BOUNCES + 1, 10), (8, POOL_MAX_OBJECTS + 1))   # (max_bounces, primitives)
    for ef, content, output, n_lens, lens_exact, bvh, mode, pool_w, (mb, n_prims) in itertools.product(
            (False, True), range(CT_ALL + 1), (0, 2), (0, 1, 3), (0, 1), (False, True), range(4), (0, 3), limits):
        if content & CT_AOV or (bvh and content & CT_VOLUMES):   # (CT_AOV comes from the output; no volumes under a BVH)
            continue
        if ef and n_lens and not lens_exact:                     # the exact flavour renders lensed scenes with the exact stepper
            continue
        req = dict(content=content, output=output, n_lens=n_lens, lens_exact=lens_exact, bvh=bvh, mode=mode, pool_w=pool_w,
                   max_bounces=mb, n_prims=n_prims, exact_flavour=ef)
        yield req


@pytest.fixture(scope="module")
def space(vt):
    """[(request, (family, row))]"""
    return [(req, select(vt, **req)) for req in requests()]


def test_exact_flavour_has_no_fast_stepper_lensed_kernels(vt):
    fast, exact = rows(vt, False), rows(vt, True)
    for f, e in zip(fast, exact):
        lens, ex = f[0], f[1]
        assert e[5] == (0 if lens and not ex else f[5])
    compiled = lambda rs: sum(bin(r[5]).count("1") for r in rs)   # kernels instantiated from the table
    assert (compiled(fast), compiled(exact)) == (58, 36)


def test_every_compiled_variant_is_reachable(vt, space):
    for ef in (False, True):
        chosen = {(row, fam) for req, (fam, row) in space if req["exact_flavour"] == ef and row is not None}
        table = rows(vt, ef)
        compiled = {(i, f) for i, r in enumerate(table) for f in FAMILIES if r[5] & f}
        assert chosen <= compiled
        assert compiled - chosen == set(), f"dead variants in the {'exact' if ef else 'fast'} flavour"


def test_row_matches_the_request(vt, space):
    tables = {ef: rows(vt, ef) for ef in (False, True)}
    for req, (fam, row) in space:
        if row is None:
            continue
        lens, exact, nl, bvh, c, fams = tables[req["exact_flavour"]][row]
        ct = req["content"] | (CT_AOV if req["output"] else 0)
        assert fams & fam and lens == (req["n_lens"] != 0) and bvh == req["bvh"] and (ct & ~c) == 0, req
        assert nl in (0, req["n_lens"]) and (not lens or exact == req["lens_exact"]), req


def test_only_pool_counters_can_be_unsupported(space):
    for req, (fam, row) in space:
        if req["mode"] != POOL_COUNTERS:
            assert row is not None, req


def test_pool_counters_unsupported_for_bvh_scenes_and_beyond_the_pool_limits(vt, space):
    for req, (fam, row) in space:
        if req["mode"] != POOL_COUNTERS:
            continue
        outside = req["pool_w"] == 0 or req["max_bounces"] > POOL_MAX_BOUNCES or (req["n_prims"] > POOL_MAX_OBJECTS and not req["bvh"])
        if req["bvh"] or outside:
            assert row is None, req
        else:
            assert fam == V_POOL_STATS
    # ... and served for the shipped lensed workloads
    assert select(vt, CT_SPHERES | CT_METAL | CT_GLASS, n_lens=1, mode=POOL_COUNTERS, pool_w=4)[1] is not None
    assert select(vt, CT_SPHERES | CT_VOLUMES, n_lens=1, lens_exact=1, mode=POOL_COUNTERS, pool_w=4, exact_flavour=True)[1] is not None


def variant(vt, fam_row, exact_flavour=False):
    fam, row = fam_row
    return fam, rows(vt, exact_flavour)[row][:5]


def test_shipped_workloads(vt):
    SMG, SV = CT_SPHERES | CT_METAL | CT_GLASS, CT_SPHERES | CT_VOLUMES
    # C1 cornell, C2 cornell2: flat fields run the lane kernel (pool_w defaults to 0 there)
    assert variant(vt, select(vt, CT_RECTS)) == (V_LANE, (0, 0, 0, 0, CT_RECTS))
    assert variant(vt, select(vt, CT_RECTS | CT_METAL)) == (V_LANE, (0, 0, 0, 0, CT_RECTS | CT_METAL))
    # C3 / C5: scene + one mass, pooled
    assert variant(vt, select(vt, SMG, n_lens=1, pool_w=4)) == (V_POOL, (1, 0, 1, 0, SMG))
    # C4-cloud, C4-cloud-lens: volumetric, so the exact flavour and (lensed) the exact stepper
    assert variant(vt, select(vt, SV, exact_flavour=True), True) == (V_LANE, (0, 0, 0, 0, SV))
    assert variant(vt, select(vt, SV, n_lens=1, lens_exact=1, pool_w=4, exact_flavour=True), True) == (V_POOL, (1, 1, 1, 0, SV))
    # a flat scene above 64 primitives gets a BVH and the pooled traversal
    assert variant(vt, select(vt, SMG | CT_RECTS, bvh=True, pool_w=3, n_prims=422)) == (V_POOL_BVH, (0, 0, 0, 1, CT_ALL & ~CT_CUBOID_LIGHT))
