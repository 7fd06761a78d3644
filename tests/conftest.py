"""Shared test plumbing.

Markers: ``gpu`` = needs a B200 (run by the driver with ``-m gpu``); everything else runs
on CPU.  The product package lives in a directory with a hyphen, so it is imported through
importlib under the module name ``cs184_raytracer_b200``.  Only tests (and bench/smoke)
touch ``oracle/``; the product never does.
"""
import ctypes as C
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
PKG_DIR = ROOT / "cs184-raytracer_b200"
ORACLE_DIR = ROOT / "oracle"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200)")
    config.addinivalue_line("markers", "slow: long-running CPU test")


def load_package():
    name = "cs184_raytracer_b200"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, PKG_DIR / "__init__.py", submodule_search_locations=[str(PKG_DIR)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def _ensure_built():
    """Build product + oracle libraries if a fresh checkout has none (CPU box: nvcc cross-compiles)."""
    need = [PKG_DIR / "lib" / "librt_b200.so", PKG_DIR / "lib" / "libas2host.so", ORACLE_DIR / "liboracle.so"]
    if all(p.exists() for p in need):
        return
    sys.path.insert(0, str(ROOT))
    import __graft_entry__
    __graft_entry__.build()


@pytest.fixture(scope="session")
def pkg():
    _ensure_built()
    return load_package()


class Oracle:
    """ctypes view of oracle/liboracle.so (the plain-C restatement)."""

    def __init__(self):
        self.lib = C.CDLL(str(ORACLE_DIR / "liboracle.so"))

    def render(self, flat, width, height, depth=10, intersection_only=False, threads=8, ids=True, samples=0):
        pkg = load_package()
        p = pkg.make_params(width, height, depth, intersection_only, samples=samples)
        rgb = np.zeros((height, width, 3))
        geom = np.zeros((height, width), np.int32) if ids else None
        face = np.zeros((height, width), np.int32) if ids else None
        counts = (C.c_uint64 * 4)()
        self.lib.oracle_render(C.cast(flat, C.c_void_p), C.byref(p), rgb.ctypes.data_as(C.c_void_p),
                               geom.ctypes.data_as(C.c_void_p) if ids else None,
                               face.ctypes.data_as(C.c_void_p) if ids else None, counts, threads)
        return rgb, geom, face, [int(c) for c in counts]

    def cast_rays(self, flat, org, direction, reverse=None):
        org = np.ascontiguousarray(org, np.float64)
        direction = np.ascontiguousarray(direction, np.float64)
        n = org.shape[0]
        rev = None if reverse is None else np.ascontiguousarray(reverse, np.uint8)
        geom = np.zeros(n, np.int32); face = np.zeros(n, np.int32); dist = np.zeros(n)
        point = np.zeros((n, 3)); normal = np.zeros((n, 3))
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        self.lib.oracle_cast_rays(C.cast(flat, C.c_void_p), C.c_int64(n), vp(org), vp(direction), vp(rev), vp(geom), vp(face),
                                  vp(dist), vp(point), vp(normal))
        return geom, face, dist, point, normal

    def trace_rays(self, flat, org, direction, depth=10, from_inside=None):
        org = np.ascontiguousarray(org, np.float64)
        direction = np.ascontiguousarray(direction, np.float64)
        n = org.shape[0]
        fi = None if from_inside is None else np.ascontiguousarray(from_inside, np.uint8)
        rgb = np.zeros((n, 3))
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        self.lib.oracle_trace_rays(C.cast(flat, C.c_void_p), C.c_int64(n), vp(org), vp(direction), depth, vp(fi), vp(rgb))
        return rgb

    def camera_rays(self, flat, width, height, pix):
        pix = np.ascontiguousarray(pix, np.int64)
        n = pix.shape[0]
        org = np.zeros((n, 3)); direction = np.zeros((n, 3))
        self.lib.oracle_camera_rays(C.cast(flat, C.c_void_p), width, height, C.c_int64(n), pix.ctypes.data_as(C.c_void_p),
                                    org.ctypes.data_as(C.c_void_p), direction.ctypes.data_as(C.c_void_p))
        return org, direction


class Reference:
    """ctypes view of oracle/_ref/libref.so: the UNMODIFIED reference hot path + our C shim."""

    def __init__(self, counting=False):
        path = ORACLE_DIR / "_ref" / ("libref_count.so" if counting else "libref.so")
        self.lib = C.CDLL(str(path))
        self.lib.ref_scene_load.restype = C.c_void_p
        self.lib.ref_scene_load.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_char_p, C.c_int]
        self.lib.ref_scene_flatten.restype = C.c_void_p
        self.lib.ref_scene_flatten.argtypes = [C.c_void_p]

    @staticmethod
    def available():
        return (ORACLE_DIR / "_ref" / "libref.so").exists()

    def load(self, *files):
        arr = (C.c_char_p * len(files))(*[str(f).encode() for f in files])
        err = C.create_string_buffer(512)
        h = self.lib.ref_scene_load(arr, len(files), err, 512)
        if not h:
            raise RuntimeError(err.value.decode())
        return C.c_void_p(h)

    def flatten(self, h):
        return C.c_void_p(self.lib.ref_scene_flatten(h))

    def render(self, h, width, height, depth=10, intersection_only=False, threads=8, ids=False, stock=False):
        rgb = np.zeros((height, width, 3))
        geom = np.zeros((height, width), np.int32) if ids else None
        sec = C.c_double(); calls = C.c_uint64()
        if stock:
            rc = self.lib.ref_render_stock(h, width, height, depth, int(intersection_only), threads, rgb.ctypes.data_as(C.c_void_p))
            assert rc == 0
        else:
            self.lib.ref_render(h, width, height, depth, int(intersection_only), threads, rgb.ctypes.data_as(C.c_void_p),
                                geom.ctypes.data_as(C.c_void_p) if ids else None, C.byref(sec), C.byref(calls))
        return rgb, geom, sec.value, int(calls.value)

    def cast_rays(self, h, org, direction, reverse=None):
        org = np.ascontiguousarray(org, np.float64)
        direction = np.ascontiguousarray(direction, np.float64)
        n = org.shape[0]
        rev = None if reverse is None else np.ascontiguousarray(reverse, np.uint8)
        geom = np.zeros(n, np.int32); dist = np.zeros(n); point = np.zeros((n, 3)); normal = np.zeros((n, 3))
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        self.lib.ref_cast_rays(h, C.c_int64(n), vp(org), vp(direction), vp(rev), vp(geom), vp(dist), vp(point), vp(normal))
        return geom, dist, point, normal

    def trace_rays(self, h, org, direction, depth=10, from_inside=None):
        org = np.ascontiguousarray(org, np.float64)
        direction = np.ascontiguousarray(direction, np.float64)
        n = org.shape[0]
        fi = None if from_inside is None else np.ascontiguousarray(from_inside, np.uint8)
        rgb = np.zeros((n, 3))
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        self.lib.ref_trace_rays(h, C.c_int64(n), vp(org), vp(direction), depth, vp(fi), vp(rgb))
        return rgb


@pytest.fixture(scope="session")
def oracle(pkg):
    return Oracle()


@pytest.fixture(scope="session")
def reference():
    if not Reference.available():
        pytest.skip("oracle/_ref/libref.so not built (needs the reference sources at build time, oracle/Makefile REF=)")
    return Reference()


@pytest.fixture(scope="session")
def live_reference():
    """The live reference where oracle/_ref is built, else None: for tests whose checks stand without it and that
    also compare with it when they can."""
    return Reference() if Reference.available() else None


@pytest.fixture(scope="session")
def manifest():
    return json.loads((GOLDEN / "ref" / "MANIFEST.json").read_text())


def scene_path(rel):
    return GOLDEN / rel


def load_ref_fixture(name, w, h):
    return np.load(GOLDEN / "ref" / f"{name}_{w}x{h}.npz")


def decode_png(path):
    from PIL import Image
    return np.array(Image.open(path).convert("RGB"))


def quantize(rgb):
    """(uint8)(clamp(v,0,1)*255.0), truncating — reference src/writers.cpp:7 restated in numpy."""
    v = np.where(1.0 < rgb, 1.0, rgb)
    v = np.where(v < 0.0, 0.0, v)
    v = np.where(np.isnan(v), 0.0, v)
    return (v * 255.0).astype(np.uint8)


@pytest.fixture(scope="session")
def gpu_renderer(pkg):
    r = pkg.Renderer(0)
    yield r
    r.close()
