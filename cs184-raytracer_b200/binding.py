"""ctypes bindings over the two product libraries.

* ``lib/librt_b200.so``  — the CUDA trace loop behind the C ABI of ``include/rt_b200.h``
  (replaces Scene::renderScene/traceRay/castRay, reference src/scene.cpp:10-167 and
  src/geometry.cpp:5-126).
* ``lib/libas2host.so``  — the C++ host (parsers, object model, flattening, PNG writer,
  synthetic scene), reference src/parsers.cpp, src/scene.h, src/writers.cpp.

There is deliberately NO fallback here: if the libraries are missing or no B200 is
present the calls raise.  Nothing in this module touches ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_DIR = Path(os.environ.get("RT_B200_LIB_DIR", PKG_DIR / "lib"))   # override: A/B builds during development

RT_OK = 0
RT_GEOM_SPHERE, RT_GEOM_TRI, RT_GEOM_MESH = 0, 1, 2
RT_LIGHT_AMBIENT, RT_LIGHT_POINT, RT_LIGHT_DIRECTIONAL = 0, 1, 2
RT_FLAG_BRUTE_FORCE = 1
RT_FLAG_COUNT_WORK = 2
RT_FLAG_TIME_KERNELS = 4
RT_FLAG_SERIAL = 8
RT_FLAG_FULL_FRAME = 16
RT_SCENE_FACES_ON_DEVICE = 1
RT_ERR_LIMIT = -6
RT_TILE_PIXELS = int(os.environ.get("RT_B200_TILE", "32")) ** 2    # must match the library build (include/rt_b200.h)


class rt_material(C.Structure):
    _fields_ = [("ka", C.c_double * 3), ("kd", C.c_double * 3), ("ks", C.c_double * 3), ("kr", C.c_double * 3),
                ("kt", C.c_double * 3), ("sp", C.c_double), ("ior", C.c_double), ("reserved_", C.c_double)]


class rt_geometry(C.Structure):
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("first_face", C.c_int64), ("num_faces", C.c_int64),
                ("fwd", C.c_double * 12), ("inv", C.c_double * 12), ("det", C.c_double), ("center", C.c_double * 3),
                ("radius", C.c_double), ("radius2", C.c_double), ("bbmin", C.c_double * 3), ("bbmax", C.c_double * 3),
                ("use_bbox", C.c_int32), ("reserved_", C.c_int32)]


class rt_light(C.Structure):
    _fields_ = [("type", C.c_int32), ("reserved_", C.c_int32), ("v", C.c_double * 3), ("color", C.c_double * 3),
                ("falloff", C.c_double)]


class rt_camera(C.Structure):
    _fields_ = [("eye", C.c_double * 3), ("ll", C.c_double * 3), ("lr", C.c_double * 3), ("ul", C.c_double * 3),
                ("ur", C.c_double * 3)]


class rt_scene(C.Structure):
    _fields_ = [("camera", rt_camera), ("num_geometries", C.c_int32), ("num_materials", C.c_int32),
                ("num_lights", C.c_int32), ("flags", C.c_uint32), ("num_faces", C.c_int64),
                ("geometries", C.POINTER(rt_geometry)), ("materials", C.POINTER(rt_material)),
                ("lights", C.POINTER(rt_light)), ("face_points", C.POINTER(C.c_double)),
                ("face_normals", C.POINTER(C.c_double))]


class rt_params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("bounce_depth", C.c_int32),
                ("intersection_only", C.c_int32), ("tile_rank", C.c_int32), ("tile_world", C.c_int32),
                ("flags", C.c_uint32), ("samples", C.c_int32), ("n_gpus", C.c_int32), ("reserved_", C.c_int32 * 3)]


class rt_stats(C.Structure):
    _fields_ = [("rays_primary", C.c_uint64), ("rays_shadow", C.c_uint64), ("rays_secondary", C.c_uint64),
                ("degenerate_rays", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("nodes_fetched", C.c_uint64 * 2), ("tris_tested", C.c_uint64 * 2), ("spheres_tested", C.c_uint64 * 2),
                ("hits", C.c_uint64), ("ms_kernel", C.c_double * 4), ("launches_kernel", C.c_uint64 * 4),
                ("ms_upload", C.c_double), ("ms_build", C.c_double), ("ms_trace", C.c_double),
                ("ms_readback", C.c_double), ("scene_bytes_h2d", C.c_uint64), ("shadow_rays_culled", C.c_uint64)]

    def as_dict(self):
        out = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            out[name] = list(v) if hasattr(v, "__len__") else v
        return out


# symbols include/rt_b200.h declares (checked by tests/test_abi_exports.py)
RT_SYMBOLS = [
    "rt_create", "rt_destroy", "rt_last_error", "rt_abi_version", "rt_scene_upload", "rt_render", "rt_render_rgb8",
    "rt_render_device", "rt_render_device_rgb8", "rt_tile_count", "rt_tile_count_total", "rt_tile_count_max",
    "rt_unpack_tiles_rgb8", "rt_unpack_tiles", "rt_primary_ids", "rt_cast_rays", "rt_get_stats",
    "rt_microbench_gather", "rt_scene_device_bytes", "rt_intersection_max", "rt_divide_device",
    "rt_shared_frame_create", "rt_shared_frame_open", "rt_shared_frame_close", "rt_microbench_node_walk",
    "rt_scene_refit",
]

_rt = None
_host = None


class RtError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def load_rt() -> C.CDLL:
    """Load librt_b200.so (fails loudly when it has not been built)."""
    global _rt
    if _rt is None:
        path = LIB_DIR / "librt_b200.so"
        if not path.exists():
            raise RtError(f"{path} is missing: run __graft_entry__.build() (there is no CPU fallback)")
        lib = C.CDLL(str(path))
        lib.rt_last_error.restype = C.c_char_p
        lib.rt_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.rt_destroy.argtypes = [C.c_void_p]
        lib.rt_scene_upload.argtypes = [C.c_void_p, C.c_void_p]
        lib.rt_scene_refit.argtypes = [C.c_void_p, C.c_void_p]
        lib.rt_render.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_render_rgb8.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_render_device.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p]
        lib.rt_render_device_rgb8.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p]
        for name in ("rt_tile_count", "rt_tile_count_total", "rt_tile_count_max"):
            getattr(lib, name).restype = C.c_int64
            getattr(lib, name).argtypes = [C.POINTER(rt_params)]
        lib.rt_unpack_tiles_rgb8.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_unpack_tiles.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_primary_ids.argtypes = [C.c_void_p, C.POINTER(rt_params), C.c_void_p, C.c_void_p]
        lib.rt_cast_rays.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.rt_get_stats.argtypes = [C.c_void_p, C.POINTER(rt_stats)]
        lib.rt_microbench_gather.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_double)]
        lib.rt_intersection_max.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        lib.rt_divide_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p]
        lib.rt_scene_device_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        lib.rt_shared_frame_create.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.c_char_p]
        lib.rt_shared_frame_open.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]
        lib.rt_shared_frame_close.argtypes = [C.c_void_p, C.c_void_p]
        lib.rt_microbench_node_walk.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        _rt = lib
    return _rt


def load_host() -> C.CDLL:
    global _host
    if _host is None:
        load_rt()
        path = LIB_DIR / "libas2host.so"
        if not path.exists():
            raise RtError(f"{path} is missing: run __graft_entry__.build()")
        lib = C.CDLL(str(path))
        lib.as2_scene_load.restype = C.c_void_p
        lib.as2_scene_load.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_char_p, C.c_int]
        lib.as2_scene_synthetic.restype = C.c_void_p
        lib.as2_scene_synthetic.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_char_p, C.c_int]
        lib.as2_write_synthetic.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_uint64, C.c_char_p, C.c_int]
        lib.as2_scene_free.argtypes = [C.c_void_p]
        lib.as2_scene_flatten.restype = C.POINTER(rt_scene)
        lib.as2_scene_flatten.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        lib.as2_scene_render.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_int]
        lib.as2_write_png_rgb8.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_int]
        lib.as2_write_png_f64.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_int]
        lib.as2_quantize_rgb8.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        lib.as2_encode_png_rgb8.restype = C.c_int64
        lib.as2_encode_png_rgb8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                            C.POINTER(C.c_int64), C.c_char_p, C.c_int]
        _host = lib
    return _host


class HostScene:
    """A scene held by the C++ host: parsed from .rti files or generated."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)
        self._flat = None

    @classmethod
    def load(cls, *files) -> "HostScene":
        lib = load_host()
        arr = (C.c_char_p * len(files))(*[os.fsencode(str(f)) for f in files])
        err = C.create_string_buffer(512)
        h = lib.as2_scene_load(arr, len(files), err, 512)
        if not h:
            raise RtError(err.value.decode())
        return cls(h)

    @classmethod
    def synthetic(cls, grid_cells=708, num_spheres=1000, seed=184) -> "HostScene":
        lib = load_host()
        err = C.create_string_buffer(512)
        h = lib.as2_scene_synthetic(grid_cells, num_spheres, seed, err, 512)
        if not h:
            raise RtError(err.value.decode())
        return cls(h)

    @property
    def flat(self):
        """POINTER(rt_scene) owned by the host scene."""
        if self._flat is None:
            err = C.create_string_buffer(512)
            p = load_host().as2_scene_flatten(self._h, err, 512)
            if not p:
                raise RtError(err.value.decode())
            p._owner = self          # the descriptor points into memory owned by this scene
            self._flat = p
        return self._flat

    def render(self, width, height, bounce_depth=10, intersection_only=False) -> np.ndarray:
        """Scene::renderScene through the C++ host (what a user of the reference calls)."""
        out = np.empty((height, width, 3), dtype=np.float64)
        err = C.create_string_buffer(512)
        rc = load_host().as2_scene_render(self._h, width, height, bounce_depth, int(intersection_only), _ptr(out), err, 512)
        if rc != 0:
            raise RtError(err.value.decode())
        return out

    def close(self):
        if self._h:
            load_host().as2_scene_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def flat_arrays(flat) -> dict:
    """Copy an rt_scene (POINTER or void*) into numpy arrays for comparisons."""
    s = C.cast(flat, C.POINTER(rt_scene)).contents
    def arr(ptr, n, typ):
        if n == 0:
            return np.zeros(0, dtype=np.uint8)
        return np.frombuffer(C.string_at(ptr, n * C.sizeof(typ)), dtype=np.uint8).copy()
    nf = s.num_faces
    return {
        "camera": np.frombuffer(bytes(s.camera), dtype=np.float64).copy(),
        "num_geometries": s.num_geometries, "num_lights": s.num_lights, "num_faces": nf,
        "geometries": arr(s.geometries, s.num_geometries, rt_geometry),
        "materials": arr(s.materials, s.num_materials, rt_material),
        "lights": arr(s.lights, s.num_lights, rt_light),
        "face_points": np.frombuffer(C.string_at(s.face_points, nf * 72), dtype=np.float64).copy() if nf else np.zeros(0),
        "face_normals": np.frombuffer(C.string_at(s.face_normals, nf * 72), dtype=np.float64).copy() if nf else np.zeros(0),
    }


def make_params(width, height, bounce_depth=10, intersection_only=False, tile_rank=0, tile_world=1, flags=0,
                samples=0, n_gpus=0) -> rt_params:
    p = rt_params()
    p.samples = int(samples)
    p.n_gpus = int(n_gpus)
    p.width, p.height, p.bounce_depth = int(width), int(height), int(bounce_depth)
    p.intersection_only = int(bool(intersection_only))
    p.tile_rank, p.tile_world, p.flags = int(tile_rank), int(tile_world), int(flags)
    return p


class Renderer:
    """Thin object wrapper over the C ABI (one rt_context)."""

    def __init__(self, device: int = -1):
        self.lib = load_rt()
        h = C.c_void_p()
        rc = self.lib.rt_create(device, C.byref(h))
        if rc != RT_OK:
            raise RtError(f"rt_create failed ({rc}): {self.lib.rt_last_error().decode()}")
        self._h = h
        self._scene_keepalive = None

    def _check(self, rc, what):
        if rc != RT_OK:
            raise RtError(f"{what} failed ({rc}): {self.lib.rt_last_error().decode()}")

    def upload(self, scene):
        """scene: HostScene, or a POINTER(rt_scene)/void* to a flat descriptor."""
        flat = scene.flat if isinstance(scene, HostScene) else scene
        self._scene_keepalive = scene
        self._check(self.lib.rt_scene_upload(self._h, C.cast(flat, C.c_void_p)), "rt_scene_upload")

    def refit(self, scene):
        """Update the uploaded scene to `scene` (HostScene or flat descriptor of the same structure) and refit the
        LBVH instead of rebuilding it (rt_scene_refit)."""
        flat = scene.flat if isinstance(scene, HostScene) else scene
        self._check(self.lib.rt_scene_refit(self._h, C.cast(flat, C.c_void_p)), "rt_scene_refit")
        self._scene_keepalive = scene

    def render(self, width, height, bounce_depth=10, intersection_only=False, flags=0, samples=0, n_gpus=0) -> np.ndarray:
        p = make_params(width, height, bounce_depth, intersection_only, flags=flags, samples=samples, n_gpus=n_gpus)
        out = np.empty((height, width, 3), dtype=np.float64)
        self._check(self.lib.rt_render(self._h, C.byref(p), _ptr(out), None, None), "rt_render")
        return out

    def render_rgb8(self, width, height, bounce_depth=10, intersection_only=False, flags=0, out=None, n_gpus=0) -> np.ndarray:
        p = make_params(width, height, bounce_depth, intersection_only, flags=flags, n_gpus=n_gpus)
        if out is None:
            out = np.empty((height, width, 3), dtype=np.uint8)
        self._check(self.lib.rt_render_rgb8(self._h, C.byref(p), _ptr(out), None, None), "rt_render_rgb8")
        return out

    def render_device(self, params: rt_params, d_out_ptr: int, rgb8=False, stream: int = 0):
        fn = self.lib.rt_render_device_rgb8 if rgb8 else self.lib.rt_render_device
        self._check(fn(self._h, C.byref(params), C.c_void_p(d_out_ptr), C.c_void_p(stream)), "rt_render_device")

    def unpack_tiles(self, params: rt_params, d_packed_ptr: int, d_frame_ptr: int, rgb8=False, stream: int = 0):
        fn = self.lib.rt_unpack_tiles_rgb8 if rgb8 else self.lib.rt_unpack_tiles
        self._check(fn(self._h, C.byref(params), C.c_void_p(d_packed_ptr), C.c_void_p(d_frame_ptr), C.c_void_p(stream)),
                    "rt_unpack_tiles")

    def primary_ids(self, width, height, flags=0):
        p = make_params(width, height, 0, flags=flags)
        g = np.empty((height, width), dtype=np.int32)
        f = np.empty((height, width), dtype=np.int32)
        self._check(self.lib.rt_primary_ids(self._h, C.byref(p), _ptr(g), _ptr(f)), "rt_primary_ids")
        return g, f

    def cast_rays(self, org, direction, reverse=None, flags=0):
        org = np.ascontiguousarray(org, dtype=np.float64)
        direction = np.ascontiguousarray(direction, dtype=np.float64)
        n = org.shape[0]
        rev = None if reverse is None else np.ascontiguousarray(reverse, dtype=np.uint8)
        geom = np.empty(n, np.int32); face = np.empty(n, np.int32); dist = np.empty(n)
        point = np.empty((n, 3)); normal = np.empty((n, 3))
        self._check(self.lib.rt_cast_rays(self._h, n, _ptr(org), _ptr(direction), _ptr(rev), flags, _ptr(geom), _ptr(face),
                                          _ptr(dist), _ptr(point), _ptr(normal)), "rt_cast_rays")
        return geom, face, dist, point, normal

    def render_host_params(self, params: rt_params, host_ptr: int, rgb8=True):
        """rt_render / rt_render_rgb8 with explicit params and a raw host pointer (pinned or shared memory)."""
        fn = self.lib.rt_render_rgb8 if rgb8 else self.lib.rt_render
        self._check(fn(self._h, C.byref(params), C.c_void_p(host_ptr), None, None), "rt_render")

    def shared_frame_create(self, nbytes: int):
        """-> (device pointer, 64-byte handle) of a frame other processes can open (CUDA IPC)."""
        ptr = C.c_void_p()
        handle = C.create_string_buffer(64)
        self._check(self.lib.rt_shared_frame_create(self._h, int(nbytes), C.byref(ptr), handle), "rt_shared_frame_create")
        return int(ptr.value), handle.raw

    def shared_frame_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        self._check(self.lib.rt_shared_frame_open(self._h, C.create_string_buffer(bytes(handle), 64), C.byref(ptr)),
                    "rt_shared_frame_open")
        return int(ptr.value)

    def shared_frame_close(self, ptr: int):
        self._check(self.lib.rt_shared_frame_close(self._h, C.c_void_p(ptr)), "rt_shared_frame_close")

    def microbench_node_walk(self, lanes=32, visits=64):
        """-> (wide-node visits per second, bytes per second through the LSU) of the node-walk ceiling probe."""
        v, b = C.c_double(), C.c_double()
        self._check(self.lib.rt_microbench_node_walk(self._h, int(lanes), int(visits), C.byref(v), C.byref(b)),
                    "rt_microbench_node_walk")
        return float(v.value), float(b.value)

    def intersection_max(self) -> float:
        v = C.c_double()
        self._check(self.lib.rt_intersection_max(self._h, C.byref(v)), "rt_intersection_max")
        return float(v.value)

    def divide_device(self, d_ptr: int, count: int, divisor: float, stream: int = 0):
        self._check(self.lib.rt_divide_device(self._h, C.c_void_p(d_ptr), int(count), float(divisor), C.c_void_p(stream)),
                    "rt_divide_device")

    def device_bytes(self):
        a, b = C.c_uint64(), C.c_uint64()
        self._check(self.lib.rt_scene_device_bytes(self._h, C.byref(a), C.byref(b)), "rt_scene_device_bytes")
        return int(a.value), int(b.value)

    def microbench_gather(self, array_bytes, loads_per_thread=64) -> float:
        g = C.c_double()
        self._check(self.lib.rt_microbench_gather(self._h, int(array_bytes), int(loads_per_thread), C.byref(g)),
                    "rt_microbench_gather")
        return float(g.value)

    def stats(self) -> dict:
        st = rt_stats()
        self._check(self.lib.rt_get_stats(self._h, C.byref(st)), "rt_get_stats")
        return st.as_dict()

    def close(self):
        if getattr(self, "_h", None):
            self.lib.rt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def tile_counts(params: rt_params):
    lib = load_rt()
    return (int(lib.rt_tile_count(C.byref(params))), int(lib.rt_tile_count_max(C.byref(params))),
            int(lib.rt_tile_count_total(C.byref(params))))


def quantize_rgb8(rgb: np.ndarray) -> np.ndarray:
    """The PNG writer's quantisation (reference src/writers.cpp:7), host implementation."""
    rgb = np.ascontiguousarray(rgb, dtype=np.float64)
    out = np.empty(rgb.shape, dtype=np.uint8)
    load_host().as2_quantize_rgb8(_ptr(rgb), rgb.size, _ptr(out))
    return out


def encode_png(rgb8: np.ndarray, threads: int = 1) -> bytes:
    """The PNG file image the host writer produces, with the deflate work cut into `threads` stripes."""
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    h, w = rgb8.shape[0], rgb8.shape[1]
    cap = int(rgb8.size * 1.01) + (1 << 16)
    out = np.empty(cap, dtype=np.uint8)
    need = C.c_int64(0)
    err = C.create_string_buffer(512)
    n = load_host().as2_encode_png_rgb8(_ptr(rgb8), w, h, threads, _ptr(out), cap, C.byref(need), err, 512)
    if n == -2:
        out = np.empty(need.value, dtype=np.uint8)
        n = load_host().as2_encode_png_rgb8(_ptr(rgb8), w, h, threads, _ptr(out), need.value, C.byref(need), err, 512)
    if n < 0:
        raise RtError(err.value.decode())
    return out[:n].tobytes()


def write_png(path, rgb8: np.ndarray):
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    err = C.create_string_buffer(512)
    if load_host().as2_write_png_rgb8(os.fsencode(str(path)), _ptr(rgb8), rgb8.shape[1], rgb8.shape[0], err, 512) != 0:
        raise RtError(err.value.decode())
