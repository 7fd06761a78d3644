"""rt_scene_refit: update an uploaded scene's geometry, faces, camera, lights and materials, and refit its LBVH.

The refit keeps the tree's topology and recomputes every box from the new primitives, padded for the new largest
|coordinate| M.  The tree only culls, so a refit scene must render exactly what a fresh upload of the same scene
renders and what the FP64 oracle renders: primary geometry and face ids and per-class ray counts equal, the FP64
frame within 1e-9 (FP64 atomics), rt_cast_rays bit for bit.  A refit of the unchanged scene rewrites the node array
byte for byte, which shows as exactly the same counted work (RT_FLAG_COUNT_WORK)."""
import ctypes as C
import re

import numpy as np
import pytest

from conftest import GOLDEN, scene_path
from test_gpu_far_coordinates import assert_cast_rays_match, cluster, load, moved, offset, unit

FP64_TOL = 1e-9
RT_ERR_INVALID, RT_ERR_NO_SCENE = -1, -4
INPUT02 = (GOLDEN / "inputs" / "input-02.rti").read_text()
TEAPOT = scene_path("inputs/teapot.obj")
SMALL_SYNTH = (60, 300)          # 7200 terrain faces + 300 spheres: two LBVH groups under a super node


# ---- descriptors ------------------------------------------------------------------------------------------------

class Desc:
    """A private copy of an rt_scene whose arrays can be edited; keeps what it points into alive."""

    def __init__(self, pkg, flat, keep=None):
        s = C.cast(flat, C.POINTER(pkg.rt_scene)).contents
        self.pkg, self.keep = pkg, [keep, flat]
        self.d = pkg.rt_scene.from_buffer_copy(s)
        ng, nl = s.num_geometries, s.num_lights
        self.geoms = (pkg.binding.rt_geometry * ng).from_buffer_copy(C.string_at(s.geometries, ng * C.sizeof(pkg.binding.rt_geometry)))
        self.lights = (pkg.binding.rt_light * nl).from_buffer_copy(C.string_at(s.lights, nl * C.sizeof(pkg.binding.rt_light)))
        self.d.geometries = C.cast(self.geoms, C.POINTER(pkg.binding.rt_geometry))
        self.d.lights = C.cast(self.lights, C.POINTER(pkg.binding.rt_light))

    @property
    def ptr(self):
        return C.pointer(self.d)

    def without_faces(self):
        self.d.face_points = None
        self.d.face_normals = None
        return self

    def with_faces(self, pts, nrm, on_device=False):
        """pts / nrm: float64 arrays [num_faces, 3, 3] (numpy, or CUDA torch tensors with on_device)."""
        self.keep += [pts, nrm]
        if on_device:
            self.d.face_points = C.cast(C.c_void_p(pts.data_ptr()), C.POINTER(C.c_double))
            self.d.face_normals = C.cast(C.c_void_p(nrm.data_ptr()), C.POINTER(C.c_double))
            self.d.flags |= self.pkg.RT_SCENE_FACES_ON_DEVICE
        else:
            self.d.face_points = pts.ctypes.data_as(C.POINTER(C.c_double))
            self.d.face_normals = nrm.ctypes.data_as(C.POINTER(C.c_double))
        return self

    def translate(self, t):
        """Every geometry, the camera and the point lights moved by t (only fwd / inv change)."""
        t = np.asarray(t, np.float64)
        for g in self.geoms:
            fwd = np.array(g.fwd).reshape(3, 4)
            inv = np.array(g.inv).reshape(3, 4)
            fwd[:, 3] += t
            inv[:, 3] -= inv[:, :3] @ t
            g.fwd[:] = list(fwd.ravel())
            g.inv[:] = list(inv.ravel())
        for name in ("eye", "ll", "lr", "ul", "ur"):
            getattr(self.d.camera, name)[:] = list(np.array(getattr(self.d.camera, name)) + t)
        for k in range(self.d.num_lights):
            if self.lights[k].type == self.pkg.binding.RT_LIGHT_POINT:
                self.lights[k].v[:] = list(np.array(self.lights[k].v) + t)
        return self


def face_arrays(pkg, flat):
    a = pkg.flat_arrays(flat)
    return a["face_points"].reshape(-1, 3, 3).copy(), a["face_normals"].reshape(-1, 3, 3).copy()


def structure(pkg, flat):
    s = C.cast(flat, C.POINTER(pkg.rt_scene)).contents
    return s.num_faces, [(s.geometries[i].type, s.geometries[i].first_face, s.geometries[i].num_faces)
                         for i in range(s.num_geometries)]


# ---- what "equal" means -----------------------------------------------------------------------------------------

def camera_rays(oracle, flat, n=6000, seed=5):
    """Rays from around the camera through the frame, with jittered directions."""
    rng = np.random.default_rng(seed)
    org, d = oracle.camera_rays(flat, 64, 48, np.arange(64 * 48))
    k = rng.integers(0, len(org), n)
    d = d[k] + rng.normal(scale=0.02, size=(n, 3)) * np.linalg.norm(d[k], axis=1)[:, None]
    return org[k], d


def snapshot(pkg, r, w, h, depth, rays, flags=0):
    """Everything a render and rt_cast_rays show of the scene on the device."""
    rgb = r.render(w, h, depth, flags=flags | pkg.RT_FLAG_COUNT_WORK)
    st = r.stats()
    geom, face = r.primary_ids(w, h, flags=flags)
    cast = r.cast_rays(rays[0], rays[1], flags=flags)
    work = [list(st["nodes_fetched"]), list(st["tris_tested"]), list(st["spheres_tested"])]
    return {"rgb": rgb, "geom": geom, "face": face, "rays": [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]],
            "work": work, "cast": cast}


def assert_same(a, b, what, work=False):
    assert np.array_equal(a["geom"], b["geom"]), f"{what}: {int((a['geom'] != b['geom']).sum())} primary geometry ids differ"
    assert np.array_equal(a["face"], b["face"]), f"{what}: primary face ids differ"
    assert a["rays"] == b["rays"], f"{what}: ray counts {a['rays']} != {b['rays']}"
    err = float(np.abs(a["rgb"] - b["rgb"]).max())
    assert err <= FP64_TOL, f"{what}: frames differ by {err}"
    for k, (x, y) in enumerate(zip(a["cast"], b["cast"])):
        assert np.array_equal(x, y), f"{what}: rt_cast_rays output {k} differs"
    if work:
        assert a["work"] == b["work"], f"{what}: counted work {a['work']} != {b['work']}"


def assert_oracle(pkg, r, oracle, flat, w, h, depth):
    """BVH and brute force both equal the oracle (ids, ray counts, FP64 frame)."""
    o_rgb, o_geom, o_face, counts = oracle.render(flat, w, h, depth)
    for flags in (0, pkg.RT_FLAG_BRUTE_FORCE):
        rgb = r.render(w, h, depth, flags=flags)
        st = r.stats()
        geom, face = r.primary_ids(w, h, flags=flags)
        assert np.array_equal(geom, o_geom), f"flags {flags}: {int((geom != o_geom).sum())} primary geometry ids differ"
        assert np.array_equal(face, o_face), f"flags {flags}: primary face ids differ"
        got = [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]]
        assert got == counts[:3], f"flags {flags}: ray counts {got} != oracle {counts[:3]}"
        err = float(np.abs(rgb - o_rgb).max())
        assert err <= FP64_TOL, f"flags {flags}: frame differs from the oracle by {err}"
    return o_geom


# ---- 1: identity and round trip -----------------------------------------------------------------------------------

def identity_scenes(pkg):
    return {"synthetic": lambda: pkg.HostScene.synthetic(*SMALL_SYNTH, 184),
            "bunny4": lambda: pkg.HostScene.load(scene_path("excess_inputs/bunny4.rti")),
            "input-02": lambda: pkg.HostScene.load(scene_path("inputs/input-02.rti"))}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synthetic", "bunny4", "input-02"])
def test_refit_of_the_unchanged_scene_is_exact(pkg, gpu_renderer, oracle, name):
    """refit(A) after upload(A) does exactly the same counted work (the node array is rewritten byte for byte), and
    so does upload A -> refit B -> refit A."""
    sc = identity_scenes(pkg)[name]()
    rays = camera_rays(oracle, sc.flat)
    r = gpu_renderer
    r.upload(sc)
    ref = snapshot(pkg, r, 96, 54, 4, rays)
    r.refit(sc)
    assert_same(snapshot(pkg, r, 96, 54, 4, rays), ref, "refit(A)", work=True)
    r.refit(Desc(pkg, sc.flat, sc).without_faces().ptr)
    assert_same(snapshot(pkg, r, 96, 54, 4, rays), ref, "refit(A) without faces", work=True)
    other = Desc(pkg, sc.flat, sc).translate((3.0, -1.5, 2.0))
    r.refit(other.ptr)
    r.refit(sc)
    assert_same(snapshot(pkg, r, 96, 54, 4, rays), ref, "refit(B) -> refit(A)", work=True)


# ---- 2: the whole scene changes ---------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["host", "device"])
def test_refit_to_another_synthetic_scene(pkg, gpu_renderer, oracle, mode):
    """Seed A refit to seed B (terrain vertices, spheres and sphere materials change; the structure does not) equals a
    fresh upload of B, brute force and the oracle."""
    import torch
    a = pkg.HostScene.synthetic(*SMALL_SYNTH, 184)
    b = pkg.HostScene.synthetic(*SMALL_SYNTH, 7)
    assert structure(pkg, a.flat) == structure(pkg, b.flat)
    assert not np.array_equal(face_arrays(pkg, a.flat)[0], face_arrays(pkg, b.flat)[0])
    rays = camera_rays(oracle, b.flat)
    r = gpu_renderer
    r.upload(b)
    fresh = snapshot(pkg, r, 96, 54, 4, rays)
    r.upload(a)
    if mode == "host":
        r.refit(b)
    else:
        pts, nrm = face_arrays(pkg, b.flat)
        d = Desc(pkg, b.flat, b).with_faces(torch.from_numpy(pts).cuda(), torch.from_numpy(nrm).cuda(), on_device=True)
        torch.cuda.synchronize()
        r.refit(d.ptr)
    assert_same(snapshot(pkg, r, 96, 54, 4, rays), fresh, f"refit A -> B ({mode} faces)")
    assert_same(snapshot(pkg, r, 96, 54, 4, rays, flags=pkg.RT_FLAG_BRUTE_FORCE), fresh, "refit A -> B, brute force")
    assert_oracle(pkg, r, oracle, b.flat, 96, 54, 4)


@pytest.mark.gpu
def test_refit_with_the_faces_kept_after_a_transform_change(pkg, gpu_renderer, oracle):
    """Only the transforms, camera and lights move: a refit without faces equals a fresh upload and the oracle."""
    a = pkg.HostScene.synthetic(*SMALL_SYNTH, 184)
    moved_desc = Desc(pkg, a.flat, a).translate((40.0, -7.25, 12.5))
    rays = camera_rays(oracle, moved_desc.ptr)
    r = gpu_renderer
    r.upload(moved_desc.ptr)
    fresh = snapshot(pkg, r, 96, 54, 4, rays)
    r.upload(a)
    r.refit(Desc(pkg, moved_desc.ptr, moved_desc).without_faces().ptr)
    assert r.stats()["scene_bytes_h2d"] < 144 * 7200
    assert_same(snapshot(pkg, r, 96, 54, 4, rays), fresh, "refit without faces")
    assert_oracle(pkg, r, oracle, moved_desc.ptr, 96, 54, 4)


@pytest.mark.gpu
def test_refit_with_deformed_faces(pkg, gpu_renderer, oracle):
    """The teapot's vertices jittered (an rt_scene assembled from numpy arrays, bbmin/bbmax recomputed as
    Mesh::updateBoundingBox does) equals a fresh upload and the oracle."""
    sc = pkg.HostScene.load(scene_path("inputs/input-02.rti"))
    pts, nrm = face_arrays(pkg, sc.flat)
    d = Desc(pkg, sc.flat, sc)
    rng = np.random.default_rng(11)
    g = d.geoms[0]
    assert g.type == pkg.binding.RT_GEOM_MESH and g.first_face == 0
    n = g.num_faces
    pts[:n] += rng.uniform(-0.05, 0.05, size=(n, 3, 3))
    g.bbmin[:] = list(pts[:n].reshape(-1, 3).min(0))
    g.bbmax[:] = list(pts[:n].reshape(-1, 3).max(0))
    d.with_faces(pts, nrm)
    rays = camera_rays(oracle, d.ptr)
    r = gpu_renderer
    r.upload(d.ptr)
    fresh = snapshot(pkg, r, 80, 45, 5, rays)
    r.upload(sc)
    r.refit(d.ptr)
    assert_same(snapshot(pkg, r, 80, 45, 5, rays), fresh, "deformed teapot")
    assert_oracle(pkg, r, oracle, d.ptr, 80, 45, 5)


# ---- 3: rigid animation -------------------------------------------------------------------------------------------------

def turntable(angle, frame):
    """input-02 with the teapot turned by `angle` about y, the camera and the first point light moved."""
    text = INPUT02.replace('obj   "teapot.obj"', f'xfr 0 {angle!r} 0\nobj "{TEAPOT}"\nxfz\nxft 0 -0.7 0')
    text = text.replace("cam   0 0 6", f"cam   {0.1 * frame!r} {0.05 * frame!r} 6")
    return text.replace("ltp   10 10 10", f"ltp   10 {10 - frame!r} {10 + 0.5 * frame!r}")


@pytest.mark.gpu
def test_turntable_with_faces_kept(pkg, gpu_renderer, oracle, tmp_path):
    """Eight frames of a turning teapot (fwd / inv / det change, faces NULL), camera and light moving: every frame
    equals the oracle."""
    r = gpu_renderer
    r.upload(load(pkg, tmp_path, turntable(0.0, 0)))
    for frame in range(1, 9):
        sc = load(pkg, tmp_path, turntable(45.0 * frame, frame), f"frame{frame}.rti")
        r.refit(Desc(pkg, sc.flat, sc).without_faces().ptr)
        assert_oracle(pkg, r, oracle, sc.flat, 80, 45, 5)


# ---- 4: far coordinates ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["r0.05", "r1", "ellipsoid"])
def test_refit_far_from_the_origin(pkg, gpu_renderer, oracle, tmp_path, shape):
    """The 125-sphere LBVH clusters, camera and lights included, refit from T = 0 to 1e5, 1e6, 1e7 and back to 0, and
    then with the eye moved 1e6 away: the box padding must follow the new M (it grows through the eye alone in the
    last step), rt_cast_rays' far-origin limit must follow it (it shrinks when the scene comes back to 0), and the
    bounding spheres must be recomputed.  Rays from close by, from the surfaces, from inside and from 1e5 away, per
    ray bit for bit against the oracle; and a render."""
    text, centres, bounds, inner = cluster(shape, 5)
    r = gpu_renderer
    r.upload(load(pkg, tmp_path, moved(text, 0.0)))
    assert r.device_bytes()[0] > 0
    rad = {"r0.05": 0.05, "r1": 1.0, "ellipsoid": 1.0}[shape]
    far_eye = text.replace(f"cam 0 0 {40 * rad!r}", "cam 0 0 1000000.0", 1)
    assert far_eye != text
    steps = [(text, 1e5), (text, 1e6), (text, 1e7), (text, 0.0), (far_eye, 0.0)]
    for k, (src, T) in enumerate(steps):
        sc = load(pkg, tmp_path, moved(src, T), f"t{k}.rti")
        r.refit(sc)
        rng = np.random.default_rng(184 + k)
        world = lambda p: offset(T) + p
        lo = (centres - bounds[:, None]).min(0)
        hi = (centres + bounds[:, None]).max(0)
        n = 12000
        org_a = world((lo + hi) / 2 + unit(rng, n) * rng.uniform(0.5, 20, n)[:, None] * rad)
        dir_a = world(rng.uniform(lo, hi, size=(n, 3))) - org_a
        g_a, _, _, p_a, _ = oracle.cast_rays(sc.flat, org_a, dir_a)
        assert (g_a >= 0).sum() >= n // 10
        org_b = p_a[g_a >= 0]
        org_c = world(centres + unit(rng, len(centres)) * 0.5 * inner[:, None])
        org_d = world((lo + hi) / 2 + unit(rng, 4000) * 1e5)
        dir_d = world(rng.uniform(lo, hi, size=(4000, 3))) - org_d
        org = np.concatenate([org_a, org_b, org_c, org_d])
        dirs = np.concatenate([dir_a, unit(rng, len(org_b)), unit(rng, len(org_c)), dir_d])
        rev = np.concatenate([np.zeros(n), rng.integers(0, 2, len(org_b)), np.ones(len(org_c)), np.zeros(4000)]).astype(np.uint8)
        og = assert_cast_rays_match(pkg, r, oracle, sc, org, dirs, rev)
        assert (og[0][-4000:] >= 0).sum() >= 400
        geom = assert_oracle(pkg, r, oracle, sc.flat, 64, 48, 3)
        assert (geom >= 0).any()


# ---- 5: the Karras fallback tree ---------------------------------------------------------------------------------------------

HEAD = ("cam 0 2 30  -10 -8 10  10 -8 10  -10 12 10  10 12 10\nlta 0.1 0.1 0.1\nltp 10 20 30 1 1 1\n"
        "ltd -0.3 -1 -0.2 0.5 0.5 0.5\nmat 0.1 0.1 0.1 0.6 0.5 0.4 0.3 0.3 0.3 10 0.3 0.3 0.3\n")


def concentric(radius, shift):
    cluster_ = "".join(f"sph {shift[0] * i!r} {shift[1] * i!r} {shift[2] * i!r} {radius(i)!r}\n" for i in range(5000))
    ring = "".join(f"sph {-40 + 2 * i} -9 -20 0.7\n" for i in range(40))
    return HEAD + cluster_ + ring


@pytest.mark.gpu
def test_refit_of_the_fallback_tree(pkg, gpu_renderer, oracle, tmp_path):
    """The 5000 concentric spheres whose optimised tree is too deep (the build keeps the even-depth Karras collapse):
    radii changed and spheres moved apart, the refit tree equals brute force and the oracle."""
    r = gpu_renderer
    r.upload(load(pkg, tmp_path, concentric(lambda i: 0.5 + 0.001 * i, (0, 0, 0))))
    assert r.stats()["kernel_launches"] == UPLOAD_LAUNCHES + 5 + 4        # the optimised attempt, then the fallback
    sc = load(pkg, tmp_path, concentric(lambda i: 0.3 + 0.0013 * i, (0.0011, -0.0007, 0.0004)), "moved.rti")
    r.refit(sc)
    rays = camera_rays(oracle, sc.flat)
    assert_same(snapshot(pkg, r, 64, 48, 3, rays), snapshot(pkg, r, 64, 48, 3, rays, flags=pkg.RT_FLAG_BRUTE_FORCE),
                "fallback tree vs brute force")
    og = oracle.cast_rays(sc.flat, *rays)
    gg = r.cast_rays(*rays)
    for x, y in zip(gg, og):
        assert np.array_equal(x, y)
    assert_oracle(pkg, r, oracle, sc.flat, 64, 48, 3)


# ---- 6: camera, lights and materials only ------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_refit_of_camera_lights_and_materials(pkg, gpu_renderer, oracle, tmp_path):
    """The eye moved to 1e6 (M grows through the eye alone), a light removed and two added, two materials swapped:
    equals a fresh upload and the oracle."""
    base = load(pkg, tmp_path, moved(INPUT02, 0.0))
    text = moved(INPUT02, 0.0).replace("cam   0 0 6", "cam   0 0 1000000.0")
    text = text.replace("ltp   -1 1 1 0.3 0.25 0.0\n", "ltp   -3 2 4 0.4 0.1 0.1\nltd   0 -1 -1 0.2 0.2 0.2\nltp   2 3 1 0.1 0.3 0.1\n")
    text = text.replace("ltp   1 1 1 0.2 0.2 0.2\n", "")
    mats = re.findall(r"^mat .*$", text, re.M)
    text = text.replace(mats[0], "@0").replace(mats[2], mats[0]).replace("@0", mats[2])
    sc = load(pkg, tmp_path, text, "changed.rti")
    assert structure(pkg, base.flat) == structure(pkg, sc.flat)
    assert C.cast(sc.flat, C.POINTER(pkg.rt_scene)).contents.num_lights == 7
    rays = camera_rays(oracle, sc.flat)
    r = gpu_renderer
    r.upload(sc)
    fresh = snapshot(pkg, r, 80, 45, 5, rays)
    r.upload(base)
    r.refit(Desc(pkg, sc.flat, sc).without_faces().ptr)
    assert_same(snapshot(pkg, r, 80, 45, 5, rays), fresh, "camera / lights / materials")
    assert_oracle(pkg, r, oracle, sc.flat, 80, 45, 5)


# ---- 7: several GPUs ----------------------------------------------------------------------------------------------------------

@pytest.fixture()
def same_device_multi(monkeypatch):
    import torch
    if torch.cuda.device_count() < 2:
        monkeypatch.setenv("RT_MULTI_SAME_DEVICE", "1")


@pytest.mark.gpu
def test_refit_reaches_the_sub_contexts(pkg, same_device_multi):
    """Render over two sub-contexts, refit, render again: the frame equals the single-device render of the refit scene."""
    a = pkg.HostScene.synthetic(*SMALL_SYNTH, 184)
    b = pkg.HostScene.synthetic(*SMALL_SYNTH, 7)
    r = pkg.Renderer(0)
    try:
        r.upload(a)
        r.render(96, 54, 4, n_gpus=2)
        r.refit(b)
        multi = r.render(96, 54, 4, n_gpus=2)
        st_multi = r.stats()
        single = r.render(96, 54, 4)
        st_single = r.stats()
    finally:
        r.close()
    assert float(np.abs(multi - single).max()) <= FP64_TOL
    for k in ("rays_primary", "rays_shadow", "rays_secondary"):
        assert st_multi[k] == st_single[k], k


# ---- 8: refusals ----------------------------------------------------------------------------------------------------------------

def refusals(pkg, sc):
    def edit(fn):
        d = Desc(pkg, sc.flat, sc)
        fn(d)
        return d

    def set_geom(field, k, value):
        return lambda d: setattr(d.geoms[k], field, value)
    s = C.cast(sc.flat, C.POINTER(pkg.rt_scene)).contents
    last_tri = max(i for i in range(s.num_geometries) if s.geometries[i].type == pkg.binding.RT_GEOM_TRI)
    sphere = min(i for i in range(s.num_geometries) if s.geometries[i].type == pkg.binding.RT_GEOM_SPHERE)
    return {
        "num_geometries": edit(lambda d: setattr(d.d, "num_geometries", s.num_geometries - 1)),
        "type": edit(set_geom("type", sphere, pkg.binding.RT_GEOM_MESH)),
        "num_faces": edit(set_geom("num_faces", 0, s.geometries[0].num_faces - 1)),
        "first_face": edit(set_geom("first_face", last_tri, s.geometries[last_tri].first_face - 2)),
        "num_faces ": edit(lambda d: setattr(d.d, "num_faces", s.num_faces + 2)),
        "face_normals": edit(lambda d: setattr(d.d, "face_normals", None)),
        "material": edit(set_geom("material", sphere, s.num_materials)),
    }


@pytest.mark.gpu
def test_refit_refusals_leave_the_scene_untouched(pkg, gpu_renderer, oracle):
    sc = pkg.HostScene.load(scene_path("inputs/input-02.rti"))
    r = gpu_renderer
    rays = camera_rays(oracle, sc.flat)
    r.upload(sc)
    before = snapshot(pkg, r, 80, 45, 5, rays)
    for field, d in refusals(pkg, sc).items():
        rc = r.lib.rt_scene_refit(r._h, C.cast(d.ptr, C.c_void_p))
        msg = r.lib.rt_last_error().decode()
        assert rc == RT_ERR_INVALID, (field, rc, msg)
        assert field.strip() in msg, (field, msg)
        if field.strip() in ("type", "first_face") or field == "num_faces":
            assert "geometry" in msg, msg
        assert_same(snapshot(pkg, r, 80, 45, 5, rays), before, f"after the refused refit ({field})", work=True)
    fresh = pkg.Renderer(0)
    try:
        rc = fresh.lib.rt_scene_refit(fresh._h, C.cast(sc.flat, C.c_void_p))
        assert rc == RT_ERR_NO_SCENE, rc
    finally:
        fresh.close()


def test_refit_on_a_null_context(pkg):
    lib = pkg.load_rt()
    assert lib.rt_scene_refit(None, None) == RT_ERR_INVALID
    assert "context" in lib.rt_last_error().decode()


# ---- 9: cost ----------------------------------------------------------------------------------------------------------------------

UPLOAD_LAUNCHES = 3 + 16          # k_scatter_codes, k_prim_bounds, k_morton, 4 radix passes x 4 kernels
OPTIMISED_BUILD = 5 + 1           # k_karras, k_refit, 2 x k_treelet, k_collapse_cost; k_pack_wide (+ 1 per wide level)


@pytest.mark.gpu
def test_refit_cost(pkg, gpu_renderer, tmp_path):
    """A refit launches one bounds pass and one kernel per wide level: no sort, no treelet, no collapse.  Without faces
    it copies no face bytes."""
    grid = "".join(f"sph {-12 + 0.35 * (i % 72)} {-12 + 0.35 * (i // 72)} {-(i % 7)} 0.15\n" for i in range(5040))
    sc = load(pkg, tmp_path, HEAD + grid)
    r = gpu_renderer
    r.upload(sc)
    wide_levels = r.stats()["kernel_launches"] - UPLOAD_LAUNCHES - OPTIMISED_BUILD
    r.refit(sc)
    assert r.stats()["kernel_launches"] == 1 + wide_levels
    # faces: the teapot scene, with and without face arrays
    t = pkg.HostScene.load(scene_path("inputs/input-02.rti"))
    s = C.cast(t.flat, C.POINTER(pkg.rt_scene)).contents
    r.upload(t)
    upload = r.stats()
    r.refit(t)
    with_faces = r.stats()
    r.refit(Desc(pkg, t.flat, t).without_faces().ptr)
    without = r.stats()
    assert with_faces["kernel_launches"] == without["kernel_launches"] + 1 < upload["kernel_launches"]
    owners = sum(1 for i in range(s.num_geometries) if s.geometries[i].num_faces > 0)
    assert with_faces["scene_bytes_h2d"] - without["scene_bytes_h2d"] == 144 * s.num_faces + 20 * owners
    assert without["scene_bytes_h2d"] < 144 * s.num_faces
    # Only the upload sends primitive codes (4 B each): the flat list, the all_prims position and code of every sphere
    # and `tri`, and those in the LBVH.  Up to 64 of them all go to the flat list.
    simple = sum(1 for i in range(s.num_geometries) if s.geometries[i].type != pkg.binding.RT_GEOM_MESH)
    assert 0 < simple <= 64
    flat, simple_in_bvh = simple, 0
    assert upload["scene_bytes_h2d"] - with_faces["scene_bytes_h2d"] == 4 * (flat + 2 * simple + simple_in_bvh)
