"""GPU parity, round 2: what round 1's verdict found unpinned or untested.

  * the BENCHMARK scene itself against the unmodified reference (fixture from ref_scene_from_flat);
  * BASELINE.json configs 2-4 at their full sizes (the sizes the stock reference aborts on);
  * face ids against the reference (ref_primary_faces), not only against the C restatement;
  * LBVH conservativeness for rays that start far outside the LBVH's own bounds (ADVICE r1);
  * deep trees (duplicate centroids), bounce depths above 255, the ray-queue pool;
  * multi-GPU inside the library (rt_params.n_gpus), frames shared between ranks / processes
    (RT_FLAG_FULL_FRAME, rt_shared_frame_*), scene arrays handed over on the device;
  * the progress cadence and the node-walk roofline probe.
Same bars as test_gpu_parity.py.
"""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_ref_fixture, quantize, scene_path

pytestmark = pytest.mark.gpu
FP64_TOL = 1e-9

SCENES = {
    **{f"input-{i:02d}": f"inputs/input-{i:02d}.rti" for i in range(1, 10)},
    "refraction3": "excess_inputs/refraction3.rti",
    "refraction": "excess_inputs/refraction.rti",
    "test": "excess_inputs/test.rti",
    "example5": "excess_inputs/example5.rti",
    "reflective_specular_test": "excess_inputs/reflective_specular_test.rti",
    "bunny4": "excess_inputs/bunny4.rti",
}


@pytest.fixture(scope="module")
def scenes(pkg):
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = pkg.HostScene.load(scene_path(SCENES[name]))
        return cache[name]
    return get


@pytest.fixture(scope="module")
def synthetic(pkg):
    return pkg.HostScene.synthetic(708, 1000, 184)


# ------------------------------------------------------------------ parity pins
def test_benchmark_scene_matches_the_reference(pkg, gpu_renderer, synthetic):
    """bench.py's headline scene (1,002,528 triangles + 1000 spheres, 8 shadow lights, depth 5) rendered by the
    UNMODIFIED reference through ref_scene_from_flat (tests/golden/make_fixtures.py) at 96x54: geometry ids,
    face ids and the castRay count exact, FP64 frame within 1e-9."""
    fx = np.load(GOLDEN / "ref" / "synthetic_96x54.npz")
    w, h, depth = 96, 54, int(fx["depth"])
    gpu_renderer.upload(synthetic)
    rgb = gpu_renderer.render(w, h, depth)
    st = gpu_renderer.stats()
    geom, face = gpu_renderer.primary_ids(w, h)
    assert np.array_equal(geom, fx["geom"])
    assert np.array_equal(face, fx["face"])
    assert st["rays_primary"] + st["rays_shadow"] + st["rays_secondary"] == int(fx["castray_calls"])
    assert st["degenerate_rays"] == 0
    assert np.abs(rgb - fx["rgb"]).max() <= FP64_TOL
    assert np.array_equal(quantize(rgb), quantize(fx["rgb"]))


@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("size", [(96, 96), (80, 45)])
def test_face_ids_match_the_reference(pkg, gpu_renderer, scenes, name, size):
    w, h = size
    fx = load_ref_fixture(name, w, h)
    gpu_renderer.upload(scenes(name))
    geom, face = gpu_renderer.primary_ids(w, h)
    assert np.array_equal(geom, fx["geom"])
    assert np.array_equal(face, fx["face"])


@pytest.mark.parametrize("name,w,h", [("input-02", 1920, 1080), ("refraction3", 3840, 2160), ("bunny4", 960, 540)])
def test_baseline_configs_at_full_size(pkg, gpu_renderer, scenes, name, w, h):
    """BASELINE.json configs[1..3] at the sizes they are quoted on (the stock reference binary aborts there,
    src/scene.cpp:21-25; the fixture comes from the patched pixel loop around the unmodified traceRay)."""
    fx = np.load(GOLDEN / "ref" / f"big_{name}_{w}x{h}.npz")
    gpu_renderer.upload(scenes(name))
    rgb = gpu_renderer.render(w, h, int(fx["depth"]))
    st = gpu_renderer.stats()
    geom, face = gpu_renderer.primary_ids(w, h)
    assert np.array_equal(geom, fx["geom"].astype(np.int32))
    assert np.array_equal(face, fx["face"])
    assert st["rays_primary"] + st["rays_shadow"] + st["rays_secondary"] == int(fx["castray_calls"])
    s = int(fx["stride"])
    assert np.abs(rgb[::s, ::s] - fx["rgb_sub"]).max() <= FP64_TOL
    diff = np.abs(quantize(rgb).astype(np.int16) - fx["rgb8"].astype(np.int16)).max(axis=2)
    assert int(diff.max()) <= 1 and float((diff == 0).mean()) >= 0.9999     # truncating quantiser at 1e-16 differences
    img = gpu_renderer.render_rgb8(w, h, int(fx["depth"]))
    d8 = np.abs(img.astype(np.int16) - fx["rgb8"].astype(np.int16)).max(axis=2)
    assert int(d8.max()) <= 1 and float((d8 == 0).mean()) >= 0.9999


# ------------------------------------------------------------------ robustness
FAR_FLOOR = """\
cam 0 6 30  -8 0 10  8 0 10  -8 9 10  8 9 10
lta 0.2 0.2 0.2
ltp 40 60 40 1 1 1
ltp 0 1.5 12 0.7 0.7 0.7
ltd -0.3 -1 -0.2 0.6 0.6 0.6
ltp -3000 80 -2000 0.8 0.8 0.8
mat 0.1 0.1 0.1 0.5 0.5 0.5 0.4 0.4 0.4 20 0.6 0.6 0.6
tri -4000 -1 -4000  4000 -1 -4000  -4000 -1 4000
tri 4000 -1 -4000  4000 -1 4000  -4000 -1 4000
mat 0.1 0.1 0.1 0.7 0.3 0.3 0.5 0.5 0.5 30 0.5 0.5 0.5
sph 2500 40 -1500 60
mat 0.1 0.1 0.1 0.3 0.5 0.8 0.6 0.6 0.6 40 0.4 0.4 0.4
xft 0 0.2 0
obj "{teapot}"
"""


def test_lbvh_is_conservative_for_far_origins(pkg, gpu_renderer, tmp_path):
    """A teapot-sized LBVH (|coordinates| < 4) next to a floor and a mirror sphere thousands of units away that stay
    in the flat list: reflection and shadow rays start at |coordinates| ~ 10^3, where the FP32 slab test errs by far
    more than a padding derived from the LBVH's own extent (ADVICE r1).  The padding now covers every primitive of
    the scene: with and without the LBVH everything must agree, also for caller-supplied far-away rays."""
    rti = tmp_path / "far_floor.rti"
    rti.write_text(FAR_FLOOR.format(teapot=str(scene_path("inputs/teapot.obj"))))
    sc = pkg.HostScene.load(rti)
    gpu_renderer.upload(sc)
    w, h, depth = 480, 270, 4
    a = gpu_renderer.render(w, h, depth)
    sa = gpu_renderer.stats()
    b = gpu_renderer.render(w, h, depth, flags=pkg.RT_FLAG_BRUTE_FORCE)
    sb = gpu_renderer.stats()
    for k in ("rays_primary", "rays_shadow", "rays_secondary", "hits"):
        assert sa[k] == sb[k], k
    assert sa["rays_secondary"] > 0
    assert np.abs(a - b).max() <= FP64_TOL
    # rays from far away (beyond every primitive: the brute-force path inside the BVH kernel) towards the teapot
    rng = np.random.default_rng(7)
    n = 100000
    org = rng.normal(size=(n, 3)) * 3.0e4
    tgt = rng.uniform(-3, 3, size=(n, 3)) + np.array([0.0, 1.5, 0.0])
    org2 = np.column_stack([rng.uniform(-3900, 3900, n), np.full(n, -1.0 + 1e-9), rng.uniform(-3900, 3900, n)])
    orgs = np.concatenate([org, org2])
    dirs = np.concatenate([tgt - org, tgt - org2])
    g1 = gpu_renderer.cast_rays(orgs, dirs)
    g2 = gpu_renderer.cast_rays(orgs, dirs, flags=pkg.RT_FLAG_BRUTE_FORCE)
    for x, y in zip(g1, g2):
        assert np.array_equal(x, y)
    assert (g1[0] == 3).sum() > 2000        # plenty of them do hit the teapot (geometry 3)


def test_deep_tree_from_duplicate_centroids(pkg, gpu_renderer, oracle, tmp_path):
    """Hundreds of primitives with the SAME centroid (concentric spheres) share one Morton code, so the Karras tree
    below that code is split on the index alone and gets deep; the build checks the depth against the traversal
    stack (RT_ERR_LIMIT instead of silently dropping subtrees) and the render equals the oracle."""
    lines = ["cam 0 0 30  -10 -10 10  10 -10 10  -10 10 10  10 10 10", "lta 0.1 0.1 0.1", "ltp 20 30 40 1 1 1",
             "ltd -1 -1 -1 0.5 0.5 0.5"]
    for i in range(300):
        lines.append(f"mat 0.1 0.1 0.1 {0.2 + 0.002 * i} 0.4 0.6 0.3 0.3 0.3 10 0.3 0.3 0.3")
        lines.append(f"sph 0 0 0 {0.5 + 0.02 * i}")
    for i in range(40):
        lines.append(f"sph {-9 + 0.45 * i} 7 0 0.3")
    rti = tmp_path / "concentric.rti"
    rti.write_text("\n".join(lines) + "\n")
    sc = pkg.HostScene.load(rti)
    gpu_renderer.upload(sc)
    w, h, depth = 120, 120, 3
    rgb = gpu_renderer.render(w, h, depth)
    st = gpu_renderer.stats()
    o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, depth)
    geom, face = gpu_renderer.primary_ids(w, h)
    assert np.array_equal(geom, o_geom) and np.array_equal(face, o_face)
    assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3]
    assert np.abs(rgb - o_rgb).max() <= FP64_TOL


def test_bounce_depth_above_255(pkg, gpu_renderer, oracle, tmp_path):
    """--bdepth 300 (the reference accepts any non-negative depth): two facing mirrors keep a ray alive for the whole
    depth, the ray-queue pool ping-pongs between two queues however deep the frame goes."""
    rti = tmp_path / "mirrors.rti"
    rti.write_text("cam 0 0 30  -4 -4 20  4 -4 20  -4 4 20  4 4 20\nlta 0.1 0.1 0.1\nltp 5 8 20 1 1 1\n"
                   "mat 0.05 0.05 0.05 0.2 0.2 0.2 0.3 0.3 0.3 10 0.95 0.95 0.95\n"
                   "tri -90000 -90000 -5  90000 -90000 -5  0 90000 -5\ntri -90000 -90000 40  90000 -90000 40  0 90000 40\n"
                   "mat 0.1 0.1 0.1 0.8 0.3 0.2 0.5 0.5 0.5 20 0 0 0\nsph 1 -1 10 1.5\n")
    sc = pkg.HostScene.load(rti)
    gpu_renderer.upload(sc)
    w, h, depth = 24, 24, 300
    rgb = gpu_renderer.render(w, h, depth)
    st = gpu_renderer.stats()
    o_rgb, _, _, counts = oracle.render(sc.flat, w, h, depth, ids=False)
    assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3]
    assert st["rays_secondary"] > 250 * 100          # rays really live for hundreds of bounces
    assert np.abs(rgb - o_rgb).max() <= FP64_TOL
    with pytest.raises(pkg.RtError):
        gpu_renderer.render(8, 8, 70000)


def test_rgb8_intersection_only_over_ranks_is_refused(pkg, gpu_renderer, scenes):
    import torch
    gpu_renderer.upload(scenes("input-02"))
    p = pkg.make_params(64, 64, 2, intersection_only=True, tile_rank=0, tile_world=2)
    out = torch.zeros(64 * 64 * 3, dtype=torch.uint8, device="cuda")
    with pytest.raises(pkg.RtError):
        gpu_renderer.render_device(p, out.data_ptr(), rgb8=True)


# ------------------------------------------------------------------ several GPUs behind the C ABI
@pytest.fixture()
def same_device_multi(monkeypatch):
    """On a one-GPU box the sub-contexts of an n_gpus > 1 render all live on that GPU: the whole multi-GPU code path
    (replication, per-device tile layouts, worker threads, resolve into the caller's frame) still runs."""
    import torch
    if torch.cuda.device_count() < 2:
        monkeypatch.setenv("RT_MULTI_SAME_DEVICE", "1")


@pytest.mark.parametrize("n", [2, 3, 8])
def test_n_gpus_inside_the_library(pkg, scenes, same_device_multi, n):
    import torch
    if torch.cuda.device_count() >= 2 and n > torch.cuda.device_count():
        pytest.skip("not enough GPUs")
    r = pkg.Renderer(0)
    try:
        sc = scenes("input-02")
        r.upload(sc)
        w, h, depth = 333, 170, 5
        one = r.render(w, h, depth)
        s1 = r.stats()
        # pageable host frame: peers store into the primary's staging frame, one copy back
        many = r.render(w, h, depth, n_gpus=n)
        sn = r.stats()
        for k in ("rays_primary", "rays_shadow", "rays_secondary", "hits"):
            assert s1[k] == sn[k], k
        assert np.abs(one - many).max() <= FP64_TOL
        # page-locked host frame: every device stores its tiles into it directly
        img1 = r.render_rgb8(w, h, depth)
        pinned = torch.empty(h, w, 3, dtype=torch.uint8).pin_memory()
        pinned.zero_()
        r.render_host_params(pkg.make_params(w, h, depth, n_gpus=n), pinned.data_ptr(), rgb8=True)
        assert np.array_equal(pinned.numpy(), img1)
        # device frame on the primary GPU: peer stores
        dframe = torch.zeros(h, w, 3, dtype=torch.uint8, device="cuda:0")
        r.render_device(pkg.make_params(w, h, depth, n_gpus=n), dframe.data_ptr(), rgb8=True)
        assert np.array_equal(dframe.cpu().numpy(), img1)
        dframe64 = torch.zeros(h, w, 3, dtype=torch.float64, device="cuda:0")
        r.render_device(pkg.make_params(w, h, depth, n_gpus=n), dframe64.data_ptr(), rgb8=False)
        assert np.abs(dframe64.cpu().numpy() - one).max() <= FP64_TOL
        # --intersection-only: the global maximum is reduced over the devices
        io1 = r.render(w, h, depth, intersection_only=True)
        ion = r.render(w, h, depth, intersection_only=True, n_gpus=n)
        assert np.array_equal(io1, ion)
        # a new scene is replicated again
        r.upload(scenes("input-05"))
        a = r.render(w, h, depth)
        b = r.render(w, h, depth, n_gpus=n)
        assert np.abs(a - b).max() <= FP64_TOL
    finally:
        r.close()


def test_n_gpus_progress_and_cli(pkg, scenes, same_device_multi, tmp_path):
    from conftest import PKG_DIR, decode_png
    out1, out2 = tmp_path / "one.png", tmp_path / "two.png"
    exe, rti = str(PKG_DIR / "bin" / "as2"), str(scene_path("inputs/input-05.rti"))
    for out, extra in ((out1, []), (out2, ["--gpus", "2"])):
        proc = subprocess.run([exe, rti, "-o", str(out), "-w", "200", "-h", "150"] + extra, capture_output=True, text=True)
        assert proc.returncode == 0, proc.stderr
        assert "Rendering scene (30000/30000) (100.0%) ..." in proc.stdout
    assert np.array_equal(decode_png(out1), decode_png(out2))


def test_full_frame_shared_by_ranks(pkg, gpu_renderer, scenes):
    """RT_FLAG_FULL_FRAME: every rank stores its tiles into ONE row-major frame (device memory, or page-locked host
    memory); together they are the single-rank frame — no gather, no unpack."""
    import torch
    gpu_renderer.upload(scenes("input-02"))
    for (w, h) in [(300, 170), (257, 65)]:
        full = gpu_renderer.render_rgb8(w, h, 5)
        full64 = gpu_renderer.render(w, h, 5)
        for world in (2, 5):
            dframe = torch.zeros(h, w, 3, dtype=torch.uint8, device="cuda")
            hframe = torch.zeros(h, w, 3, dtype=torch.uint8).pin_memory()
            d64 = torch.zeros(h, w, 3, dtype=torch.float64, device="cuda")
            for rank in range(world):
                p = pkg.make_params(w, h, 5, tile_rank=rank, tile_world=world, flags=pkg.RT_FLAG_FULL_FRAME)
                gpu_renderer.render_device(p, dframe.data_ptr(), rgb8=True)
                gpu_renderer.render_device(p, d64.data_ptr(), rgb8=False)
                gpu_renderer.render_host_params(p, hframe.data_ptr(), rgb8=True)
            torch.cuda.synchronize()
            assert np.array_equal(dframe.cpu().numpy(), full)
            assert np.array_equal(hframe.numpy(), full)
            assert np.abs(d64.cpu().numpy() - full64).max() <= FP64_TOL
    # a pageable host frame cannot be shared
    with pytest.raises(pkg.RtError):
        p = pkg.make_params(64, 64, 2, tile_rank=0, tile_world=2, flags=pkg.RT_FLAG_FULL_FRAME)
        gpu_renderer.render_host_params(p, np.zeros((64, 64, 3), np.uint8).ctypes.data, rgb8=True)


class _RawDevice:
    """__cuda_array_interface__ over a raw device pointer (uint8[n])."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}


CHILD = """
import sys
sys.path.insert(0, {tests!r})
from conftest import load_package, scene_path
pkg = load_package()
handle = bytes.fromhex(sys.argv[1])
w, h, depth, rank, world = (int(x) for x in sys.argv[2:7])
r = pkg.Renderer(0)
r.upload(pkg.HostScene.load(scene_path("inputs/input-02.rti")))
ptr = r.shared_frame_open(handle)
p = pkg.make_params(w, h, depth, tile_rank=rank, tile_world=world, flags=pkg.RT_FLAG_FULL_FRAME)
r.render_device(p, ptr, rgb8=True)
r.shared_frame_close(ptr)
r.close()
print("child ok")
"""


def test_shared_frame_between_processes(pkg, gpu_renderer, scenes, tmp_path):
    """rt_shared_frame_*: rank 0 creates the frame, a SECOND PROCESS opens the handle and its resolve kernel stores
    its tiles into rank 0's memory (CUDA IPC; over NVLink when the processes sit on different GPUs)."""
    import torch
    w, h, depth, world = 300, 170, 4, 2
    gpu_renderer.upload(scenes("input-02"))
    full = gpu_renderer.render_rgb8(w, h, depth)
    ptr, handle = gpu_renderer.shared_frame_create(w * h * 3)
    try:
        view = torch.as_tensor(_RawDevice(ptr, w * h * 3), device="cuda")      # torch view of the library's allocation
        view.zero_()
        torch.cuda.synchronize()
        p0 = pkg.make_params(w, h, depth, tile_rank=0, tile_world=world, flags=pkg.RT_FLAG_FULL_FRAME)
        gpu_renderer.render_device(p0, ptr, rgb8=True)
        script = tmp_path / "child.py"
        script.write_text(CHILD.format(tests=str(ROOT / "tests")))
        proc = subprocess.run([sys.executable, str(script), handle.hex(), str(w), str(h), str(depth), "1", str(world)],
                              capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0 and "child ok" in proc.stdout, proc.stderr[-2000:]
        assert np.array_equal(view.cpu().numpy().reshape(h, w, 3), full)
    finally:
        gpu_renderer.shared_frame_close(ptr)


def test_scene_faces_already_on_the_device(pkg, gpu_renderer, scenes):
    """RT_SCENE_FACES_ON_DEVICE: the face arrays are handed over as device pointers (how a multi-GPU caller that
    all-gathered per-rank slices over NVLink uploads a scene); same frame as the host upload."""
    import torch
    for name in ("bunny4", "input-02"):
        sc = scenes(name)
        gpu_renderer.upload(sc)
        a = gpu_renderer.render(160, 120, 4)
        flat = sc.flat.contents
        nf = flat.num_faces
        pts = np.ctypeslib.as_array(flat.face_points, shape=(nf * 9,))
        nrm = np.ctypeslib.as_array(flat.face_normals, shape=(nf * 9,))
        d_pts, d_nrm = torch.from_numpy(pts.copy()).cuda(), torch.from_numpy(nrm.copy()).cuda()
        dev = pkg.rt_scene()
        C.memmove(C.byref(dev), C.byref(flat), C.sizeof(pkg.rt_scene))
        dev.flags = pkg.RT_SCENE_FACES_ON_DEVICE
        dev.face_points = C.cast(C.c_void_p(d_pts.data_ptr()), C.POINTER(C.c_double))
        dev.face_normals = C.cast(C.c_void_p(d_nrm.data_ptr()), C.POINTER(C.c_double))
        torch.cuda.synchronize()
        gpu_renderer.upload(C.pointer(dev))
        assert gpu_renderer.stats()["scene_bytes_h2d"] < 100000
        b = gpu_renderer.render(160, 120, 4)
        assert np.array_equal(a, b) or np.abs(a - b).max() <= 1e-15
        g1, f1 = gpu_renderer.primary_ids(160, 120)
        gpu_renderer.upload(sc)
        g2, f2 = gpu_renderer.primary_ids(160, 120)
        assert np.array_equal(g1, g2) and np.array_equal(f1, f2)


# ------------------------------------------------------------------ progress, probe
def test_progress_is_reported_during_a_long_render(pkg, gpu_renderer, scenes):
    """The reference's handler runs every 100 ms (src/scene.cpp:41-44); a render of a second or so must report
    several intermediate, increasing values before the final (total, total)."""
    gpu_renderer.upload(scenes("refraction3"))
    calls = []
    CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.c_void_p)
    cb = CB(lambda done, total, user: calls.append((done, total)))
    w, h = 2000, 1500
    p = pkg.make_params(w, h, 10, samples=8)
    out = np.empty((h, w, 3))
    rc = gpu_renderer.lib.rt_render(gpu_renderer._h, C.byref(p), out.ctypes.data_as(C.c_void_p), cb, None)
    assert rc == 0
    ms = gpu_renderer.stats()["ms_trace"]
    assert calls[-1] == (w * h, w * h)
    inter = [c for c in calls[:-1]]
    assert all(0 <= a[0] < w * h for a in inter)
    assert all(a[0] < b[0] for a, b in zip(inter, inter[1:]))
    if ms > 400:
        assert len(inter) >= 2, (ms, calls)


def test_node_walk_probe(pkg, gpu_renderer, synthetic):
    gpu_renderer.upload(synthetic)
    coherent, bytes_c = gpu_renderer.microbench_node_walk(32, 64)
    divergent, _ = gpu_renderer.microbench_node_walk(1, 64)
    assert coherent > 0 and divergent > 0 and abs(bytes_c - 112 * coherent) < 1e-3 * bytes_c
    assert coherent >= divergent
    gpu_renderer.upload(pkg.HostScene.load(scene_path("inputs/input-01.rti")))      # no LBVH
    with pytest.raises(pkg.RtError):
        gpu_renderer.microbench_node_walk(32, 8)


# ------------------------------------------------------------------ INTEGRATION.md path B, compiled
def test_pathb_reference_main_on_the_b200(tmp_path):
    """oracle/_ref/as2_pathb = the reference's OWN main.cpp / parsers.cpp / options.cpp / exceptions.cpp /
    geometry.cpp / writers.cpp (+ its vendored libpng), unmodified, linked with tests/pathb/render_scene_b200.cpp
    (Scene::renderScene -> librt_b200.so) instead of src/scene.cpp.  The reference's command line of
    notes/notes-08.txt must reproduce outputs/image-08.png within the north_star gate, and the progress line the
    reference's main prints relies on the final (total, total) callback."""
    from conftest import ORACLE_DIR, decode_png
    exe = ORACLE_DIR / "_ref" / "as2_pathb"
    if not exe.exists():
        pytest.skip("oracle/_ref/as2_pathb not built (needs the reference sources at build time, tests/pathb/Makefile REF=)")
    for n, size in (("08", 1000), ("05", 1000)):
        out = tmp_path / f"image-{n}.png"
        proc = subprocess.run([str(exe), str(scene_path(f"inputs/input-{n}.rti")), "-o", str(out), "-h", str(size), "-w", str(size),
                               "-t", "8"], capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, proc.stderr[-2000:]
        assert f"Rendering scene ({size * size}/{size * size}) (100.0%) ..." in proc.stdout
        img = decode_png(out)
        gold = decode_png(GOLDEN / "outputs" / f"image-{n}.png")
        diff = np.abs(img.astype(np.int16) - gold.astype(np.int16)).max(axis=2)
        assert float((diff <= 1).mean()) >= 0.999 and int(diff.max()) <= 4


# ------------------------------------------------------------------ empty and degenerate inputs
def _scene_from_text(pkg, tmp_path, name, text):
    rti = tmp_path / name
    rti.write_text(text)
    return pkg.HostScene.load(rti)


CAM = "cam 0 0 30  -10 -10 10  10 -10 10  -10 10 10  10 10 10\n"


def test_empty_and_lightless_scenes(pkg, gpu_renderer, oracle, live_reference, tmp_path):
    """No geometry at all; geometry without any light; only an ambient light: frames, ids and ray counts equal the
    oracle's, and the unmodified reference agrees on the frame where it is built."""
    cases = {
        "nothing.rti": CAM,
        "dark.rti": CAM + "mat 0.1 0.1 0.1 0.5 0.5 0.5 0.3 0.3 0.3 10 0.5 0.5 0.5\nsph 0 0 0 4\n",
        "ambient.rti": CAM + "lta 0.4 0.5 0.6\nmat 0.5 0.4 0.3 0.5 0.5 0.5 0.3 0.3 0.3 10 0 0 0\nsph 0 0 0 4\ntri -8 -8 -3 8 -8 -3 0 8 -3\n",
        "lights_only.rti": CAM + "ltp 5 5 5 1 1 1\nltd 0 -1 0 1 1 1\nlta 1 1 1\n",
    }
    for name, text in cases.items():
        sc = _scene_from_text(pkg, tmp_path, name, text)
        gpu_renderer.upload(sc)
        for (w, h, depth) in [(40, 30, 3), (1, 1, 0)]:
            rgb = gpu_renderer.render(w, h, depth)
            st = gpu_renderer.stats()
            o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, depth)
            geom, face = gpu_renderer.primary_ids(w, h)
            assert np.array_equal(geom, o_geom) and np.array_equal(face, o_face), name
            assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3], name
            assert np.abs(rgb - o_rgb).max() <= FP64_TOL, name
        if live_reference is not None:
            href = live_reference.load(tmp_path / name)
            r_rgb, _, _, _ = live_reference.render(href, 40, 30, 3, threads=2)
            assert np.abs(gpu_renderer.render(40, 30, 3) - r_rgb).max() <= FP64_TOL, name
        img = gpu_renderer.render_rgb8(40, 30, 3)
        assert np.array_equal(img, quantize(gpu_renderer.render(40, 30, 3)))


def test_lbvh_corner_sizes(pkg, gpu_renderer, oracle, tmp_path):
    """Meshes of one and two faces (an LBVH of a single leaf / a single node) and 65 spheres (the smallest count that
    moves the spheres from the flat list into the LBVH)."""
    one = tmp_path / "one.obj"
    one.write_text("v -5 -5 0\nv 5 -5 0\nv 0 5 0\nf 1 2 3\n")
    two = tmp_path / "two.obj"
    two.write_text("v -5 -5 0\nv 5 -5 0\nv 0 5 0\nv 0 -9 1\nf 1 2 3\nf 1 4 2\n")
    head = CAM + "lta 0.1 0.1 0.1\nltp 10 20 30 1 1 1\nmat 0.1 0.1 0.1 0.6 0.5 0.4 0.3 0.3 0.3 10 0.3 0.3 0.3\n"
    spheres = "".join(f"sph {-8 + 2 * (i % 9)} {-7 + 2 * (i // 9)} {-(i % 5)} 0.8\n" for i in range(65))
    cases = {"one.rti": head + f'obj "{one}"\n', "two.rti": head + f'obj "{two}"\n', "s65.rti": head + spheres,
             "mix.rti": head + spheres + f'obj "{two}"\n'}
    for name, text in cases.items():
        sc = _scene_from_text(pkg, tmp_path, name, text)
        gpu_renderer.upload(sc)
        w, h, depth = 64, 48, 4
        rgb = gpu_renderer.render(w, h, depth)
        st = gpu_renderer.stats()
        o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, depth)
        geom, face = gpu_renderer.primary_ids(w, h)
        assert np.array_equal(geom, o_geom) and np.array_equal(face, o_face), name
        assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3], name
        assert np.abs(rgb - o_rgb).max() <= FP64_TOL, name
        b = gpu_renderer.render(w, h, depth, flags=pkg.RT_FLAG_BRUTE_FORCE)
        assert np.abs(rgb - b).max() <= FP64_TOL, name


def test_more_devices_than_tiles(pkg, scenes, same_device_multi):
    """A frame of one tile (or one pixel) rendered with n_gpus = 3: two devices own nothing and must not disturb the frame."""
    r = pkg.Renderer(0)
    try:
        r.upload(scenes("input-05"))
        for (w, h) in [(1, 1), (20, 17), (33, 31)]:
            a = r.render(w, h, 4)
            b = r.render(w, h, 4, n_gpus=3)
            assert np.abs(a - b).max() <= FP64_TOL
            assert np.array_equal(r.render_rgb8(w, h, 4), r.render_rgb8(w, h, 4, n_gpus=3))
    finally:
        r.close()


# ------------------------------------------------------------------ every scene the reference ships
ALL_LOADABLE = sorted(p for p in list((GOLDEN / "inputs").glob("*.rti")) + list((GOLDEN / "excess_inputs").glob("*.rti"))
                      if p.name not in ("teapot.rti",))   # excess teapot.rti has no teapot.obj beside it


@pytest.mark.parametrize("path", ALL_LOADABLE, ids=lambda p: p.parent.name + "/" + p.name)
def test_every_shipped_scene_matches_the_oracle(pkg, gpu_renderer, oracle, path):
    """All 25 loadable scenes of the reference tree (the oracle is pinned to the live reference on each of them in
    tests/test_oracle_vs_reference.py): hit ids, ray counts per class, FP64 frame, and per-ray castRay results."""
    sc = pkg.HostScene.load(path)
    gpu_renderer.upload(sc)
    w, h, depth = 72, 54, 6
    rgb = gpu_renderer.render(w, h, depth)
    st = gpu_renderer.stats()
    geom, face = gpu_renderer.primary_ids(w, h)
    o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, depth)
    assert np.array_equal(geom, o_geom) and np.array_equal(face, o_face)
    assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3]
    assert st["degenerate_rays"] == counts[3]
    assert np.abs(rgb - o_rgb).max() <= FP64_TOL
    rng = np.random.default_rng(11)
    n = 4000
    org, direction = oracle.camera_rays(sc.flat, 100, 100, rng.integers(0, 10000, n))
    g0, f0, d0, p0, n0 = oracle.cast_rays(sc.flat, org, direction)
    org2 = np.where((g0 >= 0)[:, None], p0, org)
    dir2 = rng.normal(size=(n, 3))
    rev = rng.integers(0, 2, n).astype(np.uint8)
    og = oracle.cast_rays(sc.flat, org2, dir2, rev)
    gg = gpu_renderer.cast_rays(org2, dir2, rev)
    for a, b in zip(gg, og):
        assert np.array_equal(a, b)
