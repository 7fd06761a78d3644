"""GPU parity: the CUDA trace loop (through the C ABI) against
  * outputs of the UNMODIFIED reference stored in tests/golden/ref/*.npz,
  * the plain-C oracle on the same seeded inputs,
  * the reference's nine golden images outputs/image-0N.png at their full sizes.
Bars: primary hit ids, per-ray hit decisions and ray counts bit-exact; FP64 framebuffer
within 1e-9 absolute (summation order of the iterative bounce loop and CUDA's pow() differ
from the recursion in the last ulps); 8-bit images within 1/255 on >= 99.9 % of pixels and no
pixel off by more than 4/255 (BASELINE.json north_star).
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, decode_png, load_ref_fixture, quantize, scene_path

pytestmark = pytest.mark.gpu

SCENES = {
    **{f"input-{i:02d}": f"inputs/input-{i:02d}.rti" for i in range(1, 10)},
    "refraction3": "excess_inputs/refraction3.rti",
    "refraction": "excess_inputs/refraction.rti",
    "test": "excess_inputs/test.rti",
    "example5": "excess_inputs/example5.rti",
    "reflective_specular_test": "excess_inputs/reflective_specular_test.rti",
    "bunny4": "excess_inputs/bunny4.rti",
}
FP64_TOL = 1e-9


@pytest.fixture(scope="module")
def scenes(pkg):
    cache = {}
    def get(name):
        if name not in cache:
            cache[name] = pkg.HostScene.load(scene_path(SCENES[name]))
        return cache[name]
    return get


@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("size", [(96, 96), (80, 45)])
def test_matches_reference_outputs(pkg, gpu_renderer, scenes, name, size):
    w, h = size
    fx = load_ref_fixture(name, w, h)
    gpu_renderer.upload(scenes(name))
    rgb = gpu_renderer.render(w, h, int(fx["depth"]))
    st = gpu_renderer.stats()
    geom, face = gpu_renderer.primary_ids(w, h)
    assert np.array_equal(geom, fx["geom"]), "primary hit geometry ids differ from the reference"
    total = st["rays_primary"] + st["rays_shadow"] + st["rays_secondary"]
    assert total == int(fx["castray_calls"]), "ray count differs from the reference's castRay call count"
    assert st["degenerate_rays"] == 0
    assert np.abs(rgb - fx["rgb"]).max() <= FP64_TOL
    assert np.array_equal(quantize(rgb), quantize(fx["rgb"]))


@pytest.mark.parametrize("name", sorted(SCENES))
def test_bvh_equals_brute_force_and_oracle(pkg, gpu_renderer, oracle, scenes, name):
    w, h = 64, 48
    sc = scenes(name)
    gpu_renderer.upload(sc)
    rgb_bvh = gpu_renderer.render(w, h, 6)
    st_bvh = gpu_renderer.stats()
    g_bvh, f_bvh = gpu_renderer.primary_ids(w, h)
    rgb_bf = gpu_renderer.render(w, h, 6, flags=pkg.RT_FLAG_BRUTE_FORCE)
    st_bf = gpu_renderer.stats()
    g_bf, f_bf = gpu_renderer.primary_ids(w, h, flags=pkg.RT_FLAG_BRUTE_FORCE)
    assert np.array_equal(g_bvh, g_bf) and np.array_equal(f_bvh, f_bf)
    for k in ("rays_primary", "rays_shadow", "rays_secondary"):
        assert st_bvh[k] == st_bf[k]
    assert np.abs(rgb_bvh - rgb_bf).max() <= FP64_TOL
    o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, 6)
    assert np.array_equal(g_bvh, o_geom) and np.array_equal(f_bvh, o_face)
    assert [st_bvh["rays_primary"], st_bvh["rays_shadow"], st_bvh["rays_secondary"]] == counts[:3]
    assert np.abs(rgb_bvh - o_rgb).max() <= FP64_TOL


@pytest.mark.parametrize("name", ["input-02", "input-05", "input-07", "input-09", "refraction3", "bunny4"])
def test_cast_rays_bit_exact(pkg, gpu_renderer, oracle, scenes, name):
    """Scene::castRay on seeded random rays (both reverseNormals values): hit ids, distance,
    point and normal must equal the oracle's doubles bit for bit."""
    sc = scenes(name)
    gpu_renderer.upload(sc)
    rng = np.random.default_rng(184)
    n = 20000
    w = h = 200
    pix = rng.integers(0, w * h, n)
    org, direction = oracle.camera_rays(sc.flat, w, h, pix)
    # second half: rays leaving primary hit points in random directions (origins ON surfaces)
    g0, f0, d0, p0, n0 = oracle.cast_rays(sc.flat, org, direction)
    hit = g0 >= 0
    org2 = np.where(hit[:, None], p0, org)
    dir2 = rng.normal(size=(n, 3))
    orgs = np.concatenate([org, org2])
    dirs = np.concatenate([direction, dir2])
    rev = rng.integers(0, 2, 2 * n).astype(np.uint8)
    og = oracle.cast_rays(sc.flat, orgs, dirs, rev)
    for flags in (0, pkg.RT_FLAG_BRUTE_FORCE):
        gg = gpu_renderer.cast_rays(orgs, dirs, rev, flags=flags)
        assert np.array_equal(gg[0], og[0]), "geometry ids"
        assert np.array_equal(gg[1], og[1]), "face ids"
        assert np.array_equal(gg[2], og[2]), "distances"
        assert np.array_equal(gg[3], og[3]), "points"
        assert np.array_equal(gg[4], og[4]), "normals"


GOLDEN_SIZES = {f"{i:02d}": (1000, 1000) for i in range(1, 9)}
GOLDEN_SIZES["09"] = (2000, 2000)


@pytest.mark.parametrize("n", sorted(GOLDEN_SIZES))
def test_golden_images(pkg, gpu_renderer, scenes, n):
    """The reference's known-answer vectors (notes/notes-0N.txt command lines, default --bdepth 10)."""
    w, h = GOLDEN_SIZES[n]
    gold = decode_png(GOLDEN / "outputs" / f"image-{n}.png")
    gpu_renderer.upload(scenes(f"input-{n}"))
    img = gpu_renderer.render_rgb8(w, h, 10)
    diff = np.abs(img.astype(np.int16) - gold.astype(np.int16)).max(axis=2)
    frac_ok = float((diff <= 1).mean())
    assert frac_ok >= 0.999, f"only {frac_ok:.5f} of pixels within 1/255"
    assert int(diff.max()) <= 4, f"max pixel error {int(diff.max())}/255"
    # device-side quantisation == host quantisation of the FP64 frame
    rgb = gpu_renderer.render(w, h, 10)
    assert np.array_equal(pkg.quantize_rgb8(rgb), img)


def test_intersection_only(pkg, gpu_renderer, scenes):
    for name in ("input-02", "input-06"):
        fx = load_ref_fixture(name, 96, 96)
        gpu_renderer.upload(scenes(name))
        rgb = gpu_renderer.render(96, 96, 10, intersection_only=True)
        assert np.array_equal(rgb[..., 0], rgb[..., 1]) and np.array_equal(rgb[..., 0], rgb[..., 2])
        assert np.array_equal(rgb[..., 0], fx["intersection_only"])


def test_host_render_scene_entry_point(pkg, scenes, gpu_renderer):
    """Scene::renderScene through the C++ host equals the direct C-ABI call."""
    sc = scenes("input-05")
    a = sc.render(120, 90, 10)
    gpu_renderer.upload(sc)
    b = gpu_renderer.render(120, 90, 10)
    assert np.abs(a - b).max() <= FP64_TOL


def test_ragged_and_tiny_frames(pkg, gpu_renderer, oracle, scenes):
    sc = scenes("input-05")
    gpu_renderer.upload(sc)
    for (w, h) in [(1, 1), (33, 31), (7, 65), (501, 499)]:
        rgb = gpu_renderer.render(w, h, 4)
        o_rgb, _, _, counts = oracle.render(sc.flat, w, h, 4, ids=False)
        st = gpu_renderer.stats()
        assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3]
        assert np.abs(rgb - o_rgb).max() <= FP64_TOL


def test_small_queue_chunks_do_not_change_the_result(pkg, scenes, monkeypatch):
    """Deep recursion through tiny ray queues (forces many chunks per level)."""
    monkeypatch.setenv("RT_QUEUE_CAP", "4096")
    r = pkg.Renderer(0)
    try:
        sc = scenes("input-06")
        r.upload(sc)
        fx = load_ref_fixture("input-06", 96, 96)
        rgb = r.render(96, 96, 10)
        st = r.stats()
        assert st["rays_primary"] + st["rays_shadow"] + st["rays_secondary"] == int(fx["castray_calls"])
        assert np.abs(rgb - fx["rgb"]).max() <= FP64_TOL
    finally:
        r.close()


def test_tile_sharding_emulated_on_one_gpu(pkg, gpu_renderer, scenes):
    """Interleaved-tile partition: render every rank's tiles (one after the other on this
    GPU), lay them out like an all_gather would, unpack, compare with the single-rank frame."""
    import torch
    sc = scenes("input-02")
    gpu_renderer.upload(sc)
    w, h = 300, 170
    full = gpu_renderer.render_rgb8(w, h, 5)
    for world in (2, 3, 8):
        p0 = pkg.make_params(w, h, 5, tile_rank=0, tile_world=world)
        _, max_tiles, total = pkg.tile_counts(p0)
        packed = torch.zeros(world, max_tiles * pkg.RT_TILE_PIXELS * 3, dtype=torch.uint8, device="cuda")
        owned = 0
        for rank in range(world):
            p = pkg.make_params(w, h, 5, tile_rank=rank, tile_world=world)
            owned += pkg.tile_counts(p)[0]
            gpu_renderer.render_device(p, packed[rank].data_ptr(), rgb8=True)
        assert owned == total
        frame = torch.empty(h, w, 3, dtype=torch.uint8, device="cuda")
        gpu_renderer.unpack_tiles(p0, packed.data_ptr(), frame.data_ptr(), rgb8=True)
        torch.cuda.synchronize()
        assert np.array_equal(frame.cpu().numpy(), full)


def test_as2_cli_renders_the_golden(pkg, tmp_path):
    """The drop-in executable end to end: same command line as notes/notes-08.txt (smaller
    thread count is irrelevant: -t is accepted and ignored), PNG within the north_star gate."""
    import subprocess
    from conftest import PKG_DIR
    out = tmp_path / "image-08.png"
    proc = subprocess.run([str(PKG_DIR / "bin" / "as2"), str(scene_path("inputs/input-08.rti")), "-o", str(out),
                           "-h", "1000", "-w", "1000", "-t", "8"], capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr
    assert "Rendering scene (1000000/1000000) (100.0%) ..." in proc.stdout
    img = decode_png(out)
    gold = decode_png(GOLDEN / "outputs" / "image-08.png")
    diff = np.abs(img.astype(np.int16) - gold.astype(np.int16)).max(axis=2)
    assert float((diff <= 1).mean()) >= 0.999 and int(diff.max()) <= 4


def test_progress_callback_contract(pkg, gpu_renderer, scenes):
    """Monotone, on the calling thread, and a final (total, total) call (src/scene.cpp:41-47)."""
    import ctypes as C
    import threading
    gpu_renderer.upload(scenes("input-05"))
    calls = []
    main_thread = threading.get_ident()
    CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.c_void_p)
    cb = CB(lambda done, total, user: calls.append((done, total, threading.get_ident())))
    p = pkg.make_params(640, 480, 3)
    out = np.empty((480, 640, 3))
    rc = gpu_renderer.lib.rt_render(gpu_renderer._h, C.byref(p), out.ctypes.data_as(C.c_void_p), cb, None)
    assert rc == 0 and calls
    assert calls[-1][:2] == (640 * 480, 640 * 480)
    assert all(a[0] <= b[0] for a, b in zip(calls, calls[1:]))
    assert all(c[2] == main_thread for c in calls)


def test_intersection_only_across_ranks(pkg, gpu_renderer, scenes):
    """--intersection-only with tile sharding: per-rank maxima are reduced by the caller
    (an all-reduce in a real multi-GPU run) before the divide; result == single-rank frame."""
    import torch
    gpu_renderer.upload(scenes("input-02"))
    w, h, world = 200, 120, 3
    full = gpu_renderer.render(w, h, 10, intersection_only=True)
    p0 = pkg.make_params(w, h, 10, intersection_only=True, tile_rank=0, tile_world=world)
    _, max_tiles, _ = pkg.tile_counts(p0)
    n = max_tiles * pkg.RT_TILE_PIXELS * 3
    packed = torch.zeros(world, n, dtype=torch.float64, device="cuda")
    maxima = []
    for rank in range(world):
        p = pkg.make_params(w, h, 10, intersection_only=True, tile_rank=rank, tile_world=world)
        gpu_renderer.render_device(p, packed[rank].data_ptr())
        maxima.append(gpu_renderer.intersection_max())
    gmax = max(maxima)
    for rank in range(world):
        gpu_renderer.divide_device(packed[rank].data_ptr(), n, gmax)
    frame = torch.empty(h, w, 3, dtype=torch.float64, device="cuda")
    gpu_renderer.unpack_tiles(p0, packed.data_ptr(), frame.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(frame.cpu().numpy(), full)


@pytest.mark.parametrize("name,size,depth", [("input-02", (320, 240), 4), ("input-03", (320, 240), 3),
                                              ("input-04", (320, 240), 3), ("input-09", (320, 240), 6),
                                              ("bunny4", (320, 180), 3)])
def test_lbvh_is_conservative_on_mesh_scenes(pkg, gpu_renderer, scenes, name, size, depth):
    """The LBVH may only cull what the exact FP64 test would reject: with and without it
    (RT_FLAG_BRUTE_FORCE tests every primitive) hit ids, ray counts per class and the FP64
    frame must agree on hundreds of thousands of primary, shadow and secondary rays."""
    w, h = size
    gpu_renderer.upload(scenes(name))
    a = gpu_renderer.render(w, h, depth)
    sa = gpu_renderer.stats()
    ga, fa = gpu_renderer.primary_ids(w, h)
    b = gpu_renderer.render(w, h, depth, flags=pkg.RT_FLAG_BRUTE_FORCE)
    sb = gpu_renderer.stats()
    gb, fb = gpu_renderer.primary_ids(w, h, flags=pkg.RT_FLAG_BRUTE_FORCE)
    assert np.array_equal(ga, gb) and np.array_equal(fa, fb)
    for k in ("rays_primary", "rays_shadow", "rays_secondary", "hits"):
        assert sa[k] == sb[k], k
    assert np.abs(a - b).max() <= FP64_TOL


def test_synthetic_scene_lbvh_vs_brute_force(pkg, gpu_renderer):
    """The benchmark scene itself (1,002,528 triangles + 1000 spheres in the LBVH, 8 shadow
    lights, depth 5) on a 96x54 sample: LBVH == brute force, and the 7680x4320 frame's
    per-class ray counts are a multiple-consistent property checked in bench runs."""
    sc = pkg.HostScene.synthetic(708, 1000, 184)
    gpu_renderer.upload(sc)
    w, h = 96, 54
    a = gpu_renderer.render(w, h, 5)
    sa = gpu_renderer.stats()
    ga, fa = gpu_renderer.primary_ids(w, h)
    b = gpu_renderer.render(w, h, 5, flags=pkg.RT_FLAG_BRUTE_FORCE)
    sb = gpu_renderer.stats()
    gb, fb = gpu_renderer.primary_ids(w, h, flags=pkg.RT_FLAG_BRUTE_FORCE)
    assert (ga >= 0).mean() > 0.5
    assert np.array_equal(ga, gb) and np.array_equal(fa, fb)
    for k in ("rays_primary", "rays_shadow", "rays_secondary", "hits"):
        assert sa[k] == sb[k], k
    assert sa["rays_secondary"] > 0 and sa["degenerate_rays"] == 0
    assert np.abs(a - b).max() <= FP64_TOL


@pytest.mark.parametrize("name", ["input-02", "input-03", "bunny4"])
@pytest.mark.parametrize("env,serial", [
    ({"RT_HIT_SORT_MIN_RAYS": "1"}, False),                               # hit sorting on every level
    ({"RT_HIT_SORT_MIN_RAYS": "1", "RT_QUEUE_CAP": "8192"}, False),       # sorted chunks of a chunked level
    ({"RT_HIT_SORT_MIN_RAYS": str(2**31)}, False),                        # sorting off: no level is that large
    ({"RT_HIT_SORT_MIN_RAYS": "1"}, True),                                # RT_FLAG_SERIAL: kernels strictly serial
], ids=["sort", "sort-chunked", "nosort", "serial"])
def test_hit_sorting_and_overlap_do_not_change_the_result(pkg, scenes, monkeypatch, name, env, serial):
    """The Morton hit sort, the shadow/trace overlap and their thresholds only reorder work: hit ids, ray
    counts and the frame (FP64 sums reorder at 1e-16) must equal the reference outputs."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    r = pkg.Renderer(0)
    try:
        sc = scenes(name)
        r.upload(sc)
        fx = load_ref_fixture(name, 96, 96)
        rgb = r.render(96, 96, int(fx["depth"]), flags=pkg.RT_FLAG_SERIAL if serial else 0)
        st = r.stats()
        assert st["rays_primary"] + st["rays_shadow"] + st["rays_secondary"] == int(fx["castray_calls"])
        assert np.abs(rgb - fx["rgb"]).max() <= FP64_TOL
        g, _ = r.primary_ids(96, 96)
        assert np.array_equal(g, fx["geom"])
    finally:
        r.close()


@pytest.mark.parametrize("name,samples", [("input-02", 2), ("input-05", 3), ("refraction3", 2), ("bunny4", 4)])
def test_supersampling_matches_the_oracle(pkg, gpu_renderer, oracle, scenes, name, samples):
    """SURVEY section 8 f-4 (the reference's TODO:2): n x n rays per pixel through the cell centres, averaged.
    samples = 1 is the reference's pixel-centre ray (all other tests); n > 1 is checked against the oracle's
    restatement of the same rule: ray counts exact, frame within the FP64 tolerance."""
    sc = scenes(name)
    gpu_renderer.upload(sc)
    w, h, depth = 61, 47, 5
    rgb = gpu_renderer.render(w, h, depth, samples=samples)
    st = gpu_renderer.stats()
    o_rgb, _, _, counts = oracle.render(sc.flat, w, h, depth, ids=False, samples=samples)
    assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3]
    assert st["rays_primary"] == w * h * samples * samples
    assert np.abs(rgb - o_rgb).max() <= FP64_TOL
    one = gpu_renderer.render(w, h, depth)
    assert np.abs(rgb - one).max() > 1e-3           # it does change edges ...
    assert np.abs(rgb.mean() - one.mean()) < 0.02    # ... and not the overall picture


def test_supersampling_argument_checks(pkg, gpu_renderer, scenes):
    gpu_renderer.upload(scenes("input-01"))
    with pytest.raises(pkg.RtError):
        gpu_renderer.render(8, 8, 2, samples=17)
    with pytest.raises(pkg.RtError):
        gpu_renderer.render(8, 8, 2, intersection_only=True, samples=2)
    a = gpu_renderer.render(8, 8, 2, samples=1)
    b = gpu_renderer.render(8, 8, 2, samples=0)
    assert np.abs(a - b).max() <= FP64_TOL      # (atomic accumulation order: equal up to 1e-16)


def test_as2_cli_supersampling_and_f64_frame(pkg, oracle, scenes, tmp_path, monkeypatch):
    """--aa N through the executable (PNG == quantised oracle frame), and the reference-style double-frame path
    of main (AS2_F64_FRAME) writes the same bytes as the default device-quantised path."""
    import subprocess
    from conftest import PKG_DIR
    exe, rti = str(PKG_DIR / "bin" / "as2"), str(scene_path("inputs/input-05.rti"))
    a, b, c = tmp_path / "a.png", tmp_path / "b.png", tmp_path / "c.png"
    for out, extra, env in ((a, ["--aa", "3"], {}), (b, [], {}), (c, [], {"AS2_F64_FRAME": "1"})):
        e = dict(os.environ, **env)
        proc = subprocess.run([exe, rti, "-o", str(out), "-w", "90", "-h", "70", "--bdepth", "4"] + extra, capture_output=True,
                              text=True, env=e)
        assert proc.returncode == 0, proc.stderr
    sc = scenes("input-05")
    o3, _, _, _ = oracle.render(sc.flat, 90, 70, 4, ids=False, samples=3)
    o1, _, _, _ = oracle.render(sc.flat, 90, 70, 4, ids=False)
    d3 = np.abs(decode_png(a).astype(np.int16) - quantize(o3).astype(np.int16))
    assert int(d3.max()) <= 1 and float((d3 == 0).mean()) > 0.999       # truncating quantiser at 1e-16 differences
    assert np.array_equal(decode_png(b), quantize(o1))
    assert np.array_equal(decode_png(b), decode_png(c))
