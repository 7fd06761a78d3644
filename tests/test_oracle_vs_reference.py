"""Pins the oracle: oracle/whitted_oracle.c against the UNMODIFIED reference hot path
(oracle/_ref/libref.so, built by oracle/Makefile from the reference's own sources) and
against outputs of that reference stored in tests/golden/ref/.  Everything here is bit-exact:
the restatement reproduces the reference's FP64 association order and both use glibc libm.
"""
import numpy as np
import pytest

from conftest import GOLDEN, decode_png, load_ref_fixture, quantize, scene_path

FIXTURE_SCENES = {
    **{f"input-{i:02d}": f"inputs/input-{i:02d}.rti" for i in range(1, 10)},
    "refraction3": "excess_inputs/refraction3.rti", "refraction": "excess_inputs/refraction.rti",
    "test": "excess_inputs/test.rti", "example5": "excess_inputs/example5.rti",
    "reflective_specular_test": "excess_inputs/reflective_specular_test.rti", "bunny4": "excess_inputs/bunny4.rti",
}
CHEAP = ["input-01", "input-05", "input-06", "input-07", "input-08", "input-09", "refraction3", "refraction", "test",
         "example5", "reflective_specular_test"]


@pytest.mark.parametrize("name", sorted(FIXTURE_SCENES))
def test_oracle_equals_stored_reference_outputs(pkg, oracle, name):
    """96x96 (80x45 for the heavy meshes): FP64 framebuffer, hit ids and ray count identical."""
    w, h = (80, 45) if name in ("input-03", "bunny4", "input-02", "input-04") else (96, 96)
    fx = load_ref_fixture(name, w, h)
    sc = pkg.HostScene.load(scene_path(FIXTURE_SCENES[name]))
    rgb, geom, face, counts = oracle.render(sc.flat, w, h, int(fx["depth"]))
    assert np.array_equal(rgb, fx["rgb"]), "framebuffer differs from the reference bit pattern"
    assert np.array_equal(geom, fx["geom"])
    assert np.array_equal(face, fx["face"]), "face ids differ from the reference's (ref_primary_faces)"
    assert sum(counts[:3]) == int(fx["castray_calls"])
    assert counts[3] == 0
    io, _, _, _ = oracle.render(sc.flat, w, h, int(fx["depth"]), intersection_only=True, ids=False)
    assert np.array_equal(io[..., 0], fx["intersection_only"])


@pytest.mark.parametrize("name", CHEAP)
def test_oracle_cast_and_trace_rays_vs_live_reference(pkg, oracle, reference, name):
    """Per-ray Scene::castRay / Scene::traceRay against the live reference library, including
    rays that START on surfaces (the +-eps `tri` pair and sphere-root logic) and both
    reverseNormals / fromInside values."""
    path = scene_path(FIXTURE_SCENES[name])
    sc = pkg.HostScene.load(path)
    h = reference.load(path)
    rng = np.random.default_rng(7)
    w = hh = 64
    pix = np.arange(w * hh)
    org, direction = oracle.camera_rays(sc.flat, w, hh, pix)
    g, f, d, p, n = oracle.cast_rays(sc.flat, org, direction)
    hit = g >= 0
    org2 = np.where(hit[:, None], p, org)
    dir2 = rng.normal(size=org.shape)
    orgs = np.concatenate([org, org2]); dirs = np.concatenate([direction, dir2])
    for rev in (0, 1):
        revs = np.full(orgs.shape[0], rev, np.uint8)
        og = oracle.cast_rays(sc.flat, orgs, dirs, revs)
        rg = reference.cast_rays(h, orgs, dirs, revs)
        assert np.array_equal(og[0], rg[0])
        assert np.array_equal(og[2], rg[1]) and np.array_equal(og[3], rg[2]) and np.array_equal(og[4], rg[3])
        fi = np.full(orgs.shape[0], rev, np.uint8)
        assert np.array_equal(oracle.trace_rays(sc.flat, orgs, dirs, 10, fi), reference.trace_rays(h, orgs, dirs, 10, fi))


def test_reference_shim_loop_equals_stock_renderScene(reference):
    """Our clamped pixel loop around the reference's traceRay == the reference's own
    Scene::renderScene where that one is safe (W*H % 2000 == 0)."""
    h = reference.load(scene_path("inputs/input-05.rti"))
    a, _, _, _ = reference.render(h, 100, 80, 10, threads=4)
    b, _, _, _ = reference.render(h, 100, 80, 10, threads=4, stock=True)
    assert np.array_equal(a, b)


def test_oracle_keeps_a_negative_zero_like_std_max(pkg, oracle, live_reference, tmp_path):
    """std::max(x, 0.0) is (x < 0.0) ? 0.0 : x, so it hands x = -0.0 on, and pow(-0.0, -1) is -inf.  On the centre
    column of test_gpu_shading's axis-aligned wall -V.R is exactly -0.0: with sp = -1 the reference's specular term
    is -inf there, with sp = -2 it is +inf.  Without the live reference this pins the oracle to the semantics of
    std::max as the C++ standard defines it; where the reference is built, the frame must also equal its own."""
    from test_gpu_shading import H_AX, W_AX, exponent_scene, write_scene
    for sp, inf in ((-1.0, -np.inf), (-2.0, np.inf)):
        sc, path = write_scene(pkg, tmp_path, f"sp_{sp}.rti", exponent_scene(sp))
        rgb, _, _, _ = oracle.render(sc.flat, W_AX, H_AX, 2, ids=False)
        centre = rgb[:, W_AX // 2, 0]
        assert (centre == inf).any() and not (centre == -inf).any()
        if live_reference is not None:
            r_rgb, _, _, _ = live_reference.render(live_reference.load(path), W_AX, H_AX, 2, threads=2)
            assert np.array_equal(rgb, r_rgb, equal_nan=True)
            assert np.array_equal(np.signbit(rgb), np.signbit(r_rgb))


GOLDEN_FULL = {"01": 1000, "05": 1000, "06": 1000, "07": 1000, "08": 1000, "09": 2000}


@pytest.mark.parametrize("n", sorted(GOLDEN_FULL))
def test_oracle_reproduces_golden_images(pkg, oracle, n):
    """The reference's known-answer vectors outputs/image-0N.png (notes/notes-0N.txt command
    lines): decoded pixels identical.  Mesh scenes 02-04 take minutes on the CPU and are
    covered at full size by the GPU suite and here at fixture size."""
    size = GOLDEN_FULL[n]
    sc = pkg.HostScene.load(scene_path(f"inputs/input-{n}.rti"))
    rgb, _, _, _ = oracle.render(sc.flat, size, size, 10, ids=False)
    gold = decode_png(GOLDEN / "outputs" / f"image-{n}.png")
    assert np.array_equal(quantize(rgb), gold)


@pytest.mark.parametrize("name,sub", [("inputs/input-05.rti", 2), ("inputs/input-06.rti", 3), ("excess_inputs/refraction3.rti", 2)])
def test_oracle_supersampling_is_the_mean_of_reference_traces(pkg, oracle, reference, name, sub):
    """SURVEY section 8 f-4.  rt_params.samples = n is defined as the mean of the reference's traceRay over the
    centres of an n x n grid inside each pixel.  The unmodified reference traces the sample rays (built here
    in numpy with Camera::calculateViewingRay's blend, src/rtbase.h:74-84); the oracle's loop must agree.
    (ref_trace_rays re-normalises the direction through the Ray constructor, hence 1e-12 and not 0.)"""
    sc = pkg.HostScene.load(scene_path(name))
    h = reference.load(scene_path(name))
    w, hh, depth = 23, 17, 4
    cam = pkg.flat_arrays(sc.flat)["camera"]
    E, LL, LR, UL, UR = (cam[3 * k:3 * k + 3] for k in range(5))
    orgs, dirs = [], []
    for r in range(hh):
        for c in range(w):
            for sj in range(sub):
                for si in range(sub):
                    rowf = (r + (sj + 0.5) / sub) / hh
                    colf = (c + (si + 0.5) / sub) / w
                    right = rowf * LR + (1.0 - rowf) * UR
                    left = rowf * LL + (1.0 - rowf) * UL
                    raw = (colf * right + (1.0 - colf) * left) - E
                    orgs.append(E)
                    dirs.append(raw)
    cols = reference.trace_rays(h, np.array(orgs), np.array(dirs), depth)
    mean = cols.reshape(hh, w, sub * sub, 3).sum(axis=2) / (sub * sub)
    rgb, _, _, counts = oracle.render(sc.flat, w, hh, depth, ids=False, samples=sub)
    assert counts[0] == w * hh * sub * sub
    assert np.abs(rgb - mean).max() <= 1e-12
    one, _, _, c1 = oracle.render(sc.flat, w, hh, depth, ids=False, samples=1)
    zero, _, _, c0 = oracle.render(sc.flat, w, hh, depth, ids=False, samples=0)
    assert np.array_equal(one, zero) and c1 == c0 and c1[0] == w * hh


def test_oracle_equals_the_reference_on_the_benchmark_scene(pkg, oracle):
    """bench.py's synthetic scene (1,002,528 triangles + 1000 spheres, seed 184) as rendered by the unmodified
    reference through ref_scene_from_flat (make_fixtures.py): the restatement must agree bit for bit, face ids
    included.  96x54 at depth 5 = 71,771 rays against a million faces each (about 20 s on 8 threads)."""
    fx = np.load(GOLDEN / "ref" / "synthetic_96x54.npz")
    cells, spheres, seed = (int(x) for x in fx["synthetic"])
    sc = pkg.HostScene.synthetic(cells, spheres, seed)
    rgb, geom, face, counts = oracle.render(sc.flat, 96, 54, int(fx["depth"]))
    assert np.array_equal(rgb, fx["rgb"])
    assert np.array_equal(geom, fx["geom"]) and np.array_equal(face, fx["face"])
    assert sum(counts[:3]) == int(fx["castray_calls"]) and counts[3] == 0
    assert (fx["geom"] == 0).any() and (fx["geom"] > 0).any()        # terrain and spheres both in view


def test_big_fixture_consistency(pkg, oracle):
    """The full-size BASELINE fixtures (8-bit frame + strided FP64 samples + ids): the cheapest one, bunny4 at
    960x540... is still minutes of CPU, so the oracle is checked on a sample of refraction3 (spheres only) instead:
    every 48th pixel in both directions via per-ray traces through the same camera."""
    fx = np.load(GOLDEN / "ref" / "big_refraction3_3840x2160.npz")
    sc = pkg.HostScene.load(scene_path("excess_inputs/refraction3.rti"))
    w, h, s = 3840, 2160, int(fx["stride"])
    rows, cols = np.arange(0, h, s)[::6], np.arange(0, w, s)[::6]
    pix = (rows[:, None] * w + cols[None, :]).ravel()
    org, direction = oracle.camera_rays(sc.flat, w, h, pix)
    rgb = oracle.trace_rays(sc.flat, org, direction, int(fx["depth"]))
    want = fx["rgb_sub"][::6, ::6].reshape(-1, 3)
    assert np.abs(rgb - want).max() <= 1e-12     # trace_rays re-normalises the (already unit) direction: not bit-identical
    g, f, _, _, _ = oracle.cast_rays(sc.flat, org, direction)
    assert np.array_equal(g, fx["geom"][::s, ::s][::6, ::6].ravel().astype(np.int32))
    assert np.array_equal(f, fx["face"][::s, ::s][::6, ::6].ravel())
    assert np.array_equal(quantize(fx["rgb_sub"]), fx["rgb8"][::s, ::s])


ALL_LOADABLE = sorted(p for p in list((GOLDEN / "inputs").glob("*.rti")) + list((GOLDEN / "excess_inputs").glob("*.rti"))
                      if p.name not in ("teapot.rti",))   # excess teapot.rti has no teapot.obj beside it


@pytest.mark.parametrize("path", ALL_LOADABLE, ids=lambda p: p.parent.name + "/" + p.name)
def test_oracle_equals_live_reference_on_every_shipped_scene(pkg, oracle, reference, path):
    """Every loadable scene the reference ships (25), not only the 15 with stored fixtures: a 40x30 frame of the
    restatement against the live unmodified reference — FP64 frame, geometry ids and castRay count bit for bit."""
    sc = pkg.HostScene.load(path)
    h = reference.load(path)
    w, hh, depth = 40, 30, 6
    rgb, geom, _, counts = oracle.render(sc.flat, w, hh, depth)
    counting = getattr(test_oracle_equals_live_reference_on_every_shipped_scene, "_counting", None)
    if counting is None:
        from conftest import Reference
        counting = Reference(counting=True)
        test_oracle_equals_live_reference_on_every_shipped_scene._counting = counting
    r_rgb, r_geom, _, calls = counting.render(counting.load(path), w, hh, depth, threads=4, ids=True)
    assert np.array_equal(rgb, r_rgb)
    assert np.array_equal(geom, r_geom)
    assert sum(counts[:3]) == calls and counts[3] == 0
    a_rgb, _, _, _ = reference.render(h, w, hh, depth, threads=4)
    assert np.array_equal(a_rgb, r_rgb)
