"""Bounce chains as deep as rt_params.bounce_depth allows (65535).

A ray between two facing mirrors spawns a reflected child at every hit, however small its weight, so its chain
only ends at the depth limit.  The render driver runs the levels of such a chain in a loop, on the calling thread
and on the worker threads of an n_gpus > 1 render alike: the depth must not be limited by a host thread's stack."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
FP64_TOL = 1e-9
MAX_DEPTH = 65535
# ka kd ks sp kr: a half-silvered mirror (the weight of a chain halves per bounce and underflows to zero long
# before the depth limit; the rays are spawned all the same)
MIRROR = "mat 0.1 0.1 0.1  0.5 0.4 0.3  0.2 0.2 0.2  10  0.5 0.5 0.5\n"
# two lights that cast shadow rays: a point light between the mirrors and a directional one along the axis
LIGHTS = "lta 0.1 0.1 0.1\nltp 0.3 0.2 0 1 1 1\nltd 0.1 0.2 -1 0.5 0.5 0.5\n"
SHADOW_LIGHTS = 2


def _rect(corner, u, v):
    """Parallelogram corner, corner + u, corner + u + v, corner + v as two `tri`s."""
    c = np.array(corner, float)
    a, b, cc, d = c, c + u, c + np.add(u, v), c + v
    return "".join("tri " + " ".join(f"{x:g}" for p in t for x in p) + "\n" for t in ((a, b, cc), (a, cc, d)))


def _scene(pkg, tmp_path, name, text):
    rti = tmp_path / name
    rti.write_text(text)
    return pkg.HostScene.load(rti)


def _mirror_pair(pkg, tmp_path):
    """Mirrors at z = -1 and z = +1, camera at the origin looking down -z: the centre ray of the image hits a
    mirror perpendicularly and bounces straight back every time."""
    cam = "cam 0 0 0  -1 -1 -1  1 -1 -1  -1 1 -1  1 1 -1\n"
    # the diagonals of the two rectangles miss the z axis
    text = cam + LIGHTS + MIRROR + _rect((-900, -800, -1), (2000, 0, 0), (0, 2000, 0)) + \
        _rect((-1100, -1200, 1), (2000, 0, 0), (0, 2000, 0))
    return _scene(pkg, tmp_path, "mirrors.rti", text)


def test_one_ray_bounces_to_the_depth_limit(pkg, gpu_renderer, tmp_path):
    gpu_renderer.upload(_mirror_pair(pkg, tmp_path))
    gpu_renderer.render(1, 1, MAX_DEPTH)
    st = gpu_renderer.stats()
    assert st["rays_primary"] == 1
    assert st["hits"] == MAX_DEPTH + 1
    assert st["rays_secondary"] == MAX_DEPTH
    assert st["rays_shadow"] == (MAX_DEPTH + 1) * SHADOW_LIGHTS
    assert st["degenerate_rays"] == 0


def test_deep_chains_match_the_oracle(pkg, gpu_renderer, oracle, tmp_path):
    """Rays near the axis stay between the mirrors for thousands of bounces: depth 1000, which the recursive
    oracle still handles, against the oracle."""
    sc = _mirror_pair(pkg, tmp_path)
    gpu_renderer.upload(sc)
    w, h, depth = 16, 16, 1000
    rgb = gpu_renderer.render(w, h, depth)
    st = gpu_renderer.stats()
    o_rgb, _, _, counts = oracle.render(sc.flat, w, h, depth, ids=False)
    assert [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]] == counts[:3]
    assert st["rays_secondary"] > 100 * w * h
    assert np.abs(rgb - o_rgb).max() <= FP64_TOL


def test_worker_threads_run_deep_chains(pkg, tmp_path, monkeypatch):
    """A closed box of mirrors with the camera and the light inside: every ray bounces until the depth runs out.  A
    64x32 frame is two tiles, one per device of an n_gpus = 2 render, so each worker thread runs 65536 levels."""
    import torch
    if torch.cuda.device_count() < 2:
        monkeypatch.setenv("RT_MULTI_SAME_DEVICE", "1")
    lo, hi = np.array([-4.0, -3.0, -5.0]), np.array([5.0, 6.0, 4.0])
    walls = ""
    for axis in range(3):
        u, v = np.zeros(3), np.zeros(3)
        i, j = [a for a in range(3) if a != axis]
        u[i], v[j] = hi[i] - lo[i], hi[j] - lo[j]
        for value in (lo[axis], hi[axis]):
            corner = lo.copy()
            corner[axis] = value
            walls += _rect(corner, u, v)
    cam = "cam 0.3 0.2 0.1  -0.7 -0.8 -0.9  1.3 -0.8 -0.9  -0.7 1.2 -0.9  1.3 1.2 -0.9\n"
    text = cam + "lta 0.1 0.1 0.1\nltp 1 1.5 -1 1 1 1\n" + MIRROR + walls
    r = pkg.Renderer(0)
    try:
        r.upload(_scene(pkg, tmp_path, "box.rti", text))
        w, h = 64, 32
        one = r.render(w, h, MAX_DEPTH)
        s1 = r.stats()
        two = r.render(w, h, MAX_DEPTH, n_gpus=2)
        s2 = r.stats()
        for k in ("rays_primary", "rays_shadow", "rays_secondary", "hits"):
            assert s1[k] == s2[k], k
        assert s1["rays_secondary"] > (MAX_DEPTH - 100) * w * h
        assert np.abs(one - two).max() <= FP64_TOL
    finally:
        r.close()
