#!/usr/bin/env python3
"""rt_scene_refit against rt_scene_upload on the 1 M-triangle synthetic scene, and what the refit tree costs a frame.

    python tools/refit_bench.py [--reps 5] [--frames 3]

Scenes: A = HostScene.synthetic(708, 1000, 184), B = the same with seed 185 (every terrain vertex and every sphere
moved, the sphere materials changed, the structure unchanged), and A under a small rigid motion (every transform,
the camera and the point lights shifted by (0.5, 0, 0.3)).

Measured, each as the median of --reps runs:
  * upload of B, and refits of A's upload to B from host faces and from device faces (RT_SCENE_FACES_ON_DEVICE, a
    torch tensor), and to the rigid motion without faces: device time (rt_stats ms_upload + ms_build, CUDA events)
    and wall time of the blocking call;
  * the 8K frame (7680x4320, depth 5, device RGB8 output, rt_stats ms_trace) after a fresh upload of B, after upload
    A + refit B, and after upload A + the rigid-motion refit; with the LBVH wide-node visits of a counted
    1920x1080 frame of each, which show what the refit tree gives up.
Prints one JSON line, with the GPU's name and power limit read in the same run.
"""
import argparse
import importlib.util
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))


def load_package():
    name = "cs184_raytracer_b200"
    spec = importlib.util.spec_from_file_location(name, ROOT / "cs184-raytracer_b200" / "__init__.py",
                                                  submodule_search_locations=[str(ROOT / "cs184-raytracer_b200")])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def gpu_info(torch):
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("refit_bench.py needs a CUDA device")
    pkg = load_package()
    from test_gpu_refit import Desc, face_arrays

    a = pkg.HostScene.synthetic(708, 1000, 184)
    b = pkg.HostScene.synthetic(708, 1000, 185)
    rigid = Desc(pkg, a.flat, a).translate((0.5, 0.0, 0.3)).without_faces()
    pts, nrm = face_arrays(pkg, b.flat)
    b_dev = Desc(pkg, b.flat, b).with_faces(torch.from_numpy(pts).cuda(), torch.from_numpy(nrm).cuda(), on_device=True)
    torch.cuda.synchronize()
    r = pkg.Renderer(0)

    def timed(call):
        t0 = time.perf_counter()
        call()
        wall = (time.perf_counter() - t0) * 1e3
        st = r.stats()
        return st["ms_upload"] + st["ms_build"], wall, st

    def medians(runs):
        return {"device_ms": round(statistics.median(x[0] for x in runs), 3),
                "wall_ms": round(statistics.median(x[1] for x in runs), 3),
                "kernel_launches": runs[-1][2]["kernel_launches"], "scene_bytes_h2d": runs[-1][2]["scene_bytes_h2d"]}

    ops = {"upload": [], "refit_host_faces": [], "refit_device_faces": [], "refit_no_faces": []}
    for _ in range(args.reps + 1):                  # the first round warms up
        ops["upload"].append(timed(lambda: r.upload(b)))
        r.upload(a)
        ops["refit_host_faces"].append(timed(lambda: r.refit(b)))
        r.upload(a)
        ops["refit_device_faces"].append(timed(lambda: r.refit(b_dev.ptr)))
        r.upload(a)
        ops["refit_no_faces"].append(timed(lambda: r.refit(rigid.ptr)))
    result = {k: medians(v[1:]) for k, v in ops.items()}

    W, H, DEPTH = 7680, 4320, 5
    out = torch.empty(H * W * 3, dtype=torch.uint8, device="cuda")
    params = pkg.make_params(W, H, DEPTH)

    def frame_and_visits():
        times = []
        for k in range(args.frames + 1):
            r.render_device(params, out.data_ptr(), rgb8=True)
            torch.cuda.synchronize()
            if k:
                times.append(r.stats()["ms_trace"])
        r.render(1920, 1080, DEPTH, flags=pkg.RT_FLAG_COUNT_WORK)
        st = r.stats()
        return {"frame_ms": round(statistics.median(times), 3), "node_visits_1080p": int(sum(st["nodes_fetched"])),
                "rays_1080p": [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]]}

    r.upload(b)
    frames = {"upload_b": frame_and_visits()}
    r.upload(a)
    r.refit(b)
    frames["upload_a_refit_b"] = frame_and_visits()
    r.upload(a)
    r.refit(rigid.ptr)
    frames["upload_a_refit_rigid"] = frame_and_visits()
    r.upload(Desc(pkg, a.flat, a).translate((0.5, 0.0, 0.3)).ptr)
    frames["upload_rigid"] = frame_and_visits()
    r.close()
    name, power = gpu_info(torch)
    print(json.dumps({"gpu": name, "power_limit": power, "scene": "synthetic(708, 1000): 1,002,528 triangles + 1000 spheres",
                      "reps": args.reps, "scene_ops": result, "frames_8k_depth5": frames}))


if __name__ == "__main__":
    main()
