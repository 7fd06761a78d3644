#!/usr/bin/env python3
"""bench.py — Mrays/s of the per-pixel trace loop (BASELINE.json metric) on 1..8 B200.

A "step" is one frame of the workload rendered by the hot path: ray generation, wavefront
trace/shade/shadow loop over all bounce levels and the device-side 8-bit resolve.  With N > 1
ranks every rank's resolve kernel stores its interleaved tiles straight into ONE frame in rank
0's memory (CUDA IPC mapping, NVLink peer stores: rt_shared_frame_* + RT_FLAG_FULL_FRAME), so
there is no gather collective and no unpack pass; `--assemble nccl` keeps round 1's
dist.gather + unpack as the A/B.  A "ray" is one reference castRay call (primary + shadow +
secondary; reference src/scene.cpp:65,91,127,134).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference]
                  [--assemble peer|nccl] [--configs all|none] [--dump-outputs DIR]

N > 1 is launched by the driver with torch.distributed.run (one rank per GPU, NCCL).
`--impl reference` times the reference's own CPU implementation of the path
(oracle/_ref/libref.so = the unmodified reference sources behind a C shim) on the host
cores, each step a bounded pixel sample of the same workload.

Only the cpu_baseline leg and `--impl reference` execute anything under oracle/.
"""
import argparse
import ctypes as C
import hashlib
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
PKG_DIR = ROOT / "cs184-raytracer_b200"
GOLDEN = ROOT / "tests" / "golden"

WORKLOADS = {
    # name: (scene spec, width, height, depth, description)
    "synthetic": (("synthetic", 708, 1000, 184), 7680, 4320, 5,
                  "BASELINE configs[4]: synthetic 1,002,528-triangle height field + 1000 spheres, 8 shadow lights, depth 5, 7680x4320"),
    "synthetic4k": (("synthetic", 708, 1000, 184), 3840, 2160, 5,
                    "configs[4] scene at 3840x2160 (the >=1 Grays/s target is stated at 4K)"),
    "teapot": (("file", "inputs/input-02.rti"), 1920, 1080, 10, "BASELINE configs[1]: teapot.obj scene at 1920x1080, depth 10"),
    "refraction3": (("file", "excess_inputs/refraction3.rti"), 3840, 2160, 10, "BASELINE configs[2]: refraction3.rti at 3840x2160"),
    "bunny": (("file", "excess_inputs/bunny4.rti"), 3840, 2160, 10, "BASELINE configs[3] stand-in: bunny.obj, 4 lights, 3840x2160"),
    "input01": (("file", "inputs/input-01.rti"), 1000, 1000, 10, "BASELINE configs[0]: input-01.rti at 1000x1000"),
}


def load_package():
    name = "cs184_raytracer_b200"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, PKG_DIR / "__init__.py", submodule_search_locations=[str(PKG_DIR)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def build_scene(pkg, spec):
    if spec[0] == "synthetic":
        return pkg.HostScene.synthetic(spec[1], spec[2], spec[3])
    return pkg.HostScene.load(GOLDEN / spec[1])


# ---------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the unmodified reference hot path on the host cores
# ---------------------------------------------------------------------------------------
class RefLib:
    def __init__(self, counting):
        path = ROOT / "oracle" / "_ref" / ("libref_count.so" if counting else "libref.so")
        if not path.exists():
            raise FileNotFoundError(str(path))
        self.lib = C.CDLL(str(path))
        self.lib.ref_scene_load.restype = C.c_void_p
        self.lib.ref_scene_load.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_char_p, C.c_int]
        self.lib.ref_scene_from_flat.restype = C.c_void_p
        self.lib.ref_scene_from_flat.argtypes = [C.c_void_p, C.c_char_p, C.c_int]

    def scene(self, pkg, spec, host_scene):
        err = C.create_string_buffer(512)
        if spec[0] == "synthetic":
            h = self.lib.ref_scene_from_flat(C.cast(host_scene.flat, C.c_void_p), err, 512)
        else:
            arr = (C.c_char_p * 1)(str(GOLDEN / spec[1]).encode())
            h = self.lib.ref_scene_load(arr, 1, err, 512)
        if not h:
            raise RuntimeError(err.value.decode())
        return C.c_void_p(h)

    def render(self, h, w, hh, depth, threads):
        rgb = np.zeros((hh, w, 3))
        sec, calls = C.c_double(), C.c_uint64()
        self.lib.ref_render(h, w, hh, depth, 0, threads, rgb.ctypes.data_as(C.c_void_p), None, C.byref(sec), C.byref(calls))
        return sec.value, int(calls.value)


def sample_size(width, height, px_budget):
    """Same camera, same aspect, fewer pixels (the ray mix is resolution independent)."""
    if width * height <= px_budget:
        return width, height
    s = (px_budget / (width * height)) ** 0.5
    return max(16, int(width * s)), max(9, int(height * s))


def reference_runs(pkg, wl_name, steps, warmup, target_s):
    """Times the reference on a bounded sample.  Returns dict(value Mrays/s, ms_per_step, ...)."""
    spec, width, height, depth, _ = WORKLOADS[wl_name]
    threads = os.cpu_count() or 1
    # silence the parsers' per-line .obj warnings
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(2)
    os.dup2(devnull, 2)
    try:
        host_scene = build_scene(pkg, spec)
        timed, counted = RefLib(False), RefLib(True)
        h_t = timed.scene(pkg, spec, host_scene)
        h_c = counted.scene(pkg, spec, host_scene)
    finally:
        os.dup2(saved, 2)
        os.close(devnull)
        os.close(saved)
    # calibrate on a tiny frame, then size the sample for ~target_s per step; the counting
    # build (castRay counter behind a linker --wrap) renders the sample once: that run gives
    # the exact ray count and doubles as the first warm-up
    cw, ch = sample_size(width, height, 12 * 7)
    t_cal, _ = timed.render(h_t, cw, ch, depth, threads)
    per_px = max(t_cal / (cw * ch), 1e-9)
    sw, sh = sample_size(width, height, max(cw * ch, int(target_s / per_px)))
    t_cnt, rays = counted.render(h_c, sw, sh, depth, threads)
    if t_cnt < 0.4 * target_s and (sw, sh) != (width, height):      # calibration was pessimistic: resize once
        sw, sh = sample_size(width, height, int(sw * sh * 0.8 * target_s / max(t_cnt, 1e-6)))
        t_cnt, rays = counted.render(h_c, sw, sh, depth, threads)
    for _ in range(max(warmup - 1, 0)):
        timed.render(h_t, sw, sh, depth, threads)
    times = [timed.render(h_t, sw, sh, depth, threads)[0] for _ in range(steps)]
    total = sum(times)
    return {
        "value": rays * steps / total / 1e6, "ms_per_step": 1e3 * total / steps, "cores": threads,
        "sample": f"{sw}x{sh} pixel subsample of the {width}x{height} frame (same camera, depth {depth}), "
                  f"{rays} rays per step, all {threads} host threads, unmodified reference traceRay/castRay",
        "rays_per_step": rays, "sample_w": sw, "sample_h": sh,
    }


# ---------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons during the timed region: NVML polled every 10 ms from a thread (the same
    counters nvidia-smi prints; the timed region of a small workload is shorter than one nvidia-smi period),
    falling back to `nvidia-smi -lms 100` when the NVML binding is unavailable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None
        self.stop_flag, self.nvml, self.source = threading.Event(), None, None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x.strip() for x in vis.split(",") if x.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = [pynvml.nvmlClocksThrottleReasonHwSlowdown, pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    pynvml.nvmlClocksThrottleReasonSwThermalSlowdown, pynvml.nvmlClocksThrottleReasonSwPowerCap]

            def poll():
                while not self.stop_flag.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.rows.append([sm, mx] + ["Active" if r & b else "Not Active" for b in bits] + [0.0])
                    except Exception:
                        pass
                    self.stop_flag.wait(0.01)
            self.nvml, self.source = pynvml, "nvml, 10 ms"
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self._physical_index()}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.source = "nvidia-smi -lms 100"

        def pump():
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            if self.thread:
                self.thread.join(timeout=2)
        elif self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            if self.thread:
                self.thread.join(timeout=2)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for k, nm in enumerate(self.NAMES):
                if str(r[2 + k]).lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.source}


# ---------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------
class RawDevice:
    """__cuda_array_interface__ over a raw device pointer, so torch can view library-owned memory."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}


# stored outputs of the UNMODIFIED reference (tests/golden/make_fixtures.py) each workload is checked against, and
# the frame size of that check (the fixture's size: full size where the reference finishes in a minute of CPU)
PARITY_FIXTURE = {
    "synthetic": ("synthetic_96x54.npz", 96, 54), "synthetic4k": ("synthetic_96x54.npz", 96, 54),
    "teapot": ("big_input-02_1920x1080.npz", 1920, 1080), "refraction3": ("big_refraction3_3840x2160.npz", 3840, 2160),
    "bunny": ("big_bunny4_960x540.npz", 960, 540), "input01": ("input-01_96x96.npz", 96, 96),
}


def parity_check(pkg, ren, wl_name):
    """Single-GPU render of the workload's scene at its fixture size against the reference's stored output:
    primary hit ids (geometry and face) and the castRay count exact, frame within 1e-9 (FP64) or equal (8-bit)."""
    fname, w, h = PARITY_FIXTURE[wl_name]
    path = GOLDEN / "ref" / fname
    if not path.exists():
        return {"against": fname, "ok": None, "note": "fixture missing"}
    fx = np.load(path)
    depth = int(fx["depth"])
    rgb = ren.render(w, h, depth)
    st = ren.stats()
    geom, face = ren.primary_ids(w, h)
    ids_ok = bool(np.array_equal(geom, fx["geom"].astype(np.int32)) and np.array_equal(face, fx["face"]))
    count_ok = st["rays_primary"] + st["rays_shadow"] + st["rays_secondary"] == int(fx["castray_calls"])
    if "rgb" in fx:
        err = float(np.abs(rgb - fx["rgb"]).max())
    else:
        s = int(fx["stride"])
        err = float(np.abs(rgb[::s, ::s] - fx["rgb_sub"]).max())
    return {"against": f"tests/golden/ref/{fname} (unmodified reference, {w}x{h}, depth {depth})", "ids_equal": ids_ok,
            "ray_count_equal": bool(count_ok), "max_abs_diff_fp64": err, "ok": bool(ids_ok and count_ok and err <= 1e-9)}


DUMP_PIXELS = 1 << 21      # --dump-outputs: frames up to this many pixels whole, larger ones as a sample of this size


def dump_outputs(out_dir, frame, height, width, rays_cls):
    """What the timed path returned in its last step, for comparing two builds output for output: the RGB8 frame as
    float32 (frame_rgb8.npy, H x W x 3), or for a frame of more than DUMP_PIXELS pixels the pixels at fixed positions
    (seed 0, sorted; frame_rgb8_sample.npy, n x 3, and their row-major indices in frame_sample_index.npy), and the
    primary / shadow / secondary ray counts (rays_per_class.npy).  At most 42 MB in all."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    if frame is not None:
        img = frame.cpu().numpy().reshape(height * width, 3)
        if height * width <= DUMP_PIXELS:
            np.save(out / "frame_rgb8.npy", img.reshape(height, width, 3).astype(np.float32))
        else:
            idx = np.unique(np.random.default_rng(0).integers(0, height * width, DUMP_PIXELS))
            np.save(out / "frame_rgb8_sample.npy", img[idx].astype(np.float32))
            np.save(out / "frame_sample_index.npy", idx.astype(np.float64))
    np.save(out / "rays_per_class.npy", np.array(rays_cls, np.float64))


def load_traffic(wl_name):
    tf = ROOT / "profiles" / "traffic.json"
    try:
        return json.loads(tf.read_text()).get(wl_name, {})
    except Exception:
        return {}


def run_workload(args, pkg, torch, dist, wl_name, headline):
    """Times one workload at the launched world size.  Returns the fields of its JSON record (rank 0) or None."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local_rank)
    spec, width, height, depth, desc = WORKLOADS[wl_name]
    steps, warmup = (args.steps, args.warmup) if headline else (min(args.steps, 5), max(min(args.warmup, 3), 3))
    nbytes = height * width * 3
    config = {"workload": f"{wl_name}: {desc}", "width": width, "height": height, "bounce_depth": depth,
              "partition": f"interleaved 32x32 tiles over {world} rank(s), scene replicated",
              "assemble": "single rank: row-major RGB8 frame on the device" if world == 1 else
                          ("peer: every rank's resolve kernel stores its tiles into rank 0's frame (CUDA IPC mapping, NVLink), "
                           "one 4-byte all-reduce per frame as the completion barrier; two frames in flight (double-buffered)" if args.assemble == "peer" else
                           "nccl: dist.gather of the packed RGB8 tiles + unpack kernel on rank 0 (round-1 path, A/B)"),
              "l2": "no explicit flush: every frame streams its ray and hit queues (80 B / 116 B per record, 10^6..10^8 records per bounce "
                    "level) through the 126 MB L2 between two uses of any scene data"}

    host_scene = build_scene(pkg, spec)
    ren = pkg.Renderer(local_rank)
    ren.upload(host_scene)
    up_stats = ren.stats()
    stream = torch.cuda.current_stream().cuda_stream
    base_flags = pkg.RT_FLAG_TIME_KERNELS
    peer = world > 1 and args.assemble == "peer"
    shared_flag = pkg.RT_FLAG_FULL_FRAME if peer else 0
    p = pkg.make_params(width, height, depth, tile_rank=rank, tile_world=world, flags=base_flags | shared_flag)
    emulate = os.environ.get("RT_BENCH_EMULATE_RANK")      # "r/n": time rank r's share of an n-rank job on one GPU (development aid)
    if emulate and world == 1:
        er, en = (int(x) for x in emulate.split("/"))
        p = pkg.make_params(width, height, depth, tile_rank=er, tile_world=en, flags=base_flags)
        config["partition"] = f"EMULATED rank {er} of {en} (its tiles only, no gather)"
    sub = int(os.environ.get("RT_BENCH_SUB", "0"))         # experiment: k sub-contexts per GPU render this rank's tiles concurrently
    if sub > 1:
        os.environ["RT_MULTI_SAME_DEVICE"] = "1"
        p.n_gpus = sub
        p.flags |= pkg.RT_FLAG_FULL_FRAME
        config["partition"] += f"; {sub} concurrent sub-contexts per GPU"
    if args.in_process > 1 and world == 1:
        # ONE process drives N GPUs through rt_params.n_gpus (what `as2 --gpus N` does): worker thread per device inside
        # the library, scene replicated with peer copies, every device's resolve kernel stores into this frame over NVLink
        p.n_gpus = args.in_process
        config["partition"] = f"interleaved 32x32 tiles over {args.in_process} GPUs of ONE process (rt_params.n_gpus), scene replicated by peer copies"
    own_tiles, max_tiles, total_tiles = pkg.tile_counts(p)
    tick = torch.zeros(1, dtype=torch.int32, device=dev)
    shared_ptr = None
    frame = gathered = packed_all = frames2 = None
    if world == 1 and emulate:
        out = torch.zeros(nbytes if sub > 1 else max_tiles * pkg.RT_TILE_PIXELS * 3, dtype=torch.uint8, device=dev)
        out_ptr = out.data_ptr()
    elif world == 1:
        frame = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out_ptr = frame.data_ptr()
    elif peer:
        # two shared frames (double buffering): frame k goes into buffer k & 1 and its completion barrier is only
        # waited for before frame k + 2 overwrites that buffer, so a rank may run one frame ahead of the slowest
        handle = [None, None]
        shared_ptr = [None, None]
        if rank == 0:
            for b in range(2):
                shared_ptr[b], handle[b] = ren.shared_frame_create(nbytes)
        dist.broadcast_object_list(handle, src=0)
        if rank != 0:
            shared_ptr = [ren.shared_frame_open(h) for h in handle]
        out_ptr = shared_ptr[0]
        if rank == 0:
            frames2 = [torch.as_tensor(RawDevice(ptr, nbytes), device=dev) for ptr in shared_ptr]
            for f in frames2:
                f.zero_()
            frame = frames2[0]
    else:
        out = torch.zeros(max_tiles * pkg.RT_TILE_PIXELS * 3, dtype=torch.uint8, device=dev)
        out_ptr = out.data_ptr()
        # rank r's tiles land in slice r of one buffer: the gather writes them in place (no concatenation pass)
        packed_all = torch.empty(world * out.numel(), dtype=torch.uint8, device=dev) if rank == 0 else None
        gathered = list(packed_all.chunk(world)) if rank == 0 else None
        frame = torch.empty(nbytes, dtype=torch.uint8, device=dev) if rank == 0 else None

    ticks = [torch.zeros(1, dtype=torch.int32, device=dev) for _ in range(2)]
    pending = [None, None]
    counter = {"k": 0}

    def assemble(pp):
        """What follows a rank's render until the frame is complete on rank 0 (round-1 path and the e2e fallback)."""
        if world == 1:
            return
        if peer:
            dist.all_reduce(tick)               # completion barrier: all ranks' peer stores have been synchronised
        else:
            dist.gather(out, gathered, dst=0)
            if rank == 0:
                ren.unpack_tiles(pp, packed_all.data_ptr(), frame.data_ptr(), rgb8=True, stream=stream)

    def drain():
        for b in range(2):
            if pending[b] is not None:
                pending[b].wait()
                pending[b] = None

    def step():
        if not peer:
            ren.render_device(p, out_ptr, rgb8=True, stream=stream)
            assemble(p)
            return
        b = counter["k"] & 1
        counter["k"] += 1
        if pending[b] is not None:
            pending[b].wait()                   # frame k - 2 is complete on every rank: its buffer may be overwritten
        ren.render_device(p, shared_ptr[b], rgb8=True, stream=stream)     # returns when this rank's tiles are stored
        pending[b] = dist.all_reduce(ticks[b], async_op=True)              # 4-byte completion barrier of frame k

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 0)):
        step()
    drain()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg = {"ms_kernel": np.zeros(4), "launches_kernel": np.zeros(4), "launches": 0}
    e0.record()
    for _ in range(steps):
        step()
        st = ren.stats()
        agg["ms_kernel"] += np.array(st["ms_kernel"]); agg["launches_kernel"] += np.array(st["launches_kernel"])
        agg["launches"] += st["kernel_launches"] + (1 if (world > 1 and rank == 0 and not peer) else 0)
    drain()                                     # the last frames' barriers belong to the timed region
    e1.record()
    sync_all()
    if peer and rank == 0:
        frame = frames2[(counter["k"] - 1) & 1]      # the frame rendered last
    clocks = sampler.stop() if rank == 0 else None
    ms_total = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    rays = torch.tensor([st["rays_primary"], st["rays_shadow"], st["rays_secondary"], agg["launches"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        dist.all_reduce(rays, op=dist.ReduceOp.SUM)
    ms_total = float(ms_total.item())
    rays_cls = [int(x) for x in rays[:3].tolist()]
    rays_frame = sum(rays_cls)
    launches_total = int(rays[3].item())
    value = rays_frame * steps / (ms_total * 1e-3) / 1e6
    if args.dump_outputs and headline and rank == 0:
        dump_outputs(args.dump_outputs, frame, height, width, rays_cls)

    # ---------------- the assembled frame against a single-rank render of the same frame (rank 0, after the timed region)
    frame_check = None
    if world > 1 and rank == 0:
        multi = frame.clone()
        single = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        ren.render_device(pkg.make_params(width, height, depth), single.data_ptr(), rgb8=True, stream=stream)
        torch.cuda.synchronize()
        diff = (multi.to(torch.int16) - single.to(torch.int16)).abs()
        frame_check = {"frame_matches_single_rank": bool(torch.equal(multi, single)), "max_abs_diff_8bit": int(diff.max().item()),
                       "values_differing": int((diff != 0).sum().item()),
                       "sha256_multi": hashlib.sha256(multi.cpu().numpy().tobytes()).hexdigest()[:16],
                       "sha256_single": hashlib.sha256(single.cpu().numpy().tobytes()).hexdigest()[:16]}
        del multi, single, diff
    if world > 1:
        dist.barrier()

    # ---------------- end-to-end: HOST buffers in, HOST frame out, every step
    #   N = 1: rt_scene_upload from (pinned) host arrays + LBVH build + rt_render_rgb8 into a pinned host frame.
    #   N > 1: every rank copies 1/N of the face arrays over its own PCIe link, one NCCL all-gather over NVLink
    #          replicates them, rt_scene_upload takes them on the device (RT_SCENE_FACES_ON_DEVICE) and builds the LBVH;
    #          the host frame lives in shared memory every rank has page-locked, and each rank's resolve kernel
    #          stores its own tiles into it over its own PCIe link (no funnel through rank 0).
    e2e = None
    if not args.no_e2e and not emulate:
        flat = host_scene.flat.contents
        cudart = torch.cuda.cudart()
        nf = int(flat.num_faces)
        pinned = []

        def pin(addr, n):
            if n and addr and cudart.cudaHostRegister(addr, n, 0) in (0, cudart.cudaError.success):
                pinned.append(addr)
                return True
            return False
        pts_addr = C.cast(flat.face_points, C.c_void_p).value
        nrm_addr = C.cast(flat.face_normals, C.c_void_p).value
        pin(pts_addr, nf * 72)
        pin(nrm_addr, nf * 72)
        shm_path = None
        host_shared = False
        if world == 1:
            host_frame = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
            host_np = host_frame.numpy()
            host_shared = True
        else:
            name = [f"/dev/shm/rt_b200_frame_{os.getpid()}_{wl_name}" if rank == 0 else None]
            dist.broadcast_object_list(name, src=0)
            shm_path = name[0]
            if rank == 0:
                np.zeros(nbytes, np.uint8).tofile(shm_path)
            dist.barrier()
            host_np = np.memmap(shm_path, dtype=np.uint8, mode="r+", shape=(nbytes,))
            ok = torch.tensor([1 if pin(host_np.ctypes.data, nbytes) else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            host_shared = bool(ok.item())
        pe = pkg.make_params(width, height, depth, tile_rank=rank, tile_world=world,
                             flags=pkg.RT_FLAG_FULL_FRAME if world > 1 else 0,
                             n_gpus=args.in_process if (args.in_process > 1 and world == 1) else 0)
        split_upload = world > 1 and nf >= 4096
        if split_upload:
            per = (nf + world - 1) // world
            pts_np = np.ctypeslib.as_array(flat.face_points, shape=(nf * 9,))
            nrm_np = np.ctypeslib.as_array(flat.face_normals, shape=(nf * 9,))
            lo, hi = min(rank * per, nf), min((rank + 1) * per, nf)
            h_slice = torch.zeros(2, per * 9, dtype=torch.float64).pin_memory()
            h_slice[0, :(hi - lo) * 9] = torch.from_numpy(pts_np[lo * 9:hi * 9])
            h_slice[1, :(hi - lo) * 9] = torch.from_numpy(nrm_np[lo * 9:hi * 9])
            d_slice = torch.empty(2, per * 9, dtype=torch.float64, device=dev)
            d_all = torch.empty(world, 2, per * 9, dtype=torch.float64, device=dev)
            d_pts = torch.empty(world * per * 9, dtype=torch.float64, device=dev)
            d_nrm = torch.empty(world * per * 9, dtype=torch.float64, device=dev)
            dev_scene = pkg.rt_scene()
            C.memmove(C.byref(dev_scene), C.byref(flat), C.sizeof(pkg.rt_scene))
            dev_scene.flags = pkg.RT_SCENE_FACES_ON_DEVICE
            dev_scene.face_points = C.cast(C.c_void_p(d_pts.data_ptr()), C.POINTER(C.c_double))
            dev_scene.face_normals = C.cast(C.c_void_p(d_nrm.data_ptr()), C.POINTER(C.c_double))

        def e2e_step():
            if split_upload:
                d_slice.copy_(h_slice, non_blocking=True)                    # 1/N of the faces over this rank's PCIe link
                dist.all_gather_into_tensor(d_all, d_slice)                   # NVLink
                d_pts.view(world, per * 9).copy_(d_all[:, 0])                # rank-major slices -> the two face arrays
                d_nrm.view(world, per * 9).copy_(d_all[:, 1])
                torch.cuda.synchronize()
                ren.upload(C.pointer(dev_scene))
            else:
                ren.upload(host_scene)
            if host_shared:
                ren.render_host_params(pe, host_np.ctypes.data, rgb8=True)   # tiles stored straight into the host frame
                if world > 1:
                    dist.all_reduce(tick)
            else:                                                            # fallback: peer frame on rank 0, one D2H
                ren.render_device(p, out_ptr, rgb8=True, stream=stream)
                assemble(p)
                if rank == 0:
                    torch.from_numpy(host_np).copy_(frames2[0] if peer else frame)
            torch.cuda.synchronize()

        e2e_step()
        sync_all()
        n_e2e = max(1, min(steps, 3))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        sync_all()
        t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        st_e = ren.stats()
        h2d = int(st_e["scene_bytes_h2d"]) + (int(h_slice.numel()) * 8 if split_upload else 0)
        h2d_t = torch.tensor([h2d], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(h2d_t, op=dist.ReduceOp.SUM)
        e2e_matches = None
        if rank == 0 and frame is not None and not emulate:
            ref8 = frame.cpu().numpy()
            d = np.abs(np.asarray(host_np).astype(np.int16) - ref8.astype(np.int16))
            e2e_matches = {"equal_to_device_frame": bool(d.max() == 0), "max_abs_diff_8bit": int(d.max())}
        e2e = {"value": rays_frame * n_e2e / float(t_e2e.item()) / 1e6, "unit": "Mrays/s",
               "h2d_bytes_per_step": int(h2d_t.item()), "d2h_bytes_per_step": nbytes,
               "ms_per_step": 1e3 * float(t_e2e.item()) / n_e2e,
               "ms_scene_upload": st_e["ms_upload"], "ms_lbvh_build": st_e["ms_build"], "steps": n_e2e,
               "host_frame": e2e_matches,
               "path": ("rt_scene_upload (pinned host arrays) + LBVH build + rt_render_rgb8 into a pinned host frame" if world == 1 else
                        ("per-rank 1/N face slices H2D + NCCL all-gather + rt_scene_upload(RT_SCENE_FACES_ON_DEVICE) + LBVH build on every rank" if split_upload
                         else "rt_scene_upload on every rank") +
                        (" + rt_render_rgb8(RT_FLAG_FULL_FRAME): every rank stores its tiles into one page-locked shared-memory host frame over its own PCIe link"
                         if host_shared else " + peer-store frame on rank 0 + one D2H"))}
        for addr in pinned:
            cudart.cudaHostUnregister(addr)
        if shm_path:
            del host_np
            if world > 1:
                dist.barrier()
            if rank == 0:
                try:
                    os.unlink(shm_path)
                except OSError:
                    pass
        if split_upload:
            ren.upload(host_scene)

    # ---------------- roofline of the traversal kernels (rank 0; its own share of the frame when N > 1)
    roofline = None
    if rank == 0:
        ptile = dict(tile_rank=p.tile_rank, tile_world=p.tile_world)
        scratch = torch.empty(max(max_tiles * pkg.RT_TILE_PIXELS * 3, nbytes if world == 1 and not emulate else 0), dtype=torch.uint8, device=dev)
        # one frame with the kernels strictly serialised: durations per kernel class that add up to the frame
        # (in the timed region k_shadow of level l runs beside k_trace / k_shade of level l+1)
        ps = pkg.make_params(width, height, depth, flags=pkg.RT_FLAG_TIME_KERNELS | pkg.RT_FLAG_SERIAL, **ptile)
        ren.render_device(ps, scratch.data_ptr(), rgb8=True, stream=stream)
        serial = ren.stats()
        pc = pkg.make_params(width, height, depth, flags=pkg.RT_FLAG_COUNT_WORK, **ptile)
        ren.render_device(pc, scratch.data_ptr(), rgb8=True, stream=stream)
        cs = ren.stats()
        names = ["k_trace", "k_shade", "k_shadow", "other"]
        ser = np.array(serial["ms_kernel"])
        dom = int(np.argmax(ser[:3]))
        node_bytes, face_bytes = ren.device_bytes()
        peak_hbm, peak_src = 6650.0, "fallback"
        try:
            mp = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
            peak_hbm, peak_src = float(mp["hbm_gbs"]), "measured"
        except Exception:
            pass
        traffic_all = load_traffic(wl_name)      # {kernel: {"dram_bytes_per_frame", "launches_per_frame", "active_lanes"}} from ncu
        if node_bytes > 0:
            walk_c, _ = ren.microbench_node_walk(32, 64)
            walk_d, _ = ren.microbench_node_walk(1, 64)
        else:
            walk_c = walk_d = None
        per_kernel = {}
        for kname, k, cls in (("k_trace", 0, 0), ("k_shadow", 1, 2)):
            ms_k = float(ser[cls])
            visits = cs["nodes_fetched"][k] / 4.0              # wide-node visits (4 child boxes each)
            nrays = (cs["rays_primary"] + cs["rays_secondary"]) if k == 0 else cs["rays_shadow"]
            ach = visits / (ms_k * 1e-3) if ms_k > 0 else 0.0
            prof = traffic_all.get(kname)
            prof = prof if isinstance(prof, dict) else {}
            tr = prof.get("dram_bytes_per_frame") if world == 1 and not emulate else None      # captured on the full single-GPU frame
            per_kernel[kname] = {
                "ms_serial_frame": ms_k, "rays": int(nrays), "node_visits": visits, "visits_per_ray": visits / max(nrays, 1),
                "exact_tests_per_ray": (cs["tris_tested"][k] + cs["spheres_tested"][k]) / max(nrays, 1),
                "achieved_gvisits_s": ach / 1e9,
                "frac_of_coherent_walk": ach / walk_c if walk_c else None,
                "frac_of_divergent_walk": ach / walk_d if walk_d else None,
                "lsu_bytes_gbs": ach * 112 / 1e9,
                "active_lanes_per_instruction_ncu": prof.get("active_lanes"),
                "dram_bytes_per_frame_ncu": tr,
                "dram_gbs": (tr / (ms_k * 1e-3) / 1e9) if (tr and ms_k > 0) else None,
                "dram_frac_of_hbm_peak": (tr / (ms_k * 1e-3) / 1e9 / peak_hbm) if (tr and ms_k > 0) else None}
        domk = names[dom] if names[dom] in per_kernel else "k_shadow"
        dk = per_kernel[domk]
        n_launch = max(serial["launches_kernel"][0 if domk == "k_trace" else 2], 1)
        roofline = {
            # The traversal kernels are bound by the rate at which L1TEX/L2 feed 112-byte node visits to partly divergent
            # warps, not by DRAM (ncu: DRAM 2 % of peak, L1TEX 80-85 %, LSU data pipe 66-82 % busy).  The ceiling is measured
            # on the real node array by rt_microbench_node_walk (the traversal's loads and nothing else, fully coherent warps).
            "bound": "l1tex-node-gather (not hbm: see dram_frac_of_hbm_peak)", "kernel": domk,
            "achieved": dk["achieved_gvisits_s"], "peak": (walk_c / 1e9) if walk_c else None, "unit": "G wide-node visits/s",
            "frac": dk["frac_of_coherent_walk"], "peak_source": "measured in this run: rt_microbench_node_walk(group=32) on the scene's LBVH",
            "traffic": (dk["dram_bytes_per_frame_ncu"] / n_launch) if dk["dram_bytes_per_frame_ncu"] else None,
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of this kernel's launches of one frame / launches (ncu --set full of the single-GPU frame, profiles/traffic.json)",
            "launches_per_step": n_launch, "ms_per_launch": dk["ms_serial_frame"] / n_launch,
            "hbm_peak_gbs": peak_hbm, "hbm_peak_source": peak_src,
            "node_walk_gvisits_s": {"coherent_warp": (walk_c / 1e9) if walk_c else None, "divergent_lanes": (walk_d / 1e9) if walk_d else None},
            "kernels": per_kernel,
            "kernel_share_of_step": float(ser[0 if domk == "k_trace" else 2] / max(serial["ms_trace"], 1e-9)),
            "ms_kernel_per_step": {n: float(v / steps) for n, v in zip(names, agg["ms_kernel"])},
            "ms_kernel_serial_frame": {n: float(v) for n, v in zip(names, serial["ms_kernel"])},
            "ms_serial_frame": float(serial["ms_trace"]),
            "duration_source": "RT_FLAG_SERIAL frame after the timed region (CUDA events around every launch on the launching stream)",
            "note": "ms_kernel_per_step: event-bracketed durations inside the timed region, where k_trace/k_shade of "
                    "bounce level l+1 run beside k_shadow of level l (brackets overlap); ms_kernel_serial_frame: one extra "
                    "frame with RT_FLAG_SERIAL, classes add up to ms_serial_frame",
            "node_array_bytes": node_bytes, "face_record_bytes": face_bytes,
            "work_per_step": {"box_tests": cs["nodes_fetched"], "tris": cs["tris_tested"], "spheres": cs["spheres_tested"],
                              "hits": cs["hits"], "shadow_lights": int(cs["rays_shadow"] // max(cs["hits"], 1)),
                              "shadow_rays_answered_without_traversal": cs["shadow_rays_culled"]}}
        del scratch

    # ---------------- parity of this workload against the stored reference output (rank 0, single-GPU render)
    parity = parity_check(pkg, ren, wl_name) if rank == 0 else None

    # ---------------- cpu baseline (rank 0, N = 1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not emulate:
        try:
            r = reference_runs(pkg, wl_name, 1, 0, target_s=12.0 if headline else 3.0)
            cpu = {"value": r["value"], "unit": "Mrays/s", "cores": r["cores"], "kind": "reference", "sample": r["sample"]}
        except FileNotFoundError as e:
            cpu = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {e}"}

    if peer and shared_ptr is not None:
        frame = frames2 = None
        torch.cuda.synchronize()
        dist.barrier()
        if rank != 0:
            for ptr in shared_ptr:
                ren.shared_frame_close(ptr)
        dist.barrier()
        if rank == 0:
            for ptr in shared_ptr:
                ren.shared_frame_close(ptr)
    ren.close()
    host_scene.close()
    if rank != 0:
        return None
    return {"value": value, "ms_per_step": ms_total / steps, "steps": steps, "warmup": warmup, "config": config,
            "rays_per_step": {"primary": rays_cls[0], "shadow": rays_cls[1], "secondary": rays_cls[2]},
            "frame_ms": ms_total / steps, "ms_scene_upload": up_stats["ms_upload"], "ms_lbvh_build": up_stats["ms_build"],
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_total, "roofline": roofline, "cpu_baseline": cpu,
            "parity": parity, "frame_check": frame_check}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline workload (the other configs of --configs all time min(K, 5))")
    ap.add_argument("--warmup", type=int, default=3,
                    help="untimed steps before them (the other configs warm up with 3)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="synthetic", choices=sorted(WORKLOADS))
    ap.add_argument("--assemble", default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = resolve kernels store into rank 0's frame over NVLink (default); nccl = gather + unpack (A/B)")
    ap.add_argument("--configs", default="all", choices=["all", "none"],
                    help="all: after the headline workload also time the other BASELINE.json configs (per_config)")
    ap.add_argument("--in-process", type=int, default=0,
                    help="single process: render with rt_params.n_gpus = N (the library drives N GPUs itself); not the driver's launch mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline workload's output of its last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus != 1:
        print(f"bench.py: --gpus {args.gpus} needs torch.distributed.run (WORLD_SIZE={world})", file=sys.stderr)
        sys.exit(2)
    pkg = load_package()

    # -------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        spec, width, height, depth, desc = WORKLOADS[args.workload]
        config = {"workload": f"{args.workload}: {desc}", "width": width, "height": height, "bounce_depth": depth}
        try:
            r = reference_runs(pkg, args.workload, args.steps, max(args.warmup, 0), target_s=6.0)
        except FileNotFoundError as e:
            print(json.dumps({"impl": "reference", "unavailable": f"reference shim not built: {e}"}))
            return
        line = {"impl": "reference", "metric": "Mrays/s (primary+shadow+secondary)", "value": r["value"], "unit": "Mrays/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "Mrays/s", "cores": r["cores"], "kind": "reference",
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # -------------------------------------------------------------- B200 arm
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    head = run_workload(args, pkg, torch, dist, args.workload, True)
    per_config = {}
    emulate = os.environ.get("RT_BENCH_EMULATE_RANK")
    if args.configs == "all" and args.workload == "synthetic" and not emulate:
        # the other BASELINE.json configurations at this N (configs[0..3]); the headline above is configs[4]
        for name in ("input01", "teapot", "refraction3", "bunny"):
            rec = run_workload(args, pkg, torch, dist, name, False)
            if rank == 0:
                rf = rec["roofline"] or {}
                per_config[name] = {
                    "workload": rec["config"]["workload"], "value": rec["value"], "unit": "Mrays/s", "ms_per_step": rec["ms_per_step"],
                    "steps": rec["steps"], "rays_per_step": rec["rays_per_step"], "gpu_launches": rec["gpu_launches"],
                    "e2e": {k: rec["e2e"][k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step")} if rec["e2e"] else None,
                    "parity": rec["parity"], "frame_check": rec["frame_check"],
                    "roofline": {"kernel": rf.get("kernel"), "frac": rf.get("frac"), "achieved": rf.get("achieved"), "peak": rf.get("peak"),
                                 "unit": rf.get("unit"), "ms_kernel_serial_frame": rf.get("ms_kernel_serial_frame")},
                    "cpu_baseline": rec["cpu_baseline"]}
    if rank == 0:
        line = {"metric": "Mrays/s (primary+shadow+secondary)", "value": head["value"], "unit": "Mrays/s", "n_gpus": world,
                "steps": head["steps"], "warmup": head["warmup"], "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": head["config"],
                "gpus_in_process": args.in_process if args.in_process > 1 else None,
                "rays_per_step": head["rays_per_step"], "frame_ms": head["frame_ms"], "ms_scene_upload": head["ms_scene_upload"],
                "ms_lbvh_build": head["ms_lbvh_build"], "clocks": head["clocks"], "e2e": head["e2e"],
                "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "cpu_baseline": head["cpu_baseline"],
                "parity": head["parity"]}
        if head["frame_check"]:
            line.update(head["frame_check"])
        if per_config:
            line["per_config"] = per_config
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
