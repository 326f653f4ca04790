#!/usr/bin/env python
"""bench.py -- throughput of the B200 draw path on BASELINE.json's workloads, self-checking.

    python bench.py --gpus N --steps K --warmup W            # this back end
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle/_ref)
    python bench.py ... --dump-outputs DIR                   # also write a fixed sample of the timed path's frames

Headline workload (default): BASELINE.json configs[4] -- the batch of independent viewpoints of the
TEXTURED ~2.5k-triangle mesh (nearest texel, gamma-2 pipeline, Gouraud) at 1920x1080 colour+z,
frame-parallel.  One STEP renders `--views` viewpoints per GPU (512: 8 GPUs x 512 = the 4096 views
of configs[4]) with ONE pass of the pipeline setup -> scan -> bin -> raster.  `value` times
dtr_b200_replay() (command list, mesh and texture resident in HBM); `e2e` times the public call path
with host buffers: record draw calls -> flush (H2D of the command block) -> read the colour frames
back into pinned host memory.  The other BASELINE configs (configs[1] mesh1080, configs[2]
mesh4k_tex, configs[3] fill4k with its sort-first band split for N > 1) are measured in the same
process and carried in `other_workloads`.

Every workload is PARITY CHECKED before its number is printed: frames rendered by the timed code
path are read back and compared bit for bit (colour and depth) with the unmodified reference
(oracle/_ref; the C restatement if that is not built), and the band-split frame assembled in rank
0's HBM is compared with rank 0's own whole-frame render.  A mismatch exits non-zero.

Prints ONE JSON line (rank 0).  See DESIGN.md §5 for the definitions behind every field.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from dtrenderer_b200 import scenes  # noqa: E402

TOTAL_VIEWS = 4096  # configs[4]: view i = rotation i*360/4096 degrees about +Y
CLEAR = (0.5, 0.0, 1.0)
WORKLOADS = {
    # frame-parallel view batches: (width, height, textured, tex_size, overlay quads per view, default views per step)
    "views1080_tex": dict(w=1920, h=1080, textured=True, tex=1024, overlays=0, views=512,
                          desc="BASELINE configs[4]: independent viewpoints of the textured 2500-triangle mesh "
                               "(1024^2 texture, nearest texel, gamma-2, Gouraud) at 1920x1080 colour+z, frame-parallel"),
    "mesh1080": dict(w=1920, h=1080, textured=False, tex=1, overlays=0, views=64,
                     desc="BASELINE configs[1]: 2500-triangle UV-sphere mesh, perspective, Gouraud, 1920x1080 colour+z"),
    "mesh4k_tex": dict(w=3840, h=2160, textured=True, tex=1024, overlays=16, views=32,
                       desc="BASELINE configs[2]: same mesh, 1024^2 texture (nearest, gamma-2) at 3840x2160 colour+z "
                            "with 16 alpha-0.5 overlay quads per frame"),
}
FILL = {"fill4k": dict(w=3840, h=2160, n=1_000_000,
                       desc="BASELINE configs[3]: fill-rate stress, 1M small random z-buffered triangles at 3840x2160; "
                            "N>1: sort-first screen bands assembled in rank 0's HBM")}
METRIC, UNIT = "shaded_gpixels_per_s", "Gpixels/s"
TRIS_PER_FRAME = 2500
SUB = 64  # views per flush in the end-to-end loop (two pinned halves of SUB frames each)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


ONE_KERNEL = "raster_opaque_kernel<true>"                       # dtr_b200_last_pass_deferred() == 2 (the default for opaque-only passes)
TWO_KERNELS = ("raster_opaque_kernel<false>", "resolve_kernel")  # == 1 (DTR_B200_FUSED=0)


def kernel_split(split, runs, stage, textured):
    """CUDA-event durations of the raster stage's kernels inside the timed region (dtr_b200_get_raster_split_ms).
    stage: 0 = the single raster kernel, 1 = visibility kernel + resolve kernel, 2 = the one-kernel opaque stage."""
    a, b = split[0] / max(runs, 1), split[1] / max(runs, 1)
    if stage == 2:
        return {ONE_KERNEL: a}
    if stage == 1:
        return {TWO_KERNELS[0]: a, TWO_KERNELS[1]: b}
    return {"raster_tex_kernel" if textured else "raster_kernel": a}


def stage_label(stage, textured):
    if stage == 2:
        return (ONE_KERNEL + " (opaque-only pass: region walk with depth test and primitive tags, then every visible pixel of the "
                "finished region shaded once from shared memory; one kernel)")
    if stage == 1:
        return (" + ".join(TWO_KERNELS) + " (opaque-only pass as two kernels: visibility, then resolve; both inside the timed interval)")
    return "raster_tex_kernel" if textured else "raster_kernel"


def load_traffic(workload, stage=0):
    """(dram bytes per frame, source) from the committed ncu capture of this workload's raster kernel(s), or
    (None, None).  A constant read from profiles/, NOT a measurement of the run that prints it.  Entries are
    keyed by workload; the capture of the one-kernel opaque stage by workload + "@one_kernel"."""
    p = os.path.join(ROOT, "profiles", "raster_traffic.json")
    if os.path.exists(p):
        try:
            e = json.load(open(p)).get(workload + "@one_kernel" if stage == 2 else workload)
            if isinstance(e, dict):
                return e.get("bytes_per_frame"), e.get("source")
        except Exception:
            pass
    return None, None


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def make_config(name, views, world):
    """The `config` object: identical for both arms (the driver compares them)."""
    if name in FILL:
        f = FILL[name]
        return {"workload": f["desc"], "width": f["w"], "height": f["h"], "triangles_per_step": f["n"],
                "parallelism": f"sort-first screen bands x{world}" if world > 1 else "single GPU, whole frame"}
    s = WORKLOADS[name]
    return {"workload": s["desc"], "width": s["w"], "height": s["h"], "triangles_per_frame": TRIS_PER_FRAME,
            "views_per_step_per_gpu": views,
            "parallelism": f"frame-parallel x{world} (independent viewpoints per GPU, no collective)",
            "l2": f"each step writes {views * 8 * s['w'] * s['h'] / 1e6:.0f} MB of frames per GPU (> 126 MB L2), "
                  "so no flush is needed between steps"}


class ViewScene:
    """The draw calls of one workload's frame, for any target exposing the renderer's call names."""

    def __init__(self, name):
        s = WORKLOADS[name]
        self.name, self.w, self.h = name, s["w"], s["h"]
        self.mesh = scenes.uv_sphere()
        self.tex = scenes.random_texture(s["tex"], s["tex"], 1, True) if s["textured"] else scenes.WHITE_TEXTURE
        self.transforms = scenes.view_transforms(TOTAL_VIEWS)  # built ONCE (10 ms of Python)
        self.overlays = [kw for nm, kw in scenes.mesh_scene(self.w, self.h, overlays=s["overlays"])[2:] if nm == "rectangle"]

    def draw_frame(self, target, view):
        """One frame through single draw calls (the reference's own call sequence)."""
        target.clear(CLEAR)
        target.mesh(self.mesh, self.tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0),
                    self.transforms[view % TOTAL_VIEWS])
        for kw in self.overlays:
            target.rectangle(**kw)

    def record_batch(self, r, first_frame, view0, n):
        """n consecutive views into frames first_frame.. of a CUDA context, batched (dtr_b200_mesh_views)."""
        for f in range(first_frame, first_frame + n):
            r.begin_frame(f)
            r.clear(CLEAR)
        ts = [self.transforms[(view0 + i) % TOTAL_VIEWS] for i in range(n)]
        r.mesh_views(self.mesh, self.tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1),
                     np.zeros((n, 3), np.float32), ts, first_frame)
        if self.overlays:
            for f in range(first_frame, first_frame + n):
                r.set_target(f)
                for kw in self.overlays:
                    r.rectangle(**kw)


DUMP_FRAMES, DUMP_PIXELS, DUMP_CROP = 512, 1 << 21, 512


def dump_outputs(out_dir, prefix, read_frame, n_frames, w, h):
    """--dump-outputs: the frames the timed path left behind after its last step, as float32 .npy files, so that
    two builds run with the same arguments (hence the same inputs) can be compared output for output.  The sample
    is fixed (seed 0): at most DUMP_FRAMES of the n_frames frames, the same DUMP_PIXELS // frames pixels of each,
    and the whole DUMP_CROP x DUMP_CROP centre of the last of those frames.  A colour pixel is split into its four bytes
    (memory order B, G, R, X), so a one-level difference in any channel shows; depth is written as stored.
    At most 2M x 20 B + 512^2 x 20 B = 47 MB.  read_frame(i) returns frame i's (colour u32, depth f32) planes."""
    rng = np.random.default_rng(0)
    frames = np.arange(n_frames) if n_frames <= DUMP_FRAMES else np.sort(rng.choice(n_frames, DUMP_FRAMES, replace=False))
    pix = np.sort(rng.choice(w * h, min(w * h, DUMP_PIXELS // len(frames)), replace=False))
    col_s = np.empty((len(frames), len(pix), 4), np.float32)
    z_s = np.empty((len(frames), len(pix)), np.float32)
    for j, f in enumerate(frames):
        col, z = read_frame(int(f))
        col_s[j] = col.reshape(-1)[pix].view(np.uint8).reshape(-1, 4)
        z_s[j] = z.reshape(-1)[pix]
    y0, x0 = max(0, (h - DUMP_CROP) // 2), max(0, (w - DUMP_CROP) // 2)
    col_c = np.ascontiguousarray(col[y0:y0 + DUMP_CROP, x0:x0 + DUMP_CROP])
    z_c = z[y0:y0 + DUMP_CROP, x0:x0 + DUMP_CROP]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("color_sample", col_s), ("depth_sample", z_s),
                    ("color_crop", col_c.view(np.uint8).reshape(*col_c.shape, 4)), ("depth_crop", z_c)):
        np.save(os.path.join(out_dir, f"{prefix}_{name}.npy"), a.astype(np.float32))


def oracle_kind():
    from oracle import dtro
    return "reference" if dtro.available("reference") else "port"


def check_view_frames(r, scene, pairs):
    """Parity: frames of the CUDA context (frame index, view index) against the oracle, colour and depth
    bit for bit.  Returns the number of frames checked; raises SystemExit on the first difference."""
    from oracle import dtro
    o = dtro.Oracle(scene.w, scene.h, oracle_kind())
    for frame, view in pairs:
        col, z = r.end_frame(frame)
        o.reset_z()
        scene.draw_frame(o, view)
        if not (np.array_equal(col, o.color()) and np.array_equal(z.view(np.uint32), o.zbuffer().view(np.uint32))):
            bad = int((col != o.color()).sum()), int((z.view(np.uint32) != o.zbuffer().view(np.uint32)).sum())
            raise SystemExit(f"bench.py: PARITY FAILURE {scene.name} frame {frame} (view {view}): {bad[0]} colour / "
                             f"{bad[1]} depth pixels differ from the {o.kind} oracle")
    o.close()
    return len(pairs)


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's own scalar path (oracle/_ref, unmodified sources) on host cores
# --------------------------------------------------------------------------------------------
_W = {}


def _cpu_init(kind, name):
    from oracle import dtro
    sc = ViewScene(name)  # view transforms, mesh and texture are built here, once per worker
    _W["scene"] = sc
    _W["o"] = dtro.Oracle(sc.w, sc.h, kind)
    _cpu_frame(0)  # warm caches / page in


def _cpu_frame(view):
    o, sc = _W["o"], _W["scene"]
    o.reset_z()
    o.reset_counters()
    t0 = time.perf_counter()
    sc.draw_frame(o, view)
    dt = time.perf_counter() - t0
    sp, tr = o.counters()
    return sp, tr, dt


class CpuPool:
    """One single-threaded reference renderer per host core (independent frames per core -- the
    deterministic way to use all cores, SURVEY.md §8c/§8d)."""

    def __init__(self, workload, cores=None):
        import multiprocessing as mp
        self.kind = oracle_kind()
        self.cores = cores or len(os.sched_getaffinity(0))
        self.pool = mp.get_context("fork").Pool(self.cores, _cpu_init, (self.kind, workload))

    def run(self, first_view, n_frames):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_frame, range(first_view, first_view + n_frames), chunksize=1)
        wall = time.perf_counter() - t0
        return sum(r[0] for r in res), sum(r[1] for r in res), wall, sum(r[2] for r in res)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline(workload, target_cpu_seconds=12.0):
    pool = CpuPool(workload)
    _, _, w1, _ = pool.run(0, pool.cores)  # calibration pass = warm-up
    per_frame = max(w1, 1e-3)
    n = int(max(pool.cores, min(TOTAL_VIEWS, target_cpu_seconds / per_frame * pool.cores)))
    n = (n // pool.cores) * pool.cores
    sp, tr, wall, busy = pool.run(0, n)
    pool.close()
    return {"value": sp / wall / 1e9, "unit": UNIT, "cores": pool.cores, "cpu": cpu_model(), "kind": pool.kind,
            "sample": f"{n} frames (views 0..{n - 1}) of the workload, one single-threaded renderer per core, "
                      f"{wall:.2f} s wall ({busy / pool.cores:.2f} s of rendering per core)",
            "frames_per_s": n / wall, "mtris_per_s": tr / wall / 1e6}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    views = args.views or WORKLOADS[args.workload]["views"]
    pool = CpuPool(args.workload)
    # a step is a bounded sample of the B200 arm's step: whole rounds over all host cores, at most SUB frames
    frames_per_step = max(1, min(SUB, views) // pool.cores) * pool.cores
    for i in range(args.warmup):
        pool.run(i * frames_per_step, frames_per_step)
    sp = tr = 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        a, b, _, _ = pool.run(i * frames_per_step, frames_per_step)
        sp += a
        tr += b
    wall = time.perf_counter() - t0
    pool.close()
    val = sp / wall / 1e9
    sample = (f"{frames_per_step} frames per step (a bounded sample of the B200 arm's {views} viewpoints per step: the "
              f"metric is a rate), one single-threaded reference renderer per host core, {args.steps} steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args.workload, views, args.gpus),
        "mtris_per_s": tr / wall / 1e6, "frames_per_s": frames_per_step * args.steps / wall,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": pool.cores, "cpu": cpu_model(), "kind": pool.kind,
                         "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# clocks: NVML polled from a thread DURING the timed regions
# --------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        self._active = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:  # noqa: BLE001
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:  # noqa: BLE001
                    pass
            time.sleep(0.002)

    def start(self):
        self._active.set()

    def pause(self):
        self._active.clear()

    def result(self):
        self._stop.set()
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
class Env:
    """Per-process CUDA / torch.distributed state shared by the workloads of one bench run."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        from dtrenderer_b200 import api, multigpu
        self.torch, self.dist, self.api, self.multigpu = torch, dist, api, multigpu
        self.rank, self.world, self.local_rank = rank, world, local_rank
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- this back end has no CPU fallback")
        torch.cuda.set_device(local_rank)
        if world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # a real (non-NULL) stream: the kernels, the copies and the timing events all go on it
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        self.clocks = ClockSampler(local_rank)
        self.launches = 0

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        t = self.torch.tensor([v], device="cuda", dtype=self.torch.int64)
        if self.world > 1:
            self.dist.all_reduce(t)
        return int(t.item())

    def events(self):
        return self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)


def measure_views(env, name, views, steps, warmup, e2e_steps, with_e2e, dump=None):
    """One frame-parallel workload on this rank's GPU: device-resident throughput (replay of one
    B-view flush), per-stage times, parity of frames rendered by the timed path, optional e2e;
    dump: directory for dump_outputs() of the frames of the last timed replay."""
    torch = env.torch
    s = WORKLOADS[name]
    w, h, B = s["w"], s["h"], views
    sub = min(SUB, B)
    scene = ViewScene(name)
    r = env.api.Renderer(w, h, max(B, 2 * sub), env.local_rank)
    r.set_stream(env.stream.cuda_stream)
    view0 = env.rank * B  # rank r renders views r*B .. r*B+B-1 (N=8, B=512: the 4096 views of configs[4])

    # one full pass to build the resident command list and count the work of a step
    r.reset_stats()
    scene.record_batch(r, 0, view0, B)
    r.flush()
    st = r.stats()
    shaded_per_step, tris_per_step = st["setPixels"], st["triangles"]
    tex_bytes = 4 * min(shaded_per_step // B, s["tex"] * s["tex"]) if s["textured"] else 0
    # SURVEY.md §8(d): one 8-byte store per pixel + 156 B per triangle + the texels touched; a blit's
    # destination pixels count once more as 8 B (read + write) -- the overlay quads of configs[2]
    blit_px = sum(max(0, min(int(kw["mx"][0]), w) - max(int(kw["mn"][0]), 0)) * max(0, min(int(kw["mx"][1]), h) - max(int(kw["mn"][1]), 0))
                  for kw in scene.overlays)
    alg_bytes = B * (8 * w * h + 156 * TRIS_PER_FRAME + tex_bytes + 8 * blit_px)

    # ---- device-resident throughput: replay() ------------------------------------------------
    for _ in range(max(warmup, 3)):
        r.replay()
    r.set_profiling(True)
    r.reset_stage_ms()
    r.reset_stats()
    env.barrier()
    e0, e1 = env.events()
    env.clocks.start()
    e0.record(env.stream)
    for _ in range(steps):
        r.replay()
    e1.record(env.stream)
    env.barrier()
    env.clocks.pause()
    ms_step = env.max_over_ranks(e0.elapsed_time(e1)) / steps
    stage, runs = r.stage_ms()
    split, _ = r.raster_split_ms()
    env.launches += r.stats()["kernelLaunches"]
    opaque_stage = r.last_pass_stage()
    # parity of what the TIMED path left in the frames: first, middle and last view of this rank
    pairs = sorted({(0, view0), (B // 2, view0 + B // 2), (B - 1, view0 + B - 1)})
    checked = check_view_frames(r, scene, pairs)
    if dump:
        cbuf, zbuf = np.empty((h, w), np.uint32), np.empty((h, w), np.float32)
        dump_outputs(dump, name + (f"_rank{env.rank}" if env.world > 1 else ""),
                     lambda f: r.end_frame(f, color_out=cbuf, z_out=zbuf), B, w, h)
    # untimed extra pass with the replay pipelining off: per-stage times in isolation (in the timed
    # region the pre-raster stages of later replays overlap the raster kernel, so their event
    # intervals include the wait for free SMs and the stages no longer add up to the step)
    r.set_replay_overlap(False)
    r.reset_stage_ms()
    for _ in range(5):
        r.replay()
    stage_iso, runs_iso = r.stage_ms()
    r.set_replay_overlap(True)
    r.set_profiling(False)

    peak, peak_src = load_peaks()
    raster_ms = stage["raster"] / max(runs, 1)
    achieved = alg_bytes / (raster_ms * 1e-3) / 1e9 if raster_ms > 0 else 0.0
    tr_frame, tr_src = load_traffic(name, opaque_stage)
    world = env.world
    out = {
        "workload": name, "value": world * shaded_per_step / (ms_step * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_step,
        "views_per_step_per_gpu": B, "shaded_fragments_per_step_per_gpu": shaded_per_step,
        "mtris_per_s": world * tris_per_step / (ms_step * 1e-3) / 1e6, "frames_per_s": world * B / (ms_step * 1e-3),
        "parity_checked": True,
        "parity": f"{checked} frames per rank of the timed replay (first, middle, last view) bit-equal in colour and depth "
                  f"to the {oracle_kind()} oracle at {w}x{h}",
        "roofline": {"bound": "hbm", "kernel": stage_label(opaque_stage, s["textured"]),
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": tr_frame * B if tr_frame else None,
                     "traffic_source": (tr_src + " (a committed capture scaled to this batch, not measured in this run)") if tr_src else None,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": raster_ms,
                     "stage_ms_per_step": {k: v / max(runs, 1) for k, v in stage.items()},
                     "raster_kernels_ms_per_step": kernel_split(split, runs, opaque_stage, s["textured"]),
                     "stage_ms_isolated": {k: v / max(runs_iso, 1) for k, v in stage_iso.items()},
                     "note": "achieved/frac use the raster kernel's CUDA-event duration inside the timed region, where "
                             "setup/scan/bin of later replays run on a second stream beside it (their stage_ms_per_step "
                             "include waiting for SMs); stage_ms_isolated = the same stages with that pipelining off"},
    }
    if not with_e2e:
        r.close()
        return out

    # ---- end to end: record -> flush (H2D) -> read the colour frames back (D2H, pinned) ------
    # A step is the same B views, issued as B/SUB flushes of SUB views; every flush uploads its command
    # block and its SUB colour planes are read back asynchronously (copy stream) into one of two pinned
    # halves, so a flush's D2H overlaps the recording and rendering of the next one.
    host = torch.empty((2, sub, h, w), dtype=torch.int32, pin_memory=True)
    nsub = B // sub
    upload = [0]

    def time_e2e(read_half, n_steps):
        turn = [0]

        def step_e2e():
            for j in range(nsub):
                half = turn[0] & 1
                turn[0] += 1
                scene.record_batch(r, half * sub, view0 + j * sub, sub)
                read_half(half)

        step_e2e()
        r.wait_reads()
        upload[0] = r.stats()["uploadBytes"]  # H2D bytes of one flush (command block + payload)
        env.barrier()
        env.clocks.start()
        e0.record(env.stream)
        for _ in range(n_steps):
            step_e2e()
        r.wait_reads()  # blocks until the last copy has landed; e1 is recorded after that
        e1.record(env.stream)
        env.barrier()
        env.clocks.pause()
        return env.max_over_ranks(e0.elapsed_time(e1)) / n_steps

    e2e_ms = time_e2e(lambda half: r.read_frames_async_ptr(half * sub, sub, host[half].data_ptr()), e2e_steps)
    # the last flush of the e2e loop, as it arrived in host memory, against the oracle (colour only)
    from oracle import dtro
    o = dtro.Oracle(w, h, oracle_kind())
    last_half = (nsub * (e2e_steps + 1) - 1) & 1
    for k in (0, sub - 1):
        o.reset_z()
        scene.draw_frame(o, view0 + (nsub - 1) * sub + k)
        if not np.array_equal(host[last_half, k].numpy().view(np.uint32), o.color()):
            raise SystemExit(f"bench.py: PARITY FAILURE {name}: e2e readback of view {view0 + (nsub - 1) * sub + k} differs")
    o.close()
    # the same loop with the on-device 24-bit DIB encode (3 bytes per pixel over PCIe); reported beside
    # `e2e`, which stays the u32 DTRRenderBuffer layout
    pitch = r.bgr24_pitch()
    host24 = torch.empty((2, sub, h, pitch), dtype=torch.uint8, pin_memory=True)
    n24 = max(2, e2e_steps // 2)
    e2e24_ms = time_e2e(lambda half: r.read_frames_bgr24_async_ptr(half * sub, sub, host24[half].data_ptr()), n24)
    # both loops end on the same views: the packed bytes must equal the u32 readback
    half24 = (nsub * (n24 + 1) - 1) & 1
    packed_ok = bool(torch.equal(host24[half24, :, :, :3 * w].reshape(sub, h, w, 3),
                                 host[last_half].view(torch.uint8).reshape(sub, h, w, 4)[..., :3]))
    if not packed_ok:
        raise SystemExit(f"bench.py: PARITY FAILURE {name}: 24-bit readback differs from the u32 readback")
    # platform ceiling of the readback alone: the same bytes, all ranks at once, no rendering
    # (last: it overwrites the pinned buffers the comparisons above read)
    e0c, e1c = env.events()
    dcol = torch.empty((sub, h, w), dtype=torch.int32, device="cuda")
    host[0].copy_(dcol, non_blocking=True)
    env.barrier()
    e0c.record(env.stream)
    for i in range(2 * nsub):
        host[i & 1].copy_(dcol, non_blocking=True)
    e1c.record(env.stream)
    env.barrier()
    d2h_ms = env.max_over_ranks(e0c.elapsed_time(e1c)) / 2
    del dcol
    out["e2e"] = {"value": world * shaded_per_step / (e2e_ms * 1e-3) / 1e9, "unit": UNIT,
                  "h2d_bytes_per_step": upload[0] * nsub, "d2h_bytes_per_step": B * 4 * w * h,
                  "ms_per_step": e2e_ms, "frames_per_s": world * B / (e2e_ms * 1e-3), "steps": e2e_steps,
                  "d2h_only_ms_per_step": d2h_ms, "frac_of_d2h_ceiling": d2h_ms / e2e_ms if e2e_ms > 0 else None,
                  "d2h_ceiling_note": "d2h_only = the same D2H bytes per step copied by all ranks at once with no rendering "
                                      "(the platform's host-ingest ceiling for this N)",
                  "readback": f"colour planes only (what the reference presents); depth stays in HBM; {nsub} flushes of "
                              f"{sub} views per step, asynchronous and double buffered (a flush's D2H overlaps the next "
                              "flush's recording and rendering)",
                  "parity_checked": True}
    out["e2e_bgr24"] = {"value": world * shaded_per_step / (e2e24_ms * 1e-3) / 1e9, "unit": UNIT,
                        "d2h_bytes_per_step": B * pitch * h, "ms_per_step": e2e24_ms, "matches_u32_readback": packed_ok,
                        "readback": "dtr_b200_read_frames_bgr24_async: colour packed on the device into 24-bit bottom-up "
                                    "DIB rows (informational; `e2e` is the DTRRenderBuffer layout)"}
    r.close()
    return out


# --------------------------------------------------------------------------------------------
# cfg 4: fill-rate stress, sort-first screen bands for N > 1
# --------------------------------------------------------------------------------------------
def _fill_cpu_init(kind, w, h):
    from oracle import dtro
    _W["o"] = dtro.Oracle(w, h, kind)


def _fill_cpu_chunk(args):
    p, color = args
    o = _W["o"]
    o.reset_z()
    o.reset_counters()
    o.clear((0, 0, 0))
    o.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
    return o.counters()


def run_fill_reference(args, rank, world):
    """Reference arm for cfg 4: every host core renders an independent frame of a bounded sample
    (triangles of the same distribution) -- whole-frame order is inherently serial in the reference,
    so independent frames are the only deterministic way to use all cores."""
    if rank != 0:
        return
    import multiprocessing as mp
    f = FILL[args.workload]
    w, h = f["w"], f["h"]
    kind = oracle_kind()
    cores = len(os.sched_getaffinity(0))
    per_core = 20000
    chunks = [scenes.small_triangles(w, h, per_core, seed=100 + i) for i in range(cores)]
    pool = mp.get_context("fork").Pool(cores, _fill_cpu_init, (kind, w, h))
    for _ in range(max(1, args.warmup)):
        pool.map(_fill_cpu_chunk, chunks, chunksize=1)
    sp = tr = 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for a, b in pool.map(_fill_cpu_chunk, chunks, chunksize=1):
            sp += a
            tr += b
    wall = time.perf_counter() - t0
    pool.close()
    pool.join()
    val = sp / wall / 1e9
    sample = f"{cores} independent 4K frames of {per_core} triangles each per step (one per host core)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": make_config(args.workload, 0, args.gpus),
        "mtris_per_s": tr / wall / 1e6,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "cpu": cpu_model(), "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}),
        flush=True)


def measure_fill(env, name, n_override, steps, warmup, e2e_steps, gather, with_e2e, band_frames=2, dump=None):
    """cfg 4 on this process group: one frame of 1M small triangles; N>1 splits the screen into
    tile-aligned bands (every rank runs setup over all triangles, bins and rasterises its band) and
    assembles the frame in rank 0's HBM.  Parity: the assembled planes == rank 0's own whole-frame
    render, and (N=1, full size) == the reference oracle.  dump: directory for dump_outputs() of the
    frame in rank 0's HBM after the timed steps."""
    torch, multigpu = env.torch, env.multigpu
    f = FILL[name]
    w, h, n = f["w"], f["h"], n_override or f["n"]
    rank, world = env.rank, env.world
    r = env.api.Renderer(w, h, 1, env.local_rank)
    r.set_stream(env.stream.cuda_stream)
    y0, y1 = multigpu.band_rows(h, world, rank, r.tile_height())
    if world > 1:
        r.set_band(y0, max(y1, y0 + 1) if y1 > y0 else h)  # (empty bands cannot occur at 4K with N <= 8)
    p, color = scenes.small_triangles(w, h, n, seed=7)  # geometry replicated on every rank
    peer = world > 1 and gather == "peer"
    nccl = world > 1 and gather == "nccl"
    if world > 1:
        r.band_comm_init_torch(env.dist)  # the library's own NCCL communicator (C ABI), bootstrapped through torch
    if peer:
        multigpu.share_frames(r, dst=0)  # ranks > 0 now rasterise straight into rank 0's planes

    def record():
        r.begin_frame(0)
        r.clear((0, 0, 0))
        r.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)

    r.reset_stats()
    record()
    r.flush()
    st = r.stats()
    shaded_per_step = env.sum_over_ranks(st["setPixels"])
    upload_bytes = st["uploadBytes"]
    alg_bytes = 8 * w * (y1 - y0) + 156 * n  # this rank's band + all triangles (every rank runs setup)

    skip_barrier = os.environ.get("DTR_BENCH_DIAG_NO_BARRIER") == "1"  # diagnostic only: what the barrier costs

    def step_resident():
        r.replay()
        if peer and not skip_barrier:
            r.band_barrier()  # stream-ordered: every band has landed in rank 0's HBM
        elif nccl:
            r.gather_bands(0, dst=0)

    for _ in range(max(warmup, 3)):
        step_resident()
    r.set_profiling(True)
    r.reset_stage_ms()
    r.reset_stats()
    env.barrier()
    e0, e1 = env.events()
    env.clocks.start()
    e0.record(env.stream)
    for _ in range(steps):
        step_resident()
    e1.record(env.stream)
    env.barrier()
    env.clocks.pause()
    ms_step = env.max_over_ranks(e0.elapsed_time(e1)) / steps
    stage, runs = r.stage_ms()
    split, _ = r.raster_split_ms()
    env.launches += r.stats()["kernelLaunches"]
    opaque_stage = r.last_pass_stage()
    r.set_profiling(False)

    # ---- two frame targets per rank (double buffering): frame i's barrier beside frame i+1's rasterisation ----
    # A second context with its own stream, its own NCCL communicator and its own mapping of rank 0's second
    # target; consecutive frames alternate between the two.  A frame is complete in rank 0's HBM when ITS
    # barrier has passed, exactly as before; what changes is that no rank waits for that before it starts
    # the next frame, which goes to the other target.  The timed interval ends when both streams are done.
    inline_ms = None
    r2 = None
    if peer and band_frames == 2 and not skip_barrier:
        inline_ms = ms_step
        r2 = env.api.Renderer(w, h, 1, env.local_rank)
        s2 = torch.cuda.Stream()
        r2.set_stream(s2.cuda_stream)
        r2.set_band(y0, max(y1, y0 + 1) if y1 > y0 else h)
        r2.band_comm_init_torch(env.dist)
        multigpu.share_frames(r2, dst=0)
        r2.begin_frame(0)
        r2.clear((0, 0, 0))
        r2.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
        with torch.cuda.stream(s2):
            r2.flush()
        pair = (r, r2)

        def run_alternating(k):
            for i in range(k):
                x = pair[i & 1]
                x.replay()
                x.band_barrier()

        run_alternating(2 * max(warmup, 3))
        env.stream.synchronize()
        s2.synchronize()
        env.barrier()
        env.clocks.start()
        e0.record(env.stream)
        s2.wait_stream(env.stream)
        run_alternating(steps)
        env.stream.wait_stream(s2)
        e1.record(env.stream)
        env.barrier()
        env.clocks.pause()
        ms_step = env.max_over_ranks(e0.elapsed_time(e1)) / steps
        env.launches += r2.stats()["kernelLaunches"]

    # ---- parity of the frame(s) the timed steps left in rank 0's HBM ---------------------------
    parity = []
    if rank == 0:
        col, z = r.end_frame(0)
        if dump:
            dump_outputs(dump, name, lambda f: (col, z), 1, w, h)
        if r2 is not None:
            col_b, z_b = r2.end_frame(0)
            if not (np.array_equal(col, col_b) and np.array_equal(z.view(np.uint32), z_b.view(np.uint32))):
                raise SystemExit(f"bench.py: PARITY FAILURE {name}: the two frame targets of the double-buffered band loop differ")
            parity.append("both frame targets of the double-buffered loop bit-equal to each other")
        if world > 1:
            whole = env.api.Renderer(w, h, 1, env.local_rank)
            whole.begin_frame(0)
            whole.clear((0, 0, 0))
            whole.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
            col1, z1 = whole.end_frame(0)
            whole.close()
            if not (np.array_equal(col, col1) and np.array_equal(z.view(np.uint32), z1.view(np.uint32))):
                raise SystemExit(f"bench.py: PARITY FAILURE {name}: the frame assembled from {world} bands differs from "
                                 "rank 0's whole-frame render")
            parity.append(f"colour+depth planes assembled from {world} bands in rank 0's HBM bit-equal to rank 0's own "
                          "whole-frame render")
        from oracle import dtro
        o = dtro.Oracle(w, h, oracle_kind())
        o.clear((0, 0, 0))
        o.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
        if not (np.array_equal(col, o.color()) and np.array_equal(z.view(np.uint32), o.zbuffer().view(np.uint32))):
            raise SystemExit(f"bench.py: PARITY FAILURE {name}: frame differs from the {o.kind} oracle")
        parity.append(f"full {w}x{h} frame of {n} triangles bit-equal in colour and depth to the {o.kind} oracle")
        o.close()
    env.barrier()

    peak, peak_src = load_peaks()
    raster_ms = stage["raster"] / max(runs, 1)
    achieved = alg_bytes / (raster_ms * 1e-3) / 1e9 if raster_ms > 0 else 0.0
    out = {
        "workload": name, "value": shaded_per_step / (ms_step * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_step,
        "scaling": "strong", "triangles_per_step": n, "shaded_fragments_per_step": shaded_per_step,
        "mtris_per_s": n / (ms_step * 1e-3) / 1e6, "frames_per_s": 1.0 / (ms_step * 1e-3),
        "parallelism": (f"sort-first bands x{world}, " + (
            "bands written into rank 0's HBM over NVLink by the raster kernel's write-back (CUDA IPC peer memory), "
            "stream-ordered NCCL barrier (dtr_b200_band_barrier)" + (
                "; two frame targets per rank used alternately: the barrier that completes frame i runs beside the "
                "rasterisation of frame i+1 (ms_per_step_one_target = the same loop with one target and the barrier in line)"
                if r2 is not None else "") if peer
            else "grouped ncclSend/ncclRecv gather (dtr_b200_gather_bands)")) if world > 1 else "single GPU, whole frame",
        "band_frames": 2 if r2 is not None else 1, "ms_per_step_one_target": inline_ms,
        "exchange_bytes_per_step_into_rank0": 8 * w * (h - multigpu.band_rows(h, world, 0, r.tile_height())[1]) if world > 1 else 0,
        "parity_checked": True, "parity": "; ".join(parity),
        "roofline": {"bound": "hbm", "kernel": stage_label(opaque_stage, False),
                     "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": raster_ms,
                     "stage_ms_per_step": {k: v / max(runs, 1) for k, v in stage.items()},
                     "raster_kernels_ms_per_step": kernel_split(split, runs, opaque_stage, False),
                     "note": "rank 0's band; this config is ALU/ordering bound, not HBM bound; the frame planes (66 MB) fit "
                             "in L2, the 160 MB of primitive records do not, L2 is not flushed between steps"},
    }
    if with_e2e:
        host = torch.empty((h, w), dtype=torch.int32, pin_memory=True)

        def step_e2e():
            record()
            r.flush()
            if peer:
                r.band_barrier()
            elif nccl:
                r.gather_bands(0, dst=0)
            if rank == 0:
                r.read_frames_ptr(0, 1, host.data_ptr())

        step_e2e()
        env.barrier()
        env.clocks.start()
        e0.record(env.stream)
        for _ in range(e2e_steps):
            step_e2e()
        e1.record(env.stream)
        env.barrier()
        env.clocks.pause()
        e2e_ms = env.max_over_ranks(e0.elapsed_time(e1)) / e2e_steps
        out["e2e"] = {"value": shaded_per_step / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": upload_bytes,
                      "d2h_bytes_per_step": 4 * w * h, "ms_per_step": e2e_ms, "steps": e2e_steps}
    if r2 is not None:
        r2.close()
    r.close()
    return out


def run_gpu_arm(args, rank, world, local_rank):
    main_is_fill = args.workload in FILL
    views = args.views or (0 if main_is_fill else WORKLOADS[args.workload]["views"])
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not main_is_fill:
        cpu = cpu_baseline(args.workload)  # before CUDA is initialised in this process (fork safety)
    env = Env(rank, world, local_rank)
    if world > 1:
        bind_to_gpu_numa_node(local_rank)
    e2e_steps = max(2, min(args.steps, args.e2e_steps))
    if main_is_fill:
        main = measure_fill(env, args.workload, args.triangles, args.steps, args.warmup, e2e_steps, args.gather, True, args.band_frames,
                            args.dump_outputs)
    else:
        main = measure_views(env, args.workload, views, args.steps, args.warmup, e2e_steps, True, args.dump_outputs)
    others = []
    if not args.no_others:
        o_steps = max(5, min(args.steps, 20))
        for name in ("mesh1080", "mesh4k_tex", "views1080_tex"):
            if name != args.workload:
                others.append(measure_views(env, name, min(WORKLOADS[name]["views"], 64), o_steps, args.warmup, 0, False))
        if not main_is_fill:
            others.append(measure_fill(env, "fill4k", args.triangles, o_steps, args.warmup, 0, args.gather, False, args.band_frames))
    clocks = env.clocks.result()
    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": main.get("scaling", "weak"), "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args.workload, views, world),
            "parity_checked": all(x.get("parity_checked") for x in [main] + others),
            "parity": main["parity"],
            "shaded_fragments_per_step": main.get("shaded_fragments_per_step_per_gpu", main.get("shaded_fragments_per_step")),
            "mtris_per_s": main["mtris_per_s"], "frames_per_s": main["frames_per_s"],
            "roofline": main["roofline"], "cpu_baseline": cpu, "e2e": main.get("e2e"),
            "other_workloads": [{k: v for k, v in o.items() if k not in ("unit",)} for o in others],
            "gpu_launches": env.launches, "clocks": clocks,
        }
        if main.get("band_frames"):
            line["band_frames"], line["ms_per_step_one_target"] = main["band_frames"], main["ms_per_step_one_target"]
        if "e2e_bgr24" in main:
            line["e2e_bgr24"] = main["e2e_bgr24"]
        print(json.dumps(line), flush=True)
    if world > 1:
        env.dist.destroy_process_group()


def bind_to_gpu_numa_node(local_rank):
    """Multi-rank runs: keep this rank's host threads -- and with them the pinned readback buffers it
    allocates next -- on the CPUs closest to its GPU (NVML's ideal affinity), so that eight ranks'
    D2H streams do not all land on one socket's memory.  Best effort; a no-op if NVML says nothing."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="views1080_tex", choices=sorted(WORKLOADS) + sorted(FILL))
    ap.add_argument("--triangles", type=int, default=0, help="fill4k: override the triangle count")
    ap.add_argument("--views", type=int, default=0, help="viewpoints (frames) per step per GPU (default: the workload's)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="measure only the main workload")
    ap.add_argument("--band-frames", type=int, default=2, choices=[1, 2],
                    help="fill4k, N>1, peer write-back: frame targets per rank. 2 = consecutive frames alternate between two "
                         "targets, so the barrier that completes frame i runs beside the rasterisation of frame i+1; "
                         "1 = one target, the barrier in line (always measured and reported as well)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="fill4k, N>1: how the bands reach rank 0 (peer-memory write-back or NCCL send/recv)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the frames the timed path rendered in its last step "
                         "to DIR/<name>.npy (float32, under 64 MB in all); see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the frames of the B200 arm's timed path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.workload in FILL:
            run_fill_reference(args, rank, world)
        else:
            run_reference_arm(args, rank, world)
    else:
        run_gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
