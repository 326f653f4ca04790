#!/usr/bin/env python
"""What render to texture (dtr_b200_frames_to_textures) costs on one GPU.

    python tools/frame_texture_cost.py [--steps 10] [--rounds 3] [--loop-steps 5]

It prints the card and its power limit, then:
  (a) frames_to_textures_kernel over 512 frames of bench.py's views1080_tex scene at k = 1 (1920x1080 frames into
      1920x1080 textures) and over 512 frames of 3840x2160 samples at k = 2 (into 1920x1080 textures), as
      algorithmic bytes (k^2 * 4 read + 4 written per texel) over kernel time (CUDA events around the call, and
      the kernel's own duration from torch.profiler), beside a device-to-device copy of as many bytes measured in
      the same run;
  (b) the impostor loop: 64 views of the textured sphere (512x512 frames), those frames turned into 64 textures,
      then 4096 bitmaps of them (32x32 on screen) drawn into one more frame.  On the device path the frames become
      textures with one dtr_b200_frames_to_textures call; on the host round trip with dtr_b200_read_frames into
      page-locked memory, the byte swizzle in numpy and 64 dtr_b200_update_texture calls.  The two loops are
      alternated, and their final frames must be equal.
Memory: about 34 GB for the 2160p sample frames, 4.3 GB of textures and 8.5 GB for the copy reference at most at once.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from bench import ViewScene  # noqa: E402
from dtrenderer_b200 import scenes  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=10, help="conversions per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the compared configurations")
    ap.add_argument("--loop-steps", type=int, default=5, help="impostor loop iterations per timed window")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    from dtrenderer_b200 import api
    from frame_texture_reference import frame_texture
    print("gpu:", gpu_info().replace("\n", " | "))
    out = {"gpu": gpu_info()}
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    # (a) the conversion kernel over 512 frames
    scene, B = ViewScene("views1080_tex"), 512
    ow, oh = scene.w, scene.h
    out["a"] = {}
    for k in (1, 2):
        r = api.Renderer(k * ow, k * oh, B, 0)
        r.set_stream(stream.cuda_stream)
        scene.record_batch(r, 0, 0, B)
        r.flush()
        r.set_readback_resolve(k)
        tids = r.frames_to_textures(0, B)
        col, _ = r.end_frame(B - 1)
        if not np.array_equal(r.read_texture(tids[-1], (oh, ow, 4)), frame_texture(col)):
            raise SystemExit(f"frame_texture_cost.py: k={k}: texture differs from the conversion of its resolved readback")
        ids = (C.c_int * B)(*tids)

        def convert():
            rc = r.lib.dtr_b200_frames_to_textures(r.ctx, 0, B, ids)
            if rc:
                raise SystemExit(f"dtr_b200_frames_to_textures failed ({rc})")

        src = torch.empty((B, oh, ow), dtype=torch.int32, device="cuda")
        dst = torch.empty_like(src)
        copy = lambda: dst.copy_(src)  # noqa: E731
        convert()
        copy()
        ms = {"convert": [], "copy": []}
        for _ in range(args.rounds):
            ms["convert"].append(timed(convert, args.steps))
            ms["copy"].append(timed(copy, args.steps))
        med = {n: float(np.median(v)) for n, v in ms.items()}
        px = B * ow * oh
        alg = {"convert": px * (k * k * 4 + 4), "copy": 2 * src.numel() * 4}
        gbs = {n: alg[n] / (med[n] * 1e-3) / 1e9 for n in med}
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                convert()
            torch.cuda.synchronize()
        tot, cnt = 0.0, 0
        for e in prof.key_averages():
            if "frames_to_textures_kernel" in e.key:
                tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                cnt += e.count
        us = tot / cnt if cnt else None
        res = {"frames": B, "samples": f"{k * ow}x{k * oh}", "texture": f"{ow}x{oh}", "ms_events": med, "all": ms,
               "algorithmic_bytes": alg, "gbs_events": gbs, "us_profiler": us,
               "gbs_profiler": alg["convert"] / (us * 1e-6) / 1e9 if us else None,
               "frac_of_copy_events": gbs["convert"] / gbs["copy"]}
        out["a"][f"k{k}"] = res
        print(f"(a) k={k}: {B} frames of {k * ow}x{k * oh} -> {ow}x{oh} textures: {med['convert']:.3f} ms (events), "
              f"{us and us / 1e3:.3f} ms (profiler), {gbs['convert']:.0f} GB/s algorithmic = "
              f"{res['frac_of_copy_events']:.2f} of this run's D2D copy ({gbs['copy']:.0f} GB/s)")
        del src, dst
        r.close()
        torch.cuda.empty_cache()

    # (b) the impostor loop, device path against the host round trip
    n, size, grid = 64, 512, 64
    mesh, tex = scenes.uv_sphere(), scenes.random_texture(256, 256, 1, True)
    ts, pos = scenes.view_transforms(n), np.zeros((n, 3), np.float32)
    cell = scenes.transform7(0.0, (0.0, 0.0, 0.0), (1.0 / 16, 1.0 / 16, 1.0))
    place = [((i % grid) * size / grid, (i // grid) * size / grid) for i in range(grid * grid)]
    host = torch.empty((n, size, size), dtype=torch.int32, pin_memory=True)
    texels = np.empty((n, size, size, 4), np.uint8)
    ctxs = {}
    for name in ("device", "host_round_trip"):
        r = api.Renderer(size, size, n + 1, 0)
        r.set_stream(stream.cuda_stream)
        tids = [r.create_texture(size, size) for _ in range(n)]
        ctxs[name] = (r, tids)
    r_dev, t_dev = ctxs["device"]
    r_host, t_host = ctxs["host_round_trip"]

    def views(r):
        for f in range(n):
            r.begin_frame(f)
            r.clear((0.5, 0.0, 1.0))
        r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos, ts, 0)

    def sprites(r, tids):
        r.begin_frame(n)
        r.clear((0.2, 0.2, 0.2))
        for i in range(grid * grid):
            r.bitmap_id(tids[i % n], place[i], cell, (1, 1, 1, 1))
        r.flush()

    host_ms = []

    def step_device():
        views(r_dev)
        r_dev.frames_to_textures(0, n, t_dev)
        sprites(r_dev, t_dev)

    def step_host():
        views(r_host)
        r_host.read_frames_ptr(0, n, host.data_ptr())
        t0 = time.perf_counter()
        b = host.numpy().view(np.uint8).reshape(n, size, size, 4)  # B, G, R, X
        texels[..., 0], texels[..., 1], texels[..., 2], texels[..., 3] = b[..., 2], b[..., 1], b[..., 0], 255
        host_ms.append((time.perf_counter() - t0) * 1e3)
        for f in range(n):
            r_host.update_texture(t_host[f], texels[f])
        sprites(r_host, t_host)

    def loop(step, r):
        step()
        r.sync()
        t0 = time.perf_counter()
        for _ in range(args.loop_steps):
            step()
        r.sync()
        return (time.perf_counter() - t0) * 1e3 / args.loop_steps

    loops = {"device": (step_device, r_dev), "host_round_trip": (step_host, r_host)}
    ms = {name: [] for name in loops}
    for _ in range(args.rounds):
        for name, (step, r) in loops.items():
            ms[name].append(loop(step, r))
    if not np.array_equal(r_dev.end_frame(n)[0], r_host.end_frame(n)[0]):
        raise SystemExit("frame_texture_cost.py: the impostor frames of the two paths differ")
    med = {name: float(np.median(v)) for name, v in ms.items()}
    out["b_impostor_loop"] = {"views": n, "frame": f"{size}x{size}", "bitmaps": grid * grid, "ms_per_iteration": med, "all": ms,
                              "host_swizzle_ms_median": float(np.median(host_ms)), "d2h_bytes": n * size * size * 4,
                              "h2d_bytes": n * size * size * 4, "speedup": med["host_round_trip"] / med["device"]}
    print(f"(b) impostor loop ({n} views of {size}x{size}, {grid * grid} bitmaps): device {med['device']:.2f} ms, "
          f"host round trip {med['host_round_trip']:.2f} ms per iteration (of which numpy swizzle "
          f"{np.median(host_ms):.2f} ms), x{out['b_impostor_loop']['speedup']:.2f}")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
