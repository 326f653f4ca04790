#!/usr/bin/env python
"""What 2x2 supersampling with the readback resolve costs on the headline workload (one GPU).

    python tools/resolve_cost.py [--views 512] [--k 2] [--steps 10] [--rounds 3]

The headline scene (bench.py's views1080_tex: the textured 2500-triangle mesh, 1024^2 texture) with --views views
rendered at 3840x2160 samples and read back at 1920x1080 (k = 2).  It prints:
  (a) replay time of the views at 2160p samples against 1080p without resolve, alternated in the same run;
  (b) resolve_frames_kernel over all the views, colour only and colour + depth, as algorithmic bytes
      (k^2 * 4 read + 4 written per plane per output pixel) over kernel time (CUDA events, and the kernel's
      own duration from torch.profiler), beside a device-to-device copy measured in the same run and the
      6547.5 GB/s copy bandwidth DESIGN.md section 5 quotes;
  (c) bench.py's end-to-end loop (8 flushes of 64 views into two pinned halves) through the resolved
      read_frames_async and the resolved bgr24 readback, beside the same loop at 1080p without resolve and the
      D2H-only ceiling of the same bytes.
Memory: 512 frames of 3840x2160 colour + depth take 34 GB, the 1080p context 8.5 GB more, the resolve
outputs 8.5 GB and the copy reference 8.5 GB: about 60 GB of device memory.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bench import SUB, ViewScene  # noqa: E402

DESIGN_COPY_GBS = 6547.5  # DESIGN.md section 5: MEASURED_PEAKS.json hbm_gbs, a device copy measured on a B200


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--views", type=int, default=512)
    ap.add_argument("--k", type=int, default=2)
    ap.add_argument("--steps", type=int, default=10, help="replays / resolves per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the compared configurations")
    ap.add_argument("--e2e-steps", type=int, default=5)
    args = ap.parse_args()

    import torch
    from dtrenderer_b200 import api
    print("gpu:", gpu_info().replace("\n", " | "))
    k, B = args.k, args.views
    scene = ViewScene("views1080_tex")
    ow, oh = scene.w, scene.h
    w, h = k * ow, k * oh
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def events():
        return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n):
        e0, e1 = events()
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / n

    big = api.Renderer(w, h, B, 0)
    small = api.Renderer(ow, oh, B, 0)
    for r in (big, small):
        r.set_stream(stream.cuda_stream)
        scene.record_batch(r, 0, 0, B)
        r.flush()
        for _ in range(3):
            r.replay()
    big.set_readback_resolve(k)
    out = {"gpu": gpu_info(), "views": B, "k": k, "samples": f"{w}x{h}", "output": f"{ow}x{oh}"}

    # check: a resolved readback equals the numpy resolve of the same frame's sample readback
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from resolve_reference import resolve_colour, resolve_depth
    big.set_readback_resolve(1)
    c1, z1 = big.end_frame(B - 1)
    big.set_readback_resolve(k)
    ck, zk = big.end_frame(B - 1)
    if not (np.array_equal(ck, resolve_colour(c1, k)) and np.array_equal(zk.view(np.uint32), resolve_depth(z1, k).view(np.uint32))):
        raise SystemExit("resolve_cost.py: resolved frame differs from the numpy resolve of its samples")

    # (a) replay time, 2160p samples against 1080p, alternated
    rep = {"1080p": [], "2160p_samples": []}
    for _ in range(args.rounds):
        rep["1080p"].append(timed(small.replay, args.steps))
        rep["2160p_samples"].append(timed(big.replay, args.steps))
    med = {n: float(np.median(v)) for n, v in rep.items()}
    out["a_replay_ms"] = {"median": med, "all": rep, "ratio": med["2160p_samples"] / med["1080p"]}
    print(f"(a) replay of {B} views: 1080p {med['1080p']:.3f} ms, 2160p samples {med['2160p_samples']:.3f} ms "
          f"(x{out['a_replay_ms']['ratio']:.2f})")

    # (b) resolve_frames_kernel over all B frames
    col = torch.empty((B, oh, ow), dtype=torch.int32, device="cuda")
    dep = torch.empty((B, oh, ow), dtype=torch.float32, device="cuda")
    lib, ctx = big.lib, big.ctx
    import ctypes as C

    def resolve(with_depth):
        rc = lib.dtr_b200_resolve_frames(ctx, 0, B, C.c_void_p(col.data_ptr()), C.c_void_p(dep.data_ptr()) if with_depth else None, None)
        if rc:
            raise SystemExit(f"dtr_b200_resolve_frames failed ({rc})")

    src = torch.empty((B, oh, ow, 2), dtype=torch.int32, device="cuda")  # 8.5 GB: as many bytes as colour + depth move
    dst = torch.empty_like(src)
    px = B * ow * oh
    res = {"colour": [], "colour_depth": [], "copy": []}
    for fn in (lambda: resolve(False), lambda: resolve(True), lambda: dst.copy_(src)):
        fn()
    for _ in range(args.rounds):
        res["colour"].append(timed(lambda: resolve(False), args.steps))
        res["colour_depth"].append(timed(lambda: resolve(True), args.steps))
        res["copy"].append(timed(lambda: dst.copy_(src), args.steps))
    ms = {n: float(np.median(v)) for n, v in res.items()}
    alg = {"colour": px * (k * k * 4 + 4), "colour_depth": 2 * px * (k * k * 4 + 4), "copy": 2 * src.numel() * 4}
    gbs = {n: alg[n] / (ms[n] * 1e-3) / 1e9 for n in ms}
    # the kernel's own duration (torch.profiler, a run of its own)
    prof_us = {}
    from torch.profiler import ProfilerActivity, profile
    for name, depth_too in (("colour", False), ("colour_depth", True)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                resolve(depth_too)
            torch.cuda.synchronize()
        tot, cnt = 0.0, 0
        for e in prof.key_averages():
            if "resolve_frames_kernel" in e.key:
                tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                cnt += e.count
        prof_us[name] = tot / cnt if cnt else None
    out["b_resolve"] = {"ms_events": ms, "algorithmic_bytes": alg, "gbs_events": gbs, "us_profiler": prof_us,
                        "gbs_profiler": {n: alg[n] / (u * 1e-6) / 1e9 for n, u in prof_us.items() if u},
                        "copy_gbs_design": DESIGN_COPY_GBS,
                        "frac_of_copy_this_run": {n: gbs[n] / gbs["copy"] for n in ("colour", "colour_depth")},
                        "frac_of_copy_design": {n: gbs[n] / DESIGN_COPY_GBS for n in ("colour", "colour_depth")}}
    for n in ("colour", "colour_depth"):
        print(f"(b) resolve_frames_kernel {n}: {ms[n]:.3f} ms (events), {prof_us[n] and prof_us[n] / 1e3:.3f} ms (profiler), "
              f"{gbs[n]:.0f} GB/s algorithmic = {gbs[n] / gbs['copy']:.2f} of this run's D2D copy ({gbs['copy']:.0f} GB/s), "
              f"{gbs[n] / DESIGN_COPY_GBS:.2f} of DESIGN's 6547.5 GB/s copy")
    del src, dst, col, dep

    # (c) bench.py's end-to-end loop
    sub = min(SUB, B)
    nsub = B // sub
    host = torch.empty((2, sub, oh, ow), dtype=torch.int32, pin_memory=True)
    pitch = big.bgr24_pitch()
    host24 = torch.empty((2, sub, oh, pitch), dtype=torch.uint8, pin_memory=True)

    def e2e(r, read_half, n_steps):
        turn = [0]

        def step():
            for j in range(nsub):
                half = turn[0] & 1
                turn[0] += 1
                scene.record_batch(r, half * sub, j * sub, sub)
                read_half(r, half)

        step()
        r.wait_reads()
        e0, e1 = events()
        e0.record(stream)
        for _ in range(n_steps):
            step()
        r.wait_reads()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / n_steps

    u32 = lambda r, half: r.read_frames_async_ptr(half * sub, sub, host[half].data_ptr())  # noqa: E731
    b24 = lambda r, half: r.read_frames_bgr24_async_ptr(half * sub, sub, host24[half].data_ptr())  # noqa: E731
    dcol = torch.empty((sub, oh, ow), dtype=torch.int32, device="cuda")

    def d2h_only():
        e0, e1 = events()
        host[0].copy_(dcol, non_blocking=True)
        e0.record(stream)
        for i in range(2 * nsub):
            host[i & 1].copy_(dcol, non_blocking=True)
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / 2

    loops = {"1080p_u32": lambda: e2e(small, u32, args.e2e_steps), "2160p_k2_u32": lambda: e2e(big, u32, args.e2e_steps),
             "1080p_bgr24": lambda: e2e(small, b24, args.e2e_steps), "2160p_k2_bgr24": lambda: e2e(big, b24, args.e2e_steps),
             "d2h_only_u32": d2h_only}
    e2e_ms = {n: [] for n in loops}
    for _ in range(args.rounds):
        for n, fn in loops.items():
            e2e_ms[n].append(fn())
    med = {n: float(np.median(v)) for n, v in e2e_ms.items()}
    out["c_e2e_ms_per_step"] = {"median": med, "all": e2e_ms, "d2h_bytes_u32": B * 4 * ow * oh, "d2h_bytes_bgr24": B * pitch * oh,
                                "frac_of_d2h_ceiling_u32": {n: med["d2h_only_u32"] / med[n] for n in ("1080p_u32", "2160p_k2_u32")}}
    for n in loops:
        print(f"(c) e2e {n}: {med[n]:.2f} ms per step of {B} views")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
