#!/usr/bin/env python
"""What drawing from device memory (dtr_b200_triangles_device) costs and saves on one GPU.

    python tools/device_geometry_cost.py [--frames 10] [--rounds 3] [--reps 20]

It prints the card and its power limit, then:
  (1) gather_device_inputs_kernel, the flush's snapshot of the 1 M-triangle arrays of bench.py's fill4k scene
      (p f32[n*9] + color f32[n*4] = 52 B per triangle, 16-byte aligned torch tensors), as bytes read + written over
      its mean kernel time from torch.profiler, beside a device-to-device copy of as many bytes measured in the same run.
      L2 is overwritten (256 MB) before every flush and every copy, so both read their source from HBM;
  (2) the dynamic fill4k loop: torch moves every triangle each frame (an integer shift of x and y), and the frame is
      begun (depth reset), cleared and drawn either through the host path (.cpu() of both tensors, dtr_b200_triangles, flush) or through
      dtr_b200_triangles_device and a flush.  Both paths run on the same torch stream (set_stream), each in its own
      3840x2160 context; the windows alternate and end with a device synchronise.  The final frames must be equal.
Memory: under 2 GB.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from dtrenderer_b200 import scenes  # noqa: E402

W, H, N = 3840, 2160, 1 << 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--frames", type=int, default=10, help="frames per timed window of the dynamic loop")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two paths")
    ap.add_argument("--reps", type=int, default=20, help="profiled flushes and copies of (1)")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    from dtrenderer_b200 import api
    info = gpu_info()
    print("gpu:", info.replace("\n", " | "))
    out = {"gpu": info}
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    p, color = scenes.small_triangles(W, H, N)
    T = scenes.DEFAULT_TRIANGLE_TRANSFORM
    tp, tc = torch.from_numpy(p.reshape(-1)).cuda(), torch.from_numpy(color.reshape(-1)).cuda()
    nbytes = (tp.numel() + tc.numel()) * 4
    scrub = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    # (1) the gather kernel against a device copy of as many bytes
    r = api.Renderer(W, H, 1, 0)
    r.set_stream(stream.cuda_stream)
    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)

    def flush_once():
        scrub.zero_()
        r.clear((0.0, 0.0, 0.0))
        r.triangles_device(tp, tc, transform=T)
        r.flush()

    def copy_once():
        scrub.zero_()
        dst.copy_(src)

    for _ in range(3):
        flush_once()
        copy_once()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            flush_once()
            copy_once()
        torch.cuda.synchronize()
    tot = {"gather": 0.0, "copy": 0.0}
    cnt = {"gather": 0, "copy": 0}
    for e in prof.key_averages():
        which = "gather" if "gather_device_inputs_kernel" in e.key else ("copy" if "Memcpy DtoD" in e.key else None)
        if which:
            tot[which] += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            cnt[which] += e.count
    if cnt["gather"] != args.reps or cnt["copy"] != args.reps:
        raise SystemExit(f"the profile holds {cnt} gather kernels / device copies, {args.reps} of each expected")
    g_us, c_us = tot["gather"] / cnt["gather"], tot["copy"] / cnt["copy"]
    g_gbs, c_gbs = 2 * nbytes / g_us / 1e3, 2 * nbytes / c_us / 1e3
    out["gather"] = {"triangles": N, "bytes": nbytes, "us_mean": {"gather": g_us, "copy": c_us}, "count": cnt,
                     "gbs_read_plus_written": {"gather": g_gbs, "copy": c_gbs}, "frac_of_copy": g_gbs / c_gbs}
    print(f"(1) gather of {N} triangles ({nbytes / 1e6:.1f} MB): {g_us:.1f} us = {g_gbs:.0f} GB/s read+written; "
          f"device copy of as many bytes {c_us:.1f} us = {c_gbs:.0f} GB/s; gather/copy = {g_gbs / c_gbs:.2f}")
    r.close()
    del src, dst

    # (2) the dynamic loop: every triangle moves every frame
    paths = {}
    for name in ("host", "device"):
        rr = api.Renderer(W, H, 1, 0)
        rr.set_stream(stream.cuda_stream)
        paths[name] = {"r": rr, "p": tp.clone(), "c": tc.clone(), "frame": 0, "ms": []}

    def move(s):
        f = s["frame"]
        s["frame"] += 1
        xy = s["p"].view(N, 3, 3)[:, :, :2]
        xy += float((f % 7) - 3)

    def frame(name):
        s = paths[name]
        move(s)
        rr = s["r"]
        rr.begin_frame(0)
        rr.clear((0.0, 0.0, 0.0))
        if name == "host":
            rr.triangles(s["p"].cpu().numpy(), s["c"].cpu().numpy(), T)
        else:
            rr.triangles_device(s["p"], s["c"], transform=T)
        rr.flush()

    for name in paths:  # warm-up
        for _ in range(2):
            frame(name)
    for _ in range(args.rounds):
        for name in paths:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.frames):
                frame(name)
            torch.cuda.synchronize()
            paths[name]["ms"].append((time.perf_counter() - t0) * 1e3 / args.frames)
    assert paths["host"]["frame"] == paths["device"]["frame"]
    ch, zh = paths["host"]["r"].end_frame(0)
    cd, zd = paths["device"]["r"].end_frame(0)
    if not (np.array_equal(ch, cd) and np.array_equal(zh.view(np.uint32), zd.view(np.uint32))):
        raise SystemExit("the final frames of the two paths differ")
    ms = {k: float(np.median(v["ms"])) for k, v in paths.items()}
    out["dynamic_fill4k"] = {"triangles": N, "frame": f"{W}x{H}", "frames_per_window": args.frames,
                             "ms_per_frame": ms, "all": {k: v["ms"] for k, v in paths.items()},
                             "speedup": ms["host"] / ms["device"], "final_frames_equal": True,
                             "uploadBytes": {k: v["r"].stats()["uploadBytes"] for k, v in paths.items()}}
    print(f"(2) dynamic fill4k ({N} moving triangles, {W}x{H}): host path {ms['host']:.2f} ms, device path "
          f"{ms['device']:.2f} ms per frame, x{ms['host'] / ms['device']:.2f}; final frames equal")
    for v in paths.values():
        v["r"].close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
