"""What the triangle id planes cost: raster-stage and step time of the bench workloads with ids off and on,
and of another build of the library (e.g. the commit before the id planes) with ids off.

    python tools/ids_cost.py --out DIR [--other-lib PATH] [--steps 20] [--reps 2]

Every arm runs in its own process (one library per process, chosen with DTR_B200_LIB); the arms alternate
rep by rep so that drift on a shared machine spreads over all of them.  Per arm: one flush, warm-up replays,
then `steps` timed replays (host clock around work that ends in a synchronise) with the per-stage events on
(dtr_b200_get_stage_ms).  Prints the card's name and power limit and a table; writes DIR/ids_cost.json.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = ("views1080_tex", "mesh1080", "mesh4k_tex", "fill4k")  # bench.py's four, at bench sizes


def run_arm(workload, ids, steps, warmup):
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    import ctypes
    from dtrenderer_b200 import api, scenes
    if not ids:  # another build may predate some entry points of the binding: bind what it has
        lib = ctypes.CDLL(api.LIB_PATH)
        api.SYMBOLS = [s for s in api.SYMBOLS if hasattr(lib, s[0])]
    if workload in bench.FILL:
        f = bench.FILL[workload]
        w, h, frames = f["w"], f["h"], 1
        p, color = scenes.small_triangles(w, h, f["n"], seed=7)
        r = api.Renderer(w, h, 1, 0)

        def record():
            r.begin_frame(0)
            r.clear((0, 0, 0))
            r.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
    else:
        s = bench.WORKLOADS[workload]
        w, h, frames = s["w"], s["h"], s["views"]
        scene = bench.ViewScene(workload)
        r = api.Renderer(w, h, frames, 0)

        def record():
            scene.record_batch(r, 0, 0, frames)
    if ids:
        r.set_id_output(True)
    record()
    r.flush()
    for _ in range(warmup):
        r.replay()
    r.sync()
    r.set_profiling(True)
    r.reset_stage_ms()
    t0 = time.perf_counter()
    for _ in range(steps):
        r.replay()
    r.sync()
    step_ms = (time.perf_counter() - t0) * 1e3 / steps
    stage, runs = r.stage_ms()
    col = r.end_frame(0)[0]
    out = {"step_ms": step_ms, "raster_ms": stage["raster"] / max(runs, 1),
           "pre_raster_ms": (stage["setup"] + stage["scan"] + stage["bin"]) / max(runs, 1),
           "frame0_color_sum": int(col.astype(np.uint64).sum())}
    if ids:
        out["frame0_ids_nonzero"] = int((r.read_ids(0, 1) > 0).sum())
    print("ARM " + json.dumps(out))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--other-lib", default="", help="libdtr_b200.so of another build, measured with ids off")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--arm", nargs=2, metavar=("WORKLOAD", "IDS"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.arm:
        return run_arm(a.arm[0], a.arm[1] == "1", a.steps, a.warmup)
    gpu = card()
    print("card (name, power limit, max SM clock):", gpu, flush=True)
    arms = [("ids_off", "", "0"), ("ids_on", "", "1")]
    if a.other_lib:
        arms.insert(0, ("other_ids_off", os.path.abspath(a.other_lib), "0"))
    res = {}
    for wl in a.workloads.split(","):
        for rep in range(a.reps):
            for name, lib, ids in arms:
                env = dict(os.environ)
                env.pop("DTR_B200_LIB", None)
                if lib:
                    env["DTR_B200_LIB"] = lib
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--out", a.out, "--steps", str(a.steps),
                                    "--warmup", str(a.warmup), "--arm", wl, ids], capture_output=True, text=True, env=env)
                line = [ln for ln in p.stdout.splitlines() if ln.startswith("ARM ")]
                if p.returncode or not line:
                    raise SystemExit(f"{wl} {name} failed ({p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-2000:]}")
                res.setdefault(wl, {}).setdefault(name, []).append(json.loads(line[0][4:]))
                print(wl, name, rep, res[wl][name][-1], flush=True)
    summary = {}
    for wl, by in res.items():
        summary[wl] = {}
        for name, runs in by.items():
            rs, ss = [x["raster_ms"] for x in runs], [x["step_ms"] for x in runs]
            summary[wl][name] = {"raster_ms_median": statistics.median(rs), "raster_ms_min": min(rs), "raster_ms_max": max(rs),
                                 "step_ms_median": statistics.median(ss), "step_ms_min": min(ss), "step_ms_max": max(ss)}
        # the same pixels whichever arm rendered them
        sums = {x["frame0_color_sum"] for runs in by.values() for x in runs}
        summary[wl]["same_frame0_colour_in_every_arm"] = len(sums) == 1
    print(f"\n{'workload':15s} {'arm':15s} {'raster ms (min..max)':>26s} {'step ms (min..max)':>26s}")
    for wl, by in summary.items():
        for name, v in by.items():
            if isinstance(v, dict):
                print(f"{wl:15s} {name:15s} {v['raster_ms_median']:9.3f} ({v['raster_ms_min']:.3f}..{v['raster_ms_max']:.3f})"
                      f" {v['step_ms_median']:9.3f} ({v['step_ms_min']:.3f}..{v['step_ms_max']:.3f})")
        print(f"{wl:15s} same frame-0 colour in every arm: {by['same_frame0_colour_in_every_arm']}")
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "ids_cost.json"), "w") as f:
        json.dump({"card": gpu, "steps": a.steps, "reps": a.reps, "runs": res, "summary": summary}, f, indent=1)


if __name__ == "__main__":
    main()
