"""Adaptive against fixed sampling on the C4 frame (scenes.demo(), 1920 x 1080, depth 8): device time, sample counts and error.

For fixed 256 spp and for rtp_render_adaptive (min 16, max 256, batch 16) at several rel_tol values it reports the device time
(rtp_stats.device_ms after a warm-up render, then several repeats), the mean and histogram of the per-pixel sample counts n_p, the
rounds and kernel launches, and the RMSE of the frame against a 1024-spp frame of the same seed. Each adaptive setting is also
compared with a fixed render at its mean sample count (rounded), the uniform render of about the same number of paths.

    python tools/adaptive_probe.py --out profiles/adaptive_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rtp_b200 import api, scenes  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def rmse(a, b):
    return float(np.sqrt(((a - b) ** 2).mean()))


def timed(fn, repeats):
    fn()  # warm-up
    ms, out = [], None
    for _ in range(repeats):
        t0 = time.perf_counter()
        out = fn()
        wall = (time.perf_counter() - t0) * 1e3
        ms.append((out[-1].device_ms, wall))
    dev = [m[0] for m in ms]
    return out, {"device_ms": dev, "device_ms_median": float(np.median(dev)), "wall_ms_median": float(np.median([m[1] for m in ms]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--depth", type=int, default=8)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--rel-tol", type=float, nargs="+", default=[0.1, 0.03, 0.01])
    ap.add_argument("--reference-spp", type=int, default=1024)
    a = ap.parse_args()
    w, h, depth, seed = a.width, a.height, a.depth, a.seed
    mn, mx, batch = 16, 256, 16

    api.init(0)
    g = api.Scene(scenes.demo())
    report = {"card": card(), "scene": "demo (C4)", "width": w, "height": h, "max_bounce": depth, "seed": seed,
              "reference_spp": a.reference_spp, "repeats": a.repeats, "adaptive": {"min_samples": mn, "max_samples": mx, "batch": batch}}
    ref = g.render(w, h, a.reference_spp, max_bounce=depth, seed=seed)[0]

    def fixed(spp):
        (img, _, st), t = timed(lambda: g.render(w, h, spp, max_bounce=depth, seed=seed), a.repeats)
        return {"spp": spp, **t, "paths": st.paths, "kernel_launches": st.kernel_launches, "rmse_vs_reference": rmse(img, ref)}

    report["fixed_256"] = fixed(256)
    print("fixed 256:", report["fixed_256"], flush=True)
    report["adaptive_runs"] = []
    for rel in a.rel_tol:
        (img, _, n, st), t = timed(lambda: g.render_adaptive(w, h, mn, mx, batch, rel_tol=rel, max_bounce=depth, seed=seed), a.repeats)
        counts = np.arange(mn, mx + 1, batch)
        hist = {int(c): int((n == c).sum()) for c in counts}
        run = {"rel_tol": rel, "abs_tol": 0.0, **t, "paths": st.paths, "mean_samples": float(n.mean()),
               "samples_histogram": hist, "rounds": int((int(n.max()) - mn) // batch + 1), "kernel_launches": st.kernel_launches,
               "rmse_vs_reference": rmse(img, ref)}
        run["fixed_at_mean_samples"] = fixed(max(1, int(round(n.mean()))))
        report["adaptive_runs"].append(run)
        print(f"rel_tol {rel}:", run, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    g.close()


if __name__ == "__main__":
    main()
