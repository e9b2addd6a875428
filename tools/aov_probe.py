"""What the albedo and normal buffers cost: rtp_render against rtp_render_aov on the frames bench.py renders.

Workloads: C1 (scenes.bunny_lambert(), 640 x 360, 16 spp, depth 8), C4 (scenes.demo(), 1920 x 1080, 256 spp, depth 8) and one 32 x 32
tile of the C1 frame at 16 spp (16,384 paths: rtp_render runs it in tail mode, rtp_render_aov as trace/shade pairs). Each workload
is warmed up with one call of each kind, then the two calls alternate for --repeats rounds; the time is rtp_stats.device_ms (CUDA
events around the call's work on the device). The colour of every rtp_render_aov call is checked against rtp_render's bytes.

    python tools/aov_probe.py --out profiles/aov_probe.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rtp_b200 import api, scenes  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def probe(g, label, w, h, spp, depth, seed, repeats, tile=None):
    def plain():
        return g.render(w, h, spp, max_bounce=depth, seed=seed, tile=tile)

    def aov():
        return g.render_aov(w, h, spp, max_bounce=depth, seed=seed, tile=tile)

    ref = plain()
    aov()
    ms = {"render": [], "render_aov": []}
    launches = {}
    for _ in range(repeats):
        a = plain()
        b = aov()
        assert a[0].tobytes() == ref[0].tobytes() and b[0].tobytes() == ref[0].tobytes() and b[1].tobytes() == ref[1].tobytes()
        ms["render"].append(a[-1].device_ms)
        ms["render_aov"].append(b[-1].device_ms)
        launches = {"render": a[-1].kernel_launches, "render_aov": b[-1].kernel_launches}
    med = {k: float(np.median(v)) for k, v in ms.items()}
    paths = int(a[-1].paths)
    return {"workload": label, "width": w, "height": h, "spp": spp, "max_bounce": depth, "tile": tile, "paths": paths,
            "device_ms": ms, "device_ms_median": med, "overhead_ms": med["render_aov"] - med["render"],
            "overhead_pct": 100.0 * (med["render_aov"] / med["render"] - 1.0), "kernel_launches": launches,
            "aov_record_bytes": 96 * paths}  # 48 B written by the shade kernel and 48 B read by aov_resolve_kernel per path


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()

    api.init(0)
    report = {"card": card(), "repeats": a.repeats, "timer": "rtp_stats.device_ms, median of alternating calls after one warm-up each",
              "runs": []}
    with api.Scene(scenes.bunny_lambert()) as g:
        report["runs"].append(probe(g, "C1: bunny Lambert + sky", 640, 360, 16, 8, a.seed, a.repeats))
        print(report["runs"][-1], flush=True)
        report["runs"].append(probe(g, "C1 scene, one 32x32 tile (tail mode for rtp_render)", 640, 360, 16, 8, a.seed, a.repeats,
                                    tile=(304, 164, 32, 32)))
        print(report["runs"][-1], flush=True)
    with api.Scene(scenes.demo()) as g:
        report["runs"].append(probe(g, "C4: demo scene", 1920, 1080, 256, 8, a.seed, a.repeats))
        print(report["runs"][-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
