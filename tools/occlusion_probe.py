"""Occlusion query (rtp_trace_occluded*) against closest hit (rtp_trace_closest*) on the same rays of the bunny scene:

    python tools/occlusion_probe.py [--steps K] [--c3-steps K3] [--out FILE.json]

Workloads: (a) shadow rays from every primary hit of the C2 camera (1920x1080, rtp_trace_closest_full) toward a point light above
the scene, d = light - p, t_min = 1e-3, t_max = 1; (b) one cosine-weighted hemisphere ray about each hit's normal (turned toward
the camera), t_max = AO_RADIUS; (c) the C3 incoherent stream (2^24 rays, bench.py's definition). For each, the device calls are
timed with CUDA events over K steps, two ray buffers rotated as bench.py does (the report says whether the pair exceeds L2),
occlusion and closest hit alternated over two rounds; every timed step writes its own output slice, and every step's occlusion
bytes are checked against that step's `leaf != MISS`. Node visits per ray come from the counted calls. The host-buffer calls are timed on workload (a). The card's name,
power limit and max SM clock are read in the same run (nvidia-smi -i <uuid> --query-gpu, read-only)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import C3_LOG2, H, W, incoherent_rays_device  # noqa: E402
from rtp_b200 import _abi as A  # noqa: E402
from rtp_b200 import api, scenes  # noqa: E402

LIGHT = np.array([1.0, 4.0, 2.0])  # above and in front of the bunny (its box: x -0.94..0.61, y 0..1.54, z -0.62..0.59)
AO_RADIUS = 0.25


def card():
    """the measured device, named by its UUID (CUDA's device order need not be nvidia-smi's)"""
    uuid = f"GPU-{torch.cuda.get_device_properties(torch.cuda.current_device()).uuid}"
    q = subprocess.run(["nvidia-smi", "-i", uuid, "--query-gpu=uuid,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    got, name, power, clock = (x.strip() for x in q.stdout.strip().split(","))
    assert got.lower() == uuid.lower(), (got, uuid)
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "uuid": uuid}


def shadow_rays(hits):
    p = hits["position"]
    r = np.zeros(len(hits), dtype=A.RAY_DTYPE)
    r["origin"], r["direction"], r["t_min"], r["t_max"] = p, LIGHT - p, 1e-3, 1.0
    return r


def ao_rays(hits, primary_dirs, seed=3):
    n = hits["normal"] / np.linalg.norm(hits["normal"], axis=1, keepdims=True)
    n = np.where((n * primary_dirs).sum(axis=1, keepdims=True) > 0.0, -n, n)  # the side the camera sees
    rng = np.random.default_rng(seed)
    u1, u2 = rng.random(len(n)), rng.random(len(n))
    r, phi = np.sqrt(u1), 2.0 * np.pi * u2
    a = np.where(np.abs(n[:, :1]) > 0.9, [[0.0, 1.0, 0.0]], [[1.0, 0.0, 0.0]])  # any vector not parallel to n
    t = np.cross(n, a)
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    b = np.cross(n, t)
    d = (r * np.cos(phi))[:, None] * t + (r * np.sin(phi))[:, None] * b + np.sqrt(np.maximum(0.0, 1.0 - u1))[:, None] * n
    rays = np.zeros(len(n), dtype=A.RAY_DTYPE)
    rays["origin"], rays["direction"], rays["t_min"], rays["t_max"] = hits["position"], d, 1e-3, AO_RADIUS
    return rays


def timed(fn, steps, warmup):
    for k in range(warmup):
        fn(k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        fn(k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def device_leg(scene, name, d_ray, steps, stream):
    """d_ray: [n, 8] float64 on the device. Returns the leg's report."""
    n = d_ray.shape[0]
    bufs = [d_ray, d_ray.clone()]  # two buffers rotated between steps, as bench.py does; whether they exceed L2 is reported with the rates
    occ = torch.empty((steps, n), dtype=torch.uint8, device="cuda")
    hit = torch.empty((steps, n, 2), dtype=torch.float64, device="cuda")
    rounds = []
    for _ in range(2):
        ms_c = timed(lambda k: scene.hit_device(bufs[k & 1].data_ptr(), n, hit[k].data_ptr(), stream), steps, 2)
        ms_o = timed(lambda k: scene.occluded_device(bufs[k & 1].data_ptr(), n, occ[k].data_ptr(), stream), steps, 2)
        leaf = hit[..., 0].view(torch.int64) & 0xFFFFFFFF
        agree = bool(((leaf != A.MISS).to(torch.uint8) == occ).all())
        rounds.append({"closest_mrays_per_s": steps * n / (ms_c * 1e-3) / 1e6, "occluded_mrays_per_s": steps * n / (ms_o * 1e-3) / 1e6,
                       "every_step_agrees": agree})
    sc_ = scene.hit_device_counted(bufs[0].data_ptr(), n, hit[0].data_ptr())
    so = scene.occluded_device_counted(bufs[0].data_ptr(), n, occ[0].data_ptr())
    frac = float(occ[0].float().mean())
    l2 = torch.cuda.get_device_properties(torch.cuda.current_device()).L2_cache_size
    rep = {"workload": name, "rays": n, "steps": steps, "occluded_fraction": frac, "rounds": rounds,
           "rotated_ray_bytes": 2 * n * 64, "l2_bytes": l2, "rotated_rays_exceed_l2": 2 * n * 64 > l2,
           "speedup_occluded_over_closest": [r["occluded_mrays_per_s"] / r["closest_mrays_per_s"] for r in rounds],
           "node_visits_per_ray": {"closest": sc_.node_visits / n, "occluded": so.node_visits / n},
           "primitive_tests_per_ray": {"closest": (sc_.triangle_tests + sc_.sphere_tests) / n, "occluded": (so.triangle_tests + so.sphere_tests) / n},
           "conservative_violations": int(sc_.conservative_violations + so.conservative_violations)}
    del occ, hit, bufs
    torch.cuda.empty_cache()
    return rep


def host_leg(scene, rays, steps):
    n = len(rays)
    h_rays = api.PinnedBuffer((n,), A.RAY_DTYPE)
    h_hits = api.PinnedBuffer((n,), A.HIT_DTYPE)
    h_occ = api.PinnedBuffer((n,), np.bool_)
    h_rays.array[:] = rays
    out = {"workload": "host buffers, workload (a)", "rays": n, "steps": steps}
    for tag, fn in (("closest", lambda: scene.hit(h_rays.array, out=h_hits.array)), ("occluded", lambda: scene.occluded(h_rays.array, out=h_occ.array))):
        fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        out[f"{tag}_mrays_per_s"] = steps * n / (time.perf_counter() - t0) / 1e6  # both calls return after their last copy is done
    _, st = scene.occluded(h_rays.array, out=h_occ.array, stats=True)
    out["agrees"] = bool((h_occ.array == (h_hits.array["leaf"] != A.MISS)).all())
    out["stats"] = {"rays": int(st.rays), "kernel_launches": int(st.kernel_launches), "device_ms": st.device_ms}
    for b in (h_rays, h_hits, h_occ):
        b.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--c3-steps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the report here (JSON)")
    args = ap.parse_args()
    api.init(0)
    stream = torch.cuda.current_stream().cuda_stream
    report = {"card": card()}
    sc = scenes.bunny_lambert()
    scene = api.Scene(sc)
    cam = api.Camera(W / H, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    primary = api.camera_rays(cam, W, H)
    full = scene.hit_full(primary)
    hit = full["leaf"] != A.MISS
    report["primary_hits"] = int(hit.sum())
    sh = shadow_rays(full[hit])
    ao = ao_rays(full[hit], primary["direction"][hit])
    legs = []
    for name, rays in (("(a) shadow rays from the C2 hits toward a point light, t_max = 1", sh), (f"(b) cosine-hemisphere AO rays, t_max = {AO_RADIUS}", ao)):
        legs.append(device_leg(scene, name, torch.from_numpy(rays.view(np.float64).reshape(-1, 8).copy()).cuda(), args.steps, stream))
        print(json.dumps(legs[-1]), flush=True)
    d3 = incoherent_rays_device(torch, 1 << C3_LOG2, torch.device("cuda"))
    legs.append(device_leg(scene, f"(c) C3: 2^{C3_LOG2} incoherent rays", d3, args.c3_steps, stream))
    print(json.dumps(legs[-1]), flush=True)
    del d3
    report["device"] = legs
    report["host"] = host_leg(scene, sh, 10)
    print(json.dumps(report["host"]), flush=True)
    print(json.dumps({"card": report["card"]}), flush=True)
    scene.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
