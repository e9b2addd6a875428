"""A/B runner: times C2 (1920x1080 primary batch) and C3 (2^22 incoherent rays) on the bunny under several environment
settings in one process (the library reads its RTP_* switches when a scene is created).
    python tools/sweep_env.py "RTP_ANY_CAP=12" "RTP_ANY_CAP=16,RTP_FREE_TREE=0" ...
The first configuration is always the default (no overrides). Checks every configuration's hits against the first."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from rtp_b200 import api, scenes


def time_batch(scene, d_rays, d_hits, reps):
    n = d_rays[0].shape[0]
    st = torch.cuda.current_stream().cuda_stream
    for k in range(10):
        scene.hit_device(d_rays[k % len(d_rays)].data_ptr(), n, d_hits.data_ptr(), st)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(reps):
        scene.hit_device(d_rays[k % len(d_rays)].data_ptr(), n, d_hits.data_ptr(), st)
    e1.record()
    torch.cuda.synchronize()
    return n * reps / (e0.elapsed_time(e1) * 1e-3) / 1e6


def main():
    configs = [""] + sys.argv[1:]
    api.init(0)
    sc = scenes.bunny_lambert()
    cam = api.Camera(1920 / 1080, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    c2 = [torch.empty((1920 * 1080, 8), dtype=torch.float64, device="cuda") for _ in range(2)]
    api.camera_rays_device(cam, 1920, 1080, c2[0].data_ptr())
    torch.cuda.synchronize()
    c2[1].copy_(c2[0])
    c3 = [torch.from_numpy(scenes.incoherent_rays(1 << 22).view(np.float64).reshape(-1, 8)).cuda()]
    h2 = torch.empty((c2[0].shape[0], 2), dtype=torch.float64, device="cuda")
    h3 = torch.empty((c3[0].shape[0], 2), dtype=torch.float64, device="cuda")
    ref2 = ref3 = None
    for rep in range(2):  # two rounds: the second shows run-to-run noise
        for cfg in configs:
            saved = {}
            for kv in filter(None, cfg.split(",")):
                k, v = kv.split("=")
                saved[k] = os.environ.get(k)
                os.environ[k] = v
            scene = api.Scene(sc)
            m2 = time_batch(scene, c2, h2, 40)
            m3 = time_batch(scene, c3, h3, 8)
            s2 = scene.hit_device_counted(c2[0].data_ptr(), c2[0].shape[0], h2.data_ptr())
            s3 = scene.hit_device_counted(c3[0].data_ptr(), c3[0].shape[0], h3.data_ptr())
            a2, a3 = h2.clone(), h3.clone()
            if ref2 is None:
                ref2, ref3 = a2, a3
            ok = bool((a2.view(torch.int64) == ref2.view(torch.int64)).all() and (a3.view(torch.int64) == ref3.view(torch.int64)).all())
            print(f"{cfg or 'default':<48} C2 {m2:8.1f}  C3 {m3:8.1f} Mrays/s   nodes/ray {s2.node_visits / s2.rays:.2f} / {s3.node_visits / s3.rays:.2f}"
                  f"  rewalks {s2.order_rewalks} / {s3.order_rewalks}  {'' if ok else 'MISMATCH'}", flush=True)
            scene.close()
            for k, v in saved.items():
                if v is None:
                    del os.environ[k]
                else:
                    os.environ[k] = v


if __name__ == "__main__":
    main()
