#!/usr/bin/env python
"""bench.py — headline measurement of the hot path on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus 1 ...            # the reference's CPU path (oracle port) on the host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU
    python bench.py ... --dump-outputs DIR                   # also save rank 0's hits of the last timed C2 step as .npy

The inputs are deterministic (camera rays of a fixed scene), so the dumps of two builds can be compared output for output.

Headline workload (BASELINE.json configs[1], "C2"): the 1920x1080 primary-ray closest-hit batch against the bunny BVH
(4,968 triangles + ground sphere, 9,937 nodes). One step = one pass of the closest-hit path over the batch (2,073,600 rays per
GPU). At N > 1 the path shards with no data-path collective: rank r traces sub-sample r of an N-times supersampled 1920x1080
primary batch (weak scaling, 2,073,600 rays per rank).

Printed JSON (ONE line, the last line rank 0 writes to stdout): `value` = C2 Mrays/s with rays and hits resident in HBM; `e2e` =
the same metric through rtp_trace_closest with pinned HOST buffers (H2D + D2H inside the timed region), next to the measured
host-link ceiling; `roofline` for the traversal kernel; `cpu_baseline` = the oracle port on the host cores. The other BASELINE
configs ride along under their own keys, each at its FULL size with a CPU arm of its own:
  `incoherent`  C3: 2^24 incoherent rays per GPU;
  `render`      C1: bunny Lambert + sky, 640x360, 16 spp, depth 8 (device-resident and through rtp_render with host buffers);
  `render_c4`   C4: demo scene 1920x1080, 256 spp TOTAL, rows dealt out over the N ranks (strong scaling), gathered on rank 0;
  `render_c4_weak`  the same scene at 32 spp per GPU (weak scaling);
  `render_c5`   C5: the 10,174,464-triangle bunny field, 3840x2160, 128 spp per GPU (= the named 1024 spp at N = 8), rows over ranks;
                scene build time (on the device) reported next to it;
  `multi_device_abi`  (N > 1) rank 0 alone drives all N GPUs through ONE rtp_render call (rtp_scene_create_multi).
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (no __pycache__ next to the package)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

W, H = 1920, 1080
N_RAYS = W * H
WORKLOAD = "C2: 1920x1080 primary-ray closest-hit batch vs bunny BVH (4968 triangles + ground sphere, 9937 nodes)"
RAY_BYTES, HIT_BYTES, WAVE_HIT_BYTES = 64, 16, 32
C3_LOG2 = 24


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-render", action="store_true", help="skip the C1 / C3 / C4 legs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the hits of the last timed C2 step to DIR/hits_{leaf,material,t}.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_hits(directory, hits):
    """The closest hits of one pass over the C2 batch, one float64 array per field of the hit record (2,073,600 values each,
    49.8 MB in all). Leaf and material ids are exact in float64 and a miss has leaf = MISS (4294967295). The hit record's t is
    +inf on a miss; the dump stores -1 there instead, so that every value is finite (a hit has t >= t_min = 1e-3)."""
    from rtp_b200 import _abi as A

    os.makedirs(directory, exist_ok=True)
    miss = hits["leaf"] == A.MISS
    arrays = {"leaf": hits["leaf"], "material": hits["material"], "t": np.where(miss, -1.0, hits["t"])}
    for field, values in arrays.items():
        np.save(os.path.join(directory, f"hits_{field}.npy"), values.astype(np.float64))


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def bind_to_gpu_local_cores(local_rank, torch):
    """One process per GPU: run this rank (and first-touch its pinned host buffers) on the cores NVML reports as local to its
    GPU, so that the host side of the e2e legs does not cross the socket interconnect. The NVML handle is taken from the CUDA
    device's PCI bus id (NVML enumerates in bus order and ignores CUDA_VISIBLE_DEVICES, so its index is not the CUDA ordinal).
    Returns (number of cores, description) or (None, reason)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(local_rank)
        bus = f"{props.pci_domain_id:08x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, mask in enumerate(words) for b in range(64) if (mask >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus), f"{bus}: cpus {min(cpus)}-{max(cpus)}"
        return None, f"{bus}: NVML reports no local cpus inside this process's affinity mask"
    except Exception as e:  # noqa: BLE001 - reported, not hidden
        return None, f"{type(e).__name__}: {e}"


# ----------------------------------------------------------------------------------------------- clocks

class ClockSampler:
    """samples SM clock / throttle reasons through NVML every 20 ms while `active`"""

    def __init__(self, torch, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.active = False
        self._stop = False
        try:
            import pynvml as nv

            nv.nvmlInit()
            self.nv = nv
            props = torch.cuda.get_device_properties(index)
            bus = f"{props.pci_domain_id:08x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
            self.h = nv.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        if nv is None:
            return
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop:
            if self.active:
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.02)

    def report(self):
        self._stop = True
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------------------------- reference arm

def run_reference(args):
    """The reference's own CPU implementation of the path (oracle port; the Rust crate cannot be built here),
    all host threads, same workload / metric / unit. Each step = one pass over the full C2 batch."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    import oracle
    from rtp_b200 import api, scenes

    sc = scenes.bunny_lambert()
    cam = api.Camera(W / H, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    o = oracle.Scene(sc)
    rays = oracle.camera_rays(cam, W, H)
    cores = os.cpu_count() or 1
    for _ in range(args.warmup):
        o.hit_full(rays, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        hits = o.hit_full(rays, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_hits(args.dump_outputs, hits)
    v = args.steps * N_RAYS / dt / 1e6
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": v, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_step_per_gpu": N_RAYS},
        "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": cores, "kind": "port",
                         "sample": f"full C2 batch (2,073,600 rays) x {args.steps} steps, oracle/rtp_oracle.c, {cores} pthreads"},
        "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- inputs

def incoherent_rays_device(torch, n, device, first=0, seed=0x00C0FFEE, stream=1):
    """BASELINE config C3 (SURVEY.md 8d), the definition of rtp_b200.scenes.incoherent_rays evaluated with torch on the device:
    ray k = draws 0..4 of stream RTP_RNG_STREAM_RAYS at counter k of the shared Philox4x32-10 generator; origin uniform on the
    sphere of radius 3 about the bunny AABB centre, target uniform in the bunny AABB. (The draws are bit-identical to the
    numpy version; cos / sin / sqrt may differ from it in the last ulp, which moves an input ray, not a result.)"""
    M = 0xFFFFFFFF
    idx = torch.arange(first, first + n, dtype=torch.int64, device=device)
    draws = []
    for block in range(3):
        c0, c1 = idx & M, (idx >> 32) & M
        c2 = torch.full_like(idx, block)
        c3 = torch.full_like(idx, stream)
        k0, k1 = seed & M, (seed >> 32) & M
        for _ in range(10):
            p0, p1 = c0 * 0xD2511F53, c2 * 0xCD9E8D57
            c0, c1, c2, c3 = (((p1 >> 32) & M) ^ c1 ^ k0) & M, p1 & M, (((p0 >> 32) & M) ^ c3 ^ k1) & M, p0 & M
            k0, k1 = (k0 + 0x9E3779B9) & M, (k1 + 0xBB67AE85) & M
        for lo, hi in ((c0, c1), (c2, c3)):
            u = (hi << 32) | lo
            draws.append(((u >> 11) & ((1 << 53) - 1)).to(torch.float64) * 2.0 ** -53)
    d = torch.stack(draws, dim=1)
    lo = torch.tensor([-0.9438, -0.00078, -0.61679], dtype=torch.float64, device=device)
    hi = torch.tensor([0.60779, 1.53609, 0.58715], dtype=torch.float64, device=device)
    centre = torch.tensor([-0.168, 0.768, -0.015], dtype=torch.float64, device=device)
    z = 2.0 * d[:, 0] - 1.0
    phi = 2.0 * math.pi * d[:, 1]
    r = torch.sqrt(torch.clamp(1.0 - z * z, min=0.0))
    origin = centre + 3.0 * torch.stack([r * torch.cos(phi), z, r * torch.sin(phi)], dim=1)
    target = lo + d[:, 2:5] * (hi - lo)
    direction = target - origin
    direction = direction / torch.sqrt((direction * direction).sum(dim=1, keepdim=True))
    rays = torch.empty((n, 8), dtype=torch.float64, device=device)
    rays[:, 0:3], rays[:, 3:6], rays[:, 6], rays[:, 7] = origin, direction, 1e-3, float("inf")
    return rays


def _camera_rays_numpy(cam, u, v):
    """render.rs:32-52 in numpy float64 (lens 0), used only to build the shifted multi-GPU input batches"""
    tan_fov = math.tan(0.5 * cam.fov)
    tx = (2.0 * u - 1.0) * tan_fov * cam.focal_dist * cam.aspect_ratio
    ty = (2.0 * v - 1.0) * tan_fov * cam.focal_dist
    tz = np.full_like(tx, -cam.focal_dist)
    n = np.sqrt(0.0 + ((tx * tx + ty * ty) + tz * tz))
    d = np.stack([tx / n, ty / n, tz / n], axis=1)
    m = np.asarray(cam.transformation.orientation)
    wd = np.stack([(m[r, 0] * d[:, 0] + m[r, 1] * d[:, 1]) + m[r, 2] * d[:, 2] for r in range(3)], axis=1)
    rays = np.empty((len(u), 8), dtype=np.float64)
    rays[:, 0:3] = np.asarray(cam.transformation.position)
    rays[:, 3:6] = wd
    rays[:, 6], rays[:, 7] = 1e-3, np.inf
    return rays


class Ctx:
    """what every leg needs"""

    def __init__(self, args, torch, dist, api, A, scenes, rank, local_rank, world, dev):
        self.args, self.torch, self.dist, self.api, self.A, self.scenes = args, torch, dist, api, A, scenes
        self.rank, self.local_rank, self.world, self.dev = rank, local_rank, world, dev
        self.stream = torch.cuda.current_stream().cuda_stream
        self.cpu_group = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t)
        return float(t.item())

    def time_device(self, fn, steps, warmup):
        """K calls of fn on the current stream between two CUDA events, barrier + synchronize on both sides; max over ranks (ms)"""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        return self.max_over_ranks(ms), ms

    def time_host(self, fn, steps, warmup):
        """K synchronous host calls, wall clock, barrier on both sides; max over ranks (s)"""
        for _ in range(warmup):
            fn()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        self.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        self.barrier()
        return self.max_over_ranks(dt)


def link_ceiling(ctx, h2d_bytes, d2h_bytes, reps=10):
    """What plain pinned copies reach on this rank's host link while every other rank does the same: one cudaMemcpyAsync H2D of
    h2d_bytes and one D2H of d2h_bytes per step on two streams (torch.Tensor.copy_ non_blocking = one cudaMemcpyAsync each), all
    ranks at once. Returns GB/s summed over both directions and over ranks: the ceiling of any host-buffer API on this box."""
    torch = ctx.torch
    hs = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hd = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    ds = torch.empty(h2d_bytes, dtype=torch.uint8, device=ctx.dev)
    dd = torch.empty(d2h_bytes, dtype=torch.uint8, device=ctx.dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    parts = 4  # a few copies in flight per direction keep both DMA engines fed across copy boundaries
    hs_p, ds_p = hs.chunk(parts), ds.chunk(parts)
    hd_p, dd_p = hd.chunk(parts), dd.chunk(parts)

    def step():
        for k in range(len(hs_p)):
            with torch.cuda.stream(s1):
                ds_p[k].copy_(hs_p[k], non_blocking=True)
            if k < len(hd_p):
                with torch.cuda.stream(s2):
                    hd_p[k].copy_(dd_p[k], non_blocking=True)

    for _ in range(2):
        step()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    ctx.barrier()
    return reps * (h2d_bytes + d2h_bytes) * ctx.world / dt / 1e9


# ----------------------------------------------------------------------------------------------- render legs

def render_leg(ctx, scene, sc, rw, rh, spp_total, name, mode, max_steps, cpu_spp=None, roofline_inputs=None):
    """One render config. mode = "weak": every rank renders spp_total samples of every pixel of its own frame copy split by SAMPLE
    range (rank r: samples [r*spp, (r+1)*spp) of a world*spp frame) and rank 0 receives the sum (NCCL reduce to the root);
    mode = "strong": ONE frame of spp_total samples, rows dealt out round-robin over the ranks (rtp_render_params.row_offset /
    row_stride), each rank renders all samples of its rows, rank 0 gathers the rows (NCCL gather): pixels bit-identical to a
    one-GPU frame. The clock sits where the reference puts it (main.rs:45,106): around the worker phase, scene build excluded."""
    torch, dist, api, A = ctx.torch, ctx.dist, ctx.api, ctx.A
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    depth = 8
    cam = api.Camera(rw / rh, sc.camera.fov, sc.camera.focal_dist, sc.camera.lens_radius, sc.camera.transformation)
    npix = rw * rh
    if mode == "weak":
        spp_frame = spp_total * world
        p = api.render_params(rw, rh, spp_frame, depth, seed=1, sample_begin=rank * spp_total, sample_end=(rank + 1) * spp_total, flags=A.RENDER_RAW_SUMS)
        my_rows = rh
    else:
        spp_frame = spp_total
        p = api.render_params(rw, rh, spp_frame, depth, seed=1, rows=(rank, world))
        my_rows = (rh - rank + world - 1) // world if rank < rh else 0
    acc = torch.zeros((npix * 4,), dtype=torch.float64, device=dev)  # full-frame layout: rgb (3 npix) then foreground (npix)
    # strong: the rows of this rank, compacted, and the gathered rows on the root
    rows_max = (rh + world - 1) // world
    send = torch.zeros((rows_max * rw * 4,), dtype=torch.float64, device=dev)
    recv = [torch.empty_like(send) for _ in range(world)] if (rank == 0 and world > 1 and mode == "strong") else None
    frame = acc.view(-1)

    def step():
        scene.render_device(p, cam, acc.data_ptr(), acc.data_ptr() + npix * 3 * 8, ctx.stream)
        if world == 1:
            return
        if mode == "weak":
            dist.reduce(acc, dst=0, op=dist.ReduceOp.SUM)
        else:
            rgb = frame[: npix * 3].view(rh, rw, 3)[rank::world]
            fg = frame[npix * 3:].view(rh, rw)[rank::world]
            send[: my_rows * rw * 3].view(my_rows, rw, 3).copy_(rgb)
            send[rows_max * rw * 3: rows_max * rw * 3 + my_rows * rw].view(my_rows, rw).copy_(fg)
            dist.gather(send, recv, dst=0)
            if rank == 0:
                for r in range(1, world):
                    nr = (rh - r + world - 1) // world
                    frame[: npix * 3].view(rh, rw, 3)[r::world].copy_(recv[r][: nr * rw * 3].view(nr, rw, 3))
                    frame[npix * 3:].view(rh, rw)[r::world].copy_(recv[r][rows_max * rw * 3: rows_max * rw * 3 + nr * rw].view(nr, rw))

    if max_steps > 1:
        scene.render_device(p, cam, acc.data_ptr(), acc.data_ptr() + npix * 3 * 8, ctx.stream)  # first call allocates the integrator's queues
    st = scene.render_device(p, cam, acc.data_ptr(), acc.data_ptr() + npix * 3 * 8, ctx.stream, stats=True)
    rays_total = ctx.sum_over_ranks(st.rays)
    trace_ms, device_ms = float(st.trace_ms), float(st.device_ms)
    steps = max(min(ctx.args.steps, max_steps), 1 if max_steps == 1 else 2)
    ms_max, _ = ctx.time_device(step, steps, 1 if max_steps == 1 else 2)
    sec = ms_max * 1e-3 / steps
    paths = npix * spp_frame
    out = {
        "workload": f"{name}, {rw}x{rh}, {spp_frame} spp in the frame ({'%d per GPU, split by sample range' % spp_total if mode == 'weak' else 'rows dealt out over %d GPU(s)' % world}), max depth {depth}",
        "scaling": mode, "samples_per_s": paths / sec, "mrays_per_s": rays_total / sec / 1e6, "ms_per_frame": sec * 1e3, "steps": steps,
        "rays_per_path": rays_total / paths,
        "collective": "none (1 GPU)" if world == 1 else ("NCCL reduce(sum, f64) of the W x H x 4 accumulation buffer to rank 0" if mode == "weak"
                                                           else "NCCL gather of each rank's rows (W x H x 4 f64 / N per rank) to rank 0; no sum: bit-identical to a one-GPU frame"),
        "launches_per_frame": int(st.kernel_launches),
    }
    if world == 1:
        # dominant kernel of the frame: the traversal launches (trace_any_kernel<OUT_WAVE>); algorithmic bytes = 64 B ray in + 32 B hit record out
        algo = int(st.rays) * (RAY_BYTES + WAVE_HIT_BYTES)
        hbm_peak, peak_src = measured_hbm_peak()
        ach = algo / (trace_ms * 1e-3) / 1e9 if trace_ms > 0 else None
        out["roofline"] = {
            "kernel": "trace_any_kernel<OUT_WAVE> (traversal launches of the wavefront integrator, summed over the frame)", "bound": "issue",
            "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": (ach / hbm_peak) if ach else None, "traffic": (roofline_inputs or {}).get("render_trace_dram_bytes_per_frame"),
            "peak_source": peak_src, "algorithmic_bytes_per_frame": algo, "bytes_per_ray": RAY_BYTES + WAVE_HIT_BYTES,
            "trace_ms_per_frame": trace_ms, "frame_device_ms": device_ms, "trace_share_of_frame": trace_ms / device_ms if device_ms else None,
            "how": "CUDA events recorded by the library around every traversal launch of one frame (rtp_stats.trace_ms), same stream",
        }
    return out


def render_e2e(ctx, scene, sc, rw, rh, spp, steps):
    """the same frame through the reference-facing call with HOST buffers: rtp_render (frame D2H inside the timed region)"""
    api = ctx.api
    cam = api.Camera(rw / rh, sc.camera.fov, sc.camera.focal_dist, sc.camera.lens_radius, sc.camera.transformation)
    rgb = api.PinnedBuffer((rh, rw, 3), np.float64)
    fg = api.PinnedBuffer((rh, rw), np.float64)
    dt = ctx.time_host(lambda: scene.render(rw, rh, spp, 8, 1, cam, out=(rgb.array, fg.array)), steps, 1)
    sec = dt / steps
    res = {"value": rw * rh * spp * ctx.world / sec, "unit": "samples/s", "ms_per_frame": sec * 1e3, "h2d_bytes_per_step": 168 + 64,
           "d2h_bytes_per_step": rw * rh * 4 * 8, "api": "rtp_render (camera + parameters in, W x H x 4 f64 frame out to pinned host memory)", "steps": steps}
    rgb.free()
    fg.free()
    return res


def cpu_render(sc, rw, rh, spp, name):
    """oracle port of the worker phase (main.rs:46-98: 32x32 LIFO tile queue, pthreads) on all host cores"""
    import oracle

    o = oracle.Scene(sc)
    cores = os.cpu_count() or 1
    from rtp_b200 import api

    cam = api.Camera(rw / rh, sc.camera.fov, sc.camera.focal_dist, sc.camera.lens_radius, sc.camera.transformation)
    t0 = time.perf_counter()
    _, _, st = o.render(rw, rh, spp, max_bounce=8, seed=1, camera=cam, threads=cores)
    dt = time.perf_counter() - t0
    return {"value": rw * rh * spp / dt, "unit": "samples/s", "mrays_per_s": st.rays / dt / 1e6, "cores": cores, "kind": "port", "seconds": dt,
            "sample": f"{name}: {rw}x{rh} at {spp} spp (of the GPU leg's spp; rays/s and samples/s do not depend on spp), oracle/rtp_oracle.c render, {cores} pthreads"}


def measured_hbm_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_roofline_inputs():
    """ncu-derived numbers of the traversal kernel (profiles/r02_roofline_inputs.json, written from the committed ncu summaries)"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_roofline_inputs.json")))
    except Exception:
        return {}


# ----------------------------------------------------------------------------------------------- our arm

def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from rtp_b200 import _abi as A
    from rtp_b200 import api, scenes

    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    affinity, affinity_how = bind_to_gpu_local_cores(local_rank, torch) if world > 1 else (None, "single GPU: not bound")
    api.init(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    ctx = Ctx(args, torch, dist, api, A, scenes, rank, local_rank, world, dev)
    # a host-side group: ranks that only wait (multi_device_leg) must not park a spinning NCCL kernel on their GPU
    ctx.cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    sampler = ClockSampler(torch, local_rank) if rank == 0 else None
    roof_in = load_roofline_inputs()

    sc = scenes.bunny_lambert()
    scene = api.Scene(sc)
    cam = api.Camera(W / H, sc.camera.fov, sc.camera.focal_dist, 0.0, sc.camera.transformation)
    stream = ctx.stream

    # --- inputs: this rank's primary batch, generated on the device by the camera kernel (render.rs:32-52) -----------
    # two distinct ray buffers are rotated so that no step can reuse its rays from L2 (2 x 132.7 MB > 126 MB L2)
    d_rays = [torch.empty((N_RAYS, 8), dtype=torch.float64, device=dev) for _ in range(2)]
    if world == 1:
        api.camera_rays_device(cam, W, H, d_rays[0].data_ptr(), stream)
    else:
        # rank r = sub-sample r of a world-times supersampled frame: shift the pixel centres by (r+0.5)/world - 0.5
        i = np.tile(np.arange(W, dtype=np.float64), H)
        j = np.repeat(np.arange(H, dtype=np.float64), W)
        off = (rank + 0.5) / world
        d_rays[0].copy_(torch.from_numpy(_camera_rays_numpy(cam, (i + off) / W, (j + off) / H)))
    d_rays[1].copy_(d_rays[0])
    d_hits = torch.empty((N_RAYS, 2), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    # the numpy camera that makes the shifted N > 1 batches is the device camera kernel bit for bit (checked at the unshifted centre)
    inputs_ok = None
    if rank == 0:
        i = np.tile(np.arange(W, dtype=np.float64), H)
        j = np.repeat(np.arange(H, dtype=np.float64), W)
        centre = torch.empty((N_RAYS, 8), dtype=torch.float64, device=dev)
        api.camera_rays_device(cam, W, H, centre.data_ptr(), stream)
        torch.cuda.synchronize()
        inputs_ok = bool(centre.cpu().numpy().tobytes() == _camera_rays_numpy(cam, (i + 0.5) / W, (j + 0.5) / H).tobytes())
        del centre

    # --- value: device-resident batch, CUDA events on the launching stream ------------------------------------------------
    k_ = [0]

    def c2_step():
        scene.hit_device(d_rays[k_[0] & 1].data_ptr(), N_RAYS, d_hits.data_ptr(), stream)
        k_[0] += 1

    if sampler:
        sampler.active = True
    ms_max, ms_own = ctx.time_device(c2_step, args.steps, max(args.warmup, 3))
    if sampler:
        sampler.active = False
    if args.dump_outputs and rank == 0:  # before the legs below overwrite d_hits
        dump_hits(args.dump_outputs, d_hits.cpu().numpy().view(A.HIT_DTYPE).reshape(-1))
    value = args.steps * N_RAYS * world / (ms_max * 1e-3) / 1e6
    kernel_ms = ms_own / args.steps  # one traversal launch (+ one empty deferred launch) per step, back to back on one stream
    launches_per_step = 2 if scene.info().any_order else 1

    # --- e2e: host buffers through rtp_trace_closest (chunked H2D -> kernel -> D2H pipeline inside the call) -----------
    h_rays = api.PinnedBuffer((N_RAYS,), A.RAY_DTYPE)
    h_hits = api.PinnedBuffer((N_RAYS,), A.HIT_DTYPE)
    h_rays.array.view(np.float64).reshape(-1, 8)[:] = d_rays[0].cpu().numpy()
    _, st = scene.hit(h_rays.array, out=h_hits.array, stats=True)
    e2e_launches = int(st.kernel_launches)
    e2e_steps = max(3, min(args.steps, 50))
    if sampler:
        sampler.active = True
    dt = ctx.time_host(lambda: scene.hit(h_rays.array, out=h_hits.array), e2e_steps, max(args.warmup, 1))
    if sampler:
        sampler.active = False
    e2e_value = e2e_steps * N_RAYS * world / dt / 1e6
    scene.hit_device(d_rays[0].data_ptr(), N_RAYS, d_hits.data_ptr(), stream)
    torch.cuda.synchronize()
    same = bool((torch.from_numpy(h_hits.array.view(np.float64).reshape(-1, 2).copy()).to(dev).view(torch.int64) == d_hits.view(torch.int64)).all())
    ceiling = link_ceiling(ctx, N_RAYS * RAY_BYTES, N_RAYS * HIT_BYTES)
    e2e_gbs = e2e_value * 1e6 * (RAY_BYTES + HIT_BYTES) / 1e9

    # --- e2e, camera-driven: the same batch through rtp_trace_camera (H2D = the camera, rays made on the device, D2H = hits) ----
    dtc = ctx.time_host(lambda: scene.hit_camera(cam, W, H, out=h_hits.array), e2e_steps, 1)
    e2e_camera = e2e_steps * N_RAYS * world / dtc / 1e6
    same_cam = bool((torch.from_numpy(h_hits.array.view(np.float64).reshape(-1, 2).copy()).to(dev).view(torch.int64) == d_hits.view(torch.int64)).all()) if world == 1 else None
    ceiling_d2h = link_ceiling(ctx, 4096, N_RAYS * HIT_BYTES)

    # --- roofline inputs: work counters of one counted pass (outside any timed region) ---------------------------------
    cst = scene.hit_device_counted(d_rays[0].data_ptr(), N_RAYS, d_hits.data_ptr())

    incoherent = render = render_c4 = render_c4_weak = multi_abi = render_c5 = None
    if not args.no_render:
        # --- C3: 2^24 incoherent rays per rank (1.07 GB of rays, 268 MB of hits per rank) ----------------------------------
        n3 = 1 << C3_LOG2
        d3 = incoherent_rays_device(torch, n3, dev, first=rank * n3)
        h3 = torch.empty((n3, 2), dtype=torch.float64, device=dev)
        reps3 = max(3, min(args.steps, 10))
        ms3, _ = ctx.time_device(lambda: scene.hit_device(d3.data_ptr(), n3, h3.data_ptr(), stream), reps3, 2)
        c3 = scene.hit_device_counted(d3.data_ptr(), n3, h3.data_ptr())
        v3 = reps3 * n3 * world / (ms3 * 1e-3) / 1e6
        incoherent = {"workload": f"C3: 2^{C3_LOG2} incoherent rays per GPU vs bunny BVH (1.07 GB of rays per GPU > L2)", "mrays_per_s": v3, "ms_per_step": ms3 / reps3, "steps": reps3,
                      "hbm_frac_of_stream": v3 / world * 1e6 * (RAY_BYTES + HIT_BYTES) / 1e9 / measured_hbm_peak()[0],
                      "per_ray": {"node_visits": c3.node_visits / n3, "leaf_gates": c3.leaf_gates / n3, "triangle_tests": c3.triangle_tests / n3, "sphere_tests": c3.sphere_tests / n3,
                                  "deferred_to_in_order": int(c3.order_rewalks), "conservative_violations": int(c3.conservative_violations)}}
        if rank == 0 and not args.no_cpu:
            incoherent["cpu_baseline"] = cpu_trace(sc, d3[: 1 << 20].cpu().numpy(), "first 2^20 rays of the C3 batch")
        del d3, h3
        torch.cuda.empty_cache()

        # --- C1 (640x360, 16 spp, depth 8): device-resident frame, the same through rtp_render, CPU arm -----------------------
        render = render_leg(ctx, scene, sc, 640, 360, 16, "C1: bunny Lambert + sky", "weak", 20, roofline_inputs=roof_in)
        render["e2e"] = render_e2e(ctx, scene, sc, 640, 360, 16, max(3, min(args.steps, 10)))
        if rank == 0 and not args.no_cpu:
            render["cpu_baseline"] = cpu_render(sc, 640, 360, 16 if world == 1 else 4, "C1")

        # --- C4 (demo scene 1920x1080, 256 spp): strong scaling by rows, weak scaling at 32 spp per GPU, CPU arm -----------
        sc4 = scenes.demo()
        scene4 = api.Scene(sc4)
        render_c4 = render_leg(ctx, scene4, sc4, 1920, 1080, 256, "C4: demo scene (glass bunny, Lambert bunny, earthmap sphere, light, metal ground, sky)", "strong", 3, roofline_inputs=None)
        render_c4_weak = render_leg(ctx, scene4, sc4, 1920, 1080, 32, "C4 scene", "weak", 3)
        if world == 1:
            render_c4["e2e"] = render_e2e(ctx, scene4, sc4, 1920, 1080, 256, 2)
        if rank == 0 and not args.no_cpu:
            render_c4["cpu_baseline"] = cpu_render(sc4, 1920, 1080, 1, "C4")
        scene4.close()
        del scene4

        # --- one host call, N devices: rank 0 drives every GPU through rtp_scene_create_multi + rtp_render (rows over devices) ---
        if world > 1:
            multi_abi = multi_device_leg(ctx, sc4, 1920, 1080, 64)

        # --- C5: the 2,048-copy bunny field (10,174,464 triangles), 3840x2160; 1024 spp across 8 GPUs is the named config, so the
        #     frame carries 128 spp per GPU (1024 at N = 8), rows dealt out over the ranks; scene built on each rank's device ---------
        if os.environ.get("RTP_BENCH_C5", "1") != "0":
            t0 = time.perf_counter()
            sc5 = scenes.bunny_field(64, 32)
            t1 = time.perf_counter()
            scene5 = api.Scene(sc5)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            render_c5 = render_leg(ctx, scene5, sc5, 3840, 2160, 128 * world, "C5: 64x32 bunny field, 10,174,464 triangles + ground sphere" + ("" if world == 8 else f" (subset of the named config: {128 * world} of 1024 spp on {world} of 8 GPUs)"), "strong", 1)
            render_c5["scene_build_s"] = ctx.max_over_ranks(t2 - t1)
            render_c5["scene_description_s"] = t1 - t0
            render_c5["scene_build_how"] = "rtp_scene_create: validation on the host, then leaf boxes, reference order, SAH culling tree, records, 4-wide collapse and any-order tables on the device (rtp_build.cu); max over ranks"
            render_c5["device_bytes"] = int(scene5.info().device_bytes)
            if rank == 0 and not args.no_cpu:
                t0 = time.perf_counter()
                render_c5["cpu_baseline"] = cpu_render(sc5, 480, 270, 1, "C5 scene")
                render_c5["cpu_baseline"]["includes"] = "oracle Bvh::new over 10,174,465 leaves is outside the timed region, like the GPU scene build"
            scene5.close()
            del scene5, sc5

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, peak_src = measured_hbm_peak()
    algo_bytes = N_RAYS * (RAY_BYTES + HIT_BYTES)
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    clocks = sampler.report()
    sm_hz = (clocks["sm_mhz"] or 1965) * 1e6
    # f64 work of the reference algorithm per launch (SURVEY.md §8d): 24 ops per slab test, 75 per triangle test, 20 per sphere test
    f64_ops = 24 * cst.leaf_gates + 75 * cst.triangle_tests + 20 * cst.sphere_tests  # inner nodes are culled in f32
    fp64_peak, fp64_src = 148 * 64 * sm_hz, "148 SM x 64 FP64 lanes x median SM clock during the run (nominal)"
    try:
        import ctypes

        g = ctypes.c_double(0.0)
        if A.load().rtp_probe_fp64(ctypes.byref(g)) == 0 and g.value > 0:
            fp64_peak, fp64_src = g.value * 1e9, "measured: rtp_probe_fp64 (independent DMUL+DADD chains, best of 3)"
    except Exception:
        pass
    scene_bytes = 128 * cst.node_visits + 128 * (cst.triangle_tests + cst.sphere_tests)  # one 128 B DWide per node visit, one 128 B DPrim per tested leaf
    issue = roof_in.get("c2", {})
    warp_inst = issue.get("warp_instructions_per_launch")
    issue_peak = 148 * 4 * sm_hz  # one warp instruction per SM sub-partition per cycle
    line = {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": WORKLOAD,
            "rays_per_step_per_gpu": N_RAYS, "sharding": "rank r traces sub-sample r of a world-times supersampled primary batch; no data-path collective",
            "l2": "inputs larger than L2: two 132.7 MB ray buffers are rotated between steps (265 MB > 126 MB L2); no flush needed",
            "host_cores_bound_per_rank": affinity, "host_cores_bound_how": affinity_how,
            "inputs": "rays made by camera_rays_kernel (N = 1) / by its numpy restatement at shifted pixel centres (N > 1)", "numpy_camera_equals_device_kernel_bits": inputs_ok,
        },
        "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": N_RAYS * RAY_BYTES, "d2h_bytes_per_step": N_RAYS * HIT_BYTES,
                "steps": e2e_steps, "api": "rtp_trace_closest (pinned host buffers, 256Ki-ray chunks on 3 streams)", "gpu_launches_per_step": e2e_launches,
                "matches_device_result": same, "link_gbs": e2e_gbs, "link_ceiling_gbs": ceiling, "frac_of_link_ceiling": e2e_gbs / ceiling if ceiling else None,
                "link_ceiling_how": "plain pinned cudaMemcpyAsync copies, no kernel: the batch's 132.7 MB H2D and its 33.2 MB D2H per step, four copies per direction on two streams, every rank at once, wall clock, summed over ranks"},
        "e2e_camera": {"value": e2e_camera, "unit": "Mrays/s", "h2d_bytes_per_step": 168, "d2h_bytes_per_step": N_RAYS * HIT_BYTES, "steps": e2e_steps,
                       "api": "rtp_trace_camera: Camera::shoot (render.rs:32-52) on the device + closest hit; the reference never materialises a ray array, its input is the camera",
                       "matches_device_result": same_cam, "link_gbs": e2e_camera * 1e6 * HIT_BYTES / 1e9, "link_ceiling_gbs": ceiling_d2h,
                       "cpu_arm": "cpu_baseline below: the oracle's camera rays + closest hits are the same call on the CPU (camera ray generation is < 2 % of its time)"},
        "gpu_launches": args.steps * launches_per_step,
        "gpu_launches_note": "per step: one trace_any_kernel launch + one launch of the in-order kernel over the (normally empty) deferred list",
        "clocks": clocks,
        "roofline": {
            "kernel": "trace_any_kernel<COUNT=false, OUT_HIT> (pure any-order walk, DESIGN.md 4b/6)",
            "bound": "issue", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": issue.get("dram_bytes_per_launch"), "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": kernel_ms,
            "binding": {"resource": "instruction issue (scene is cache-resident; HBM carries only the 80 B/ray stream)",
                        "issue_slot_frac": (warp_inst / (kernel_ms * 1e-3) / issue_peak) if warp_inst else None,
                        "issue_slot_frac_how": "warp instructions per launch (ncu smsp__inst_executed.sum, profiles/r02_roofline_inputs.json) / live kernel time / (148 SM x 4 schedulers x SM clock)",
                        "ncu_issue_active_frac": issue.get("issue_active_frac"), "ncu_lanes_per_instruction": issue.get("lanes_per_instruction"),
                        "ncu_l1_hit_frac": issue.get("l1_hit_frac"), "ncu_warp_occupancy_frac": issue.get("warp_occupancy_frac"), "source": issue.get("source")},
            "fp64": {"ops_per_launch": f64_ops, "achieved_gops": f64_ops / (kernel_ms * 1e-3) / 1e9, "peak_gops": fp64_peak / 1e9,
                     "frac": f64_ops / (kernel_ms * 1e-3) / fp64_peak, "peak_source": fp64_src},
            "l2": {"bytes_per_launch": scene_bytes, "achieved_gbs": scene_bytes / (kernel_ms * 1e-3) / 1e9,
                   "note": "128 B culling node per node visit + 128 B primitive record per leaf test, served by L1/L2"},
            "per_ray": {"node_visits": cst.node_visits / N_RAYS, "leaf_gates": cst.leaf_gates / N_RAYS, "triangle_tests": cst.triangle_tests / N_RAYS, "sphere_tests": cst.sphere_tests / N_RAYS,
                        "deferred_to_in_order": int(cst.order_rewalks), "conservative_violations": int(cst.conservative_violations)},
        },
    }
    for key, val in (("incoherent", incoherent), ("render", render), ("render_c4", render_c4), ("render_c4_weak", render_c4_weak), ("render_c5", render_c5), ("multi_device_abi", multi_abi)):
        if val is not None:
            line[key] = val
    if not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(sc, cam)
    sys.stderr.flush()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def multi_device_leg(ctx, sc, rw, rh, spp):
    """rank 0 alone: ONE rtp_render call renders the frame on all N GPUs (rows dealt out inside the library, each device copies its
    rows straight into the pinned host frame). The other ranks wait at the barrier; their contexts stay idle."""
    api, world = ctx.api, ctx.world
    res = None
    ctx.barrier()
    ctx.torch.cuda.synchronize()
    ctx.dist.barrier(group=ctx.cpu_group)
    if ctx.rank == 0:
        try:
            cam = api.Camera(rw / rh, sc.camera.fov, sc.camera.focal_dist, sc.camera.lens_radius, sc.camera.transformation)
            multi = api.Scene(sc, device_mask=(1 << world) - 1)
            rgb = api.PinnedBuffer((rh, rw, 3), np.float64)
            out = {}
            for mask_n in (1, world):
                mask = (1 << mask_n) - 1
                multi.render(rw, rh, spp, 8, 1, cam, out=(rgb.array, None), device_mask=mask)
                t0 = time.perf_counter()
                reps = 2
                for _ in range(reps):
                    multi.render(rw, rh, spp, 8, 1, cam, out=(rgb.array, None), device_mask=mask)
                out[mask_n] = (time.perf_counter() - t0) / reps
                if mask_n == 1:
                    ref = rgb.array.copy()
            res = {"workload": f"C4 scene {rw}x{rh} at {spp} spp through ONE rtp_render call on a scene made by rtp_scene_create_multi", "api": "rtp_render, params.device_mask",
                   "ms_per_frame_1_device": out[1] * 1e3, f"ms_per_frame_{world}_devices": out[world] * 1e3, "speedup": out[1] / out[world],
                   "samples_per_s": rw * rh * spp / out[world], "bit_identical_to_1_device": bool((ref.view(np.int64) == rgb.array.view(np.int64)).all()),
                   "collective": "none: rows round-robin over devices, each device copies its rows to the host frame"}
            rgb.free()
            multi.close()
            # the C2 batch through ONE rtp_trace_closest call: its 256 Ki-ray chunks are dealt out over the devices, so every
            # device's host link carries a share of the 80 B/ray stream
            from rtp_b200 import _abi as A2

            scb = ctx.scenes.bunny_lambert()
            camb = api.Camera(W / H, scb.camera.fov, scb.camera.focal_dist, 0.0, scb.camera.transformation)
            h_rays = api.PinnedBuffer((N_RAYS,), A2.RAY_DTYPE)
            h_hits = api.PinnedBuffer((N_RAYS,), A2.HIT_DTYPE)
            h_rays.array[:] = api.camera_rays(camb, W, H)
            rates = {}
            for mask_n in (1, world):
                with api.Scene(scb, device_mask=(1 << mask_n) - 1) as sb:
                    sb.hit(h_rays.array, out=h_hits.array)
                    t0 = time.perf_counter()
                    reps = 10
                    for _ in range(reps):
                        sb.hit(h_rays.array, out=h_hits.array)
                    rates[mask_n] = reps * N_RAYS / (time.perf_counter() - t0) / 1e6
                    if mask_n == 1:
                        ref_hits = h_hits.array.copy()
            res["trace_closest_host_buffers"] = {"mrays_per_s_1_device": rates[1], f"mrays_per_s_{world}_devices": rates[world], "speedup": rates[world] / rates[1],
                                                 "bit_identical_to_1_device": bool(ref_hits.tobytes() == h_hits.array.tobytes()),
                                                 "api": "rtp_trace_closest on a multi-device scene (pinned host buffers)"}
            h_rays.free()
            h_hits.free()
        except Exception as e:  # noqa: BLE001 - the leg is reported as failed, the headline stands
            res = {"error": f"{type(e).__name__}: {e}"}
    ctx.dist.barrier(group=ctx.cpu_group)  # the waiting ranks sit in a gloo (host) barrier: their GPUs stay idle for rank 0
    return res


def cpu_trace(sc, rays_f64, what):
    """oracle port of batched Hittable::hit on all host cores over a bounded sample of a device batch"""
    import oracle
    from rtp_b200 import _abi as A

    o = oracle.Scene(sc)
    rays = np.ascontiguousarray(rays_f64).view(A.RAY_DTYPE).reshape(-1)
    cores = os.cpu_count() or 1
    o.hit_full(rays[: 1 << 16], threads=cores)
    t0 = time.perf_counter()
    o.hit_full(rays, threads=cores)
    dt = time.perf_counter() - t0
    return {"value": len(rays) / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": f"{what} ({len(rays)} rays), oracle/rtp_oracle.c with {cores} pthreads"}


def cpu_baseline(sc, cam):
    """oracle port (kind 'port': the Rust reference cannot be compiled here) on all host cores, bounded sample: 6 passes
    over the full C2 batch (~15 core-seconds)."""
    import oracle

    o = oracle.Scene(sc)
    rays = oracle.camera_rays(cam, W, H)
    cores = os.cpu_count() or 1
    o.hit_full(rays, threads=cores)
    reps = 6
    t0 = time.perf_counter()
    for _ in range(reps):
        o.hit_full(rays, threads=cores)
    dt = time.perf_counter() - t0
    out = {"value": reps * N_RAYS / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
           "sample": f"{reps} passes over the full C2 batch (2,073,600 rays each), oracle/rtp_oracle.c with {cores} pthreads, gcc -O3 -ffp-contract=off"}
    # the reference ships with 4 worker threads hard-coded (main.rs:27): the same port at 4 threads, 2 passes
    t0 = time.perf_counter()
    for _ in range(2):
        o.hit_full(rays, threads=4)
    out["as_shipped_4_threads"] = {"value": 2 * N_RAYS / (time.perf_counter() - t0) / 1e6, "unit": "Mrays/s", "cores": 4}
    return out


if __name__ == "__main__":
    main()
