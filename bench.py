#!/usr/bin/env python
"""bench.py — Msamples/s (and Mrays/s) of the render hot path on BASELINE config C3
(cbbunny_area_light_transforms.glb, 1920x1080, 256 spp, depth 8, light samples 4), N GPUs of one node.

  python bench.py --gpus N --steps K --warmup W            # this backend (libraytracing_cuda.so)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host cores
  python bench.py --dump-outputs DIR                       # + the planes of the last timed step as DIR/<plane>.npy

A step = one full render of the frame (one pass of the hot path over one batch of synthetic-free, fixed
input: the scene fixture committed under tests/golden/scenes). See DESIGN.md "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

WORKLOADS = {
    # name: (fixture, width, height, spp, depth, light samples)
    "C3": ("cbbunny_area_light_transforms", 1920, 1080, 256, 8, 4),
    "C2": ("cb", 512, 512, 64, 8, 1),
    "C4": ("cb_texture", 1920, 1080, 128, 8, 4),
    "C3s": ("cbbunny_area_light", 1920, 1080, 256, 8, 4),
    # BASELINE config C5: 16,777,216-triangle displaced UV-sphere (4096 x 2048 quads, seed 42) inside the cb.glb box, 4K
    "C5": ("cb", 3840, 2160, 256, 8, 1),
    "C5s": ("cb", 1920, 1080, 32, 8, 1),     # same mesh, 1080p / 32 spp (quick check of the HBM-bound regime)
    # the general shade kernel (k_shade<Surface>: every non-Diffuse material): the reference's builtin Cornell box with a
    # rough-conductor / rough-dielectric sphere (test_scenes/mod.rs), 1000x1000, 64 spp, point light
    "CM": ("builtin:rough_metal", 1000, 1000, 64, 8, 4),
    "CD": ("builtin:rough_dielectric", 1000, 1000, 64, 8, 4),
}
SYNTHETIC = {"C5": (4096, 2048), "C5s": (4096, 2048)}
# Tile edge of the multi-GPU deal: BASELINE names 64x64 tiles for C5; the other frames concentrate their cost in part of the
# raster (C3: the box covers a quarter of it), where 16x16 tiles balance the ranks to < 1 %.
TILE_SIZE = {"C5": 64, "C5s": 64}
CPU_SPP = {"C3": 16, "C3s": 16, "C2": 64}   # bounded CPU sample: ~10-30 s of host work on a 16-thread box


DATA_NOTE = "scene fixture (reference asset; C5: procedural mesh generated in-process, seed 42)"


def load_workload(name, synthetic_tris=0):
    import raytracing_cuda as rc
    fixture, w, h, spp, depth, ls = WORKLOADS[name]
    if fixture.startswith("builtin:"):
        import math
        import numpy as np
        t = [t for t in rc.test_scenes.all_test_scenes() if t.name == fixture.split(":")[1]][0]
        sc = t.scene_func()
        sc.camera = rc.Camera.lookat_camera_perspective((0.0, 1.0 + 3.4, 0.4), (0, 0, 0.75), (0, 0, 1), False,
                                                        float(np.float32(37.8) * np.float32(math.pi / 180)), w, h)   # cornell_box()'s camera
        st = rc.RaytracerSettings(samples_per_pixel=spp, max_ray_depth=depth, light_sample_count=ls)
        return sc, st
    sc = rc.Scene.load_npz(os.path.join(ROOT, "tests", "golden", "scenes", fixture + ".npz"))
    if name in SYNTHETIC:
        sc = rc.test_scenes.synthetic_mesh_scene(sc, *SYNTHETIC[name])
    sc.camera = sc.camera.with_raster_size(w, h)
    st = rc.RaytracerSettings(samples_per_pixel=spp, max_ray_depth=depth, light_sample_count=ls)
    if name == "C4":   # BASELINE config C4: "with normal,uv AOVs (texture fetch + AOV path)"
        st.outputs = rc.AovFlags.BEAUTY | rc.AovFlags.NORMALS | rc.AovFlags.UV_COORDS
    return sc, st


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (B200_PROFILING.md recipe). Sampled through NVML in-process
    (nvidia_ml_py): forking `nvidia-smi` every 200 ms takes the driver lock for tens of ms and stalled kernel launches of the
    process being measured (gaps of 5-10 % of a step with the subprocess sampler, A/B logs under profiles/); the
    `nvidia-smi` query stays as the fallback when NVML cannot be loaded."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.source = index, [], False, "nvidia-smi"
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: match the CUDA device by its PCI bus id
            import torch
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.handle = h
                        break
            self.nvml, self.source = pynvml, "nvml"
        except Exception:
            self.nvml = None

    def sample(self):
        if self.nvml is not None:
            n = self.nvml
            sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            bits = [n.nvmlClocksEventReasonHwSlowdown, n.nvmlClocksEventReasonHwThermalSlowdown,
                    n.nvmlClocksEventReasonSwThermalSlowdown, n.nvmlClocksEventReasonSwPowerCap]
            return [str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits]
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        return [c.strip() for c in out.splitlines()[0].split(",")] if out else None

    def run(self):
        while not self.stop_flag:
            try:
                row = self.sample()
                if row:
                    self.rows.append(row)
            except Exception:
                pass
            time.sleep(0.05 if self.nvml is not None else 0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "source": self.source}


DUMP_BYTES = 64_000_000
DUMP_SAMPLE_PIXELS = 1 << 20   # x at most 13 float32 channels, + their float64 indices: 63 MB


def dump_outputs(path, planes):
    """--dump-outputs: the planes the timed path handed back in its last step (rank 0 after the combine: the full frame) as
    <path>/<plane>.npy, float32 [H, W, C]. When the frame's planes come to more than DUMP_BYTES together, every plane is written
    at the same fixed, seeded sample of DUMP_SAMPLE_PIXELS pixels instead ([N, C], in raster order), and pixel_index.npy
    (float64, exact) holds their flat y * W + x indices. One-channel planes (mip_level, debug_depth) keep their channel axis,
    [H, W, 1], where a RenderOutput holds them as [H, W]."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {name: t.cpu().numpy() for name, t in planes.items()}
    h, w = next(iter(arrays.values())).shape[:2]
    if sum(a.nbytes for a in arrays.values()) > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(42).choice(h * w, size=DUMP_SAMPLE_PIXELS, replace=False))
        arrays = {name: a.reshape(h * w, -1)[idx] for name, a in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return json.load(open(path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_cpu_reference(scene, settings, spp_sample, threads, steps, warmup):
    """The reference algorithm (oracle restatement: scalar BVH2 + Moller-Trumbore + identical shading, 64x64
    tile queue over std::thread) on the host cores, on a bounded sample of the workload: the full raster at
    `spp_sample` samples per pixel."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    import copy
    oracle_py.use_native_build()   # -O3 -march=native, compiled on THIS host (BASELINE.md: the CPU arm is built for the box it runs on)
    st = copy.copy(settings)
    st.samples_per_pixel = spp_sample
    times, rays = [], 0
    for i in range(warmup + steps):
        _, stats = oracle_py.render(scene, st, num_threads=threads)
        if i >= warmup:
            times.append(stats["render_ms"] / 1e3)
            rays = stats["primary_rays"] + stats["bounce_rays"] + stats["shadow_rays"]
    n = scene.camera.raster_width * scene.camera.raster_height * spp_sample
    t = sum(times) / len(times)
    return n / t / 1e6, rays / t / 1e6, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-spp", type=int, default=0, help="spp of the bounded CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tile-size", type=int, default=0, help="tile edge of the multi-GPU deal (0 = per workload: 64 for C5, else 16)")
    ap.add_argument("--partition", default="tiles", choices=["tiles", "samples"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the planes of the last timed step to DIR/<plane>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    fixture, W, H, spp, depth, ls = WORKLOADS[args.workload]
    what = (f"{fixture}.glb" if not fixture.startswith("builtin:") else f"builtin scene '{fixture.split(':')[1]}'") + (f" + synthetic displaced UV-sphere {SYNTHETIC[args.workload][0]}x{SYNTHETIC[args.workload][1]} quads (seed 42)"
                               if args.workload in SYNTHETIC else "")
    tile = args.tile_size or TILE_SIZE.get(args.workload, 16)
    part = (f"{tile}x{tile} tiles round-robin" if args.partition == "tiles" else "sample ranges of every pixel")
    config = {"workload": f"{args.workload}: {what} {W}x{H}, {spp} spp, depth {depth}, light samples {ls}, "
                          f"independent sampler, seed 42" + (", beauty + normal + uv planes" if args.workload == "C4" else ""),
              "triangles": None, "partition": f"{part} over {world} GPU(s), scene replicated, 1 NCCL collective per frame (tiles: gather of the owned pixels to rank 0; samples: sum-reduce)",
              "l2": "every step re-streams ~17 GB of wavefront state per batch through L2 (>> 126 MB) and a 512 MiB buffer is "
                    "written between timed steps; the 3 MB BVH is L2-resident by design"}

    if args.impl == "reference":
        if rank != 0:
            return
        sc, st = load_workload(args.workload)
        threads = os.cpu_count() or 1
        cpu_spp = args.cpu_spp or CPU_SPP.get(args.workload, 4)
        ms, mr, t = run_cpu_reference(sc, st, cpu_spp, threads, args.steps, args.warmup)
        config["triangles"] = sc.triangle_count()
        config["partition"] = f"64x64 tiles popped from a queue by {threads} host threads (lib.rs:481-504, 706-805)"
        config["l2"] = "n/a (host cores)"
        line = {"impl": "reference", "metric": "Msamples/s", "value": ms, "unit": "Msamples/s", "mrays_per_s": mr, "n_gpus": 0,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": DATA_NOTE,
                "config": config,
                "cpu_baseline": {"value": ms, "unit": "Msamples/s", "cores": threads, "kind": "port",
                                 "sample": f"full {W}x{H} raster at {cpu_spp} spp (of {spp}), depth {depth}, light samples {ls}"},
                "e2e": {"value": ms, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import numpy as np
    import torch
    import raytracing_cuda as rc
    from raytracing_cuda import _ffi
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sc, st = load_workload(args.workload)
    config["triangles"] = sc.triangle_count()
    dr = rc.multi_gpu.DistributedRenderer(sc, rank, world, device_id=local_rank, partition=args.partition, tile_size=tile,
                                          collect_stats=_ffi.STATS_KERNEL_TIMES)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def one_step():
        """render this rank's tiles into HBM planes + (N > 1) one NCCL collective to rank 0 (DistributedRenderer.combine). Device ms of the step = the
        library's CUDA events around the whole render on its launching stream (rtcuda_stats.render_ms: every kernel of
        every batch plus the launch gaps between them) + (N > 1) torch CUDA events around the reduce, taken after a
        barrier so that the wait for a slower rank is not counted twice (the job time is the max over ranks anyway)."""
        flush.zero_()
        torch.cuda.synchronize()
        planes = dr.render_local(st)
        stats = dr.renderer.stats()
        ms = stats["render_ms"]
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dr.combine(planes)   # tiles: gather of the owned pixels to rank 0; samples: sum-reduce
            e1.record()
            torch.cuda.synchronize()
            red = e0.elapsed_time(e1)
            ms += red
            stats = dict(stats, reduce_ms=red)
        return ms, stats, planes

    for _ in range(args.warmup):
        one_step()
    clocks = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("BENCH_NO_CLOCKS"):   # (diagnostic switch: A/B of the sampler's own footprint)
        clocks.start()
    sync_all()
    total_ms, agg = 0.0, {}
    wall0 = time.time()
    for _ in range(args.steps):
        ms, stats, planes = one_step()
        total_ms += ms
        for k in ("samples", "primary_rays", "bounce_rays", "shadow_rays", "primary_rays_culled", "kernel_launches", "extend_launches", "shade_launches",
                  "shadow_launches", "extend_ms", "shade_ms", "shadow_ms", "gather_ms", "other_ms", "render_ms", "reduce_ms"):
            agg[k] = agg.get(k, 0) + stats.get(k, 0.0)
    sync_all()
    wall = time.time() - wall0
    clocks.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, planes)
    t = torch.tensor([total_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
    cnt = torch.tensor([agg["samples"], agg["primary_rays"] + agg["bounce_rays"] + agg["shadow_rays"], agg["kernel_launches"], agg["primary_rays_culled"]],
                       dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    per_rank = None
    if world > 1:   # every rank's own device time per step (balance of the deal), gathered for the report
        mine = torch.tensor([agg["render_ms"] / args.steps], dtype=torch.float64, device=f"cuda:{local_rank}")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [round(float(x.item()), 3) for x in allr]
    job_s = float(t.item()) / 1e3
    samples, rays, launches, culled = (float(x) for x in cnt.tolist())

    # ---- end to end through the public API with HOST buffers: rc.render(scene, settings) per step =
    # context + scene upload (H2D) + device BVH build + render + D2H of the frame (raytracing_cpu::render also
    # builds its acceleration structures inside every call, lib.rs:655)
    e2e_steps = args.steps
    holder = sc.to_desc(own_arrays=True)
    h2d = int(holder.geometry_bytes + holder.image_bytes.nbytes)
    e2e_each = []
    if world == 1:
        def e2e_call(record):
            t_call = time.time()
            with rc.CudaRenderer(sc, rc.multi_gpu.backend_settings_for_rank(rank, world, local_rank)) as r:
                t_up = time.time()
                out = r.render(st)
                t_rn = time.time()
                if record:
                    e2e_each.append({"upload_build_ms": 1e3 * (t_up - t_call), "render_d2h_ms": 1e3 * (t_rn - t_up), "device_render_ms": r.stats()["render_ms"],
                                     "bvh_build_device_ms": r.stats()["bvh_build_ms"], "setup_ms": r.setup_ms})
            return out
        e2e_what = "raytracing_cuda.render(scene, settings): rtcuda_init + scene_upload (H2D, device BVH build) + render + D2H frame"
    else:
        # N GPUs through the public API = ONE call from ONE process: rc.render(scene, settings, CudaBackendSettings(num_devices=N)).
        # The library replicates the scene (geometry sliced over the GPUs' PCIe links, forwarded over NVLink), builds the BVH on
        # every GPU, deals the tiles, and every GPU copies its owned pixels into the caller's host frame. Rank 0 makes the call;
        # the other torchrun ranks wait at the barrier (their GPUs are driven by rank 0's process during this leg).
        multi_bs = rc.CudaBackendSettings(num_devices=world, device_ids=list(range(world)), tile_size=tile)

        def e2e_call(record):
            if rank != 0:
                return None
            t_call = time.time()
            out = rc.render(sc, st, multi_bs)
            if record:
                e2e_each.append({"call_ms": 1e3 * (time.time() - t_call)})
            return out
        e2e_what = (f"raytracing_cuda.render(scene, settings, CudaBackendSettings(num_devices={world})) from one process (rank 0): rtcuda_init on {world} GPUs + "
                    "scene_upload (H2D slices + NVLink forward, device BVH build per GPU) + render of the tile deal + D2H of the owned pixels into the host frame")
    sync_all()
    if world > 1 and rank != 0:
        # wait on the rendezvous store (host side): an NCCL barrier would park a spinning kernel on this rank's GPU while rank 0's
        # process renders on it
        dist.distributed_c10d._get_default_store().wait(["bench_e2e_done"])
        e2e_s = 0.0
    else:
        if args.warmup:
            e2e_call(False)   # one untimed call: the first allocation of a second set of path-state buffers pays the driver's page mapping
        torch.cuda.synchronize()
        e0 = time.time()
        for _ in range(e2e_steps):
            e2e_call(True)
        e2e_s = (time.time() - e0)
        if world > 1:
            rc._ffi.load_library().rtcuda_release_cached_memory()   # rank 0's arenas on the other ranks' GPUs
            dist.distributed_c10d._get_default_store().set("bench_e2e_done", "1")
    sync_all()
    d2h = int(W * H * 4 * sum(ch for _n, flag, ch, _dt in rc.RenderOutput._PLANES if rc.AovFlags(st.outputs) & flag))

    if rank != 0:
        dr.close()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the three hot kernels, the dominant one first (DESIGN.md "Kernels" / SURVEY 8d):
    #   traversal kernels  bytes = rays * (80 * nodes/ray + 48 * prims/ray + 64)   (N from one instrumented, untimed render)
    #   shade              bytes = vertices * 160 + 32 * shadow rays emitted (+ texel bytes, not counted)
    # duration = CUDA events around every launch of the class inside the timed region (rtcuda_stats, the library's own stream).
    # `bound`: for the L2-resident scenes (C1-C4: BVH <= 3 MB) the traversal kernels are limited by instruction issue, not by HBM
    # — the algorithmic GB/s below are served by L1 / L2; the ncu counters of the same build (profiles/, per-launch durations
    # within 5 % of the CUDA-event ones) say how busy the issue slots are and how many of 32 lanes an instruction carries.
    with rc.CudaRenderer(sc, rc.multi_gpu.backend_settings_for_rank(rank, world, local_rank, collect_stats=_ffi.STATS_COUNTERS, tile_size=tile)) as rs:
        rs.render_device(st, {"beauty": dr.planes_for(rc.AovFlags.BEAUTY)["beauty"].data_ptr()})
        cs = rs.stats()
    peak, peak_src = peaks()
    ncu = {}
    npath = os.path.join(ROOT, "profiles", "ncu_counters.json")   # written by scripts/ncu_counters.py from an `ncu --set full` capture of this build
    if os.path.exists(npath):
        ncu = json.load(open(npath)).get(args.workload, {}) if world == 1 else {}
    ext_rays = cs["primary_rays"] - cs["primary_rays_culled"] + cs["bounce_rays"]   # rays k_extend walked (culled camera rays never reach it)
    sh_rays = cs["shadow_rays"]
    steps = args.steps

    def kernel_block(name, what, nbytes, items, item_name, ms_total, launches, extra):
        sec = ms_total / 1e3 / steps
        ach = nbytes / sec / 1e9 if sec > 0 else None
        c = ncu.get(name, {})
        blk = {"kernel": what, "bound": c.get("bound", "hbm"), "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if ach else None,
               "traffic": c.get("dram_bytes_per_launch"), "peak_source": peak_src,
               "algorithmic_bytes_per_" + item_name: nbytes / max(1, items), item_name + "s_per_step": items,
               "launches_per_step": launches / steps, "ms_per_step": 1e3 * sec, "ms_per_launch": 1e3 * sec / max(1.0, launches / steps),
               "share_of_step": ms_total / max(1e-9, agg["render_ms"])}
        for k in ("issue_active_pct", "lanes_per_inst", "dram_pct_of_peak", "l2_hit_pct", "ncu_ms_per_launch", "ncu_source"):
            if k in c:
                blk[k] = c[k]
        if blk["traffic"] and sec > 0 and launches:
            blk["dram_gbs"] = blk["traffic"] * (launches / steps) / sec / 1e9
            blk["dram_frac"] = blk["dram_gbs"] / peak
        blk.update(extra)
        return blk

    k_shadow = kernel_block("k_shadow", "k_shadow (any-hit BVH8 traversal of the shadow-ray queue)",
                            80 * cs["shadow_nodes"] + 48 * cs["shadow_prims"] + 64 * sh_rays, sh_rays, "ray", agg["shadow_ms"], agg["shadow_launches"],
                            {"nodes_per_ray": cs["shadow_nodes"] / max(1, sh_rays), "prims_per_ray": cs["shadow_prims"] / max(1, sh_rays)})
    k_shade = kernel_block("k_shade", "k_shade (material + next-event estimation + BSDF sampling)",
                           160 * cs["shaded_vertices"] + 32 * sh_rays, cs["shaded_vertices"], "vertex", agg["shade_ms"], agg["shade_launches"],
                           {"shadow_rays_per_vertex": sh_rays / max(1, cs["shaded_vertices"])})
    k_extend = kernel_block("k_extend", "k_extend (closest-hit BVH8 traversal)",
                            80 * cs["extend_nodes"] + 48 * cs["extend_prims"] + 64 * ext_rays, ext_rays, "ray", agg["extend_ms"], agg["extend_launches"],
                            {"nodes_per_ray": cs["extend_nodes"] / max(1, ext_rays), "prims_per_ray": cs["extend_prims"] / max(1, ext_rays),
                             "primary_rays_culled_per_step": cs["primary_rays_culled"]})
    blocks = sorted([k_shadow, k_shade, k_extend], key=lambda b: -b["ms_per_step"])
    roofline = dict(blocks[0])
    roofline["other_kernels"] = blocks[1:]
    timed = {k: agg[k] for k in ("extend_ms", "shade_ms", "shadow_ms", "gather_ms", "other_ms")}
    roofline["kernel_share_of_step"] = {k: v / agg["render_ms"] for k, v in timed.items()}
    roofline["kernel_share_of_step"]["untimed_ms(resolve, finalize, memsets, gaps)"] = 1.0 - sum(timed.values()) / agg["render_ms"]
    # whole-step cross-check: every algorithmic byte of the step over the step's time stays below the measured HBM peak only if ... it need not:
    # the BVH bytes come from L1 / L2. Reported so that the reader can see by how much.
    roofline["whole_step_algorithmic_gbs"] = sum(b["achieved"] * b["ms_per_step"] for b in blocks if b["achieved"]) / (1e3 * job_s / steps)

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        threads = os.cpu_count() or 1
        cpu_spp = args.cpu_spp or CPU_SPP.get(args.workload, 4)
        ms, mr, tcpu = run_cpu_reference(sc, st, cpu_spp, threads, 1, 0)
        cpu = {"value": ms, "unit": "Msamples/s", "mrays_per_s": mr, "cores": threads, "kind": "port", "seconds": tcpu,
               "sample": f"full {W}x{H} raster at {cpu_spp} spp (of {spp}), depth {depth}, light samples {ls}"}

    # rays: every sample is one primary ray; `culled` of them end at the scene-bounds test in ray generation (or before: pixels
    # outside the scene's raster rectangle) and are never traversed — mrays_traced_per_s leaves them out.
    line = {"metric": "Msamples/s", "value": samples / job_s / 1e6, "unit": "Msamples/s", "mrays_per_s": rays / job_s / 1e6,
            "mrays_traced_per_s": (rays - culled) / job_s / 1e6,
            "msamples_reaching_the_scene_per_s": (samples - culled) / job_s / 1e6,
            "north_star_unit_note": "target '>= 2 Gsamples-rays/s': value is SAMPLES/s (camera samples, 74 % of C3's end at the scene-bounds test); "
                                    "mrays_traced_per_s counts primary + bounce + shadow rays actually walked through the BVH",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * job_s / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": DATA_NOTE, "config": config,
            "wall_s_timed_region": wall, "clocks": clocks.summary(),
            "rank0_ms_per_step": {"render": agg["render_ms"] / args.steps, "collective": agg["reduce_ms"] / args.steps},
            "render_ms_per_rank": per_rank,
            "e2e": {"value": (W * H * spp * e2e_steps) / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "breakdown": e2e_each,
                    "what": e2e_what},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}
    print(json.dumps(line))
    dr.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
