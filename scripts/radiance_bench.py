"""radiance_bench.py — samples per second of rtcuda_radiance_device on fixed ray sets, beside the renderer's own rate on the same
scene and settings.

On C3 (cbbunny_area_light_transforms, 1080p, 256 spp, depth 8, 4 light samples) and C5 (the 16.8 M-triangle mesh in the cb box, 4K,
256 spp, depth 8, 1 light sample), at the bench settings of bench.py, two ray sets are built on the device with torch:
  camera  pinhole rays through the pixel centres of the bench raster, [near, far]: the frame's paths without the per-sample primary
          walk (the radiance call traces each ray's first segment once, then spp paths from its hit);
  probes  from the closest hits of the camera set (t_min offset), cosine-distributed about the reversed camera ray, at 64 spp.
Rates are samples over the LIVE rays (rays whose first segment hits something; neither scene has an environment light) per second
of the call. A call is timed with a host clock around the blocking _device call after torch.cuda.synchronize(); the median of
--repeats calls after one warm-up call is reported. The renderer's rate is msamples_reaching_the_scene_per_s of bench.py, from one
render with RTCUDA_STATS_KERNEL_TIMES in the same run: (samples - culled primary rays) / render_ms. The share of a call spent in
k_radiance_prep / k_trace / k_radiance_live / the wavefront (k_raygen_rays, extend, shade, shadow, gather, resolve, finalize) comes
from torch.profiler over one more call, run after the timed ones.

usage: python scripts/radiance_bench.py [--workloads C3,C5] [--repeats 5] [--out profiles/r11_radiance.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.dont_write_bytecode = True

from trace_bench import gpu_info, primary_rays  # noqa: E402

PROBE_SPP = 64


def time_call(torch, fn, repeats):
    fn()   # warm-up
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), times


def kernel_shares(torch, fn):
    """device time per stage of one call (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    stages = {"prep": 0.0, "k_trace": 0.0, "live_list": 0.0, "wavefront": 0.0}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        if not us or "memset" in e.key.lower() or "memcpy" in e.key.lower():
            continue
        k = "prep" if "k_radiance_prep" in e.key else "k_trace" if "k_trace" in e.key else "live_list" if "k_radiance_live" in e.key else "wavefront"
        stages[k] += us / 1e3
    total = sum(stages.values())
    return {"device_ms": stages, "share": {k: v / total for k, v in stages.items()} if total else {}}


def run_workload(torch, rc, bench, name, repeats):
    scene, st = bench.load_workload(name)
    cam = scene.camera
    assert cam.kind == rc._ffi.CAMERA_PINHOLE
    gen = torch.Generator(device="cuda")
    gen.manual_seed(42)
    res = {"workload": name, "raster": [cam.raster_width, cam.raster_height], "triangles": int(scene.triangle_count()),
           "settings": {"spp": st.samples_per_pixel, "depth": st.max_ray_depth, "light_samples": st.light_sample_count}, "sets": {}}
    with rc.CudaRenderer(scene, rc.CudaBackendSettings(collect_stats=rc._ffi.STATS_KERNEL_TIMES)) as r:
        r.render(st)
        s = r.stats()
        reaching = s["samples"] - s["primary_rays_culled"]
        res["render"] = {"samples": s["samples"], "samples_reaching_the_scene": reaching, "render_ms": s["render_ms"],
                         "msamples_reaching_the_scene_per_s": reaching / s["render_ms"] / 1e3,
                         "extend_ms": s["extend_ms"], "shade_ms": s["shade_ms"], "shadow_ms": s["shadow_ms"], "gather_ms": s["gather_ms"]}

        def measure(rays, settings):
            n = rays.shape[0]
            t = torch.empty(n, device="cuda")
            ids = torch.empty((n, 2), device="cuda", dtype=torch.int32)
            torch.cuda.synchronize()
            r.trace_device(rays.data_ptr(), n, t.data_ptr(), ids.data_ptr(), None)
            live = int((ids[:, 0] != -1).sum())
            out = torch.empty((n, 3), device="cuda")
            fn = lambda: r.radiance_device(rays.data_ptr(), n, settings, out.data_ptr())
            med, times = time_call(torch, fn, repeats)
            spp = settings.samples_per_pixel
            rec = {"rays": n, "live_rays": live, "spp": spp, "median_s": med, "times_s": times,
                   "msamples_per_s_over_live_rays": live * spp / med / 1e6, "mean_radiance": float(out.mean())}
            rec.update(kernel_shares(torch, fn))
            return rec, t, ids

        cam_rays = primary_rays(torch, cam)
        rec, t, ids = measure(cam_rays, st)
        res["sets"]["camera"] = rec
        hit = ids[:, 0] != -1
        back = -cam_rays[hit, 4:7]
        pts = cam_rays[hit, 0:3] + cam_rays[hit, 4:7] * t[hit][:, None]
        eps = 1e-4 * float((pts.max(dim=0).values - pts.min(dim=0).values).norm())
        # cosine-distributed directions about `back`: a unit vector on the sphere added to the axis, normalised
        u = torch.nn.functional.normalize(torch.randn(back.shape, device="cuda", generator=gen), dim=1)
        d = torch.nn.functional.normalize(back + u, dim=1)
        probes = torch.empty((pts.shape[0], 8), device="cuda")
        probes[:, 0:3], probes[:, 3], probes[:, 4:7], probes[:, 7] = pts, eps, d, float("inf")
        st_probe = rc.RaytracerSettings(samples_per_pixel=PROBE_SPP, max_ray_depth=st.max_ray_depth, light_sample_count=st.light_sample_count)
        res["sets"]["probes"] = measure(probes.contiguous(), st_probe)[0]
        res["sets"]["probes"]["t_min"] = eps
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C3,C5")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_radiance.json"))
    args = ap.parse_args()
    import torch
    import raytracing_cuda as rc
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("radiance_bench.py needs a CUDA device")
    result = {"gpu": gpu_info(), "repeats": args.repeats,
              "timing": "host clock around the blocking _device call after torch.cuda.synchronize(); median after one warm-up call",
              "workloads": []}
    for name in args.workloads.split(","):
        w = run_workload(torch, rc, bench, name, args.repeats)
        result["workloads"].append(w)
        for set_name, s in w["sets"].items():
            print(f"{name} {set_name:7s} {s['msamples_per_s_over_live_rays']:9.1f} Msamples/s over {s['live_rays']} live rays x {s['spp']} spp "
                  f"(median {1e3 * s['median_s']:.1f} ms; shares {({k: round(v, 3) for k, v in s['share'].items()})}) | render "
                  f"{w['render']['msamples_reaching_the_scene_per_s']:.1f} Msamples/s reaching the scene")
    print(f"{result['gpu']['name']}, power limit {result['gpu']['power_limit']}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
