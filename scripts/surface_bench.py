"""surface_bench.py — rays per second of the surface query (rtcuda_trace_surfaces_device) beside the closest-hit query
(rtcuda_trace_rays_device with t, ids and barycentrics) on the same ray sets, and k_surface_finish's share of the call.

The ray sets are those of scripts/trace_bench.py on C3 (cbbunny_area_light_transforms, 1080p) and C5 (the 16.8 M-triangle mesh in
the cb box, 4K): `primary` (pinhole rays through the pixel centres, [near, far]) and `incoherent` (uniform directions from the
primary set's closest hits, t_min offset). Every timed call carries >= 64 Mi rays (the set tiled). A call is timed with a host
clock around the blocking _device call, after torch.cuda.synchronize(); the median of --repeats calls after one warm-up call is
reported, the two queries alternating. After the timed calls of a set, torch.profiler (CUDA activities) traces one more call of
each query and its kernel times are summed by kernel name: k_surface_finish's share of the surface call's kernel time.

usage: python scripts/surface_bench.py [--workloads C3,C5] [--repeats 5] [--out profiles/r12_surfaces.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
sys.dont_write_bytecode = True

import trace_bench  # noqa: E402  (ray sets, tiling, GPU name and power limit)


def kernel_times(torch, fn):
    """{kernel name: (device ms, launches)} of one call of fn under torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                out[e.key] = (t / 1e3, e.count)
    return out


def run_workload(torch, rc, bench, name, repeats):
    scene, st = bench.load_workload(name)
    cam = scene.camera
    assert cam.kind == rc._ffi.CAMERA_PINHOLE
    gen = torch.Generator(device="cuda")
    gen.manual_seed(42)
    res = {"workload": name, "raster": [cam.raster_width, cam.raster_height], "triangles": int(scene.triangle_count()), "sets": {}}
    with rc.CudaRenderer(scene) as r:
        prim = trace_bench.primary_rays(torch, cam)
        n_set = prim.shape[0]
        t = torch.empty(n_set, device="cuda")
        ids = torch.empty((n_set, 2), device="cuda", dtype=torch.int32)
        uv = torch.empty((n_set, 2), device="cuda")
        torch.cuda.synchronize()
        r.trace_device(prim.data_ptr(), n_set, t.data_ptr(), ids.data_ptr(), uv.data_ptr())
        hit = ids[:, 0] != -1
        pts = prim[hit, 0:3] + prim[hit, 4:7] * t[hit][:, None]
        m = pts.shape[0]
        lo, hi = pts.min(dim=0).values, pts.max(dim=0).values
        eps = 1e-4 * float((hi - lo).norm())
        inc = torch.empty((m, 8), device="cuda")
        inc[:, 0:3], inc[:, 3] = pts, eps
        inc[:, 4:7] = torch.nn.functional.normalize(torch.randn((m, 3), device="cuda", generator=gen), dim=1)
        inc[:, 7] = float("inf")
        del t, ids, uv, pts
        for set_name, base in (("primary", prim), ("incoherent", inc)):
            rays = trace_bench.tile(torch, base)
            n = rays.shape[0]
            surf = torch.empty((n, 16), device="cuda")
            t = torch.empty(n, device="cuda")
            ids = torch.empty((n, 2), device="cuda", dtype=torch.int32)
            uv = torch.empty((n, 2), device="cuda")
            calls = {"surfaces": lambda: r.surfaces_device(rays.data_ptr(), n, surf.data_ptr()),
                     "trace_rays": lambda: r.trace_device(rays.data_ptr(), n, t.data_ptr(), ids.data_ptr(), uv.data_ptr())}
            for fn in calls.values():
                fn()   # warm-up
            times = {k: [] for k in calls}
            for _ in range(repeats):
                for k, fn in calls.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    times[k].append(time.perf_counter() - t0)
            s = {"set_rays": base.shape[0], "rays": n, "hit_fraction": float((surf[:, 10].view(torch.int32) != -1).float().mean())}
            for k in calls:
                med = statistics.median(times[k])
                s[k] = {"median_s": med, "times_s": times[k], "mrays_per_s": n / med / 1e6}
            # the records agree with the closest-hit query (t bits and ids)
            s["t_and_ids_match_trace_rays"] = bool(torch.equal(surf[:, 3].view(torch.int32), t.view(torch.int32)) and
                                                   torch.equal(surf[:, 10:12].view(torch.int32), ids))
            s["ratio_surfaces_over_trace_rays_time"] = s["surfaces"]["median_s"] / s["trace_rays"]["median_s"]
            # after the timing: one traced call of each query
            ks, kt = kernel_times(torch, calls["surfaces"]), kernel_times(torch, calls["trace_rays"])
            total = sum(v[0] for v in ks.values())
            fin = sum(v[0] for k, v in ks.items() if "k_surface_finish" in k)
            s["profile"] = {"surfaces_kernels_ms": {k: v[0] for k, v in ks.items()}, "trace_rays_kernels_ms": {k: v[0] for k, v in kt.items()},
                            "surfaces_kernel_ms_total": total, "k_surface_finish_ms": fin, "k_surface_finish_share": fin / total if total else None}
            res["sets"][set_name] = s
            del surf, t, ids, uv, rays
            torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C3,C5")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(HERE), "profiles", "r12_surfaces.json"))
    args = ap.parse_args()
    import torch
    import raytracing_cuda as rc
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("surface_bench.py needs a CUDA device")
    result = {"gpu": trace_bench.gpu_info(), "min_rays_per_call": trace_bench.MIN_RAYS, "repeats": args.repeats,
              "timing": "host clock around the blocking _device call after torch.cuda.synchronize(); median after one warm-up "
                        "call; the two queries alternate; trace_rays writes t, ids and barycentrics",
              "profile": "torch.profiler (CUDA activities), one call per query and set, traced after that set's timed calls",
              "workloads": []}
    names = args.workloads.split(",")
    for name in names:
        w = run_workload(torch, rc, bench, name, args.repeats)
        result["workloads"].append(w)
        for set_name, s in w["sets"].items():
            print(f"{name} {set_name:10s} surfaces {s['surfaces']['mrays_per_s']:9.1f} Mrays/s | trace_rays "
                  f"{s['trace_rays']['mrays_per_s']:9.1f} Mrays/s ({s['rays']} rays, hit {s['hit_fraction']:.3f}, "
                  f"t/ids match {s['t_and_ids_match_trace_rays']}) | k_surface_finish {s['profile']['k_surface_finish_ms']:.2f} ms of "
                  f"{s['profile']['surfaces_kernel_ms_total']:.2f} ms kernel time")
    print(f"{result['gpu']['name']}, power limit {result['gpu']['power_limit']}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
