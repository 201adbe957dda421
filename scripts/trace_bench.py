"""trace_bench.py — rays per second of the ray-query kernels (rtcuda_trace_rays_device / rtcuda_occluded_device) on fixed ray
sets, beside the renderer's own extend / shadow rates on the same scene.

On C3 (cbbunny_area_light_transforms, 1080p) and C5 (the 16.8 M-triangle mesh in the cb box, 4K), three seeded ray sets are
built on the device with torch:
  primary     pinhole rays through the pixel centres, from the camera matrices, [near, far];
  incoherent  from the closest hits of the primary set, uniform directions on the sphere, t_min offset; closest hit and occlusion;
  shadow      from those hit points to uniform points on the area light's triangles, t_max just below 1; occlusion only.
Every timed call carries >= 64 Mi rays (the set tiled). A call is timed with a host clock around the blocking _device call,
after torch.cuda.synchronize(); the median of --repeats calls after one warm-up call is reported. The renderer's rates come from
one render with RTCUDA_STATS_KERNEL_TIMES: (primary - culled + bounce rays) / extend_ms and shadow rays / shadow_ms.

usage: python scripts/trace_bench.py [--workloads C3,C5] [--repeats 5] [--out profiles/r10_trace_rays.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

MIN_RAYS = 64 << 20


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in out.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def primary_rays(torch, cam):
    """camera_ray (rt_integrator.h) for a pinhole camera at the pixel centres, in float32: [W*H, 8]"""
    W, H = cam.raster_width, cam.raster_height
    dev = "cuda"
    r2c = torch.tensor(cam.raster_to_camera.forward, device=dev)
    c2w = torch.tensor(cam.camera_to_world.forward, device=dev)
    ys, xs = torch.meshgrid(torch.arange(H, device=dev, dtype=torch.float32) + 0.5, torch.arange(W, device=dev, dtype=torch.float32) + 0.5,
                            indexing="ij")
    raster = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.zeros(W * H, device=dev), torch.ones(W * H, device=dev)], dim=1)
    cp = raster @ r2c.T
    cp = cp[:, :3] / cp[:, 3:]
    d = torch.nn.functional.normalize(torch.nn.functional.normalize(cp, dim=1) @ c2w[:3, :3].T, dim=1)
    o = (c2w[:3, 3] / c2w[3, 3]).expand_as(d)
    rays = torch.empty((W * H, 8), device=dev)
    rays[:, 0:3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o, cam.near_clip, d, cam.far_clip
    return rays


def light_points(torch, scene, n, gen):
    """uniform points on the triangles of the scene's first area light (area-weighted), world space"""
    light = [l for l in scene.lights if l.kind == 2][0]
    inst = [tf for s, tf in scene.instances if s == light.shape][0]
    mesh = scene.shapes[light.shape].shape
    v = torch.tensor(mesh.vertices, device="cuda", dtype=torch.float32)
    m = torch.tensor(inst.forward, device="cuda")
    v = v @ m[:3, :3].T + m[:3, 3]
    tri = torch.tensor(mesh.tris.astype("int64"), device="cuda")
    p0, p1, p2 = v[tri[:, 0]], v[tri[:, 1]], v[tri[:, 2]]
    area = torch.linalg.cross(p1 - p0, p2 - p0).norm(dim=1)
    k = torch.multinomial(area, n, replacement=True, generator=gen)
    u, w = torch.rand(n, device="cuda", generator=gen), torch.rand(n, device="cuda", generator=gen)
    s = u.sqrt()
    return p0[k] * (1 - s)[:, None] + p1[k] * (s * (1 - w))[:, None] + p2[k] * (s * w)[:, None]


def tile(torch, rays):
    reps = -(-MIN_RAYS // rays.shape[0])
    return rays.repeat(reps, 1).contiguous()


def time_call(torch, fn, repeats):
    fn()   # warm-up
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), times


def run_workload(torch, rc, bench, name, repeats):
    scene, st = bench.load_workload(name)
    cam = scene.camera
    assert cam.kind == rc._ffi.CAMERA_PINHOLE
    gen = torch.Generator(device="cuda")
    gen.manual_seed(42)
    res = {"workload": name, "raster": [cam.raster_width, cam.raster_height], "triangles": int(scene.triangle_count()), "sets": {}}
    with rc.CudaRenderer(scene, rc.CudaBackendSettings(collect_stats=rc._ffi.STATS_KERNEL_TIMES)) as r:
        # the renderer's own traversal rates on this scene (one render, kernel times on)
        r.render(st)
        s = r.stats()
        ext_rays = s["primary_rays"] - s["primary_rays_culled"] + s["bounce_rays"]
        res["render"] = {"spp": st.samples_per_pixel, "extend_rays": ext_rays, "extend_ms": s["extend_ms"],
                         "extend_mrays_per_s": ext_rays / s["extend_ms"] / 1e3, "shadow_rays": s["shadow_rays"], "shadow_ms": s["shadow_ms"],
                         "shadow_mrays_per_s": s["shadow_rays"] / s["shadow_ms"] / 1e3}

        def query(rays, mode):
            n = rays.shape[0]
            if mode == "closest":
                t = torch.empty(n, device="cuda")
                ids = torch.empty((n, 2), device="cuda", dtype=torch.int32)
                uv = torch.empty((n, 2), device="cuda")
                fn = lambda: r.trace_device(rays.data_ptr(), n, t.data_ptr(), ids.data_ptr(), uv.data_ptr())
            else:
                occ = torch.empty(n, device="cuda", dtype=torch.uint8)
                fn = lambda: r.occluded_device(rays.data_ptr(), n, occ.data_ptr())
            med, times = time_call(torch, fn, repeats)
            out = {"rays": n, "median_s": med, "times_s": times, "mrays_per_s": n / med / 1e6}
            if mode == "closest":
                out["hit_fraction"] = float((ids[:, 0] != -1).float().mean())
            else:
                out["occluded_fraction"] = float(occ.float().mean())
            return out, (t, ids) if mode == "closest" else None

        prim = primary_rays(torch, cam)
        n_set = prim.shape[0]
        res["sets"]["primary"] = {"set_rays": n_set}
        res["sets"]["primary"]["closest"], (t, ids) = query(tile(torch, prim), "closest")
        # hit points of the primary set (the first n_set rays of the tiled call are the set itself)
        hit = ids[:n_set, 0] != -1
        pts = prim[hit, 0:3] + prim[hit, 4:7] * t[:n_set][hit][:, None]
        m = pts.shape[0]
        lo, hi = pts.min(dim=0).values, pts.max(dim=0).values
        eps = 1e-4 * float((hi - lo).norm())
        inc = torch.empty((m, 8), device="cuda")
        inc[:, 0:3], inc[:, 3] = pts, eps
        inc[:, 4:7] = torch.nn.functional.normalize(torch.randn((m, 3), device="cuda", generator=gen), dim=1)
        inc[:, 7] = float("inf")
        inc_t = tile(torch, inc)
        res["sets"]["incoherent"] = {"set_rays": m, "t_min": eps, "closest": query(inc_t, "closest")[0], "occluded": query(inc_t, "occluded")[0]}
        del inc_t
        sh = torch.empty((m, 8), device="cuda")
        sh[:, 0:3], sh[:, 3] = pts, eps
        sh[:, 4:7] = light_points(torch, scene, m, gen) - pts
        sh[:, 7] = 0.999
        res["sets"]["shadow"] = {"set_rays": m, "t_min": eps, "t_max": 0.999, "occluded": query(tile(torch, sh), "occluded")[0]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C3,C5")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_trace_rays.json"))
    args = ap.parse_args()
    import torch
    import raytracing_cuda as rc
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("trace_bench.py needs a CUDA device")
    result = {"gpu": gpu_info(), "min_rays_per_call": MIN_RAYS, "repeats": args.repeats,
              "timing": "host clock around the blocking _device call after torch.cuda.synchronize(); median after one warm-up call",
              "workloads": []}
    for name in args.workloads.split(","):
        w = run_workload(torch, rc, bench, name, args.repeats)
        result["workloads"].append(w)
        rr = w["render"]
        for set_name, s in w["sets"].items():
            for mode in ("closest", "occluded"):
                if mode in s:
                    print(f"{name} {set_name:10s} {mode:8s} {s[mode]['mrays_per_s']:9.1f} Mrays/s ({s[mode]['rays']} rays, "
                          f"median {1e3 * s[mode]['median_s']:.1f} ms) | render extend {rr['extend_mrays_per_s']:.1f} Mrays/s, "
                          f"shadow {rr['shadow_mrays_per_s']:.1f} Mrays/s")
    print(f"{result['gpu']['name']}, power limit {result['gpu']['power_limit']}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
