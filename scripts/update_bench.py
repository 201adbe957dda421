"""Cost of rtcuda_scene_update (CudaRenderer.update) against a fresh upload, and what a refit does to the wide tree.

For each workload (C3, C5 of bench.py):
  * host wall time and device time (stats update_ms) of an identity update, a camera-only update, a small rigid motion of
    one instance and a motion that triggers the rebuild, against constructing a fresh CudaRenderer (upload_and_build);
  * one instance moved by 0, 1, 5, 20, 50 % of the scene extent: SAH cost of the refitted tree against a fresh build's, and
    extend_ms + shadow_ms (CUDA events, RTCUDA_STATS_KERNEL_TIMES) and nodes / primitives fetched per ray after the refit
    against after a fresh build. The refits here run with RTCUDA_TEST_REFIT_MAX_GROWTH set very high, so that the table
    shows the refit's cost also where the library would rebuild (the table REFIT_MAX_GROWTH is chosen from).
Writes one JSON document (--out). Needs a GPU."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

import raytracing_cuda as rc  # noqa: E402
from bench import load_workload  # noqa: E402
from scene_motion import moved, scatter, trs  # noqa: E402

TIMES, COUNTERS = rc._ffi.STATS_KERNEL_TIMES, rc._ffi.STATS_COUNTERS


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def world_bounds(sc):
    lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
    for si, tf in sc.instances:
        sh = sc.shapes[si].shape
        if isinstance(sh, rc.Mesh):
            v = sh.vertices.astype(np.float64)
            w = v @ tf.forward[:3, :3].T.astype(np.float64) + tf.forward[:3, 3]
            lo, hi = np.minimum(lo, w.min(0)), np.maximum(hi, w.max(0))
    return lo, hi


def _mesh_tris(sc, i):
    sh = sc.shapes[sc.instances[i][0]]
    return len(sh.shape.tris) if isinstance(sh.shape, rc.Mesh) and sh.area_light is None else 0


def timed_update(r, b, reps):
    walls, devs, kinds = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        r.update(b[0])
        walls.append(1e3 * (time.perf_counter() - t0))
        s = r.stats()
        devs.append(s["update_ms"]); kinds.append(s["bvh_last_update"])
        b = b[::-1]   # alternate the two states, so that every call has something to do
    return {"host_ms_median": statistics.median(walls), "update_ms_median": statistics.median(devs), "host_ms": walls, "update_ms": devs,
            "bvh_last_update": kinds}


def trace_figures(r, st):
    r.render(st)   # warm
    r.render(st)
    s = r.stats()
    return s


def per_ray(s):
    rays = s["primary_rays"] - s["primary_rays_culled"] + s["bounce_rays"] + s["shadow_rays"]
    return s["nodes_fetched"] / max(1, rays), s["prims_fetched"] / max(1, rays)


def run(name, spp, reps):
    a, st = load_workload(name)
    st.samples_per_pixel = spp
    lo, hi = world_bounds(a)
    extent = float(np.max(hi - lo))
    k = max(range(len(a.instances)), key=lambda i: _mesh_tris(a, i))   # the largest mesh that is not an emitter
    out = {"workload": name, "raster": [a.camera.raster_width, a.camera.raster_height], "spp_for_trace_figures": spp,
           "triangles": a.triangle_count(), "moving_instance": k, "scene_extent": extent}
    # update costs
    t0 = time.perf_counter()
    r = rc.CudaRenderer(a)
    out["fresh_renderer"] = {"host_ms": 1e3 * (time.perf_counter() - t0), "upload_and_build_ms": r.setup_ms["upload_and_build"],
                             "bvh_build_ms": r.stats()["bvh_build_ms"]}
    r.update(moved(a))   # first update: the built tree's cost (node pass over the unchanged primitives)
    out["first_identity_update"] = {"update_ms": r.stats()["update_ms"], "bvh_sah_cost": r.stats()["bvh_sah_cost"]}
    out["identity"] = timed_update(r, [moved(a), moved(a)], reps)
    out["camera_only"] = timed_update(r, [moved(a, camera=trs((0.05 * extent, 0, 0))), moved(a)], reps)
    out["rigid_motion_1pct"] = timed_update(r, [moved(a, instances={k: trs((0.01 * extent, 0, 0))}), moved(a)], reps)
    sc = scatter(a, seed=3, extent=0.75 * extent)
    out["scatter_rebuild"] = timed_update(r, [sc, a], reps)
    r.close()
    # refit against fresh build, one instance moved
    os.environ["RTCUDA_TEST_REFIT_MAX_GROWTH"] = "1e30"
    rows = []
    rt = rc.CudaRenderer(a, rc.CudaBackendSettings(collect_stats=TIMES))
    rn = rc.CudaRenderer(a, rc.CudaBackendSettings(collect_stats=COUNTERS))
    for pct in (0, 1, 5, 20, 50):
        b = moved(a, instances={k: trs((0.01 * pct * extent, 0.0, 0.0))})
        row = {"moved_pct_of_extent": pct}
        for label, renderers in (("refit", (rt, rn)), ("fresh", None)):
            if renderers is None:
                renderers = (rc.CudaRenderer(b, rc.CudaBackendSettings(collect_stats=TIMES)), rc.CudaRenderer(b, rc.CudaBackendSettings(collect_stats=COUNTERS)))
            for x in renderers:
                x.update(b)
            sah = renderers[0].stats()["bvh_sah_cost"]
            s = trace_figures(renderers[0], st)
            c = trace_figures(renderers[1], st)
            npr, ppr = per_ray(c)
            row[label] = {"bvh_sah_cost": sah, "extend_plus_shadow_ms": s["extend_ms"] + s["shadow_ms"], "extend_ms": s["extend_ms"],
                          "shadow_ms": s["shadow_ms"], "nodes_per_ray": npr, "prims_per_ray": ppr, "render_ms": s["render_ms"],
                          "bvh_last_update": renderers[0].stats()["bvh_last_update"]}
            if label == "fresh":
                for x in renderers:
                    x.close()
        row["sah_growth"] = row["refit"]["bvh_sah_cost"] / row["fresh"]["bvh_sah_cost"]
        row["trace_time_ratio"] = row["refit"]["extend_plus_shadow_ms"] / row["fresh"]["extend_plus_shadow_ms"]
        rows.append(row)
        print(name, json.dumps({k2: row[k2] for k2 in ("moved_pct_of_extent", "sah_growth", "trace_time_ratio")}), flush=True)
    del os.environ["RTCUDA_TEST_REFIT_MAX_GROWTH"]
    rt.close(); rn.close()
    out["refit_vs_fresh"] = rows
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="C3,C5")
    ap.add_argument("--spp", default="C3:16,C5:4", help="samples per pixel of the trace figures, per workload")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    spp = dict((k, int(v)) for k, v in (x.split(":") for x in args.spp.split(",")))
    doc = {"device": device_info(), "note": "host_ms: wall time of CudaRenderer.update (includes Scene.to_desc); update_ms: CUDA events "
           "around the device work of the update. Trace figures at reduced samples per pixel (spp_for_trace_figures), rendered twice, "
           "the second render reported.", "workloads": []}
    for name in args.workloads.split(","):
        doc["workloads"].append(run(name, spp.get(name, 4), args.reps))
        print(name, "done", flush=True)
    doc["device_after"] = device_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
