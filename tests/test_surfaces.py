"""`-m gpu`: surface queries through the library (CudaRenderer.surfaces / surfaces_device): agreement with the oracle's HitInfo and
albedo per ray, t and ids bit-identical to the closest-hit query, bit-identical records across host / device arrays, ray order,
GPU counts, BVH builders and scene updates, agreement with the first-hit AOV planes of a render, no effect on renders or stats,
and the device variant's pointer checks.

Measured on a B200 (2^16 seeded rays per scene, tests/ray_sets.py): on C2, C3, the texture zoo and C3 with the watertight test
every id agreed with the oracle and no field was outside the tolerances; on the sphere scene 12 of 34,673 hit rays (3.5e-4) had
a uv outside it (the sphere uv is the one field computed with acosf / sinf, whose device and host results may round
differently). Camera rays agreed with the first-hit planes on all 186,252 hit pixels of C2. The oracle gates are those of the ray-query tests (parity.py's
ID_AGREEMENT and AOV_OUTLIER_FRAC, and PLANE_ATOL["albedo"] for the albedo), since the traversal's world-space test runs in the
FMA-contracted translation unit."""
import numpy as np
import pytest

from conftest import load_scene, texture_zoo_scene
from parity import AOV_ATOL, AOV_OUTLIER_FRAC, AOV_RTOL, ID_AGREEMENT, NONE_ID, PLANE_ATOL
from ray_sets import query_rays
from scene_motion import moved, trs
from surface_compare import bits, compare_surfaces, is_miss_record

pytestmark = pytest.mark.gpu

INVALID_ARGUMENT = 1

SCENES = {
    # name: (scene factory, oracle brute force, seed)
    "C2": (lambda rc: load_scene("cb", 512, 512), True, 11),
    "C3": (lambda rc: load_scene("cbbunny_area_light_transforms", 480, 270), False, 12),
    "sphere_scene": (lambda rc: rc.test_scenes.sphere_scene(), True, 13),
    "texture_zoo": (lambda rc: texture_zoo_scene(), True, 14),
}


@pytest.fixture(scope="module")
def hs():
    import hostsim_surfaces_py
    hostsim_surfaces_py.build()
    return hostsim_surfaces_py


@pytest.mark.parametrize("name,watertight", [("C2", False), ("C3", False), ("sphere_scene", False), ("texture_zoo", False), ("C3", True)])
def test_surfaces_match_the_reference(rc, hs, name, watertight):
    make, brute, seed = SCENES[name]
    sc = make(rc)
    rays, invalid = query_rays(sc, seed=seed)
    with rc.CudaRenderer(sc, rc.CudaBackendSettings(watertight=watertight)) as r:
        got = r.surfaces(rays).records
        h = r.trace(rays)
    rep = compare_surfaces(got, hs.oracle_trace_surfaces(sc, rays, brute_force=brute))
    print(name, "watertight" if watertight else "", rep)
    assert rep["hit_rays"] > rep["rays"] // 3
    assert rep["id_agreement"] >= ID_AGREEMENT, rep
    assert rep["outlier_frac"] <= AOV_OUTLIER_FRAC, rep
    assert rep["material_light_mismatches"] == 0, rep
    assert is_miss_record(got[invalid]).all()
    # t and the ids are the closest-hit query's, bit for bit
    assert np.array_equal(got["t"].view(np.uint32), h.t.view(np.uint32))
    assert np.array_equal(got["geom_id"], h.instance) and np.array_equal(got["prim_id"], h.primitive)
    assert np.array_equal(is_miss_record(got), h.instance == NONE_ID)


def _c3_rays(rc):
    sc = load_scene("cbbunny_area_light_transforms", 320, 180)
    return sc, query_rays(sc, seed=21)[0]


def _device_surfaces(r, rays, device="cuda"):
    import torch
    n = rays.shape[0]
    d_rays = torch.from_numpy(rays).to(device)
    out = torch.full((n, 16), -1.0, dtype=torch.float32, device=device)
    torch.cuda.synchronize(device)
    r.surfaces_device(d_rays.data_ptr(), n, out.data_ptr())
    return out


def test_host_and_device_variants_and_ray_order_give_the_same_records(rc):
    import torch
    from raytracing_cuda.backend import SURFACE_DTYPE
    sc, rays = _c3_rays(rc)
    n = rays.shape[0]
    with rc.CudaRenderer(sc) as r:
        host = r.surfaces(rays).records
        perm = np.random.default_rng(5).permutation(n)
        shuffled = r.surfaces(np.ascontiguousarray(rays[perm])).records
        assert np.array_equal(bits(host), bits(shuffled[np.argsort(perm)]))
        out = _device_surfaces(r, rays)
        assert np.array_equal(bits(host), bits(out.cpu().numpy().view(SURFACE_DTYPE).reshape(n)))
        # the integer words read through an int32 view
        ints = out.view(torch.int32).cpu().numpy().view(np.uint32)
        assert np.array_equal(ints[:, 10], host["geom_id"]) and np.array_equal(ints[:, 15], host["light"])


def test_multi_device_contexts_give_the_one_gpu_records(rc):
    import torch
    from raytracing_cuda.backend import SURFACE_DTYPE
    sc, rays = _c3_rays(rc)
    with rc.CudaRenderer(sc) as r:
        one = r.surfaces(rays).records
    configs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for ids in configs:
        with rc.CudaRenderer(sc, rc.CudaBackendSettings(device_ids=ids)) as r:
            assert np.array_equal(bits(one), bits(r.surfaces(rays).records))
            out = _device_surfaces(r, rays, f"cuda:{ids[0]}")
            assert np.array_equal(bits(one), bits(out.cpu().numpy().view(SURFACE_DTYPE).reshape(-1)))


def test_lbvh_tree_gives_the_same_records(rc, monkeypatch):
    sc, rays = _c3_rays(rc)
    with rc.CudaRenderer(sc) as r:
        ploc = r.surfaces(rays).records
    monkeypatch.setenv("RTCUDA_BUILDER", "lbvh")
    with rc.CudaRenderer(sc) as r:
        assert np.array_equal(bits(ploc), bits(r.surfaces(rays).records))


@pytest.mark.parametrize("rebuild", [False, True])
def test_updated_scene_gives_the_fresh_upload_records(rc, monkeypatch, rebuild):
    a, rays = _c3_rays(rc)
    b = moved(a, instances={5: trs((0.12, -0.08, 0.02), (0, 0, 1), 0.4), 6: trs((0.1, 0.05, -0.03))})
    with rc.CudaRenderer(b) as r:
        fresh = r.surfaces(rays).records
    with rc.CudaRenderer(a) as r:
        before = r.surfaces(rays).records
        if rebuild:
            monkeypatch.setenv("RTCUDA_TEST_REFIT_MAX_GROWTH", "0")
        r.update(b)
        monkeypatch.delenv("RTCUDA_TEST_REFIT_MAX_GROWTH", raising=False)
        assert r.stats()["bvh_last_update"] == (3 if rebuild else 2)
        assert np.array_equal(bits(fresh), bits(r.surfaces(rays).records))
    assert not np.array_equal(bits(before), bits(fresh))


def _close(a, b, atol, rtol):
    a, b = np.asarray(a, np.float64).reshape(len(a), -1), np.asarray(b, np.float64).reshape(len(b), -1)
    return (np.abs(a - b) <= atol + rtol * np.abs(b)).all(axis=1)


def test_camera_rays_agree_with_the_first_hit_planes(rc):
    """The un-jittered camera rays k_aov traces (pixel centres through raster_to_camera and camera_to_world, [near, far]),
    rebuilt in numpy, against one C2 render's NORMALS / ALBEDO / UV_COORDS / DEBUG_IDS / DEBUG_DEPTH planes: on >= 99.9 % of the
    hit pixels the ids agree and normal / uv / t are within the AOV tolerance and the albedo within PLANE_ATOL. cb's albedos
    are constant, so the render's texture footprint does not matter. The numpy rays differ from the kernel's in the last bits
    (float64 here), so a pixel whose ray grazes an edge may flip."""
    sc = load_scene("cb", 512, 512)
    cam = sc.camera
    W, H = cam.raster_width, cam.raster_height
    ys, xs = np.meshgrid(np.arange(H, dtype=np.float64) + 0.5, np.arange(W, dtype=np.float64) + 0.5, indexing="ij")
    raster = np.stack([xs.ravel(), ys.ravel(), np.zeros(W * H), np.ones(W * H)], axis=1)
    cp = raster @ np.asarray(cam.raster_to_camera.forward, np.float64).T
    cp = cp[:, :3] / cp[:, 3:]
    c2w = np.asarray(cam.camera_to_world.forward, np.float64)
    assert cam.kind == rc._ffi.CAMERA_PINHOLE
    d = (cp / np.linalg.norm(cp, axis=1, keepdims=True)) @ c2w[:3, :3].T
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = np.broadcast_to(c2w[:3, 3] / c2w[3, 3], d.shape)
    rays = rc.make_rays(o, d, cam.near_clip, cam.far_clip)
    A = rc.AovFlags
    st = rc.RaytracerSettings(outputs=A.NORMALS | A.ALBEDO | A.UV_COORDS | A.DEBUG_IDS | A.DEBUG_DEPTH, samples_per_pixel=1)
    with rc.CudaRenderer(sc) as r:
        out = r.render(st)
        s = r.surfaces(rays)
    ids = out.debug_ids.reshape(-1, 2)
    got = np.stack([s.instance, s.primitive], axis=1)
    hit = (ids[:, 0] != NONE_ID) | (got[:, 0] != NONE_ID)
    ok = (got == ids).all(axis=1)
    ok &= _close(s.normal, out.normals.reshape(-1, 3), AOV_ATOL, AOV_RTOL)
    ok &= _close(s.uv, out.uv.reshape(-1, 2), AOV_ATOL, AOV_RTOL)
    ok &= _close(s.t, out.debug_depth.reshape(-1), AOV_ATOL, AOV_RTOL)
    ok &= _close(s.albedo, out.albedo.reshape(-1, 3), PLANE_ATOL["albedo"], 0.0)
    agree = float(ok[hit].mean())
    print(f"camera rays: {agree:.6f} of {int(hit.sum())} hit pixels agree")
    assert hit.sum() > W * H // 4 and agree >= 0.999


def test_surfaces_leave_renders_and_stats_alone(rc):
    sc, rays = _c3_rays(rc)
    A = rc.AovFlags
    st = rc.RaytracerSettings(outputs=A.BEAUTY | A.NORMALS | A.ALBEDO | A.DEBUG_IDS | A.DEBUG_DEPTH, samples_per_pixel=4,
                              light_sample_count=2)
    with rc.CudaRenderer(sc, rc.CudaBackendSettings(collect_stats=rc._ffi.STATS_COUNTERS)) as r:
        before = r.render(st)
        s0 = r.stats()
        r.surfaces(rays)
        _device_surfaces(r, rays)
        assert r.stats() == s0
        after = r.render(st)
    for p in ("beauty", "normals", "albedo", "debug_ids", "debug_depth"):
        assert np.array_equal(getattr(before, p), getattr(after, p)), p


def test_device_variant_checks_its_pointers(rc):
    import torch
    sc, rays = _c3_rays(rc)
    lib = rc._ffi.load_library()
    with rc.CudaRenderer(sc) as r:
        d = torch.from_numpy(rays).cuda()
        out = torch.empty((rays.shape[0] + 1, 16), dtype=torch.float32, device="cuda")
        host_out = np.empty((4, 16), np.float32)
        torch.cuda.synchronize()
        r.surfaces_device(d.data_ptr(), 0, out.data_ptr())   # count 0: nothing to do
        st = lib.rtcuda_trace_surfaces_device(r._scene, d.data_ptr(), 4, host_out.ctypes.data)
        assert st == INVALID_ARGUMENT and b"not device memory" in lib.rtcuda_last_error()
        st = lib.rtcuda_trace_surfaces_device(r._scene, rays.ctypes.data, 4, out.data_ptr())
        assert st == INVALID_ARGUMENT and b"not device memory" in lib.rtcuda_last_error()
        st = lib.rtcuda_trace_surfaces_device(r._scene, d.data_ptr(), 4, out.data_ptr() + 8)
        assert st == INVALID_ARGUMENT and b"16-byte aligned" in lib.rtcuda_last_error()
        st = lib.rtcuda_trace_surfaces_device(r._scene, d.data_ptr() + 8, 4, out.data_ptr())
        assert st == INVALID_ARGUMENT and b"16-byte aligned" in lib.rtcuda_last_error()
