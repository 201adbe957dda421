"""`-m gpu`: ray queries through the library (CudaRenderer.trace / occluded and the device-pointer variants): agreement with the
oracle's traverse_bvh per ray, occlusion == closest hit found, bit-identical results across the host / device variants, ray
order, GPU counts, BVH builders and scene updates, agreement with the first-hit AOV pass, and no effect on renders or stats.

Measured on a B200 (2^16 seeded rays per scene, tests/ray_sets.py): on C2, C3, the sphere scene and C3 with the watertight test
every id agreed with the oracle on every ray that hit in either, and no t / u / v was outside the AOV tolerance; the gates are
parity.py's (0.9999, 2e-3), since the traversal's world-space test runs in the FMA-contracted translation unit."""
import numpy as np
import pytest

from conftest import load_scene
from parity import AOV_OUTLIER_FRAC, ID_AGREEMENT
from ray_sets import compare, query_rays
from scene_motion import moved, trs

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF
INVALID_ARGUMENT = 1


def _trace(r, rays):
    h = r.trace(rays)
    return h.t, np.stack([h.instance, h.primitive], axis=1), h.barycentrics, r.occluded(rays).astype(np.uint8)


def _same(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8))


SCENES = {
    # name: (scene factory, oracle brute force, seed)
    "C2": (lambda rc: load_scene("cb", 512, 512), True, 11),
    "C3": (lambda rc: load_scene("cbbunny_area_light_transforms", 480, 270), False, 12),
    "sphere_scene": (lambda rc: rc.test_scenes.sphere_scene(), True, 13),
}


@pytest.mark.parametrize("name,watertight", [("C2", False), ("C3", False), ("sphere_scene", False), ("C3", True)])
def test_queries_match_the_reference(rc, oracle, name, watertight):
    make, brute, seed = SCENES[name]
    sc = make(rc)
    rays, degenerate = query_rays(sc, seed=seed)
    with rc.CudaRenderer(sc, rc.CudaBackendSettings(watertight=watertight)) as r:
        got = _trace(r, rays)
    rep = compare(got, oracle.trace_rays(sc, rays, brute_force=brute))
    print(name, "watertight" if watertight else "", rep)
    assert rep["hit_rays"] > rep["rays"] // 3
    assert rep["id_agreement"] >= ID_AGREEMENT, rep
    assert rep["outlier_frac"] <= AOV_OUTLIER_FRAC, rep
    assert (got[1][degenerate] == NONE).all() and (got[3][degenerate] == 0).all()
    assert (got[0][degenerate] == np.inf).all() and (got[2][degenerate] == 0).all()
    # any hit and closest hit run the same primitive tests: occlusion is "a closest hit exists", bit for bit
    assert np.array_equal(got[3], (got[1][:, 0] != NONE).astype(np.uint8))


def _c3_rays(rc):
    sc = load_scene("cbbunny_area_light_transforms", 320, 180)
    return sc, query_rays(sc, seed=21)[0]


def test_host_and_device_variants_and_ray_order_give_the_same_results(rc):
    import torch
    sc, rays = _c3_rays(rc)
    n = rays.shape[0]
    with rc.CudaRenderer(sc) as r:
        host = _trace(r, rays)
        perm = np.random.default_rng(5).permutation(n)
        shuffled = _trace(r, np.ascontiguousarray(rays[perm]))
        inv = np.argsort(perm)
        _same(host, [a[inv] for a in shuffled])
        d_rays = torch.from_numpy(rays).cuda()
        t = torch.empty(n, dtype=torch.float32, device="cuda")
        ids = torch.empty((n, 2), dtype=torch.int32, device="cuda")
        uv = torch.empty((n, 2), dtype=torch.float32, device="cuda")
        occ = torch.empty(n, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        r.trace_device(d_rays.data_ptr(), n, t.data_ptr(), ids.data_ptr(), uv.data_ptr())
        r.occluded_device(d_rays.data_ptr(), n, occ.data_ptr())
        dev = (t.cpu().numpy(), ids.cpu().numpy().view(np.uint32), uv.cpu().numpy(), occ.cpu().numpy())
        _same(host, dev)
        t.fill_(-1.0)   # one output alone
        r.trace_device(d_rays.data_ptr(), n, t.data_ptr(), None, None)
        assert np.array_equal(t.cpu().numpy().view(np.uint32), host[0].view(np.uint32))


def test_multi_device_contexts_give_the_one_gpu_results(rc):
    import torch
    sc, rays = _c3_rays(rc)
    with rc.CudaRenderer(sc) as r:
        one = _trace(r, rays)
    configs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for ids in configs:
        with rc.CudaRenderer(sc, rc.CudaBackendSettings(device_ids=ids)) as r:
            _same(one, _trace(r, rays))
            d_rays = torch.from_numpy(rays).to(f"cuda:{ids[0]}")
            t = torch.empty(rays.shape[0], dtype=torch.float32, device=f"cuda:{ids[0]}")
            torch.cuda.synchronize(ids[0])
            r.trace_device(d_rays.data_ptr(), rays.shape[0], t.data_ptr(), None, None)
            assert np.array_equal(t.cpu().numpy().view(np.uint32), one[0].view(np.uint32))


def test_lbvh_tree_gives_the_same_results(rc, monkeypatch):
    sc, rays = _c3_rays(rc)
    with rc.CudaRenderer(sc) as r:
        ploc = _trace(r, rays)
    monkeypatch.setenv("RTCUDA_BUILDER", "lbvh")
    with rc.CudaRenderer(sc) as r:
        _same(ploc, _trace(r, rays))


@pytest.mark.parametrize("rebuild", [False, True])
def test_updated_scene_gives_the_fresh_upload_results(rc, monkeypatch, rebuild):
    a, rays = _c3_rays(rc)
    b = moved(a, instances={5: trs((0.12, -0.08, 0.02), (0, 0, 1), 0.4), 6: trs((0.1, 0.05, -0.03))})
    with rc.CudaRenderer(b) as r:
        fresh = _trace(r, rays)
    with rc.CudaRenderer(a) as r:
        before = _trace(r, rays)
        if rebuild:
            monkeypatch.setenv("RTCUDA_TEST_REFIT_MAX_GROWTH", "0")
        r.update(b)
        monkeypatch.delenv("RTCUDA_TEST_REFIT_MAX_GROWTH", raising=False)
        assert r.stats()["bvh_last_update"] == (3 if rebuild else 2)
        _same(fresh, _trace(r, rays))
    assert not np.array_equal(before[1], fresh[1])


def test_camera_rays_agree_with_the_first_hit_pass(rc):
    """The un-jittered camera rays k_aov traces (pixel centres through raster_to_camera and camera_to_world, [near, far]),
    rebuilt in numpy, queried: ids agree with the DEBUG_IDS plane of a C2 render on >= 99.9 % of the hit pixels (measured on a
    B200: all 186,252). The numpy rays differ from the kernel's in the last bits (float64 here), so a pixel whose ray grazes an
    edge may flip."""
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
    st = rc.RaytracerSettings(outputs=rc.AovFlags.DEBUG_IDS, samples_per_pixel=1)
    with rc.CudaRenderer(sc) as r:
        ids = r.render(st).debug_ids.reshape(-1, 2)
        h = r.trace(rays)
    got = np.stack([h.instance, h.primitive], axis=1)
    hit = (ids[:, 0] != NONE) | (got[:, 0] != NONE)
    agree = float((got[hit] == ids[hit]).all(axis=1).mean())
    print(f"camera rays: {agree:.6f} of {int(hit.sum())} hit pixels agree")
    assert hit.sum() > W * H // 4 and agree >= 0.999


def test_queries_leave_renders_and_stats_alone(rc):
    sc, rays = _c3_rays(rc)
    A = rc.AovFlags
    st = rc.RaytracerSettings(outputs=A.BEAUTY | A.NORMALS | A.DEBUG_IDS | A.DEBUG_DEPTH, samples_per_pixel=4, light_sample_count=2)
    with rc.CudaRenderer(sc, rc.CudaBackendSettings(collect_stats=rc._ffi.STATS_COUNTERS)) as r:
        before = r.render(st)
        s0 = r.stats()
        _trace(r, rays)
        assert r.stats() == s0
        after = r.render(st)
    for p in ("beauty", "normals", "debug_ids", "debug_depth"):
        assert np.array_equal(getattr(before, p), getattr(after, p)), p


def test_device_variants_check_their_pointers(rc):
    import torch
    sc, rays = _c3_rays(rc)
    lib = rc._ffi.load_library()
    with rc.CudaRenderer(sc) as r:
        d = torch.from_numpy(rays).cuda()
        t = torch.empty(rays.shape[0] + 1, dtype=torch.float32, device="cuda")
        host_t = np.empty(rays.shape[0], np.float32)
        torch.cuda.synchronize()
        r.trace_device(d.data_ptr(), 0, t.data_ptr(), None, None)   # count 0: nothing to do
        r.occluded_device(d.data_ptr(), 0, t.data_ptr())
        st = lib.rtcuda_trace_rays_device(r._scene, d.data_ptr(), 4, host_t.ctypes.data, None, None)
        assert st == INVALID_ARGUMENT and b"not device memory" in lib.rtcuda_last_error()
        st = lib.rtcuda_trace_rays_device(r._scene, rays.ctypes.data, 4, t.data_ptr(), None, None)
        assert st == INVALID_ARGUMENT and b"not device memory" in lib.rtcuda_last_error()
        st = lib.rtcuda_trace_rays_device(r._scene, t.data_ptr() + 4, 4, t.data_ptr(), None, None)
        assert st == INVALID_ARGUMENT and b"16-byte aligned" in lib.rtcuda_last_error()
        st = lib.rtcuda_occluded_device(r._scene, d.data_ptr() + 8, 4, t.data_ptr())
        assert st == INVALID_ARGUMENT and b"16-byte aligned" in lib.rtcuda_last_error()
