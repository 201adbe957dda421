"""`-m gpu`: rtcuda_scene_update (CudaRenderer.update). After an update every plane equals the frame of a fresh CudaRenderer on
the updated scene, bit for bit: traversal keeps the closest t (ties to the larger (geom, prim)) and tests boxes conservatively,
so a refitted tree, a rebuilt tree and a fresh build render the same pixels."""
import numpy as np
import pytest

from conftest import load_scene
from scene_motion import about, moved, scatter, trs

pytestmark = pytest.mark.gpu

PLANES = ("beauty", "normals", "albedo", "uv", "mip_level", "debug_ids", "debug_depth")


def _all(rc):
    A = rc.AovFlags
    return A.BEAUTY | A.NORMALS | A.ALBEDO | A.UV_COORDS | A.MIP_LEVEL | A.DEBUG_IDS | A.DEBUG_DEPTH


def _fresh(rc, scene, st, **backend):
    with rc.CudaRenderer(scene, rc.CudaBackendSettings(**backend)) as r:
        return r.render(st), r.stats()


def _assert_same(a, b):
    for p in PLANES:
        x, y = getattr(a, p), getattr(b, p)
        assert (x is None) == (y is None), p
        assert x is None or np.array_equal(x, y), p


def _c3_motion(s):
    """bunny translated and turned, emitter and its light moved together, camera moved"""
    return moved(s, instances={5: about((0.0, 0.0, 0.3), trs((0.12, -0.08, 0.02), (0, 0, 1), 0.4)), 6: trs((0.1, 0.05, -0.03))},
                 lights={0: trs((0.1, 0.05, -0.03))}, camera=trs((0.15, -0.2, 0.05), (0, 0, 1), 0.05))


@pytest.mark.parametrize("which", ["C2", "C3"])
def test_refit_gives_the_fresh_upload_frame(rc, which):
    if which == "C2":
        a = load_scene("cb", 512, 512)
        b = moved(a, instances={2: trs((0.05, 0.0, 0.02)), 5: trs((0.1, -0.05, -0.02))}, lights={0: trs((0.1, -0.05, -0.02))},
                  camera=trs((0.1, 0.1, 0.0), (0, 0, 1), 0.03))
        st = rc.RaytracerSettings(outputs=_all(rc), samples_per_pixel=8)
    else:
        a = load_scene("cbbunny_area_light_transforms", 480, 270)
        b = _c3_motion(a)
        st = rc.RaytracerSettings(outputs=_all(rc), samples_per_pixel=8, light_sample_count=4)
    with rc.CudaRenderer(a) as r:
        before = r.render(st)
        r.update(b)
        s = r.stats()
        assert s["bvh_last_update"] == 2 and s["bvh_sah_cost"] > 1.0 and s["update_ms"] > 0.0
        after = r.render(st)
    fresh, _ = _fresh(rc, b, st)
    _assert_same(after, fresh)
    assert not np.array_equal(before.beauty, after.beauty)


def _aov_fetches(r, rc):
    """BVH nodes / primitives the first-hit AOV pass fetches: one thread walks one ray, so the counts are a function of the
    tree (the persistent extend / shadow kernels count per warp phase, which depends on how rays are dealt to warps)"""
    A = rc.AovFlags
    r.render(rc.RaytracerSettings(outputs=A.NORMALS | A.DEBUG_IDS, samples_per_pixel=1))
    s = r.stats()
    return s["nodes_fetched"], s["prims_fetched"]


def test_rebuild_gives_the_fresh_upload_frame_and_tree(rc, monkeypatch):
    """the rebuild path, forced through the rule's test hook: instance motions that trip the rule are rare (every instance
    is a subtree of its own, which a rigid motion keeps intact: DESIGN.md "Scene updates")"""
    a = load_scene("cbbunny_area_light_transforms", 320, 180)
    b = scatter(a, seed=3, extent=1.5)
    st = rc.RaytracerSettings(outputs=_all(rc), samples_per_pixel=4, light_sample_count=2)
    with rc.CudaRenderer(a, rc.CudaBackendSettings(collect_stats=1)) as r:
        monkeypatch.setenv("RTCUDA_TEST_REFIT_MAX_GROWTH", "0")
        r.update(b)
        monkeypatch.delenv("RTCUDA_TEST_REFIT_MAX_GROWTH")
        s = r.stats()
        assert s["bvh_last_update"] == 3
        after = r.render(st)
        fetched = _aov_fetches(r, rc)
    with rc.CudaRenderer(b, rc.CudaBackendSettings(collect_stats=1)) as f:
        fresh = f.render(st)
        assert _aov_fetches(f, rc) == fetched and f.stats()["bvh_node_count"] == s["bvh_node_count"]
        f.update(b)   # an identity update reports the built tree's cost
        assert f.stats()["bvh_sah_cost"] == s["bvh_sah_cost"]
    _assert_same(after, fresh)


def test_identity_update_changes_nothing(rc):
    a = load_scene("cbbunny_area_light_transforms", 320, 180)
    st = rc.RaytracerSettings(outputs=_all(rc), samples_per_pixel=4)
    with rc.CudaRenderer(a, rc.CudaBackendSettings(collect_stats=1)) as r:
        before = r.render(st)
        f0 = _aov_fetches(r, rc)
        r.update(moved(a))
        s1 = r.stats()
        assert s1["bvh_last_update"] == 0 and s1["bvh_sah_cost"] > 1.0
        after = r.render(st)
        f1 = _aov_fetches(r, rc)
    _assert_same(after, before)
    assert f1 == f0


def test_camera_update_drops_the_captured_frame_graph(rc):
    """frames of >= 2^22 paths are captured as a CUDA graph on their second launch and replayed from the third; the graph
    holds the old camera in its kernel parameters"""
    a = load_scene("cb", 1920, 1080)
    b = moved(a, camera=trs((0.2, -0.1, 0.05), (0, 0, 1), 0.06))
    st = rc.RaytracerSettings(samples_per_pixel=8, light_sample_count=1)
    with rc.CudaRenderer(a) as r:
        frames = [r.render(st).beauty for _ in range(3)]
        assert np.array_equal(frames[0], frames[2])
        r.update(b)
        assert r.stats()["bvh_last_update"] == 1
        after = r.render(st).beauty
    fresh, _ = _fresh(rc, b, st)
    assert np.array_equal(after, fresh.beauty) and not np.array_equal(after, frames[0])


def test_camera_update_recomputes_the_culled_pixels(rc):
    a = load_scene("cbbunny_area_light_transforms", 480, 270)
    b = moved(a, camera=trs((0.0, 0.8, 0.0)))   # backs away: the box covers fewer pixels
    st = rc.RaytracerSettings(samples_per_pixel=4, light_sample_count=2)
    with rc.CudaRenderer(a) as r:
        r.render(st)
        d0 = r.stats()["pixels_dropped"]
        r.update(b)
        after = r.render(st)
        d1 = r.stats()["pixels_dropped"]
    fresh, fs = _fresh(rc, b, st)
    assert np.array_equal(after.beauty, fresh.beauty)
    assert d1 == fs["pixels_dropped"] and d1 != d0


@pytest.mark.parametrize("n", [2, 4])
def test_multi_device_update(rc, n):
    import torch
    from test_gpu_parity import _device_ids
    a = load_scene("cbbunny_area_light_transforms", 256, 144)
    b = _c3_motion(a)
    A = rc.AovFlags
    st = rc.RaytracerSettings(outputs=A.BEAUTY | A.NORMALS | A.DEBUG_IDS, samples_per_pixel=6, light_sample_count=2)
    fresh, _ = _fresh(rc, b, st)
    ids = _device_ids(n)
    with rc.CudaRenderer(a, rc.CudaBackendSettings(num_devices=len(ids), device_ids=ids, tile_size=16)) as r:
        dev = f"cuda:{ids[0]}"
        beauty = torch.zeros((144, 256, 3), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        r.render_device(st, {"beauty": beauty.data_ptr()})   # rank 0 now holds the other ranks' tile tables
        r.update(b)
        assert r.stats()["bvh_last_update"] == 2
        _assert_same(r.render(st), fresh)
        normals = torch.zeros_like(beauty)
        r.render_device(st, {"beauty": beauty.data_ptr(), "normals": normals.data_ptr()})
        assert np.array_equal(beauty.cpu().numpy(), fresh.beauty) and np.array_equal(normals.cpu().numpy(), fresh.normals)
        acc = torch.zeros_like(beauty)
        torch.cuda.synchronize()
        for lo, hi in ((0, 2), (2, 6)):
            r.render_samples_accumulate_device(st, lo, hi, acc.data_ptr())
        inv = torch.tensor(1.0 / 6, dtype=torch.float32)
        np.testing.assert_allclose((acc.cpu() * inv).numpy(), fresh.beauty, rtol=2e-6, atol=1e-7)


def test_topology_mismatch_is_refused_and_leaves_the_scene(rc):
    import copy
    a = load_scene("cbbunny_area_light_transforms", 160, 90)
    st = rc.RaytracerSettings(outputs=_all(rc), samples_per_pixel=2)
    fewer = moved(a)
    fewer.instances = fewer.instances[:-1]
    other_shape = moved(a, instances={5: trs((0.1, 0, 0))})
    other_shape.instances[5] = (4, other_shape.instances[5][1])
    bigger = moved(a)
    bigger.camera = a.camera.with_raster_size(320, 180)
    other_light = moved(a)
    other_light.lights[0] = copy.copy(other_light.lights[0])
    other_light.lights[0].kind = rc._ffi.LIGHT_POINT
    with rc.CudaRenderer(a) as r:
        before = r.render(st)
        for bad in (fewer, other_shape, bigger, other_light):
            with pytest.raises(rc._ffi.RtCudaError, match="INVALID_ARGUMENT"):
                r.update(bad)
            _assert_same(r.render(st), before)
