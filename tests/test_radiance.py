"""`-m gpu`: radiance along caller-supplied rays through the library (CudaRenderer.radiance / radiance_device): agreement with the
oracle's ray_radiance per ray, bit-identical results across host / device arrays, GPU counts, batch sizes, stream-base slices, BVH
builders and scene updates, statistical agreement with render() on jittered camera rays, no effect on renders or stats (including
a captured frame graph across a re-carve of the path-state arena), and the device variant's pointer checks.

Oracle parity uses 2^14 seeded rays per scene (tests/ray_sets.py) at 16 spp and depth 5 with the default beauty gates of
tests/parity.py (SPECULAR_GATES for the rough-metal box): the wavefront kernels contract multiply-adds and use approximate division,
so paths agree with the oracle to rounding until a rounding flips a branch. The figures of each run are printed; measured on a
B200 (p50 / p99 / diverged of the per-ray difference over the reference's mean): C2 3.7e-8 / 3.7e-7 / 0, C3 1.6e-7 / 4.3e-6 /
1.8e-4, environment scene 0 / 2.1e-7 / 0, rough-metal box 1.9e-7 / 1.8e-5 / 8.7e-5; camera rays vs render z = -1.66."""
import numpy as np
import pytest

from conftest import load_scene
from parity import SPECULAR_GATES, beauty_close, mean_luminance_z
from radiance_rays import jittered_camera_rays
from ray_sets import query_rays
from scene_motion import moved, trs

pytestmark = pytest.mark.gpu

INVALID_ARGUMENT = 1
SETTINGS = dict(samples_per_pixel=16, max_ray_depth=5)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _env(rc):
    return rc.test_scenes.environment_lighting_scene(rc.test_scenes.synthetic_environment_map())


SCENES = {
    # name: (scene factory, seed, gates)
    "C2": (lambda rc: load_scene("cb", 512, 512), 31, {}),
    "C3": (lambda rc: load_scene("cbbunny_area_light_transforms", 480, 270), 32, {}),
    "sphere_scene": (lambda rc: rc.test_scenes.sphere_scene(), 33, None),   # no light: exactly 0
    "environment": (_env, 34, {}),
    "rough_metal": (lambda rc: rc.test_scenes.rough_metal_scene(), 35, SPECULAR_GATES),
}


@pytest.mark.parametrize("name", sorted(SCENES))
def test_radiance_matches_the_reference(rc, oracle, name):
    make, seed, gates = SCENES[name]
    sc = make(rc)
    rays, invalid = query_rays(sc, n=1 << 14, seed=seed)
    st = rc.RaytracerSettings(**SETTINGS)
    with rc.CudaRenderer(sc) as r:
        got = r.radiance(rays, st)
    ref, _ = oracle.radiance(sc, st, rays)
    assert got.shape == (len(rays), 3) and got.dtype == np.float32
    assert not got[invalid].any()
    if gates is None:
        assert not got.any() and not ref.any()
        return
    rep = {}
    ok = beauty_close(got, ref, report=rep, **gates)
    print(name, rep)
    assert rep["pixels"] > len(rays) // 4
    assert ok, rep


def _c3(rc):
    sc = load_scene("cbbunny_area_light_transforms", 320, 180)
    return sc, query_rays(sc, n=1 << 14, seed=41)[0]


def test_host_device_batches_and_slices_give_the_same_bits(rc):
    import torch
    sc, rays = _c3(rc)
    n = len(rays)
    st = rc.RaytracerSettings(**SETTINGS)
    with rc.CudaRenderer(sc) as r:
        host = r.radiance(rays, st)
        d_rays = torch.from_numpy(rays).cuda()
        d_out = torch.full((n, 3), -1.0, dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        r.radiance_device(d_rays.data_ptr(), n, st, d_out.data_ptr())
        assert np.array_equal(_bits(host), _bits(d_out.cpu().numpy()))
        a, b = 5000, 12000
        assert np.array_equal(_bits(host[a:b]), _bits(r.radiance(np.ascontiguousarray(rays[a:b]), st, stream_base=a)))
        assert not np.array_equal(_bits(host[a:b]), _bits(r.radiance(np.ascontiguousarray(rays[a:b]), st, stream_base=a + 1)))
    with rc.CudaRenderer(sc, rc.CudaBackendSettings(max_paths_in_flight=4096)) as r:
        assert np.array_equal(_bits(host), _bits(r.radiance(rays, st)))


def test_multi_device_contexts_give_the_one_gpu_results(rc):
    import torch
    sc, rays = _c3(rc)
    st = rc.RaytracerSettings(**SETTINGS)
    with rc.CudaRenderer(sc) as r:
        one = r.radiance(rays, st)
    configs = [[0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for ids in configs:
        with rc.CudaRenderer(sc, rc.CudaBackendSettings(device_ids=ids)) as r:
            assert np.array_equal(_bits(one), _bits(r.radiance(rays, st))), ids
            d_rays = torch.from_numpy(rays).to(f"cuda:{ids[0]}")
            d_out = torch.empty((len(rays), 3), dtype=torch.float32, device=f"cuda:{ids[0]}")
            torch.cuda.synchronize(ids[0])
            r.radiance_device(d_rays.data_ptr(), len(rays), st, d_out.data_ptr())
            assert np.array_equal(_bits(one), _bits(d_out.cpu().numpy())), ids


def test_lbvh_tree_gives_the_same_results(rc, monkeypatch):
    sc, rays = _c3(rc)
    st = rc.RaytracerSettings(**SETTINGS)
    with rc.CudaRenderer(sc) as r:
        ploc = r.radiance(rays, st)
    monkeypatch.setenv("RTCUDA_BUILDER", "lbvh")
    with rc.CudaRenderer(sc) as r:
        assert np.array_equal(_bits(ploc), _bits(r.radiance(rays, st)))


def test_updated_scene_gives_the_fresh_upload_results(rc):
    a, rays = _c3(rc)
    b = moved(a, instances={5: trs((0.12, -0.08, 0.02), (0, 0, 1), 0.4), 6: trs((0.1, 0.05, -0.03))})
    st = rc.RaytracerSettings(**SETTINGS)
    with rc.CudaRenderer(b) as r:
        fresh = r.radiance(rays, st)
    with rc.CudaRenderer(a) as r:
        before = r.radiance(rays, st)
        r.update(b)
        assert np.array_equal(_bits(fresh), _bits(r.radiance(rays, st)))
    assert not np.array_equal(_bits(before), _bits(fresh))


def test_camera_rays_agree_with_the_renderer(rc):
    """64 jittered camera rays per pixel (numpy, own RNG) at 1 spp each, averaged per pixel, against render() at 64 spp with another
    seed: the mean luminance differs by less than 3 standard errors (the different-seed rule of the parity tests)"""
    sc = load_scene("cbbunny_area_light_transforms", 96, 64)
    cam = sc.camera
    assert cam.kind == rc._ffi.CAMERA_PINHOLE
    per = 64
    rays = jittered_camera_rays(cam, per, seed=3)
    with rc.CudaRenderer(sc) as r:
        rad = r.radiance(rays, rc.RaytracerSettings(samples_per_pixel=1, seed=1234))
        img = r.render(rc.RaytracerSettings(samples_per_pixel=per, seed=99)).beauty
    mean = rad.astype(np.float64).reshape(cam.raster_height, cam.raster_width, per, 3).mean(axis=2)
    z = mean_luminance_z(mean, img.astype(np.float64), per, per)
    print(f"camera rays vs render: z = {z:.3f}, mean {mean.mean():.6f} vs {img.mean():.6f}")
    assert abs(z) < 3.0 and img.mean() > 0


def test_radiance_leaves_renders_graphs_and_stats_alone(rc):
    """A frame large enough for the captured frame graph (>= 4 Mi paths), rendered twice so the graph is captured; then a radiance
    call whose wavefront has more slots but fewer light samples per slot, so the arena is carved anew inside the same allocation;
    then two more frames. Every frame is the same bits and the stats are those of the last render."""
    sc = load_scene("cbbunny_area_light_transforms", 320, 180)
    st = rc.RaytracerSettings(samples_per_pixel=128, light_sample_count=8)
    rays, _ = query_rays(sc, n=1 << 18, seed=43)
    with rc.CudaRenderer(sc, rc.CudaBackendSettings(collect_stats=rc._ffi.STATS_COUNTERS)) as r:
        frames = [r.render(st).beauty for _ in range(2)]
        s0 = r.stats()
        assert s0["samples"] >= 1 << 22
        # ~2.6e5 live rays x 64 spp > the frame's 7.4e6 paths, at 196 B of path state per slot instead of 532: more slots
        # carved from the arena the frame sized
        rad = r.radiance(rays, rc.RaytracerSettings(samples_per_pixel=64, light_sample_count=1))
        assert (rad.max(axis=1) > 0).mean() > 0.5
        assert r.stats() == s0
        frames += [r.render(st).beauty for _ in range(2)]
    for f in frames[1:]:
        assert np.array_equal(_bits(frames[0]), _bits(f))


def test_device_variant_checks_its_pointers(rc):
    import torch
    sc, rays = _c3(rc)
    lib = rc._ffi.load_library()
    st = rc.RaytracerSettings(samples_per_pixel=1).to_c()
    import ctypes as C
    with rc.CudaRenderer(sc) as r:
        d = torch.from_numpy(rays).cuda()
        out = torch.empty((len(rays) + 1, 3), dtype=torch.float32, device="cuda")
        host_out = np.empty((len(rays), 3), np.float32)
        torch.cuda.synchronize()
        assert lib.rtcuda_radiance_device(r._scene, C.byref(st), d.data_ptr(), 0, 0, out.data_ptr()) == 0   # count 0: nothing to do
        status = lib.rtcuda_radiance_device(r._scene, C.byref(st), d.data_ptr(), 4, 0, host_out.ctypes.data)
        assert status == INVALID_ARGUMENT and b"not device memory" in lib.rtcuda_last_error()
        status = lib.rtcuda_radiance_device(r._scene, C.byref(st), rays.ctypes.data, 4, 0, out.data_ptr())
        assert status == INVALID_ARGUMENT and b"not device memory" in lib.rtcuda_last_error()
        status = lib.rtcuda_radiance_device(r._scene, C.byref(st), d.data_ptr() + 8, 4, 0, out.data_ptr())
        assert status == INVALID_ARGUMENT and b"16-byte aligned" in lib.rtcuda_last_error()
