"""rtcuda_radiance's bodies on the CPU (hostsim_radiance in tests/hostsim/hostsim.cpp: prep, k_trace's walk, the live list,
raygen_rays and the wavefront's extend / shade / shadow / gather / resolve) against the reference, the oracle's ray_radiance per
ray and sample over the ray's normalised range (oracle_radiance in oracle/rays.cpp).

Measured (2^12 seeded rays per scene, tests/ray_sets.py, 8 spp, depth 5; per-ray relative difference = max over channels over the
mean of the reference, over the rays that carry light in either; "diverged" = share of those beyond 1 %):

    scene                           rays   p50      p99      diverged
    cb                              2715   2.0e-8   2.4e-7   0
    cbbunny_area_light_transforms   2770   1.7e-7   4.6e-6   1.1e-3 (3 rays)
    reused mesh                     2735   4.0e-8   3.1e-6   0
    environment scene               4056   0        0        0
    rough-metal box                 2840   1.2e-8   7.4e-6   0
    sphere scene (no light)         every ray exactly 0 in both

The prepared rays agree bit for bit. The gates below are tightened to these figures, well inside parity.py's default beauty
gates (2e-5 / 2e-3 / 5e-3) and SPECULAR_GATES; the rough-metal box keeps more room for lobe flips than the diffuse scenes."""
import numpy as np
import pytest

from conftest import instanced_bunnies_scene, load_scene
from parity import beauty_close
from radiance_rays import emitter_rays, outgoing_rays
from ray_sets import query_rays

SETTINGS = dict(samples_per_pixel=8, max_ray_depth=5)
DIFFUSE_GATES = dict(p50=1e-6, p99=5e-5, diverged=2e-3)
SPECULAR_HARNESS_GATES = dict(p50=1e-6, p99=1e-4, diverged=1e-2)

SCENES = {
    # name: (scene factory, seed, gates)
    "cb": (lambda rc: load_scene("cb", 64, 64), 1, DIFFUSE_GATES),
    "sphere_scene": (lambda rc: rc.test_scenes.sphere_scene(), 2, None),   # no light: every ray returns exactly 0
    "cbbunny_area_light_transforms": (lambda rc: load_scene("cbbunny_area_light_transforms", 64, 64), 3, DIFFUSE_GATES),
    "reused_mesh": (lambda rc: instanced_bunnies_scene(), 4, DIFFUSE_GATES),
    "environment": (lambda rc: rc.test_scenes.environment_lighting_scene(rc.test_scenes.synthetic_environment_map()), 5, DIFFUSE_GATES),
    "rough_metal": (lambda rc: rc.test_scenes.rough_metal_scene(), 6, SPECULAR_HARNESS_GATES),
}


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_radiance_matches_the_reference(rc, hostsim, oracle, name):
    make, seed, gates = SCENES[name]
    sc = make(rc)
    rays, invalid = query_rays(sc, n=1 << 12, seed=seed)
    st = rc.RaytracerSettings(**SETTINGS)
    got, prep = hostsim.radiance(sc, st, rays)
    ref, ref_prep = oracle.radiance(sc, st, rays)
    assert np.array_equal(_bits(prep), _bits(ref_prep))   # the normalisation is the same float arithmetic
    if gates is None:
        assert not got.any() and not ref.any()
        return
    rep = {}
    ok = beauty_close(got, ref, report=rep, **gates)
    print(name, rep)
    assert rep["pixels"] > len(rays) // 4
    assert ok, rep
    assert not got[invalid].any() and not ref[invalid].any()


def test_depth_0_returns_the_emitter_radiance_of_the_closest_hit(rc, hostsim):
    """max_ray_depth = 0: a ray whose closest hit is an area emitter returns exactly its radiance (2 spp: the mean of two equal
    samples is exact); every other ray returns 0"""
    sc = load_scene("cbbunny_area_light_transforms", 64, 64)
    rays = np.concatenate([emitter_rays(sc, 1024, seed=7), query_rays(sc, n=1024, seed=8)[0]])
    got, prep = hostsim.radiance(sc, rc.RaytracerSettings(samples_per_pixel=2, max_ray_depth=0), rays)
    _, ids, _, _ = hostsim.trace_rays(sc, prep)
    expect = np.zeros_like(got)
    on_light = np.zeros(len(rays), bool)
    for i, g in enumerate(ids[:, 0]):
        if g != 0xFFFFFFFF:
            light = sc.shapes[sc.instances[g][0]].area_light
            if light is not None:
                expect[i] = np.float32(sc.lights[light].b)
                on_light[i] = True
    assert on_light.sum() > 256
    assert np.array_equal(_bits(got), _bits(expect))


@pytest.mark.parametrize("environment", [False, True])
def test_invalid_rays_return_exactly_zero(rc, hostsim, oracle, environment):
    sc = rc.test_scenes.environment_lighting_scene(rc.test_scenes.synthetic_environment_map()) if environment else load_scene("cb", 64, 64)
    rays, invalid = query_rays(sc, n=1 << 12, seed=9)
    st = rc.RaytracerSettings(samples_per_pixel=2, max_ray_depth=3)
    got, _ = hostsim.radiance(sc, st, rays)
    ref, _ = oracle.radiance(sc, st, rays)
    assert invalid.sum() > 0
    assert np.array_equal(_bits(got[invalid]), np.zeros((invalid.sum(), 3), np.uint32))
    assert np.array_equal(_bits(ref[invalid]), np.zeros((invalid.sum(), 3), np.uint32))


def test_rays_leaving_the_scene_return_the_environment(rc, hostsim, oracle):
    sc = rc.test_scenes.environment_lighting_scene(rc.test_scenes.synthetic_environment_map())
    rays = outgoing_rays(sc, 2048, seed=10)
    st = rc.RaytracerSettings(samples_per_pixel=4, max_ray_depth=5)
    got, _ = hostsim.radiance(sc, st, rays)
    one, _ = oracle.radiance(sc, rc.RaytracerSettings(samples_per_pixel=1, max_ray_depth=0), rays)
    assert (one.max(axis=1) > 0).all()
    np.testing.assert_allclose(got, one, rtol=1e-6, atol=0)


def test_direction_length_does_not_matter(rc, hostsim):
    """directions x 2 and both bounds x 1/2 (exact in float) normalise to the same ray: bit-identical radiance"""
    sc = load_scene("cbbunny_area_light_transforms", 64, 64)
    rays, _ = query_rays(sc, n=1 << 11, seed=11)
    scaled = rays.copy()
    scaled[:, 4:7] *= 2
    scaled[:, [3, 7]] *= 0.5
    st = rc.RaytracerSettings(**SETTINGS)
    a, pa = hostsim.radiance(sc, st, rays)
    b, pb = hostsim.radiance(sc, st, scaled)
    assert np.array_equal(_bits(pa), _bits(pb)) and np.array_equal(_bits(a), _bits(b))


def test_batches_and_slices_give_the_same_bits(rc, hostsim):
    sc = load_scene("cbbunny_area_light_transforms", 64, 64)
    rays, _ = query_rays(sc, n=1 << 11, seed=12)
    st = rc.RaytracerSettings(**SETTINGS)
    full, _ = hostsim.radiance(sc, st, rays)
    small, _ = hostsim.radiance(sc, st, rays, capacity=1024)
    assert np.array_equal(_bits(full), _bits(small))
    a, b = 700, 1500
    part, _ = hostsim.radiance(sc, st, rays[a:b], stream_base=a)
    assert np.array_equal(_bits(full[a:b]), _bits(part))
    shifted, _ = hostsim.radiance(sc, st, rays[a:b], stream_base=a + 1)   # the key, not the position, selects the stream
    assert not np.array_equal(_bits(full[a:b]), _bits(shifted))
