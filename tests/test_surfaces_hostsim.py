"""The surface-query body of the CUDA library (rt_query.h: the traversal k_trace runs, then the k_surface_finish body) on the CPU,
against the reference: the oracle's traverse_bvh per ray over the ray's own [t_min, t_max] and the winner's HitInfo (point,
normal, uv, material, light) with get_albedo at a zero footprint (oracle_trace_surfaces in oracle/rays.cpp), brute force on
the small scenes, over the oracle's BVH2 on the bunny scenes. The harness's surface and closest-hit queries
(tests/hostsim/hostsim.cpp) build the same scene the same way, so their t and ids can be compared bit for bit.

Measured (2^16 seeded rays per scene, tests/ray_sets.py): on cb, the sphere scene, cbbunny_area_light_transforms (C3), the
reused-mesh scene (normals through rotations and non-uniform scales), the texture zoo (every texture kind, format, wrap mode and
filter feeding the albedo), the rough-metal box, and C3 with the watertight test, every id agrees on every ray that hits in
either result, no t / point / normal / uv is outside the AOV tolerance of tests/parity.py (1e-4 + 2e-5 relative), no albedo is
outside PLANE_ATOL["albedo"], material and light agree on every hit, and invalid rays give the miss record bit for bit. The
harness's t and ids are rtcuda_trace_rays's bit for bit. The gates below are those figures: no outlier, except 2e-4 (about 10
rays) with the watertight test, whose re-test the ray-query tests have seen flip a few rays."""
import numpy as np
import pytest

from conftest import instanced_bunnies_scene, load_scene, texture_zoo_scene
from ray_sets import query_rays
from surface_compare import compare_surfaces, is_miss_record

SCENES = {
    # name: (scene factory, oracle in brute-force mode, seed)
    "cb": (lambda rc: load_scene("cb", 64, 64), True, 1),
    "sphere_scene": (lambda rc: rc.test_scenes.sphere_scene(), True, 2),
    "cbbunny_area_light_transforms": (lambda rc: load_scene("cbbunny_area_light_transforms", 64, 64), False, 3),
    "reused_mesh": (lambda rc: instanced_bunnies_scene(), False, 4),
    "texture_zoo": (lambda rc: texture_zoo_scene(), True, 5),
    "rough_metal": (lambda rc: rc.test_scenes.rough_metal_scene(), True, 6),
}


def _check(hostsim, oracle, sc, rays, invalid, brute, outlier_gate):
    got = hostsim.trace_surfaces(sc, rays)
    ref = oracle.trace_surfaces(sc, rays, brute_force=brute)
    rep = compare_surfaces(got, ref)
    print(rep)
    assert rep["hit_rays"] > rep["rays"] // 3, rep
    assert rep["id_mismatches"] == 0, rep
    assert rep["outlier_frac"] <= outlier_gate, rep
    assert rep["material_light_mismatches"] == 0, rep
    assert is_miss_record(got[invalid]).all() and is_miss_record(ref[invalid]).all()
    # t and the ids are those of the closest-hit query, bit for bit
    t, ids, _, _ = hostsim.trace_rays(sc, rays)
    assert np.array_equal(got["t"].view(np.uint32), t.view(np.uint32))
    assert np.array_equal(got["geom_id"], ids[:, 0]) and np.array_equal(got["prim_id"], ids[:, 1])
    # a miss of the closest-hit query is the miss record
    assert np.array_equal(is_miss_record(got), ids[:, 0] == 0xFFFFFFFF)
    return got


@pytest.mark.parametrize("name", sorted(SCENES))
def test_surfaces_match_the_reference(rc, hostsim, oracle, name):
    make, brute, seed = SCENES[name]
    sc = make(rc)
    rays, invalid = query_rays(sc, seed=seed)
    _check(hostsim, oracle, sc, rays, invalid, brute, 0.0)


def test_watertight_surfaces_match_the_reference(rc, hostsim, oracle, monkeypatch):
    monkeypatch.setenv("HOSTSIM_WATERTIGHT", "1")
    sc = load_scene("cbbunny_area_light_transforms", 64, 64)
    rays, invalid = query_rays(sc, seed=7)
    _check(hostsim, oracle, sc, rays, invalid, False, 2e-4)


def test_surface_fields(rc, hostsim):
    """what a caller relies on without a reference: unit normals, the point on the ray at t for triangles, the instance's
    material and light"""
    sc = load_scene("cbbunny_area_light_transforms", 64, 64)
    rays, _ = query_rays(sc, seed=8)
    got = hostsim.trace_surfaces(sc, rays)
    hit = got["geom_id"] != 0xFFFFFFFF
    np.testing.assert_allclose(np.linalg.norm(got["normal"][hit].astype(np.float64), axis=1), 1.0, atol=1e-6)
    on_ray = rays[hit, 0:3].astype(np.float64) + rays[hit, 4:7].astype(np.float64) * got["t"][hit, None]
    np.testing.assert_allclose(got["point"][hit], on_ray, atol=1e-5)
    for g in np.unique(got["geom_id"][hit]):
        shape = sc.shapes[sc.instances[g][0]]
        light = shape.area_light if shape.area_light is not None else 0xFFFFFFFF
        sel = got["geom_id"] == g
        assert (got["material"][sel] == shape.material).all() and (got["light"][sel] == light).all()
