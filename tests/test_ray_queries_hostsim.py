"""The ray-query bodies of the CUDA library (rt_query.h: the traversal k_trace runs, then the k_trace_finish body) on the CPU,
against the reference: the oracle's traverse_bvh per ray over the ray's own [t_min, t_max] (tests/hostsim/oracle_query.cpp),
brute force on the small scenes, over the oracle's BVH2 on the bunny scenes.

Measured (2^16 seeded rays per scene, tests/ray_sets.py): with Moller-Trumbore on cb, the sphere scene,
cbbunny_area_light_transforms and the reused-mesh scene, every id agrees on every ray that hits in either result and no t / u / v
is outside the AOV tolerance of tests/parity.py (1e-4 + 2e-5 relative): the winning triangle is re-tested in object space the
reference's way. With the watertight test 3 of 44,829 hit rays (6.7e-5) are outside it, all ids agreeing. The gates below are
those figures (watertight: 10x), tighter than parity.py's 0.9999 / 2e-3."""
import pytest

from conftest import instanced_bunnies_scene, load_scene
from ray_sets import compare, query_rays

NONE = 0xFFFFFFFF

SCENES = {
    # name: (scene factory, oracle in brute-force mode, seed)
    "cb": (lambda rc: load_scene("cb", 64, 64), True, 1),
    "sphere_scene": (lambda rc: rc.test_scenes.sphere_scene(), True, 2),
    "cbbunny_area_light_transforms": (lambda rc: load_scene("cbbunny_area_light_transforms", 64, 64), False, 3),
    "reused_mesh": (lambda rc: instanced_bunnies_scene(), False, 4),
}


@pytest.fixture(scope="module")
def hq():
    import hostsim_query_py
    hostsim_query_py.build()
    return hostsim_query_py


def _check(got, ref, degenerate, outlier_gate):
    rep = compare(got, ref)
    assert rep["hit_rays"] > rep["rays"] // 3, rep
    assert rep["id_mismatches"] == 0, rep
    assert rep["outlier_frac"] <= outlier_gate, rep
    for res in (got, ref):
        ids, occ = res[1], res[3]
        assert (ids[degenerate] == NONE).all() and (occ[degenerate] == 0).all()
        assert (occ == (ids[:, 0] != NONE)).all()
    return rep


@pytest.mark.parametrize("name", sorted(SCENES))
def test_queries_match_the_reference(rc, hq, name):
    make, brute, seed = SCENES[name]
    sc = make(rc)
    rays, degenerate = query_rays(sc, seed=seed)
    _check(hq.trace_rays(sc, rays), hq.oracle_trace_rays(sc, rays, brute_force=brute), degenerate, 0.0)


def test_watertight_queries_match_the_reference(rc, hq, monkeypatch):
    monkeypatch.setenv("HOSTSIM_WATERTIGHT", "1")
    sc = load_scene("cbbunny_area_light_transforms", 64, 64)
    rays, degenerate = query_rays(sc, seed=5)
    _check(hq.trace_rays(sc, rays), hq.oracle_trace_rays(sc, rays), degenerate, 6.7e-4)


def test_misses_and_ranges(rc, hq):
    """a miss is (inf, NONE, NONE, 0, 0); t_max below the hit's t misses, t_min = t_max = t hits (inclusive bounds)"""
    import numpy as np
    sc = load_scene("cb", 64, 64)
    rays = rc.make_rays([[0.0, 0.0, 0.75]] * 4, [[0.0, 0.0, -1.0], [0.0, 0.0, -1.0], [0.0, 0.0, -1.0], [0.0, 0.0, 0.0]])
    t, ids, uv, occ = hq.trace_rays(sc, rays[:1])
    assert ids[0, 0] != NONE and t[0] > 0
    rays[1, 7] = np.nextafter(t[0], np.float32(0))
    rays[2, 3] = rays[2, 7] = t[0]
    t2, ids2, uv2, occ2 = hq.trace_rays(sc, rays)
    assert t2[1] == np.inf and (ids2[1] == NONE).all() and (uv2[1] == 0).all() and occ2[1] == 0
    assert t2[2] == t[0] and (ids2[2] == ids[0]).all() and occ2[2] == 1
    assert t2[3] == np.inf and (ids2[3] == NONE).all() and occ2[3] == 0
