"""The scene-update refit (rt_build.h refit_prims_body / refit_nodes_body, api.cu update_scene) run by the CPU harness: a refit
with unchanged transforms reproduces the built tree, and build(A) -> update to B -> render gives the frame of build(B) -> render,
bit for bit, on every plane, after a refit and after a rebuild."""
import math

import numpy as np
import pytest

from conftest import load_scene
from scene_motion import about, moved, trs


def _bits(a):
    """float32 words as u32, with -0.0 read as +0.0 (the only difference min / max of equal boxes can make: fminf(-0, +0)
    may return either, and the refit unions a leaf's boxes in slot order where the build merged them in tree order)"""
    b = np.ascontiguousarray(a).view(np.uint32)
    return np.where(b == 0x80000000, 0, b)


def sphere_in_box(rc, w=64, h=64):
    """the builtin Cornell box (point light) with a diffuse sphere instance"""
    b = rc.test_scenes.cornell_box()
    tex = b.add_constant_texture((0.5, 0.6, 0.7, 1.0))
    mat = b.add_material(rc.Material(rc._ffi.MATERIAL_DIFFUSE, albedo=tex))
    b.add_shape_at_position(rc.test_scenes.Sphere((0, 0, 0), 0.4), mat, (0.2, -0.1, 0.6))
    sc = b.build()
    sc.camera = rc.Camera.lookat_camera_perspective((0.0, 4.4, 0.4), (0, 0, 0.75), (0, 0, 1), False, math.radians(37.8), w, h)
    return sc


def _scene(rc, name):
    return sphere_in_box(rc) if name == "sphere" else load_scene(name, 96, 54)


def _settings(rc):
    A = rc.AovFlags
    return rc.RaytracerSettings(outputs=A.BEAUTY | A.NORMALS | A.ALBEDO | A.UV_COORDS | A.MIP_LEVEL | A.DEBUG_IDS | A.DEBUG_DEPTH,
                                samples_per_pixel=2)


PLANES = ("beauty", "normals", "albedo", "uv", "mip_level", "debug_ids", "debug_depth")


def _assert_same_frame(a, b):
    for p in PLANES:
        assert np.array_equal(getattr(a, p), getattr(b, p)), p


@pytest.mark.parametrize("name", ["cb", "cbbunny_area_light_transforms", "sphere"])
def test_refit_with_unchanged_transforms_reproduces_the_tree(rc, hostsim, name):
    nodes_b, nodes_r, prims_b, prims_r, (sah_b, sah_r) = hostsim.refit_identity(_scene(rc, name))
    assert len(nodes_b) and len(prims_b)
    assert np.array_equal(_bits(prims_b), _bits(prims_r))
    assert np.array_equal(_bits(nodes_b), _bits(nodes_r))
    assert sah_b == sah_r and sah_b > 1.0


MOTIONS = {
    # (scene, scene -> moved copy)
    "translated_instance": ("cbbunny_area_light_transforms", lambda s: moved(s, instances={5: trs((0.15, -0.1, 0.05))})),
    "rotated_nonuniform_scaled_instance": ("cbbunny_area_light_transforms",
                                           lambda s: moved(s, instances={5: about((0.0, 0.0, 0.3), trs((0, 0, 0), (0.3, 0.2, 1.0), 0.7, (1.2, 0.7, 0.9)))})),
    "moved_sphere": ("sphere", lambda s: moved(s, instances={5: trs((-0.3, 0.2, 0.1))})),
    "moved_area_light": ("cbbunny_area_light_transforms", lambda s: moved(s, instances={6: trs((0.2, 0.1, -0.05))}, lights={0: trs((0.2, 0.1, -0.05))})),
    "moved_point_light": ("sphere", lambda s: moved(s, lights={0: trs((0.3, -0.2, -0.3))})),
    "moved_camera": ("cb", lambda s: moved(s, camera=trs((0.2, -0.3, 0.1), (0, 0, 1), 0.08))),
}


@pytest.mark.parametrize("motion", sorted(MOTIONS))
def test_refit_renders_the_frame_of_a_fresh_build(rc, hostsim, motion):
    name, move = MOTIONS[motion]
    a = _scene(rc, name)
    b = move(a)
    st = _settings(rc)
    fresh, _ = hostsim.render(b, st)
    upd, _, (last, sah) = hostsim.update_render(a, b, st)
    assert last == 2 and sah > 1.0
    _assert_same_frame(upd, fresh)
    if motion != "moved_camera" and "light" not in motion:   # the instance moved on screen
        assert not np.array_equal(upd.debug_ids, hostsim.render(a, st)[0].debug_ids)


@pytest.mark.parametrize("motion", ["translated_instance", "moved_sphere", "moved_area_light"])
def test_rebuild_renders_the_frame_of_a_fresh_build(rc, hostsim, motion):
    name, move = MOTIONS[motion]
    a = _scene(rc, name)
    b = move(a)
    st = _settings(rc)
    fresh, fs = hostsim.render(b, st)
    upd, us, (last, sah) = hostsim.update_render(a, b, st, max_growth=0.0)   # the rule then always asks for the rebuild
    assert last == 3 and sah > 1.0
    _assert_same_frame(upd, fresh)
    assert (us["nodes_fetched"], us["prims_fetched"]) == (fs["nodes_fetched"], fs["prims_fetched"])   # the same tree as a fresh build
