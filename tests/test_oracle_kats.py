"""Pins the CPU oracle against every known-answer test the reference holds for the path (SURVEY §8c) and
against published vectors of the third-party generators it restates."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_scene


def fa(v):
    return (C.c_float * len(v))(*v)


def test_sphere_uv_off_center(oracle):
    # crates/raytracing-cpu/src/geometry.rs:342-373
    out = (C.c_float * 6)()
    hit = oracle.lib().oracle_ray_sphere(fa([0, 3, 0]), 1.0, fa([0, 0, 0]), fa([0, 1, 0]), 0.0, 1e30, out)
    assert hit == 1
    t, u, v, nx, ny, nz = list(out)
    assert abs(t - 2.0) < 1e-5
    assert abs(nx) < 1e-5 and abs(ny + 1.0) < 1e-5 and abs(nz) < 1e-5
    assert abs(u - 0.75) < 1e-4 and abs(v - 0.5) < 1e-4


def test_make_orthonormal_basis(oracle):
    # crates/raytracing-cpu/src/geometry.rs:22-47
    z = np.array([0.262, -0.151, 0.370], dtype=np.float32)
    z = z / np.linalg.norm(z)
    x, y = (C.c_float * 3)(), (C.c_float * 3)()
    oracle.lib().oracle_make_orthonormal_basis(fa(z.tolist()), x, y)
    x, y = np.array(list(x)), np.array(list(y))
    assert abs(np.dot(x, y)) < 1e-6 and abs(np.dot(x, z)) < 1e-6 and abs(np.dot(y, z)) < 1e-6
    assert abs(np.linalg.norm(x) - 1) < 1e-6 and abs(np.linalg.norm(y) - 1) < 1e-6
    assert np.allclose(np.cross(x, y), z, atol=1e-6)


@pytest.mark.parametrize("length", [1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 97])
def test_permute_is_permutation(oracle, length):
    # crates/raytracing-cpu/src/sample.rs:256-275
    seen = sorted(oracle.lib().oracle_permute(i, length, 0x12345678) for i in range(length))
    assert seen == list(range(length))


def test_pcg32_published_vectors(oracle):
    # pcg32-demo (pcg-c-basic): pcg32_srandom_r(42, 54) -> first six outputs; rand_pcg::Lcg64Xsh32::new(42, 54)
    # is the same initialisation (state = (state + inc) * M + inc)
    out = (C.c_uint32 * 6)()
    oracle.lib().oracle_pcg32_stream(42, 54, 6, out)
    assert list(out) == [0xa15c02b7, 0x7b47f409, 0xba1d3330, 0x83d2f293, 0xbfa4784b, 0xcbed606e]


def test_fxhash_structure(oracle):
    # rustc-hash 2.x: hash = (hash + x) * K, finish = rotate_left(26). No vector ships with the reference
    # (parity unpinned, SURVEY appendix C); this pins the restated arithmetic itself.
    K = 0xf1357aea2e62a9c5
    M = (1 << 64) - 1
    rotl = lambda v, r: ((v << r) | (v >> (64 - r))) & M
    assert oracle.lib().oracle_fxhash_u64(42) == rotl((42 * K) & M, 26)
    h = 0
    for v in (3, 5, 7):
        h = ((h + v) * K) & M
    assert oracle.lib().oracle_fxhash_u32x3(3, 5, 7) == rotl(h, 26)


def test_fxhasher_constants_against_compiled_rustc_hash(oracle):
    """Evidence for the two constants the reference's tests do not pin (SURVEY appendix C: multiplier K and the rotate of
    `finish`): Rust extension modules that link rustc-hash 2.x (tokenizers 0.22.2, tiktoken 0.12.0, outlines_core 0.2.14) carry K
    as a 64-bit immediate, and the `rol r64, 26` of `finish()` follows it. rustc-hash 2.0.0 rotated by 20; 1.x used another K.
    The machine code that follows each K in those modules is stored in tests/golden/rustc_hash_k_windows.npz
    (tests/golden/make_rustc_hash_windows.py). The oracle's FxHasher must use the K and the rotate found there."""
    K = bytes.fromhex("c5a9622eea7a35f1")           # 0xf1357aea2e62a9c5, little endian
    z = np.load(os.path.join(GOLDEN, "rustc_hash_k_windows.npz"))
    assert {s.split(":")[0].split()[0] for s in z["sources"]} == {"tiktoken", "tokenizers", "outlines_core"}
    rol26 = rol20 = with_k = 0
    for row in z["windows"]:
        assert bytes(row[:8]) == K
        with_k += 1
        window = bytes(row[8:])
        for j in range(len(window) - 3):   # rol r64, imm8 = REX.W(48/49) C1 /0 ib
            if window[j] in (0x48, 0x49) and window[j + 1] == 0xC1 and 0xC0 <= window[j + 2] <= 0xC7:
                rol26 += window[j + 3] == 26
                rol20 += window[j + 3] == 20
    assert rol26 >= 5 and rol20 == 0, (with_k, rol26, rol20)
    k, m = int.from_bytes(K, "little"), (1 << 64) - 1
    for x in (1, 42, 0xdeadbeef, m):
        h = (x * k) & m
        assert oracle.lib().oracle_fxhash_u64(x) == ((h << 26) | (h >> 38)) & m, x


def test_uniform_f32_is_24bit(oracle, rc):
    st = rc.RaytracerSettings().to_c()
    out = (C.c_float * 64)()
    oracle.lib().oracle_sampler_stream(C.byref(st), 3, 4, 5, 64, out)
    v = np.array(list(out), dtype=np.float64)
    assert ((v >= 0) & (v < 1)).all()
    assert np.allclose(v * 2 ** 24, np.round(v * 2 ** 24))


def test_range_u32_in_range(oracle):
    for s in range(50):
        assert 0 <= oracle.lib().oracle_range_u32(s, 7, 0, 2) < 2
        assert 10 <= oracle.lib().oracle_range_u32(s, 9, 10, 13) < 13


def test_triangle_inclusive_edges(oracle):
    # geometry.rs:301-340: u, v, u+v bounds are inclusive; t bounds are inclusive; no back-face culling
    tri = fa([0, 0, 0, 1, 0, 0, 0, 1, 0])
    out = (C.c_float * 3)()
    assert oracle.lib().oracle_ray_triangle(tri, fa([0.0, 0.0, 1.0]), fa([0, 0, -1]), 0.0, 10.0, out) == 1      # vertex
    assert oracle.lib().oracle_ray_triangle(tri, fa([0.5, 0.5, 1.0]), fa([0, 0, -1]), 0.0, 10.0, out) == 1      # hypotenuse
    assert oracle.lib().oracle_ray_triangle(tri, fa([0.25, 0.25, -1.0]), fa([0, 0, 1]), 0.0, 10.0, out) == 1    # back face
    assert abs(out[0] - 1.0) < 1e-6
    assert oracle.lib().oracle_ray_triangle(tri, fa([0.25, 0.25, 1.0]), fa([0, 0, -1]), 0.0, 1.0, out) == 1     # t == t_max
    assert oracle.lib().oracle_ray_triangle(tri, fa([0.25, 0.25, 1.0]), fa([0, 0, -1]), 0.0, 0.99, out) == 0
    assert oracle.lib().oracle_ray_triangle(tri, fa([0.25, 0.25, 1.0]), fa([1, 0, 0]), 0.0, 10.0, out) == 0     # parallel


@pytest.mark.parametrize("name,w,h", [("cb", 96, 96), ("cbbunny_area_light_transforms", 96, 54)])
def test_bvh_equals_brute_force(oracle, rc, name, w, h):
    """self-consistency: the BVH2 closest hit is the brute-force closest hit (BVH-independent answers)"""
    sc = load_scene(name, w, h)
    A = rc.AovFlags
    st = rc.RaytracerSettings(outputs=A.NORMALS | A.UV_COORDS | A.DEBUG_IDS | A.DEBUG_DEPTH)
    a, _ = oracle.render(sc, st)
    b, _ = oracle.render(sc, st, brute_force=True)
    assert np.array_equal(a.debug_depth, b.debug_depth)
    assert (a.debug_ids == b.debug_ids).all(axis=-1).mean() > 0.999   # equal-t ties may pick another primitive
    assert np.abs(a.normals - b.normals).max() < 1e-5 or (a.debug_ids == b.debug_ids).all(axis=-1).mean() < 1.0


def test_sphere_scene_c1_facts(oracle, rc):
    """BASELINE config C1: builtin `sphere`, normals only, 400x400 (test_scenes/mod.rs:150-176, 605-623)"""
    sc = rc.test_scenes.sphere_scene()
    st = rc.test_scenes.all_test_scenes()[0].settings_func()
    st.samples_per_pixel, st.max_ray_depth = 4, 5
    out, stats = oracle.render(sc, st)
    assert out.beauty is None and out.normals.shape == (400, 400, 3)
    assert stats["aov_rays"] == 160000 and stats["primary_rays"] == 0
    n = out.normals
    hit = np.abs(n).sum(axis=2) > 0
    assert np.allclose(np.linalg.norm(n[hit], axis=1), 1.0, atol=1e-5)
    # the sphere (r=1 at distance 3, yfov 45deg) covers a centred disc; the centre normal faces the camera (+z)
    assert n[200, 200, 2] > 0.9999 and not hit[0, 0]
    assert abs(hit.mean() - np.pi * (400 * np.tan(np.arcsin(1 / 3)) / (2 * np.tan(np.radians(22.5)))) ** 2 / 160000) < 5e-3


def test_white_furnace_energy(oracle, rc):
    """a diffuse sphere of albedo a under a constant environment L reflects at most L: every pixel <= L,
    and the directly visible background equals L"""
    env = np.full((4, 8, 3), 0.5, dtype=np.float32)
    sc = rc.test_scenes.environment_lighting_scene(env)
    sc.camera = rc.Camera.lookat_camera_perspective((0, 0, 0), (0, 1, 0), (0, 0, 1), False, 0.66, 48, 48)
    out, _ = oracle.render(sc, rc.RaytracerSettings(samples_per_pixel=16))
    assert out.beauty.max() <= 0.5 + 1e-5
    assert abs(out.beauty[0, 0, 0] - 0.5) < 1e-6
