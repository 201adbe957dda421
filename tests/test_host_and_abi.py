"""CPU-side checks: the C-ABI library loads and exports every symbol include/rtcuda.h declares (no compute
calls without a GPU), ctypes mirrors match the compiled struct sizes, scene importers, host vocabulary."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_scene


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "rtcuda.h")).read()
    return sorted(set(re.findall(r"RTCUDA_API\s+[\w\s\*]+?\b(rtcuda_\w+)\s*\(", hdr)))


def test_header_declares_the_binding_surface(rc):
    assert declared_symbols() == sorted(rc._ffi.EXPORTED_SYMBOLS)


def test_library_exports_every_declared_symbol(rc):
    path = rc._ffi.LIB_PATH
    assert os.path.exists(path), "libraytracing_cuda.so is not built: run __graft_entry__.build()"
    lib = C.CDLL(path)
    for sym in declared_symbols():
        assert hasattr(lib, sym), sym


def test_abi_struct_sizes_match_ctypes(rc):
    lib = rc._ffi.load_library()   # raises on version / size mismatch
    sizes = (C.c_uint32 * 32)()
    n = lib.rtcuda_abi_struct_sizes(sizes, 32)
    assert n == len(rc._ffi.ABI_STRUCTS)
    assert lib.rtcuda_abi_version() == rc._ffi.ABI_VERSION


def test_no_cpu_fallback_without_device(rc):
    """Without a GPU the backend must fail loudly (NO_DEVICE), never render on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(rc._ffi.RtCudaError, match="NO_DEVICE"):
        rc.render(rc.test_scenes.sphere_scene(), rc.RaytracerSettings(outputs=rc.AovFlags.NORMALS))


def test_missing_library_fails_loudly(rc, tmp_path):
    with pytest.raises(rc._ffi.RtCudaError, match="no CPU fallback"):
        rc._ffi.load_library(str(tmp_path / "libraytracing_cuda.so"))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "opencl-raytracing_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".h", ".cu", ".cuh", ".cpp")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle_py" not in src and "liboracle" not in src and "hostsim" not in src.replace("tests/hostsim", ""), f


def test_default_settings_match_reference(rc):
    s = rc.RaytracerSettings()   # renderer/mod.rs:100-117
    assert (s.max_ray_depth, s.accumulate_bounces, s.light_sample_count, s.samples_per_pixel, s.seed) == (8, True, 4, 32, None)
    assert s.sampler.kind == "independent" and s.outputs == rc.AovFlags.BEAUTY
    assert int(rc.AovFlags.FIRST_HIT_AOVS) == 2 | 4 | 8 | 16


def test_gltf_fixture_facts():
    cb = load_scene("cb")
    assert (cb.camera.raster_width, cb.camera.raster_height) == (1066, 600)   # (600 * 1.7777778) as usize
    assert cb.triangle_count() == 12 and len(cb.instances) == 6 and len(cb.lights) == 1
    assert cb.lights[0].b == (1.0, 1.0, 1.0)   # emissive_factor only; emissive_strength ignored (scene.rs:411)
    bun = load_scene("cbbunny_area_light_transforms", 1920, 1080)
    assert bun.triangle_count() == 28588 and (bun.camera.raster_width, bun.camera.raster_height) == (1920, 1080)
    tex = load_scene("cb_texture")
    assert tex.triangle_count() == 972 and tex.images[0].shape == (461, 530, 3)
    assert tex.textures[0].filter == 2 and tex.textures[0].wrap == 0   # trilinear / repeat


def test_camera_matrices_are_consistent(rc):
    cam = rc.test_scenes.sphere_scene().camera
    ident = cam.raster_to_camera.forward.astype(np.float64) @ cam.raster_to_camera.inverse.astype(np.float64)
    assert np.allclose(ident, np.eye(4), atol=1e-4)
    # raster centre looks down -z towards the sphere
    p = cam.raster_to_camera.apply_point([200.0, 200.0, 0.0])
    assert abs(p[0]) < 1e-4 and abs(p[1]) < 1e-4


def test_scene_desc_round_trip(rc):
    sc = load_scene("cbbunny_area_light_transforms")
    h = sc.to_desc()
    d = h.desc
    assert d.tri_count == 28588 and d.instance_count == 7 and d.light_count == 1
    assert d.shapes[d.lights[0].shape].area_light == 0
    # own_arrays: every mesh points at its own numpy arrays, nothing is concatenated, same counts
    o = sc.to_desc(own_arrays=True)
    assert o.desc.tri_count == 0 and o.desc.vertex_count == 0 and o.geometry_bytes == h.geometry_bytes
    for i, bp in enumerate(sc.shapes):
        sh, ref = o.desc.shapes[i], d.shapes[i]
        assert (sh.vertex_count, sh.tri_count) == (ref.vertex_count, ref.tri_count) and bool(sh.vertices) and bool(sh.tris)
        assert np.array_equal(np.ctypeslib.as_array(sh.tris, shape=(sh.tri_count * 3,)), np.asarray(bp.shape.tris, dtype=np.uint32).ravel())
        assert bool(sh.normals) == (ref.normal_offset != rc._ffi.NONE) and bool(sh.uvs) == (ref.uv_offset != rc._ffi.NONE)


def test_tile_owner_map(rc):
    m = rc.multi_gpu.tile_owner_map(200, 130, 3)
    assert m.shape == (130, 200) and m[0, 0] == 0 and m[0, 64] == 1 and m[0, 128] == 2 and m[64, 0] == (4 % 3)


def test_synthetic_mesh_generator(rc):
    m = rc.test_scenes.procedural_sphere_mesh(64, 32)
    assert m.vertices.shape == (65 * 33, 3) and m.tris.shape[0] == 2 * 64 * 32 - 2 * 64
    r = np.linalg.norm(m.vertices, axis=1)
    assert r.min() > 0.44 and r.max() < 0.56
    assert np.allclose(np.linalg.norm(m.normals, axis=1), 1.0, atol=1e-4)
    m2 = rc.test_scenes.procedural_sphere_mesh(64, 32)
    assert np.array_equal(m.vertices, m2.vertices)


def test_exr_round_trip(rc, tmp_path):
    """the driver's EXR files: channel names of crates/cli/src/main.rs:398-467, sorted, f32, bit-exact round trip"""
    rng = np.random.default_rng(1)
    out = rc.RenderOutput.allocate(37, 23, rc.AovFlags.BEAUTY | rc.AovFlags.NORMALS | rc.AovFlags.UV_COORDS | rc.AovFlags.MIP_LEVEL)
    for plane in ("beauty", "normals", "uv", "mip_level"):
        getattr(out, plane)[...] = rng.standard_normal(getattr(out, plane).shape).astype(np.float32)
    ch = rc.exr.channels_of_render_output(out, rc.AovFlags.BEAUTY | rc.AovFlags.NORMALS | rc.AovFlags.UV_COORDS | rc.AovFlags.MIP_LEVEL)
    assert sorted(ch) == ["B", "G", "Mip Level", "Normal.X", "Normal.Y", "Normal.Z", "R", "U", "V"]
    path = str(tmp_path / "a.exr")
    rc.exr.write_exr(path, ch)
    back, w, h = rc.exr.read_exr(path)
    assert (w, h) == (37, 23) and list(back) == sorted(ch)
    for k in ch:
        assert np.array_equal(back[k], ch[k])
    import cv2   # an independent reader agrees on the RGB planes
    os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")
    img = cv2.imread(path, cv2.IMREAD_UNCHANGED)
    if img is not None:
        assert np.array_equal(img[..., 2], ch["R"]) and np.array_equal(img[..., 0], ch["B"])


def test_flip_and_mse_metrics(rc):
    rng = np.random.default_rng(0)
    a = rng.random((48, 64, 3))
    assert rc.imagecmp.flip(a, a, hdr=False) == 0.0
    assert rc.imagecmp.mse_maxdiff(a, a) == (0.0, 0.0)
    b = np.clip(a + 0.02 * rng.standard_normal(a.shape), 0, 1)
    c = np.clip(a + 0.2 * rng.standard_normal(a.shape), 0, 1)
    fb, fc = rc.imagecmp.flip(a, b, hdr=False), rc.imagecmp.flip(a, c, hdr=False)
    assert 0.0 < fb < fc <= 1.0
    black, white = np.zeros((32, 32, 3)), np.ones((32, 32, 3))
    assert rc.imagecmp.flip(black, white, hdr=False) > 0.9     # the largest possible achromatic error maps close to 1


def test_cli_argument_surface(rc, capsys):
    """flag surface of crates/cli/src/main.rs:20-107 (+ raster override); list-scenes prints the builtin names as JSON"""
    from raytracing_cuda import cli
    assert cli.main(["list-scenes"]) == 0
    import json
    names = json.loads(capsys.readouterr().out)
    assert names[:4] == ["sphere", "cube", "cube_orthographic", "checkered_plane"]
    a = cli.build_parser().parse_args(["--scene-name", "sphere", "-s", "4", "-d", "5", "-l", "2", "--sampler", "stratified", "-o", "x.exr",
                                       "full", "--aov", "n,u", "--no-beauty"])
    assert (a.spp, a.ray_depth, a.light_samples, a.sampler, a.aov, a.no_beauty) == (4, 5, 2, "stratified", "n,u", True)
    p = cli.build_parser().parse_args(["--scene-name", "cube", "pixel", "10", "20", "3", "1"])
    assert (p.x, p.y, p.sample_count, p.sample_offset) == (10, 20, 3, 1)
    assert cli.main([]) == 1 and cli.main(["--scene-name", "cube", "-t", "4", "full"]) == 1
    m = cli.backend_settings_from_args(cli.build_parser().parse_args(["--scene-name", "cube", "--devices", "0,2,3", "--tile-size", "16", "full"]))
    assert (m.num_devices, list(m.device_ids)[:3], m.tile_size) == (3, [0, 2, 3], 16)
    one = cli.backend_settings_from_args(cli.build_parser().parse_args(["--scene-name", "cube", "--gpu", "1", "full"]))
    assert (one.num_devices, one.device_id) == (0, 1)


def test_partition_helpers():
    """multi-GPU host logic: every pixel has one owner at any tile size; sample ranges tile [0, spp) without gaps"""
    import raytracing_cuda as rc
    for tile in (64, 16, 8):
        own = rc.multi_gpu.tile_owner_map(200, 136, 3, tile=tile)
        assert own.shape == (136, 200) and set(np.unique(own)) == {0, 1, 2}
        assert (own[:tile, :tile] == 0).all() and own[0, tile] == 1
    for spp, world in ((256, 8), (5, 8), (7, 2), (1, 1)):
        rs = [rc.multi_gpu.sample_range_for_rank(spp, r, world) for r in range(world)]
        assert rs[0][0] == 0 and rs[-1][1] == spp and all(a[1] == b[0] for a, b in zip(rs, rs[1:]))
        assert max(h - l for l, h in rs) - min(h - l for l, h in rs) <= 1


def test_nonfinite_warnings_follow_the_reference():
    """lib.rs:813-854: raster order, channel names, 'NaN' / 'infty', first 10 then the total"""
    from raytracing_cuda.backend import warn_nonfinite
    img = np.zeros((4, 5, 3), dtype=np.float32)
    assert warn_nonfinite(img, log=lambda m: None) == 0
    img[0, 3, 1] = np.nan
    img[2, 1, 0] = np.inf
    img[2, 1, 2] = -np.inf
    img[3, :, :] = np.nan
    msgs = []
    assert warn_nonfinite(img, log=msgs.append) == 18
    assert msgs[0] == "G component of (3, 0) is NaN" and msgs[1] == "R component of (1, 2) is infty" and msgs[2] == "B component of (1, 2) is infty"
    assert len(msgs) == 11 and msgs[-1] == "encountered 18 NaN and infty values in radiance buffer"


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the oracle port on the host cores; no GPU involved): one JSON line with the keys the driver reads"""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C2", "--cpu-spp", "1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Msamples/s" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("C2")


def _bench_module(monkeypatch):
    import importlib.util
    import sys
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)   # restored after the test (bench.py sets it)
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_dump_outputs_whole_or_sampled(tmp_path, monkeypatch):
    """bench.py --dump-outputs: whole planes while they fit DUMP_BYTES, else every plane at the same fixed sample of pixels"""
    import torch
    bench = _bench_module(monkeypatch)
    planes = {"beauty": torch.rand(48, 64, 3), "debug_depth": torch.rand(48, 64, 1)}
    bench.dump_outputs(str(tmp_path / "whole"), planes)
    assert sorted(os.listdir(tmp_path / "whole")) == ["beauty.npy", "debug_depth.npy"]
    for name, t in planes.items():
        assert np.array_equal(np.load(tmp_path / "whole" / f"{name}.npy"), t.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    monkeypatch.setattr(bench, "DUMP_SAMPLE_PIXELS", 100)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), planes)
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 100 and (np.diff(idx) > 0).all()
    assert np.array_equal(idx, np.load(tmp_path / "b" / "pixel_index.npy"))
    for name, t in planes.items():
        a = np.load(tmp_path / "a" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy().reshape(48 * 64, -1)[idx.astype(np.int64)])


def test_bench_rejects_zero_steps():
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=60)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_bench_dumps_the_frame_of_the_timed_steps(rc, tmp_path, monkeypatch):
    """bench.py --steps K --dump-outputs DIR: K timed steps (and K end-to-end calls), and DIR/beauty.npy is the frame the
    renderer returns for the same workload"""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C2", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2 and len(d["e2e"]["breakdown"]) == 2
    assert sorted(os.listdir(tmp_path)) == ["beauty.npy"]
    sc, st = _bench_module(monkeypatch).load_workload("C2")
    with rc.CudaRenderer(sc) as r:
        frame = r.render(st).beauty
    assert np.array_equal(np.load(tmp_path / "beauty.npy"), frame)
    assert d["config"]["workload"].startswith("C2")


def test_integration_patch_applies(tmp_path):
    """integration/reference.patch is a real diff against the reference tree: it applies cleanly to copies of the files it
    names (only where /root/reference exists: the GPU box does not have it), and the Rust crate only calls entry points and
    constants that include/rtcuda.h declares"""
    import re
    import shutil
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    patch = os.path.join(root, "integration", "reference.patch")
    text = open(patch).read()
    files = re.findall(r"^\+\+\+ b/(\S+)", text, flags=re.M)
    assert len(files) == 6 and "crates/cli/src/main.rs" in files and "visual-testing/src/rttest/runner.py" in files
    header = open(os.path.join(root, "include", "rtcuda.h")).read()
    rust = open(os.path.join(root, "integration", "crates", "raytracing-cuda", "src", "lib.rs")).read()
    for name in set(re.findall(r"ffi::(rtcuda_\w+|RTCUDA_\w+)", rust)):
        base = re.sub(r"^rtcuda_(\w+?_kind|image_format|status)_(RTCUDA_\w+)$", r"\2", name)   # bindgen's name for a C enum constant
        assert re.search(r"\b" + re.escape(base) + r"\b", header), f"{name} is not in rtcuda.h"
    if not os.path.isdir("/root/reference"):
        pytest.skip("reference tree absent")
    for f in files:
        dst = tmp_path / f
        dst.parent.mkdir(parents=True, exist_ok=True)
        shutil.copy(os.path.join("/root/reference", f), dst)
        os.chmod(dst, 0o644)
    r = subprocess.run(["patch", "-p1", "--dry-run", "-i", patch], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_ply_importer_variants(rc):
    """Mesh::from_ply_reader conventions (mesh.rs:25-170): (s, t) texture coordinates as well as (u, v), CRLF headers, extra
    elements and trailing face properties in binary files"""
    import struct
    hdr = ("ply\r\nformat binary_little_endian 1.0\r\nelement vertex 4\r\nproperty float x\r\nproperty float y\r\nproperty float z\r\n"
           "property float s\r\nproperty float t\r\nelement edge 2\r\nproperty int a\r\nproperty int b\r\n"
           "element face 2\r\nproperty list uchar int vertex_indices\r\nproperty uchar flags\r\nend_header\r\n").encode()
    verts = [(0, 0, 0, 0, 0), (1, 0, 0, 1, 0), (1, 1, 0, 1, 1), (0, 1, 0, 0, 1)]
    body = b"".join(struct.pack("<5f", *v) for v in verts) + struct.pack("<4i", 0, 1, 1, 2)
    body += struct.pack("<B3iB", 3, 0, 1, 2, 9) + struct.pack("<B3iB", 3, 0, 2, 3, 9)
    m = rc.scene.mesh_from_ply_bytes(hdr + body)
    assert m.vertices.shape == (4, 3) and m.tris.tolist() == [[0, 1, 2], [0, 2, 3]]
    assert m.uvs is not None and m.uvs.tolist() == [[0, 0], [1, 0], [1, 1], [0, 1]]
    bad = rc.test_scenes.cube_scene()
    bad.shapes[0].shape.normals = bad.shapes[0].shape.normals[:-1]
    with pytest.raises(ValueError, match="one entry per vertex"):
        bad.to_desc(own_arrays=True)
