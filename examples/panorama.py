#!/usr/bin/env python
"""An equirectangular panorama, a camera the scene format does not have, through CudaRenderer.radiance: one ray per pixel from a
point inside the Cornell box (longitude across, latitude down, z up), the path tracer's radiance along each, written to EXR.
CudaRenderer.surfaces on the same rays gives the G-buffer the panorama camera lacks: the shading normal and the albedo at each
pixel's first hit, written next to it as <out>_normal.exr and <out>_albedo.exr (denoiser guides, for instance).

  python examples/panorama.py [out.exr] [width] [spp]    # default panorama.exr, 1024 x 512, 64 spp
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_cuda as rc
from raytracing_cuda import exr

out_path = sys.argv[1] if len(sys.argv) > 1 else "panorama.exr"
W = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
spp = int(sys.argv[3]) if len(sys.argv) > 3 else 64
H = W // 2
scene = rc.Scene.load_npz(os.path.join(ROOT, "tests/golden/scenes/cbbunny_area_light_transforms.npz"))
eye = (0.0, 0.0, 0.75)                              # inside the box (x, y in [-1, 1], z in [0, 1.5])
phi = (np.arange(W) + 0.5) / W * 2 * np.pi - np.pi   # longitude
theta = (np.arange(H) + 0.5) / H * np.pi            # angle from +z
th, ph = np.meshgrid(theta, phi, indexing="ij")
d = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)], axis=-1).reshape(-1, 3)
rays = rc.make_rays(eye, d)
with rc.CudaRenderer(scene) as r:
    radiance = r.radiance(rays, rc.RaytracerSettings(samples_per_pixel=spp)).reshape(H, W, 3)
    surf = r.surfaces(rays)
stem = os.path.splitext(out_path)[0]
planes = {out_path: radiance, stem + "_normal.exr": surf.normal.reshape(H, W, 3), stem + "_albedo.exr": surf.albedo.reshape(H, W, 3)}
for path, img in planes.items():
    exr.write_exr(path, {c: np.ascontiguousarray(img[..., k], np.float32) for k, c in enumerate("RGB")})
print(f"{out_path}: {W}x{H}, {spp} spp, mean radiance {radiance.mean():.5f}; "
      f"{stem}_normal.exr, {stem}_albedo.exr: {int((surf.instance != rc._ffi.NONE).sum())} of {W * H} rays hit")
