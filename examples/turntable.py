#!/usr/bin/env python
"""Animation through rtcuda_scene_update: the camera orbits the scene and one instance spins, and every frame is an update of
the uploaded scene (the BVH is refitted on the device, nothing is uploaded again) plus a progressive accumulation from a zeroed
device plane.

  python examples/turntable.py [scene.npz] [frames] [spp]    # prints update_ms and render_ms per frame
"""
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import torch                      # only used as the owner of the device plane
import raytracing_cuda as rc
from scene_motion import moved, trs

scene = rc.Scene.load_npz(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests/golden/scenes/cbbunny_area_light_transforms.npz"))
frames = int(sys.argv[2]) if len(sys.argv) > 2 else 24
spp = int(sys.argv[3]) if len(sys.argv) > 3 else 16
spinning = max(range(len(scene.instances)), key=lambda i: len(getattr(scene.shapes[scene.instances[i][0]].shape, "tris", ())))
settings = rc.RaytracerSettings(samples_per_pixel=spp)
with rc.CudaRenderer(scene) as r:
    plane = torch.zeros((r.height, r.width, 3), dtype=torch.float32, device="cuda:0")
    for f in range(frames):
        a = 2 * math.pi * f / frames
        frame = moved(scene, instances={spinning: trs(angle=2 * a)},
                      camera=trs(angle=0.25 * math.sin(a)))   # the camera swings about the world z axis
        r.update(frame)
        update_ms = r.stats()["update_ms"]
        plane.zero_()
        torch.cuda.synchronize()
        r.render_samples_accumulate_device(settings, 0, spp, plane.data_ptr())
        image = (plane / spp).cpu().numpy()           # <- what a viewer would show
        print(f"frame {f:3d}  update {update_ms:6.3f} ms ({['none', 'camera / lights', 'refit', 'rebuild'][r.stats()['bvh_last_update']]})"
              f"  render {r.stats()['render_ms']:7.1f} ms  mean {image.mean():.6f}")
