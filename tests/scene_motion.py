"""Scene motions for the scene-update tests (rtcuda_scene_update): copies of a scene with moved instances, lights or camera.
The copies share the shapes, materials and textures of the original, so they have its topology."""
import copy

import numpy as np

import raytracing_cuda as rc
from raytracing_cuda.geometry import Transform


def trs(translate=(0.0, 0.0, 0.0), axis=(0.0, 0.0, 1.0), angle=0.0, scale=(1.0, 1.0, 1.0)):
    """T * R(axis, angle) * S with its inverse (float64, rounded once)"""
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    R = np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)
    M = np.eye(4)
    M[:3, :3] = R @ np.diag(np.asarray(scale, dtype=np.float64))
    M[:3, 3] = translate
    f = M.astype(np.float32)
    return Transform(f, np.linalg.inv(f.astype(np.float64)).astype(np.float32))


def about(center, m):
    """the motion m applied about `center` instead of the origin"""
    c = np.asarray(center, dtype=np.float64)
    return trs(-c).compose(m).compose(trs(c))


def moved(scene, instances=None, camera=None, lights=None):
    """A copy of `scene` in which instance i is followed by the Transform instances[i], the camera by `camera`, and light k
    by the Transform lights[k] (position / direction, light_to_world)."""
    out = copy.copy(scene)
    out.instances = list(scene.instances)
    for i, m in (instances or {}).items():
        si, tf = out.instances[i]
        out.instances[i] = (si, tf.compose(m))
    if camera is not None:
        c = copy.copy(scene.camera)
        c.camera_to_world = scene.camera.camera_to_world.compose(camera)
        c.world_to_raster = camera.invert().compose(scene.camera.world_to_raster)
        out.camera = c
    out.lights = [copy.copy(l) for l in scene.lights]
    for k, m in (lights or {}).items():
        l = out.lights[k]
        if l.kind == rc._ffi.LIGHT_DIFFUSE_AREA:
            ltw = np.eye(4, dtype=np.float32) if l.light_to_world is None else np.asarray(l.light_to_world, dtype=np.float32).reshape(4, 4)
            l.light_to_world = (m.forward.astype(np.float64) @ ltw.astype(np.float64)).astype(np.float32)
        elif l.kind == rc._ffi.LIGHT_POINT:
            l.a = tuple(float(x) for x in (m.forward.astype(np.float64) @ np.array([*l.a, 1.0]))[:3].astype(np.float32))
        else:
            l.a = tuple(float(x) for x in (m.forward[:3, :3].astype(np.float64) @ np.array(l.a)).astype(np.float32))
    return out


def scatter(scene, seed, extent):
    """every instance thrown `extent` away in a random direction and spun: a motion no refit serves well"""
    rng = np.random.default_rng(seed)
    moves = {i: trs(rng.normal(size=3) * extent, rng.normal(size=3), float(rng.uniform(0, 6.28))) for i in range(len(scene.instances))}
    return moved(scene, instances=moves)
