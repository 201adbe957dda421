"""Ray sets of the radiance tests (CPU and GPU): rays aimed at a scene's area emitter, rays leaving the scene, and jittered camera
rays built in numpy from the scene's own camera."""
import numpy as np

from ray_sets import scene_bounds


def emitter_rays(scene, n, seed=0):
    """float32 [n, 8]: origins uniform in the scene's bounds, aimed at uniform points on the triangles of its first area emitter"""
    rng = np.random.default_rng(seed)
    lo, hi = scene_bounds(scene)
    shape_index, tf = next((si, tf) for si, tf in scene.instances if scene.shapes[si].area_light is not None)
    mesh = scene.shapes[shape_index].shape
    v = np.asarray(mesh.vertices, np.float64)
    m = np.asarray(tf.forward, np.float64)
    tri = v[np.asarray(mesh.tris).reshape(-1, 3)] @ m[:3, :3].T + m[:3, 3]
    k = rng.integers(0, len(tri), n)
    a, b = rng.random(n), rng.random(n)
    flip = a + b > 1
    a[flip], b[flip] = 1 - a[flip], 1 - b[flip]
    target = tri[k, 0] + a[:, None] * (tri[k, 1] - tri[k, 0]) + b[:, None] * (tri[k, 2] - tri[k, 0])
    o = lo + rng.random((n, 3)) * (hi - lo)
    rays = np.zeros((n, 8), np.float32)
    rays[:, 0:3], rays[:, 4:7], rays[:, 7] = o, target - o, np.inf
    return rays


def outgoing_rays(scene, n, seed=0):
    """float32 [n, 8]: rays that start outside the scene's bounding sphere and point away from it (they hit nothing)"""
    rng = np.random.default_rng(seed)
    lo, hi = scene_bounds(scene)
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    rays = np.zeros((n, 8), np.float32)
    rays[:, 0:3] = (lo + hi) / 2 + u * 2 * np.linalg.norm(hi - lo)
    rays[:, 4:7], rays[:, 7] = u, np.inf
    return rays


def jittered_camera_rays(camera, per_pixel, seed=0):
    """float32 [H * W * per_pixel, 8]: pinhole camera rays through uniform points of each pixel (raster_to_camera, then
    camera_to_world), pixel-major, over the camera clip"""
    rng = np.random.default_rng(seed)
    W, H = camera.raster_width, camera.raster_height
    ys, xs = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
    xs = np.repeat(xs.ravel(), per_pixel) + rng.random(W * H * per_pixel)
    ys = np.repeat(ys.ravel(), per_pixel) + rng.random(W * H * per_pixel)
    raster = np.stack([xs, ys, np.zeros_like(xs), np.ones_like(xs)], axis=1)
    cp = raster @ np.asarray(camera.raster_to_camera.forward, np.float64).T
    cp = cp[:, :3] / cp[:, 3:]
    c2w = np.asarray(camera.camera_to_world.forward, np.float64)
    d = (cp / np.linalg.norm(cp, axis=1, keepdims=True)) @ c2w[:3, :3].T
    rays = np.zeros((len(d), 8), np.float32)
    rays[:, 0:3] = c2w[:3, 3] / c2w[3, 3]
    rays[:, 3], rays[:, 4:7], rays[:, 7] = camera.near_clip, d, camera.far_clip
    return rays
