"""Seeded query-ray sets and the comparison of two query results (the ray-query tests, CPU and GPU)."""
import itertools

import numpy as np

from parity import AOV_ATOL, AOV_RTOL, NONE_ID


def scene_bounds(scene):
    """world-space box of every instance (mesh vertices, sphere boxes) of a raytracing_cuda Scene"""
    lo, hi = np.full(3, np.inf), np.full(3, -np.inf)
    for shape_index, tf in scene.instances:
        shape = scene.shapes[shape_index].shape
        if hasattr(shape, "vertices"):
            pts = np.asarray(shape.vertices, np.float64)
        else:
            pts = np.asarray(shape.center, np.float64) + shape.radius * np.array(list(itertools.product((-1, 1), repeat=3)), np.float64)
        m = np.asarray(tf.forward, np.float64)
        p = pts @ m[:3, :3].T + m[:3, 3]
        lo, hi = np.minimum(lo, p.min(axis=0)), np.maximum(hi, p.max(axis=0))
    return lo, hi


def _unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def query_rays(scene, n=1 << 16, seed=0):
    """float32 [n, 8] packed rays over the scene's bounds, in five kinds (shuffled):
      inside      origins uniform in the bounds, uniform directions, [0, inf];
      outside     origins on a sphere around the bounds, aimed at points inside them, [0, inf];
      short       like `inside`, t_max uniform in [0, half the bounds' diagonal] (ends inside geometry or short of it);
      offset      like `inside`, t_min uniform in [0, half the diagonal];
      degenerate  zero direction, NaN components, t_min > t_max (1 % of the set; every one must miss)."""
    rng = np.random.default_rng(seed)
    lo, hi = scene_bounds(scene)
    ext = hi - lo
    diag = float(np.linalg.norm(ext))
    center = (lo + hi) / 2
    k = n // 100
    m = (n - k) // 4
    inside = lo + rng.random((3 * m, 3)) * ext
    d_in = _unit(rng.normal(size=(3 * m, 3)))
    o_out = center + _unit(rng.normal(size=(n - k - 3 * m, 3))) * diag
    d_out = lo + rng.random((len(o_out), 3)) * ext - o_out
    rays = np.zeros((n, 8), np.float64)
    rays[:3 * m, 0:3], rays[:3 * m, 4:7] = inside, d_in
    rays[:3 * m, 7] = np.inf
    rays[m:2 * m, 7] = rng.random(m) * diag / 2
    rays[2 * m:3 * m, 3] = rng.random(m) * diag / 2
    rays[3 * m:n - k, 0:3], rays[3 * m:n - k, 4:7] = o_out, d_out
    rays[3 * m:n - k, 7] = np.inf
    deg = rays[n - k:]
    deg[:, 0:3] = lo + rng.random((k, 3)) * ext
    deg[:, 4:7] = _unit(rng.normal(size=(k, 3)))
    deg[:, 7] = np.inf
    kind = np.arange(k) % 4
    deg[kind == 0, 4:7] = 0.0                                          # zero direction
    deg[kind == 1, rng.integers(0, 3, (kind == 1).sum())] = np.nan     # NaN origin component
    deg[kind == 2, 4 + rng.integers(0, 3, (kind == 2).sum())] = np.nan  # NaN direction component
    deg[kind == 3, 3], deg[kind == 3, 7] = 1.0, 0.5                    # t_min > t_max
    degenerate = np.zeros(n, bool)
    degenerate[n - k:] = True
    perm = rng.permutation(n)
    return np.ascontiguousarray(rays[perm].astype(np.float32)), degenerate[perm]


def compare(got, ref):
    """figures of a query result (t, ids [N, 2], barycentrics [N, 2], ...) against a reference: id agreement over the rays that
    hit in either, and the fraction of those rays whose t or barycentrics are outside the AOV tolerance of tests/parity.py
    (a ray whose ids disagree counts as an outlier)"""
    t, ids, uv = got[0], got[1], got[2]
    rt, rids, ruv = ref[0], ref[1], ref[2]
    hit = (ids[:, 0] != NONE_ID) | (rids[:, 0] != NONE_ID)
    same = (ids == rids).all(axis=1)
    both = hit & same & (ids[:, 0] != NONE_ID)

    def bad(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        with np.errstate(invalid="ignore"):   # misses: inf - inf (only rays that hit in both are looked at)
            x = ~(np.abs(a - b) <= AOV_ATOL + AOV_RTOL * np.abs(b))
        return x.any(axis=1) if x.ndim == 2 else x

    outliers = (hit & ~same) | (both & (bad(t, rt) | bad(uv, ruv)))
    n_hit = max(1, int(hit.sum()))
    return {"rays": len(t), "hit_rays": int(hit.sum()), "id_agreement": float(same[hit].mean()) if hit.any() else 1.0,
            "id_mismatches": int((hit & ~same).sum()), "outlier_frac": float(outliers.sum()) / n_hit}

