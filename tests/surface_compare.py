"""Comparison of two surface-query results (SURFACE_DTYPE records, rtcuda_trace_surfaces) for the surface tests, CPU and GPU."""
import numpy as np

from parity import AOV_ATOL, AOV_RTOL, NONE_ID, PLANE_ATOL

FLOAT_FIELDS = ("t", "point", "normal", "uv")


def miss_record():
    """the record of a miss or an invalid ray: t = +inf, zeros, NONE ids / material / light"""
    from raytracing_cuda.backend import SURFACE_DTYPE
    r = np.zeros((), SURFACE_DTYPE)
    r["t"] = np.inf
    for f in ("geom_id", "prim_id", "material", "light"):
        r[f] = NONE_ID
    return r


def is_miss_record(rec):
    """bool [N]: the record is the miss record bit for bit"""
    return (rec.view(np.uint32).reshape(len(rec), 16) == miss_record()[None].view(np.uint32)).all(axis=1)


def bits(rec):
    return np.ascontiguousarray(rec).view(np.uint8)


def compare_surfaces(got, ref):
    """figures of surface records against a reference, over the rays that hit in either: id agreement; the fraction of those rays
    that are outliers (ids disagree, or t / point / normal / uv outside the AOV tolerance of tests/parity.py, or albedo outside
    PLANE_ATOL["albedo"]); and the rays whose ids agree but whose material or light differ. NaN matches NaN: the reference's
    sphere uv is NaN where rounding puts |cos phi| above 1 (points next to the y = 0 meridian), and HitInfo::uv reproduces it."""
    ids, rids = np.stack([got["geom_id"], got["prim_id"]], 1), np.stack([ref["geom_id"], ref["prim_id"]], 1)
    hit = (ids[:, 0] != NONE_ID) | (rids[:, 0] != NONE_ID)
    same = (ids == rids).all(axis=1)
    both = hit & same & (ids[:, 0] != NONE_ID)

    def bad(a, b, atol, rtol):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        with np.errstate(invalid="ignore"):   # misses: inf - inf (only rays that hit in both are looked at)
            x = ~((np.abs(a - b) <= atol + rtol * np.abs(b)) | (np.isnan(a) & np.isnan(b)))
        return x.reshape(len(x), -1).any(axis=1)

    field_bad = {f: both & bad(got[f], ref[f], AOV_ATOL, AOV_RTOL) for f in FLOAT_FIELDS}
    field_bad["albedo"] = both & bad(got["albedo"], ref["albedo"], PLANE_ATOL["albedo"], 0.0)
    outliers = (hit & ~same) | np.logical_or.reduce(list(field_bad.values()))
    n_hit = max(1, int(hit.sum()))
    return {"rays": len(got), "hit_rays": int(hit.sum()), "id_agreement": float(same[hit].mean()) if hit.any() else 1.0,
            "id_mismatches": int((hit & ~same).sum()), "outlier_frac": float(outliers.sum()) / n_hit,
            "outliers": {f: int(v.sum()) for f, v in field_bad.items()},
            "material_light_mismatches": int((both & ((got["material"] != ref["material"]) | (got["light"] != ref["light"]))).sum())}
