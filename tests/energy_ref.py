"""numpy statement of the encircled-energy contract of include/ort_b200.h (ort_spot_energy_dev): the distances d of the
kept rays of one set, the curve counts by searchsorted and the energy radii by sort -- what the device must equal bit for
bit."""
import math

import numpy as np


def distances(ex, ey, cy, metric):
    """d per ray; numpy evaluates these operations one by one, never contracted"""
    ex, ey = np.asarray(ex, dtype=np.float64), np.asarray(ey, dtype=np.float64)
    dy = ey - np.float64(cy)
    if metric == "circle":
        return np.sqrt(ex * ex + dy * dy)
    return np.maximum(np.abs(ex), np.abs(dy))


def rank_k(q, n):
    """1-based rank of the energy radius of fraction q over n kept rays"""
    return min(max(int(math.ceil(np.float64(q) * np.float64(n))), 1), n)


def energy(d, radii, fracs):
    """(counts int64 [R], radius float64 [Q]) of the distances d of one set's kept rays"""
    s = np.sort(np.asarray(d, dtype=np.float64))           # NaN last
    counts = np.searchsorted(s, np.asarray(radii, dtype=np.float64), side="right").astype(np.int64)
    n = len(s)
    radius = np.array([s[rank_k(q, n) - 1] if n else np.nan for q in fracs], dtype=np.float64)
    return counts, radius


def set_energy(ex, ey, mask, n_kept, mean_y, radii, fracs, metric="circle", center="centroid"):
    """one set: ex / ey full grid with mask (uint8, kept == 1) or compacted (mask None: the first n_kept entries)"""
    ex, ey = np.asarray(ex), np.asarray(ey)
    if mask is None:
        ex, ey = ex[:n_kept], ey[:n_kept]
    else:
        keep = np.asarray(mask) == 1
        ex, ey = ex[keep], ey[keep]
    cy = mean_y if center == "centroid" else 0.0
    return energy(distances(ex, ey, cy, metric), radii, fracs)
