"""Seeded points of interest on a context's DEM square, for the labels tests and tools/annotate_bench.py.

    summits(h, count, seed)   -> (count, 3) float64 lat, lon, ele: vertices that are the highest of their 9 x 9
                                 neighbourhood, drawn at random (seeded) from all such vertices of the square
"""
import numpy as np


def vertex_latlon(h, i, j):
    """lat, lon of mosaic vertex (i east, j north) of context h: the inverse of horizonator_move()'s cell coordinates."""
    d = h.context.dems
    cpd = float(d.cells_per_deg)
    lon = d.origin_dem_lon_lat[0] + (np.asarray(i, np.float64) + d.origin_dem_cellij[0]) / cpd
    lat = d.origin_dem_lon_lat[1] + (np.asarray(j, np.float64) + d.origin_dem_cellij[1]) / cpd
    return lat, lon


def summits(h, count, seed=0, mosaic=None):
    from scipy.ndimage import maximum_filter
    z = h.mosaic() if mosaic is None else mosaic
    peak = (z == maximum_filter(z, size=9, mode="nearest")) & (z > 0)
    j, i = np.nonzero(peak)
    pick = np.random.default_rng(seed).choice(len(j), size=min(count, len(j)), replace=False)
    lat, lon = vertex_latlon(h, i[pick], j[pick])
    return np.stack([lat, lon, z[j[pick], i[pick]].astype(np.float64)], axis=1)
