"""Shared helpers of the test-suite: tolerances, comparisons, oracle glue."""

from __future__ import annotations

import numpy as np

RTOL = 1e-5  # north_star: fp32 state within 1e-5 relative


def rel_err(got, ref, scale=None):
    """|got - ref| / max(|ref|, 1)  (relative above 1, absolute below)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    s = np.maximum(np.abs(ref), 1.0) if scale is None else np.maximum(np.asarray(scale, dtype=np.float64), 1.0)
    return np.abs(got - ref) / s


def heading_err(got, ref):
    """Heading compared modulo 2*pi."""
    d = np.asarray(got, dtype=np.float64) - np.asarray(ref, dtype=np.float64)
    return np.abs((d + np.pi) % (2 * np.pi) - np.pi)


def assert_state_close(got: dict, ref: dict, mask=None, rtol=RTOL, what=""):
    """x, y, speed within rtol of max(|ref|,1); heading modulo 2 pi; vx, vy relative to max(|v|,1)."""
    m = slice(None) if mask is None else mask
    vscale = np.maximum(np.sqrt(np.asarray(ref["vx"], dtype=np.float64) ** 2 + np.asarray(ref["vy"], dtype=np.float64) ** 2), 1.0)
    worst = {}
    for k in ("x", "y", "speed"):
        worst[k] = float(np.max(rel_err(got[k], ref[k])[m], initial=0.0))
    worst["heading"] = float(np.max(heading_err(got["heading"], ref["heading"])[m], initial=0.0))
    for k in ("vx", "vy"):
        worst[k] = float(np.max(rel_err(got[k], ref[k], vscale)[m], initial=0.0))
    bad = {k: v for k, v in worst.items() if not v <= rtol}
    assert not bad, f"{what} state mismatch beyond {rtol}: {bad} (all: {worst})"
    return worst


def parking_like_objects():
    """Walls and obstacles the way ParkingLotGenerator builds them (map/generator/generate_parking_lot.py:122-205,354-385):
    Area polygons - a long wall, a block big enough to swallow a car, an L-shaped (concave) obstacle, a kerb stone smaller
    than a car - plus an open kerb line."""
    from tactics2d_b200.map import polygons_to_segments

    polys = [
        [(-30, 18), (30, 18), (30, 19), (-30, 19)],                          # wall
        [(-25, -20), (-5, -20), (-5, -4), (-25, -4)],                        # block: a car fits inside
        [(4, -18), (16, -18), (16, -6), (12, -6), (12, -14), (4, -14)],      # L shape: its notch is outside the polygon
        [(20.0, 5.0), (20.8, 5.0), (20.8, 5.4), (20.0, 5.4)],                # smaller than a car
    ]
    lines = [[(-30, -26), (0, -27), (30, -26)]]
    return polygons_to_segments(polys, lines)
