"""The map tile compiler (tactics2d_b200/csrc/t2d_tile.h), compiled for the host by tests/hostsim/tilesim.cpp: the blob
K1 and the lidar kernel read, checked against float64 geometry without a GPU.  K1 trusts these properties and checks none
of them: a fine clearance byte that is too high, or a segment missing from a cell list, loses a collision silently."""

import ctypes as C
import functools
import os
import subprocess

import numpy as np
import pytest

from tactics2d_b200._lib import MapTileC
from tests.util import parking_like_objects

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLEAR_QUANT = 0.125
T2D_E_INVALID = -1

HEADER = np.dtype([
    ("n_seg", "<i4"), ("gx", "<i4"), ("gy", "<i4"), ("n_items", "<i4"),
    ("x0", "<f4"), ("y0", "<f4"), ("inv_cell", "<f4"), ("cell", "<f4"),
    ("off_seg", "<u4"), ("off_cell", "<u4"), ("off_items", "<u4"), ("total_bytes", "<u4"),
    ("unused", "<u4"), ("fine", "<i4"), ("off_dcell", "<u4"), ("off_ditems", "<u4"), ("dil", "<f4"), ("n_ditems", "<i4"),
    ("off_objfirst", "<u4"), ("n_poly", "<i4"), ("off_poly", "<u4"), ("off_pbox", "<u4"), ("off_fine", "<u4"),
    ("smem_bytes", "<u4"), ("bxmin", "<f4"), ("bxmax", "<f4"), ("bymin", "<f4"), ("bymax", "<f4"), ("has_bounds", "<i4"),
    ("pad", "<u4", (3,)),
])
assert HEADER.itemsize == 128


@pytest.fixture(scope="session")
def tilesim():
    """g++ build of the tile compiler header - test harness only."""
    src = os.path.join(ROOT, "tests", "hostsim", "tilesim.cpp")
    out = os.path.join(ROOT, "tests", "hostsim", "_tilesim.so")
    deps = [src, os.path.join(ROOT, "tactics2d_b200", "csrc", "t2d_tile.h"), os.path.join(ROOT, "include", "t2d_b200.h")]
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", out, src])
    lib = C.CDLL(out)
    lib.ts_compile.restype = C.c_int
    lib.ts_compile.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                               C.c_void_p, C.c_char_p, C.c_int]
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def _arrays(seg, poly_start=None, bounds=None):
    seg = None if seg is None else np.ascontiguousarray(np.asarray(seg, np.float32).reshape(-1, 4))
    ps = None if poly_start is None else np.ascontiguousarray(np.asarray(poly_start, np.int32))
    b = None if bounds is None else np.ascontiguousarray(np.asarray(bounds, np.float32))
    return seg, ps, b


def compile_tiles(lib, tiles, cell_size, reach, table=False):
    """tiles: [(segments, poly_start, bounds, n_seg, n_poly)] (n_seg / n_poly None: taken from the arrays).  Returns
    (code, error text, blob bytes, offsets or None)."""
    rows = (MapTileC * len(tiles))()
    keep = []   # the arrays the rows point into stay alive until the call returns
    for i, (seg, ps, b, n_seg, n_poly) in enumerate(tiles):
        seg, ps, b = _arrays(seg, ps, b)
        keep.append((seg, ps, b))
        rows[i].segments, rows[i].poly_start, rows[i].bounds = _ptr(seg), _ptr(ps), _ptr(b)
        rows[i].n_seg = (0 if seg is None else len(seg)) if n_seg is None else n_seg
        rows[i].n_poly = (0 if ps is None else len(ps) - 1) if n_poly is None else n_poly
    offsets = np.zeros(len(tiles), np.uint32) if table else None
    err = C.create_string_buffer(512)
    n = C.c_int64(0)
    cap = 1 << 22
    while True:
        out = np.zeros(cap, np.uint8)
        code = lib.ts_compile(rows, len(tiles), cell_size, reach, _ptr(out), cap, C.byref(n), _ptr(offsets), err, len(err))
        if code != 0 or n.value <= cap:
            return code, err.value.decode(), out[:n.value].copy() if code == 0 else None, offsets
        cap = n.value


def compile_one(lib, seg, poly_start=None, bounds=None, cell_size=0.0, reach=0.0, n_seg=None, n_poly=None):
    return compile_tiles(lib, [(seg, poly_start, bounds, n_seg, n_poly)], cell_size, reach)[:3]


# ------------------------------------------------------------------------------------------------------------- inputs
def _input_names():
    from tactics2d_b200.map import list_tiles

    tiles = list_tiles()
    return sorted(tiles + [t + "_areas" for t in tiles if t.startswith(("inD", "rounD"))]
                  + ["parking", "grid_walls", "one_segment", "zero_length"])


INPUT_NAMES = _input_names()


@functools.lru_cache(maxsize=None)
def tile_input(name):
    """(segments, poly_start or None, bounds or None) of one named input, built on first use."""
    from tactics2d_b200 import synthetic
    from tactics2d_b200.map import load_areas, load_collidable_segments, polygons_to_segments

    if name == "parking":
        return (*parking_like_objects(), (-40.0, 40.0, -40.0, 40.0))
    if name == "grid_walls":
        return synthetic.grid_wall_segments(), None, (-8.0, 208.0, -8.0, 208.0)
    if name == "one_segment":
        return [[1.0, 2.0, 7.5, -3.0]], None, None
    if name == "zero_length":
        return [[4.0, 4.0, 4.0, 4.0]], None, (0.0, 10.0, 0.0, 10.0)
    tile = name[:-len("_areas")] if name.endswith("_areas") else name
    seg, bounds = load_collidable_segments(tile)
    if tile == name:
        return seg, None, bounds
    # an Area with holes goes in as its exterior: the ring check wants every edge of an object to chain to the next,
    # which the exterior and hole rings placed back to back do not
    seg, ps = polygons_to_segments([a.outer if a.inners else a for a in load_areas(tile)])
    return seg, ps, bounds


PARAMS = [(cell, reach) for cell in (0.0, 3.0) for reach in (0.0, 2.9, 40.0)]


# ------------------------------------------------------------------------------------------------------------- geometry
def _point_seg_dist(px, py, s):
    """float64 distance of points to segments (x1, y1, x2, y2) in the last axis; shapes broadcast."""
    x1, y1, x2, y2 = s[..., 0], s[..., 1], s[..., 2], s[..., 3]
    dx, dy, ux, uy = x2 - x1, y2 - y1, px - x1, py - y1
    dd = dx * dx + dy * dy
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.clip(np.where(dd > 0.0, (ux * dx + uy * dy) / dd, 0.0), 0.0, 1.0)
    return np.hypot(ux - t * dx, uy - t * dy)


def _point_box_dist(px, py, b):
    ox = np.maximum(np.maximum(b[..., 0] - px, px - b[..., 1]), 0.0)
    oy = np.maximum(np.maximum(b[..., 2] - py, py - b[..., 3]), 0.0)
    return np.hypot(ox, oy)


def seg_box_dist(s, b):
    """float64 distance of segments s (x1, y1, x2, y2) to closed boxes b (x0, x1, y0, y1), shapes broadcast: 0 where they
    meet (separating axes: x, y and the segment's normal), else the least distance of an endpoint to the box or of a box
    corner to the segment."""
    x1, y1, x2, y2 = s[..., 0], s[..., 1], s[..., 2], s[..., 3]
    bx0, bx1, by0, by1 = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    nx, ny = y1 - y2, x2 - x1
    meet = ((np.minimum(x1, x2) <= bx1) & (np.maximum(x1, x2) >= bx0) & (np.minimum(y1, y2) <= by1) & (np.maximum(y1, y2) >= by0)
            & (np.abs((0.5 * (bx0 + bx1) - x1) * nx + (0.5 * (by0 + by1) - y1) * ny)
               <= 0.5 * (bx1 - bx0) * np.abs(nx) + 0.5 * (by1 - by0) * np.abs(ny)))
    d = np.minimum(_point_box_dist(x1, y1, b), _point_box_dist(x2, y2, b))
    for cx, cy in ((bx0, by0), (bx0, by1), (bx1, by0), (bx1, by1)):
        d = np.minimum(d, _point_seg_dist(cx, cy, s))
    return np.where(meet, 0.0, d)


def _points_in_rings(px, py, seg, poly_start):
    """[P] bool: the point lies inside one of the rings (even-odd over each ring's edges)."""
    inside = np.zeros(len(px), bool)
    for p in range(len(poly_start) - 1):
        e = seg[poly_start[p]:poly_start[p + 1]]
        x1, y1, x2, y2 = (e[:, k][None, :] for k in range(4))
        with np.errstate(divide="ignore", invalid="ignore"):
            cross = ((y1 > py[:, None]) != (y2 > py[:, None])) & (px[:, None] < (x2 - x1) * (py[:, None] - y1) / (y2 - y1) + x1)
        inside |= (cross.sum(1) & 1).astype(bool)
    return inside


def _cell_boxes(x0, y0, size, nx, ny):
    ix, iy = np.meshgrid(np.arange(nx), np.arange(ny))          # row-major: index iy * nx + ix
    bx0 = x0 + ix.ravel() * size
    by0 = y0 + iy.ravel() * size
    return np.stack([bx0, bx0 + size, by0, by0 + size], 1)


def _box_gaps(x0, y0, size, nx, ny, seg):
    """Gaps between the bounding boxes of the segments and the columns [nx, S] / rows [ny, S] of a grid: the hypotenuse
    of a column's and a row's gap is a lower bound of the distance between a segment and that cell, a cheap cull before
    the exact distance."""
    def gap(lo, s0, s1):
        return np.maximum(np.maximum(s0[None, :] - (lo + size)[:, None], lo[:, None] - s1[None, :]), 0.0)
    return (gap(x0 + np.arange(nx) * size, np.minimum(seg[:, 0], seg[:, 2]), np.maximum(seg[:, 0], seg[:, 2])),
            gap(y0 + np.arange(ny) * size, np.minimum(seg[:, 1], seg[:, 3]), np.maximum(seg[:, 1], seg[:, 3])))


# ------------------------------------------------------------------------------------------------------------- checks
def _section(blob, off, dtype, count):
    return np.frombuffer(blob[off:off + np.dtype(dtype).itemsize * count].tobytes(), dtype)


def _check_lists(blob, off_start, off_items, h, seg, reach):
    """Cell lists: cell_start never decreases and ends at the item count, every list is strictly ascending, and lists
    every segment within `reach` of the cell's closed box."""
    gx, gy = int(h["gx"]), int(h["gy"])
    n_cells = gx * gy
    start = _section(blob, off_start, "<u4", n_cells + 1).astype(np.int64)
    n_items = int(start[-1])
    items = _section(blob, off_items, "<u2", n_items).astype(np.int64)
    assert start[0] == 0 and np.all(np.diff(start) >= 0)
    cell_of = np.repeat(np.arange(n_cells), np.diff(start))
    same_cell = cell_of[1:] == cell_of[:-1]
    assert np.all(items[1:][same_cell] > items[:-1][same_cell]), "a cell list is not strictly ascending"
    assert np.all(items < len(seg))
    listed = np.zeros((n_cells, len(seg)), bool)
    listed[cell_of, items] = True
    x0, y0, cell = float(h["x0"]), float(h["y0"]), float(h["cell"])
    gap_x, gap_y = _box_gaps(x0, y0, cell, gx, gy, seg)
    near = np.hypot(gap_x[None, :, :], gap_y[:, None, :]).reshape(n_cells, len(seg)) <= reach
    ci, si = np.nonzero(near & ~listed)
    d = seg_box_dist(seg[si], _cell_boxes(x0, y0, cell, gx, gy)[ci])
    missing = d <= reach
    assert not missing.any(), f"segment {si[missing][0]} missing from cell {ci[missing][0]}"
    return n_items


def _check_fine(blob, h, seg, poly_start):
    """Fine clearance field: byte x CLEAR_QUANT is at most the distance from the fine cell's box to the static geometry
    (0 when the cell centre lies inside a ring)."""
    k = int(h["fine"])
    nx, ny = int(h["gx"]) * k, int(h["gy"]) * k
    assert h["off_fine"] + nx * ny <= h["total_bytes"]
    bound = _section(blob, int(h["off_fine"]), np.uint8, nx * ny).astype(np.float64).reshape(ny, nx) * CLEAR_QUANT
    x0, y0, fc = float(h["x0"]), float(h["y0"]), float(h["cell"]) / k
    if poly_start is not None and len(poly_start) > 1:
        iy, ix = np.nonzero(bound > 0)          # a zero byte claims nothing
        inside = _points_in_rings(x0 + (ix + 0.5) * fc, y0 + (iy + 0.5) * fc, seg, poly_start)
        assert not inside.any(), f"fine cell ({ix[inside][0]}, {iy[inside][0]}) lies inside a ring but has clearance"
    # only a segment whose box comes closer than the claimed clearance can contradict it: gather those pairs row by row
    gap_x, gap_y = _box_gaps(x0, y0, fc, nx, ny, seg)
    cells, segs = [], []
    for iy in range(ny):
        r = bound[iy]
        sel = np.nonzero(gap_y[iy] < r.max())[0]
        ix, j = np.nonzero(np.hypot(gap_x[:, sel], gap_y[iy, sel][None, :]) < r[:, None])
        cells.append(iy * nx + ix)
        segs.append(sel[j])
    ci, si = np.concatenate(cells), np.concatenate(segs)
    d = seg_box_dist(seg[si], _cell_boxes(x0, y0, fc, nx, ny)[ci])
    bad = d < bound.ravel()[ci]
    assert not bad.any(), f"fine cell {ci[bad][0]}: clearance {bound.ravel()[ci[bad][0]]} > distance {d[bad][0]}"


def check_blob(blob, seg, poly_start, bounds):
    h = np.frombuffer(blob[:128].tobytes(), HEADER)[0]
    seg64 = np.asarray(seg, np.float64).reshape(-1, 4)
    n_seg, gx, gy = int(h["n_seg"]), int(h["gx"]), int(h["gy"])
    n_poly = 0 if poly_start is None else len(poly_start) - 1
    assert n_seg == len(seg64) and int(h["n_poly"]) == n_poly
    assert h["total_bytes"] == len(blob) and h["smem_bytes"] == h["off_fine"] and h["unused"] == 0
    if bounds is None:
        assert h["has_bounds"] == 0
    else:
        assert h["has_bounds"] == 1 and [h["bxmin"], h["bxmax"], h["bymin"], h["bymax"]] == list(np.float32(bounds))
    # layout: the sections in the order they are written, 16-byte aligned, none overlapping the next
    cells = gx * gy
    order = [("off_seg", n_seg * 16), ("off_cell", (cells + 1) * 4), ("off_items", int(h["n_items"]) * 2),
             ("off_dcell", (cells + 1) * 4), ("off_ditems", int(h["n_ditems"]) * 2), ("off_objfirst", n_seg * 2),
             ("off_poly", (n_poly + 1) * 4), ("off_pbox", n_poly * 16), ("off_fine", cells * int(h["fine"]) ** 2)]
    end = 128
    for name, size in order:
        off = int(h[name])
        assert off % 16 == 0 and off >= end, (name, off, end)
        end = off + size
    assert end <= h["total_bytes"]
    assert bytes(blob[h["off_seg"]:h["off_seg"] + n_seg * 16]) == np.asarray(seg, np.float32).tobytes()
    # coarse lists: every segment that meets a cell's closed box; dilated lists: every segment within dil of it
    assert _check_lists(blob, int(h["off_cell"]), int(h["off_items"]), h, seg64, 0.0) == h["n_items"]
    assert _check_lists(blob, int(h["off_dcell"]), int(h["off_ditems"]), h, seg64, float(h["dil"])) == h["n_ditems"]
    _check_fine(blob, h, seg64, poly_start)
    # objects: an open segment is its own object, a ring edge belongs to the ring's first edge
    objfirst = _section(blob, int(h["off_objfirst"]), "<u2", n_seg)
    want = np.arange(n_seg)
    for p in range(n_poly):
        want[poly_start[p]:poly_start[p + 1]] = poly_start[p]
    assert np.array_equal(objfirst, want)
    pstart = _section(blob, int(h["off_poly"]), "<i4", n_poly + 1)
    assert np.array_equal(pstart, np.zeros(1, np.int32) if n_poly == 0 else poly_start)
    pbox = _section(blob, int(h["off_pbox"]), "<f4", 4 * n_poly).reshape(-1, 4)
    s32 = np.asarray(seg, np.float32).reshape(-1, 4)
    for p in range(n_poly):
        v = s32[poly_start[p]:poly_start[p + 1], :2]
        assert np.array_equal(pbox[p], [v[:, 0].min(), v[:, 0].max(), v[:, 1].min(), v[:, 1].max()])
    return h


# ------------------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("cell_size,reach", PARAMS)
@pytest.mark.parametrize("name", INPUT_NAMES)
def test_tile_blob(tilesim, name, cell_size, reach):
    seg, ps, bounds = tile_input(name)
    code, err, blob = compile_one(tilesim, seg, ps, bounds, cell_size, reach)
    assert code == 0, err
    h = check_blob(blob, seg, ps, bounds)
    assert h["gx"] >= 1 and h["gy"] >= 1


def test_bounds_only_tile(tilesim):
    code, err, blob = compile_one(tilesim, None, bounds=(-5.0, 6.0, 7.0, 9.5), cell_size=3.0, reach=2.9)
    assert code == 0, err
    assert len(blob) == 128
    h = np.frombuffer(blob.tobytes(), HEADER)[0]
    assert h["n_seg"] == 0 and h["gx"] == 0 and h["gy"] == 0 and h["has_bounds"] == 1
    assert (h["bxmin"], h["bxmax"], h["bymin"], h["bymax"]) == (-5.0, 6.0, 7.0, 9.5)
    assert h["total_bytes"] == h["smem_bytes"] == h["off_fine"] == 128


SQUARE = [[0, 0, 4, 0], [4, 0, 4, 4], [4, 4, 0, 4], [0, 4, 0, 0]]
RINGS = "poly_start: rings must be ascending, inside the segment list and have >= 3 edges"


@pytest.mark.parametrize("kw,msg", [
    (dict(seg=SQUARE, n_seg=-1), "n_seg must be in 0..32767"),
    (dict(seg=SQUARE, n_seg=32768), "n_seg must be in 0..32767"),
    (dict(seg=None, n_seg=4), "segments is NULL"),
    (dict(seg=SQUARE, n_poly=1), "poly_start is NULL"),
    (dict(seg=SQUARE, poly_start=[0, 4], n_poly=-1), "poly_start is NULL"),
    (dict(seg=SQUARE, bounds=(1.0, 0.0, 0.0, 1.0)), "bounds must be (xmin<=xmax, ymin<=ymax)"),
    (dict(seg=SQUARE, bounds=(0.0, 1.0, 2.0, 1.0)), "bounds must be (xmin<=xmax, ymin<=ymax)"),
    (dict(seg=[[0, 0, np.nan, 1]]), "segments must be finite"),
    (dict(seg=[[0, 0, 1, np.inf]]), "segments must be finite"),
    (dict(seg=SQUARE, poly_start=[0, 2]), RINGS),                        # fewer than 3 edges
    (dict(seg=SQUARE, poly_start=[0, 5]), RINGS),                        # beyond the segment list
    (dict(seg=SQUARE, poly_start=[-1, 3]), RINGS),
    (dict(seg=SQUARE + SQUARE, poly_start=[4, 0, 8]), RINGS),            # not ascending
    (dict(seg=SQUARE[:3] + [[0, 4, 0, 1]], poly_start=[0, 4]), "poly_start: a ring's edges must chain and close"),
    (dict(seg=[SQUARE[0], SQUARE[2], SQUARE[1], SQUARE[3]], poly_start=[0, 4]), "poly_start: a ring's edges must chain and close"),
])
def test_rejections(tilesim, kw, msg):
    code, err, blob = compile_one(tilesim, kw.get("seg"), kw.get("poly_start"), kw.get("bounds"), n_seg=kw.get("n_seg"),
                                  n_poly=kw.get("n_poly"))
    assert (code, err, blob) == (T2D_E_INVALID, msg, None)


def test_map_table(tilesim):
    names = ["highD_1", "parking", "one_segment", "inD_2_areas", "grid_walls"]
    tiles = [(*tile_input(k), None, None) for k in names]
    tiles.insert(2, (None, None, (0.0, 100.0, -50.0, 50.0), None, None))    # bounds only
    code, err, table, offsets = compile_tiles(tilesim, tiles, 0.0, 2.9, table=True)
    assert code == 0, err
    end = 0
    for t, off in zip(tiles, offsets):
        _, _, blob = compile_one(tilesim, t[0], t[1], t[2], 0.0, 2.9)
        assert off % 128 == 0 and off >= end
        assert not table[end:off].any()
        assert np.array_equal(table[off:off + len(blob)], blob)
        end = off + len(blob)
    assert len(table) == (end + 127) // 128 * 128 and not table[end:].any()
    # a rejected tile rejects the table with its own message
    tiles[3] = (SQUARE, [0, 2], None, None, None)
    assert compile_tiles(tilesim, tiles, 0.0, 2.9, table=True)[:3] == (T2D_E_INVALID, RINGS, None)
