// t2d_tile.h - the map tile format and its host compiler.
//
// A tile is the static geometry of one map: the segments in list order (+ which of them close up to polygons), a uniform
// grid over their bounding box grown by one cell, per cell the ascending list of the segments that touch it and the
// "dilated" list of those within one cell of it, the fine clearance field, the tile's boundary box.  compile_tile writes
// one tile's blob, compile_map_table packs several of them; K1 and the lidar kernel read the sections through MapHeader.
// This header is the only definition of the format.  It is plain C++ apart from the device accessors, so that g++ can
// compile the tile compiler for host tests.
#ifndef T2D_TILE_H
#define T2D_TILE_H

#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "../../include/t2d_b200.h"

namespace t2d {

struct MapHeader {   // 128 bytes, start of a tile's blob
  int32_t n_seg, gx, gy, n_items;
  float x0, y0, inv_cell, cell;
  uint32_t off_seg, off_cell, off_items, total_bytes;
  uint32_t unused;      // zero; keeps the fields below at their offsets
  int32_t fine;         // the fine clearance field has (gx * fine) x (gy * fine) cells, one byte each (global memory)
  // "dilated" lists: cell c lists (ascending) every segment that comes within `dil` metres of the cell's box, so that a
  // participant whose bounding radius is <= dil finds all its candidates in the ONE cell under its centre (the grid
  // covers the segments' bounding box grown by dil: a centre outside it cannot reach a segment)
  uint32_t off_dcell, off_ditems;
  float dil;
  int32_t n_ditems;
  uint32_t off_objfirst;   // uint16 per segment: first segment of the object (polygon / polyline piece) it belongs to
  int32_t n_poly;          // closed rings among the segments (Area.geometry polygons)
  uint32_t off_poly;       // int32 [n_poly + 1]: ring p = segments [start[p], start[p + 1])
  uint32_t off_pbox;       // float4 per ring: xmin, xmax, ymin, ymax
  uint32_t off_fine;       // the fine clearance field (bytes), last section of the blob
  uint32_t smem_bytes;     // = off_fine: the part worth staging into shared memory
  float bxmin, bxmax, bymin, bymax;   // Map.boundary of the tile (OutBound)
  int32_t has_bounds;
  uint32_t pad[3];
};
constexpr float CLEAR_QUANT = 0.125f;   // metres per unit of the byte-quantised fine clearance field
static_assert(sizeof(MapHeader) == 128, "MapHeader must be 128 bytes");

#if defined(__CUDACC__)
// The sections of a map blob (in shared or in global memory: the accessors are inlined, the address space is known).
struct MapView {
  const float4* seg;
  const uint32_t* cell_start;
  const uint16_t* items;
  const uint32_t* dcell_start;
  const uint16_t* ditems;
};
__device__ __forceinline__ MapView map_view(const unsigned char* blob, const MapHeader& mh) {
  MapView v;
  v.seg = reinterpret_cast<const float4*>(blob + mh.off_seg);
  v.cell_start = reinterpret_cast<const uint32_t*>(blob + mh.off_cell);
  v.items = reinterpret_cast<const uint16_t*>(blob + mh.off_items);
  v.dcell_start = reinterpret_cast<const uint32_t*>(blob + mh.off_dcell);
  v.ditems = reinterpret_cast<const uint16_t*>(blob + mh.off_ditems);
  return v;
}
#endif

inline bool point_in_ring(const float* seg, int s0, int s1, double px, double py) {   // even-odd over the ring's edges
  bool in = false;
  for (int i = s0; i < s1; ++i) {
    const double x1 = seg[4 * i], y1 = seg[4 * i + 1], x2 = seg[4 * i + 2], y2 = seg[4 * i + 3];
    if ((y1 > py) != (y2 > py) && px < (x2 - x1) * (py - y1) / (y2 - y1) + x1) in = !in;
  }
  return in;
}

// One tile's blob.  reach: the largest bounding radius of the type table (0: none set).  Returns T2D_OK, or
// T2D_E_INVALID with the reason in `err`.
inline int compile_tile(const t2d_map_tile& t, float cell_size, float reach, std::vector<unsigned char>& blob, std::string& err) {
  auto reject = [&](const char* msg) {
    err = msg;
    return T2D_E_INVALID;
  };
  const float* segments = t.segments;
  const int n_seg = t.n_seg;
  if (n_seg < 0 || n_seg > T2D_MAX_SEGMENTS) return reject("n_seg must be in 0..32767");
  if (n_seg > 0 && !segments) return reject("segments is NULL");
  if (t.n_poly < 0 || (t.n_poly > 0 && !t.poly_start)) return reject("poly_start is NULL");
  if (t.bounds && !(t.bounds[0] <= t.bounds[1] && t.bounds[2] <= t.bounds[3])) return reject("bounds must be (xmin<=xmax, ymin<=ymax)");
  for (int p = 0; p < t.n_poly; ++p) {
    const int s0 = t.poly_start[p], s1 = t.poly_start[p + 1];
    if (s0 < 0 || s1 > n_seg || s1 - s0 < 3 || (p > 0 && s0 < t.poly_start[p])) return reject("poly_start: rings must be ascending, inside the segment list and have >= 3 edges");
    for (int i = s0; i < s1; ++i) {   // a ring: every edge ends where the next one starts, the last one at the first one's start
      const int j = i + 1 < s1 ? i + 1 : s0;
      if (segments[4 * i + 2] != segments[4 * j] || segments[4 * i + 3] != segments[4 * j + 1]) return reject("poly_start: a ring's edges must chain and close");
    }
  }
  MapHeader mh{};
  mh.n_seg = n_seg; mh.n_poly = t.n_poly;
  mh.has_bounds = t.bounds ? 1 : 0;
  if (t.bounds) { mh.bxmin = t.bounds[0]; mh.bxmax = t.bounds[1]; mh.bymin = t.bounds[2]; mh.bymax = t.bounds[3]; }
  if (n_seg == 0) {   // bounds only
    mh.gx = mh.gy = 0; mh.total_bytes = mh.smem_bytes = mh.off_fine = sizeof(MapHeader);
    blob.assign(sizeof(MapHeader), 0);
    memcpy(blob.data(), &mh, sizeof(mh));
    return T2D_OK;
  }
  float xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
  for (int i = 0; i < n_seg * 4; ++i)
    if (!std::isfinite(segments[i])) return reject("segments must be finite");
  for (int i = 0; i < n_seg; ++i) {
    const float* s = segments + 4 * i;
    xmin = std::min(xmin, std::min(s[0], s[2])); xmax = std::max(xmax, std::max(s[0], s[2]));
    ymin = std::min(ymin, std::min(s[1], s[3])); ymax = std::max(ymax, std::max(s[1], s[3]));
  }
  const float span = std::max(xmax - xmin, ymax - ymin);
  float cell = cell_size > 0.0f ? cell_size : 8.0f;
  // keep the grid small enough for shared memory: at most 64 x 64 cells over the box grown by one cell (the dilation)
  while (span / cell > 62.0f) cell *= 2.0f;
  // reach of the dilated lists: the largest bounding radius of the type table (as the kernel inflates it) when a table is
  // set - shorter lists in dense maps - else one cell; a participant that reaches further takes the out-of-line walk
  const float dil = reach > 0.0f ? std::min(cell, reach * 1.0002f + 2e-3f) : cell;
  const float margin = 1e-3f * std::max(1.0f, std::max(std::fabs(xmin) + std::fabs(xmax), std::fabs(ymin) + std::fabs(ymax)) * 1e-3f);
  const float x0 = xmin - dil - margin, y0 = ymin - dil - margin;
  const int gx = std::max(1, (int)std::floor((xmax + dil + margin - x0) / cell) + 1);
  const int gy = std::max(1, (int)std::floor((ymax + dil + margin - y0) / cell) + 1);
  const float inv = 1.0f / cell;
  // cells[c] lists (ascending) the segments that pass within `grow` of cell c's box (conservatively: the segment's line
  // against the box grown by `grow` on every side)
  auto bin_segments = [&](float grow) {
    std::vector<std::vector<uint16_t>> cells((size_t)gx * gy);
    for (int i = 0; i < n_seg; ++i) {
      const float* s = segments + 4 * i;
      const float g = grow + margin;
      const float sx0 = std::min(s[0], s[2]) - g, sx1 = std::max(s[0], s[2]) + g;
      const float sy0 = std::min(s[1], s[3]) - g, sy1 = std::max(s[1], s[3]) + g;
      int cx0 = std::max(0, (int)std::floor((sx0 - x0) * inv)), cx1 = std::min(gx - 1, (int)std::floor((sx1 - x0) * inv));
      int cy0 = std::max(0, (int)std::floor((sy0 - y0) * inv)), cy1 = std::min(gy - 1, (int)std::floor((sy1 - y0) * inv));
      for (int cy = cy0; cy <= cy1; ++cy)
        for (int cx = cx0; cx <= cx1; ++cx) {
          // exact-enough cull: does the segment's line pass within the grown cell box?
          const float bx0 = x0 + cx * cell - g, bx1 = x0 + (cx + 1) * cell + g;
          const float by0 = y0 + cy * cell - g, by1 = y0 + (cy + 1) * cell + g;
          const double dx = (double)s[2] - s[0], dy = (double)s[3] - s[1];
          const double hx = 0.5 * ((double)bx1 - bx0), hy = 0.5 * ((double)by1 - by0);
          const double mx = 0.5 * ((double)bx1 + bx0), my = 0.5 * ((double)by1 + by0);
          const double cr = std::fabs(((double)s[0] - mx) * dy - ((double)s[1] - my) * dx);
          if (cr > hx * std::fabs(dy) + hy * std::fabs(dx) + 1e-6 * (std::fabs(dx) + std::fabs(dy) + 1.0)) continue;
          cells[(size_t)cy * gx + cx].push_back((uint16_t)i);
        }
    }
    return cells;
  };
  const std::vector<std::vector<uint16_t>> cells = bin_segments(0.0f);
  // the dilated lists serve participants with reach r <= dil from the cell under their centre: every segment within r
  // of the centre is within dil of that cell's box (+ a 0.1 % + 1 mm guard for the fp32 cell index)
  const std::vector<std::vector<uint16_t>> dcells = bin_segments(dil * 1.001f + 1e-3f);
  size_t n_items = 0, n_ditems = 0;
  for (auto& v : cells) n_items += v.size();
  for (auto& v : dcells) n_ditems += v.size();
  int fine = 4;   // bounded host work: cells x segments <= ~1e8 distance evaluations
  while (fine > 1 && (double)gx * gy * fine * fine * n_seg > 1e8) fine >>= 1;
  mh.gx = gx; mh.gy = gy; mh.n_items = (int)n_items; mh.n_ditems = (int)n_ditems; mh.fine = fine;
  mh.x0 = x0; mh.y0 = y0; mh.inv_cell = inv; mh.cell = cell; mh.dil = dil;
  auto up16 = [](size_t v) { return (v + 15) / 16 * 16; };
  mh.off_seg = (uint32_t)up16(sizeof(MapHeader));
  mh.off_cell = (uint32_t)up16(mh.off_seg + (size_t)n_seg * 16);
  mh.off_items = (uint32_t)up16(mh.off_cell + ((size_t)gx * gy + 1) * 4);
  mh.off_dcell = (uint32_t)up16(mh.off_items + n_items * 2);
  mh.off_ditems = (uint32_t)up16(mh.off_dcell + ((size_t)gx * gy + 1) * 4);
  mh.off_objfirst = (uint32_t)up16(mh.off_ditems + n_ditems * 2);
  mh.off_poly = (uint32_t)up16(mh.off_objfirst + (size_t)n_seg * 2);
  mh.off_pbox = (uint32_t)up16(mh.off_poly + ((size_t)t.n_poly + 1) * 4);
  mh.off_fine = (uint32_t)up16(mh.off_pbox + (size_t)t.n_poly * 16);
  mh.smem_bytes = mh.off_fine;   // the fine field is read through L1 / L2, everything in front of it may be staged
  mh.total_bytes = (uint32_t)up16(mh.off_fine + (size_t)gx * fine * gy * fine);
  blob.assign(mh.total_bytes, 0);
  memcpy(blob.data(), &mh, sizeof(mh));
  memcpy(blob.data() + mh.off_seg, segments, (size_t)n_seg * 16);
  auto write_lists = [&](const std::vector<std::vector<uint16_t>>& lists, uint32_t off_start, uint32_t off_items) {
    uint32_t* cs = reinterpret_cast<uint32_t*>(blob.data() + off_start);
    uint16_t* it = reinterpret_cast<uint16_t*>(blob.data() + off_items);
    uint32_t acc = 0;
    for (size_t ci = 0; ci < lists.size(); ++ci) {
      cs[ci] = acc;
      for (uint16_t sg : lists[ci]) it[acc++] = sg;
    }
    cs[lists.size()] = acc;
  };
  write_lists(cells, mh.off_cell, mh.off_items);
  write_lists(dcells, mh.off_dcell, mh.off_ditems);
  // the object a segment belongs to, named by the object's first segment: an open polyline piece is its own object, the
  // edges of a polygon share the polygon's first edge (StaticCollision.update reports the first OBJECT hit, collision.py:37-43)
  uint16_t* objfirst = reinterpret_cast<uint16_t*>(blob.data() + mh.off_objfirst);
  for (int i = 0; i < n_seg; ++i) objfirst[i] = (uint16_t)i;
  int32_t* pstart = reinterpret_cast<int32_t*>(blob.data() + mh.off_poly);
  float* pbox = reinterpret_cast<float*>(blob.data() + mh.off_pbox);
  for (int p = 0; p < t.n_poly; ++p) {
    const int s0 = t.poly_start[p], s1 = t.poly_start[p + 1];
    pstart[p] = s0;
    float bx0 = INFINITY, bx1 = -INFINITY, by0 = INFINITY, by1 = -INFINITY;
    for (int i = s0; i < s1; ++i) {
      objfirst[i] = (uint16_t)s0;
      bx0 = std::min(bx0, segments[4 * i]); bx1 = std::max(bx1, segments[4 * i]);
      by0 = std::min(by0, segments[4 * i + 1]); by1 = std::max(by1, segments[4 * i + 1]);
    }
    pbox[4 * p] = bx0; pbox[4 * p + 1] = bx1; pbox[4 * p + 2] = by0; pbox[4 * p + 3] = by1;
  }
  pstart[t.n_poly] = t.n_poly > 0 ? t.poly_start[t.n_poly] : 0;
  // fine clearance field: lower bound of the distance from any point of a fine cell to the nearest segment
  // (distance from the cell centre minus the half diagonal); ZERO inside a polygon - a pose deep inside an obstacle
  // touches no edge but intersects the Area all the same.  Bytes of CLEAR_QUANT metres, fine x fine per grid cell, read
  // through L1 / L2.
  auto centre_dist = [&](double px, double py) {
    for (int p = 0; p < t.n_poly; ++p)
      if (px >= pbox[4 * p] && px <= pbox[4 * p + 1] && py >= pbox[4 * p + 2] && py <= pbox[4 * p + 3] &&
          point_in_ring(segments, t.poly_start[p], t.poly_start[p + 1], px, py))
        return 0.0;
    double best = INFINITY;
    for (int i = 0; i < n_seg; ++i) {
      const float* sg = segments + 4 * i;
      const double dx = (double)sg[2] - sg[0], dy = (double)sg[3] - sg[1], ux = px - sg[0], uy = py - sg[1];
      const double dd = dx * dx + dy * dy;
      double tt = dd > 0.0 ? (ux * dx + uy * dy) / dd : 0.0;
      tt = std::min(1.0, std::max(0.0, tt));
      const double ex = ux - tt * dx, ey = uy - tt * dy;
      best = std::min(best, ex * ex + ey * ey);
    }
    return std::sqrt(best);
  };
  uint8_t* fine_field = blob.data() + mh.off_fine;
  {
    const double fc = (double)cell / fine;
    const double half_diag = 0.5 * std::sqrt(2.0) * fc * 1.001 + 2.0 * margin + 1e-3 * fc;
    for (int iy = 0; iy < gy * fine; ++iy)
      for (int ix = 0; ix < gx * fine; ++ix) {
        const double d = centre_dist((double)x0 + (ix + 0.5) * fc, (double)y0 + (iy + 0.5) * fc) - half_diag;
        const double q = std::floor(std::max(0.0, d) / CLEAR_QUANT);
        fine_field[(size_t)iy * gx * fine + ix] = (uint8_t)std::min(255.0, q);
      }
  }
  return T2D_OK;
}

// The blobs of n_tiles tiles back to back in `all`, every one starting 128-byte aligned at offsets[i].  Returns T2D_OK, or
// the rejection of the first tile that fails.
inline int compile_map_table(const t2d_map_tile* tiles, int n_tiles, float cell_size, float reach, std::vector<unsigned char>& all,
                             std::vector<uint32_t>& offsets, std::string& err) {
  all.clear();
  offsets.assign((size_t)std::max(n_tiles, 0), 0);
  std::vector<unsigned char> blob;
  for (int i = 0; i < n_tiles; ++i) {
    if (int r = compile_tile(tiles[i], cell_size, reach, blob, err)) return r;
    offsets[i] = (uint32_t)all.size();
    all.insert(all.end(), blob.begin(), blob.end());
    all.resize((all.size() + 127) / 128 * 128, 0);
  }
  return T2D_OK;
}

}  // namespace t2d

#endif  // T2D_TILE_H
