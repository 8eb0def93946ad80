// ray_lists.h — the per-(cell, ray) candidate lists of the sensor sweep: their layout, the host set-up both builders
// share, and the host reference builder (cat_ray_lists_host).  Environments build their lists on the device
// (ray_lists_kernel.cuh), which writes the same words.  Included by cat_b200.cu inside its anonymous namespace.
// maps.ray_lists() is the numpy statement of the same construction (tests/test_maps.py compares the two).
//
// The sensor's ray directions are fixed (entity.py:182), so for ray index i the fat rays of every origin inside
// a grid cell sweep the cell translated along direction i: in the ray's own frame (t along, w across) a region
// inside the rectangle [t0, t1 + L] x [w0, w1] of the cell's projections.  Edge e — its plane offset by rsum and
// the bevel circle of radius rsum at its end vertex, exactly what cpPolyShapeSegmentQuery tests — can be the first
// thing such a ray touches only if
//   (1) its segment comes within rsum of that rectangle,
//   (2) the ray runs against the edge's normal or the next edge's (the bevel's exposed arc spans the two; a hit on
//       the hidden part of the circle lies inside the rounded hull, behind an earlier hit of the same hull),
//   (3) some point of the cell lies in front of one of those two planes (the per-origin rule of the rasteriser).
// Every entry carries a lower bound of the hit distance valid for the whole cell; a list is sorted by it, so a
// lane walking the list stops as soon as the hit it already holds is nearer than the next bound.  The lists are
// conservative supersets and each listed edge still gets the exact arithmetic, so results never depend on them.
//
// Storage: slot[cell * R + ray] = 4 words; entry = (bf16 bits of the bound, truncated = rounded down) << 16 | edge id.
// Lists of up to 4 entries live in the slot (padded with kRayEnd); longer ones keep 3 entries there and a link
// (bit 31 | word offset, a multiple of 4) to a chunk of the overflow array, which again holds up to 4 entries or
// 3 entries and a link to the next chunk.  A link word read as a float is negative, i.e. "a bound nobody is under".
#pragma once
// needs <algorithm>, <thread>, <vector>, <math.h>, <string.h> (included by cat_b200.cu before its anonymous namespace)

constexpr uint32_t kRayEnd = 0x7F80FFFFu;    // bound = +inf: stops every walk
constexpr uint32_t kRayLink = 0x80000000u;

struct RayListGrid {
  float x0 = 0.f, y0 = 0.f, cell = 0.f, inv_cell = 0.f;
  int nx = 0, ny = 0;
};

struct RayLists {
  RayListGrid g;
  std::vector<uint32_t> slots;   // [nx * ny * R][4]
  std::vector<uint32_t> ovf;     // word 0..3 unused (a zero link offset would read as "no overflow")
};

namespace raylist_detail {

// parameter interval of p0 + lam * dp inside [lo, hi]
inline void clip_slab(double p0, double dp, double lo, double hi, double& l0, double& l1) {
  if (dp == 0.0) {
    if (p0 < lo || p0 > hi) { l0 = 1e300; l1 = -1e300; }
    return;
  }
  double a = (lo - p0) / dp, b = (hi - p0) / dp;
  if (a > b) std::swap(a, b);
  if (a > l0) l0 = a;
  if (b < l1) l1 = b;
}

inline double point_rect_dist(double px, double py, double l, double b, double r, double t) {
  const double dx = std::max(std::max(l - px, px - r), 0.0), dy = std::max(std::max(b - py, py - t), 0.0);
  return sqrt(dx * dx + dy * dy);
}

inline uint32_t bound_bits(double lb) {
  // bf16 truncation of a non-negative float rounds towards zero: the stored bound never exceeds the true one
  float f = (float)(lb * (1.0 - 1e-6) - 1e-3);
  if (!(f > 0.f)) f = 0.f;
  uint32_t u;
  memcpy(&u, &f, 4);
  return u & 0xFFFF0000u;
}

}  // namespace raylist_detail

// What both builders (this one and the device one, ray_lists_kernel.cuh) take from the host: the list grid, the sensor
// reach, the rays' directions (cos / sin of the host's libm) and per edge its start vertex A and the next edge's normal.
struct RayListSetup {
  RayListGrid g;
  double gx0 = 0.0, gy0 = 0.0, cell = 0.0, L = 0.0, rs = 0.0;
  std::vector<double> ux, uy;          // [R]
  std::vector<double> ax, ay, nnx, nny; // [E]
};

// `cell` <= 0: automatic.  Grid = bounding box of the hulls grown by the sensor reach: an origin outside it cannot
// see any wall, so the kernel treats "outside the grid" as "empty lists".
static void ray_list_setup(const CatMapDesc* map, int R, double L, double rsum, double cell, RayListSetup* s) {
  const int H = map->n_hulls, E = map->n_edges;
  const double eps = 1e-2, rs = rsum + eps, reach = L + rs + 1.0;
  double bl = 1e300, bb = 1e300, br = -1e300, bt = -1e300;
  for (int h = 0; h < H; ++h) {
    bl = std::min(bl, map->hull_bb[4 * h]); bb = std::min(bb, map->hull_bb[4 * h + 1]);
    br = std::max(br, map->hull_bb[4 * h + 2]); bt = std::max(bt, map->hull_bb[4 * h + 3]);
  }
  const double gx0 = bl - reach, gy0 = bb - reach, gw = br - bl + 2 * reach, gh = bt - bb + 2 * reach;
  // automatic: about 64k cells, not below 6 units (narrower strips = shorter lists = fewer edge tests and fewer overflow
  // links per ray).  Measured on agh-map x 16384, us per step: 308 / 248 / 208 / 198 / 187 at 48 / 32 / 19 / 16 / 12 units
  // with the first list kernel; 137 / 129 / 124 / 121 / 120 at 13.6 / 10 / 8 / 6.8 / 6.3 units with the final one
  // (33 / 58 / 88 / 120 / 136 MB of lists: HBM is not the scarce resource here).
  if (!(cell > 0.0)) {
    double target = 65536.0, min_cell = 6.0;
    if (const char* e = getenv("CAT_RAY_LIST_CELLS")) { const double v = atof(e); if (v >= 64.0) target = v; }          // tuning knobs
    if (const char* e = getenv("CAT_RAY_LIST_MIN_CELL")) { const double v = atof(e); if (v >= 1.0) min_cell = v; }
    cell = std::max(min_cell, sqrt(gw * gh / target));
  }
  const int nx = std::max(1, (int)ceil(gw / cell)), ny = std::max(1, (int)ceil(gh / cell));
  s->g.x0 = (float)gx0; s->g.y0 = (float)gy0; s->g.cell = (float)cell; s->g.inv_cell = (float)(1.0 / cell);
  s->g.nx = nx; s->g.ny = ny;
  s->gx0 = gx0; s->gy0 = gy0; s->cell = cell; s->L = L; s->rs = rs;

  // per edge: A (start), B (end = vert[e]), n, next normal
  s->ax.assign(E, 0.0); s->ay.assign(E, 0.0); s->nnx.assign(E, 0.0); s->nny.assign(E, 0.0);
  for (int h = 0; h < H; ++h) {
    const int o = map->hull_off[h], e1 = map->hull_off[h + 1];
    for (int e = o; e < e1; ++e) {
      const int p = e > o ? e - 1 : e1 - 1, q = e + 1 < e1 ? e + 1 : o;
      s->ax[e] = map->vert[2 * p]; s->ay[e] = map->vert[2 * p + 1];
      s->nnx[e] = map->normal[2 * q]; s->nny[e] = map->normal[2 * q + 1];
    }
  }
  s->ux.resize(R); s->uy.resize(R);
  for (int i = 0; i < R; ++i) {
    const double th = i * (2.0 * M_PI / R);
    s->ux[i] = cos(th); s->uy[i] = sin(th);
  }
}

// The reference builder (host threads): cat_ray_lists_host.  Environments build their lists with the device builder,
// which gives the same words.
static void build_ray_lists(const CatMapDesc* map, int R, double L, double rsum, double cell, RayLists* out) {
  using namespace raylist_detail;
  const int H = map->n_hulls, E = map->n_edges;
  const double eps = 1e-2;
  RayListSetup su;
  ray_list_setup(map, R, L, rsum, cell, &su);
  out->g = su.g;
  const double rs = su.rs, gx0 = su.gx0, gy0 = su.gy0;
  cell = su.cell;
  const int nx = su.g.nx, ny = su.g.ny;
  const std::vector<double>& ax = su.ax, &ay = su.ay, &nnx = su.nnx, &nny = su.nny, &ux = su.ux, &uy = su.uy;
  // (2) per (ray, edge), direction only
  std::vector<uint8_t> against((size_t)R * E);
  for (int i = 0; i < R; ++i)
    for (int e = 0; e < E; ++e)
      against[(size_t)i * E + e] = (ux[i] * map->normal[2 * e] + uy[i] * map->normal[2 * e + 1] < 1e-4) ||
                                   (ux[i] * nnx[e] + uy[i] * nny[e] < 1e-4);

  out->slots.assign((size_t)nx * ny * R * 4, kRayEnd);
  std::vector<std::vector<uint32_t>> row_ovf(ny);

  auto do_row = [&](int cy) {
    std::vector<int> cand;
    std::vector<double> cand_lb;
    std::vector<uint32_t> lst;
    std::vector<uint32_t>& ovf = row_ovf[cy];
    for (int cx = 0; cx < nx; ++cx) {
      // the cell rectangle, grown a little: the kernel bins the origin in fp32
      const double cl = gx0 + cx * cell - 0.05, cb = gy0 + cy * cell - 0.05, cr = cl + cell + 0.1, ct = cb + cell + 0.1;
      const double cxs[4] = {cl, cr, cr, cl}, cys[4] = {cb, cb, ct, ct};
      cand.clear(); cand_lb.clear();
      for (int h = 0; h < H; ++h) {
        const double* hb = map->hull_bb + 4 * h;
        const double dx = std::max(std::max(hb[0] - cr, cl - hb[2]), 0.0), dy = std::max(std::max(hb[1] - ct, cb - hb[3]), 0.0);
        if (dx * dx + dy * dy > (L + rs) * (L + rs)) continue;
        for (int e = map->hull_off[h]; e < map->hull_off[h + 1]; ++e) {
          const double bx = map->vert[2 * e], by = map->vert[2 * e + 1];
          // (3) some corner in front of plane e or of the next plane
          double pd = -1e300, pdn = -1e300;
          for (int c = 0; c < 4; ++c) {
            pd = std::max(pd, (cxs[c] - bx) * map->normal[2 * e] + (cys[c] - by) * map->normal[2 * e + 1]);
            pdn = std::max(pdn, (cxs[c] - bx) * nnx[e] + (cys[c] - by) * nny[e]);
          }
          if (!(pd > -eps || pdn > -eps)) continue;
          // Euclidean distance rectangle <-> segment AB (0 when they intersect)
          const double abx = bx - ax[e], aby = by - ay[e];
          double l0 = 0.0, l1 = 1.0;
          clip_slab(ax[e], abx, cl, cr, l0, l1);
          clip_slab(ay[e], aby, cb, ct, l0, l1);
          double d = 0.0;
          if (l0 > l1) {
            d = std::min(point_rect_dist(ax[e], ay[e], cl, cb, cr, ct), point_rect_dist(bx, by, cl, cb, cr, ct));
            const double l2 = std::max(abx * abx + aby * aby, 1e-300);
            for (int c = 0; c < 4; ++c) {
              double tt = ((cxs[c] - ax[e]) * abx + (cys[c] - ay[e]) * aby) / l2;
              tt = std::min(std::max(tt, 0.0), 1.0);
              const double qx = cxs[c] - (ax[e] + abx * tt), qy = cys[c] - (ay[e] + aby * tt);
              d = std::min(d, sqrt(qx * qx + qy * qy));
            }
          }
          if (d - rs >= L) continue;
          cand.push_back(e);
          cand_lb.push_back(d - rs);
        }
      }
      for (int i = 0; i < R; ++i) {
        double t0 = 1e300, t1 = -1e300, w0 = 1e300, w1 = -1e300;
        for (int c = 0; c < 4; ++c) {
          const double t = cxs[c] * ux[i] + cys[c] * uy[i], w = -cxs[c] * uy[i] + cys[c] * ux[i];
          t0 = std::min(t0, t); t1 = std::max(t1, t); w0 = std::min(w0, w); w1 = std::max(w1, w);
        }
        lst.clear();
        const uint8_t* ag = against.data() + (size_t)i * E;
        for (size_t q = 0; q < cand.size(); ++q) {
          const int e = cand[q];
          if (!ag[e]) continue;
          const double tA = ax[e] * ux[i] + ay[e] * uy[i], wA = -ax[e] * uy[i] + ay[e] * ux[i];
          const double tB = map->vert[2 * e] * ux[i] + map->vert[2 * e + 1] * uy[i];
          const double wB = -map->vert[2 * e] * uy[i] + map->vert[2 * e + 1] * ux[i];
          double l0 = 0.0, l1 = 1.0;
          clip_slab(tA, tB - tA, t0 - rs, t1 + L + rs, l0, l1);   // (1)
          clip_slab(wA, wB - wA, w0 - rs, w1 + rs, l0, l1);
          if (l0 > l1) continue;
          const double tmin = std::min(tA + l0 * (tB - tA), tA + l1 * (tB - tA));
          const double lb = std::max(std::max(tmin - rs - t1, cand_lb[q]), 0.0);
          if (lb >= L) continue;
          lst.push_back(bound_bits(lb) | (uint32_t)e);
        }
        std::sort(lst.begin(), lst.end());
        uint32_t* slot = out->slots.data() + ((size_t)(cy * nx + cx) * R + i) * 4;
        if (lst.size() <= 4) {
          for (size_t q = 0; q < lst.size(); ++q) slot[q] = lst[q];
        } else {
          slot[0] = lst[0]; slot[1] = lst[1]; slot[2] = lst[2];
          slot[3] = kRayLink | (uint32_t)ovf.size();          // row-relative; rebased below (ovf_links)
          size_t q = 3;
          for (;;) {
            const size_t left = lst.size() - q;
            if (left <= 4) {
              for (size_t j = 0; j < 4; ++j) ovf.push_back(j < left ? lst[q + j] : kRayEnd);
              break;
            }
            ovf.push_back(lst[q]); ovf.push_back(lst[q + 1]); ovf.push_back(lst[q + 2]);
            ovf.push_back(kRayLink | (uint32_t)(ovf.size() + 1));   // the next chunk follows
            q += 3;
          }
        }
      }
    }
  };

  unsigned nthr = std::thread::hardware_concurrency();
  nthr = std::max(1u, std::min(nthr, 16u));
  if ((size_t)nx * ny * R * (size_t)E < 4000000) nthr = 1;
  if (nthr == 1) {
    for (int cy = 0; cy < ny; ++cy) do_row(cy);
  } else {
    std::vector<std::thread> pool;
    for (unsigned t = 0; t < nthr; ++t)
      pool.emplace_back([&, t]() { for (int cy = (int)t; cy < ny; cy += (int)nthr) do_row(cy); });
    for (auto& th : pool) th.join();
  }
  // concatenate the rows' overflow arrays and rebase the links
  out->ovf.assign(4, kRayEnd);
  for (int cy = 0; cy < ny; ++cy) {
    const uint32_t base = (uint32_t)out->ovf.size();
    uint32_t* rowslots = out->slots.data() + (size_t)cy * nx * R * 4;
    for (size_t s = 0; s < (size_t)nx * R; ++s)
      if (rowslots[4 * s + 3] & kRayLink) rowslots[4 * s + 3] += base;
    for (size_t q = 3; q < row_ovf[cy].size(); q += 4)
      if (row_ovf[cy][q] & kRayLink) row_ovf[cy][q] += base;
    out->ovf.insert(out->ovf.end(), row_ovf[cy].begin(), row_ovf[cy].end());
  }
}
