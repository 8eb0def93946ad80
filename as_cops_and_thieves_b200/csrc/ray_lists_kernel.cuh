// ray_lists_kernel.cuh — device builder of the per-(cell, ray) candidate lists of the sensor sweep.  Included by
// cat_b200.cu after ray_lists.h, whose build_ray_lists is the reference: this builder writes exactly its words (the same
// slots, the same overflow array, the same link offsets), from the same host set-up (ray_list_setup: grid, ray
// directions, per-edge vertices and next normals).
//
// Bit-exactness: every fp64 expression of the host builder is written here with __dmul_rn / __dadd_rn / __dsub_rn in the
// host's order of operations, so nvcc fuses nothing into an FMA; fp64 division and square root are IEEE on the device;
// min / max keep std::min / std::max's argument order.
//
// Passes (one CTA per grid cell in each, grid-stride over the cells):
//   1. candidates: count, then write, the edges that pass the per-cell filter (hull reach, facing corner, segment
//      distance) with their per-cell lower bound — in global memory, unordered (a list is sorted at the end);
//   2. lists, count: one warp per ray, the entries of the (cell, ray) list from the cell's candidates (staged in shared
//      memory when they fit, read from global memory otherwise); the entries and overflow words of each list;
//   3. a scan over the cells (single CTA) of the overflow words and of the entries of the lists too long for on-chip
//      sorting;
//   4. lists, fill: each warp collects its list's entries (shared memory up to kRlSortCap entries, a global scratch area
//      otherwise), ranks every entry among them (ascending as uint32, as std::sort) and stores it at its final word.
// The overflow offset of a list is 4 + the overflow words of the lists before it in (cy, cx, ray) order: the host appends
// its chunks row by row, in (cx, ray) order within a row, after 4 unused words.
#pragma once

constexpr int kRlThreads = 256;           // 8 warps per CTA
constexpr int kRlCandCap = 2048;          // candidates of a cell staged in shared memory (more: read from global memory)
constexpr int kRlSortCap = 256;           // entries of a list sorted in shared memory (more: the global scratch area)

struct RayListDev {
  // map (fp64, from the host description and ray_list_setup)
  int H, E, R, nx, ny;
  const double* vert;       // [E][2]
  const double* normal;     // [E][2]
  const double* a;          // [E][2] start vertex of edge e
  const double* nn;         // [E][2] normal of the next edge of the hull
  const double* hull_bb;    // [H][4]
  const int32_t* ehull;     // [E]
  const double* u;          // [R][2] cos, sin
  double gx0, gy0, cell, L, rs;
  // work
  unsigned long long* cand_off;   // [cells + 1] after the scan (pass 1 writes the counts)
  int32_t* cand_e;
  double* cand_lb;
  uint32_t* n_list;               // [cells * R] entries per list
  unsigned long long* words;      // [cells + 1] overflow words per cell -> exclusive scan
  unsigned long long* longs;      // [cells + 1] entries of the cell's lists longer than kRlSortCap -> exclusive scan
  uint32_t* long_buf;
  // output
  uint32_t* slots;                // [cells * R][4]
  uint32_t* ovf;
};

namespace rldev {

__device__ __forceinline__ double dmax(double a, double b) { return (a < b) ? b : a; }   // std::max
__device__ __forceinline__ double dmin(double a, double b) { return (b < a) ? b : a; }   // std::min

__device__ __forceinline__ void clip_slab(double p0, double dp, double lo, double hi, double& l0, double& l1) {
  if (dp == 0.0) {
    if (p0 < lo || p0 > hi) { l0 = 1e300; l1 = -1e300; }
    return;
  }
  double a = __dsub_rn(lo, p0) / dp, b = __dsub_rn(hi, p0) / dp;
  if (a > b) { const double t = a; a = b; b = t; }
  if (a > l0) l0 = a;
  if (b < l1) l1 = b;
}

__device__ __forceinline__ double hypot_rn(double x, double y) {
  return __dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
}

__device__ __forceinline__ double point_rect_dist(double px, double py, double l, double b, double r, double t) {
  const double dx = dmax(dmax(__dsub_rn(l, px), __dsub_rn(px, r)), 0.0), dy = dmax(dmax(__dsub_rn(b, py), __dsub_rn(py, t)), 0.0);
  return hypot_rn(dx, dy);
}

__device__ __forceinline__ uint32_t bound_bits(double lb) {
  float f = __double2float_rn(__dsub_rn(__dmul_rn(lb, 1.0 - 1e-6), 1e-3));
  if (!(f > 0.f)) f = 0.f;
  return __float_as_uint(f) & 0xFFFF0000u;
}

// the cell rectangle, grown a little (ray_lists.h)
struct CellRect { double cl, cb, cr, ct; };
__device__ __forceinline__ CellRect cell_rect(const RayListDev& p, int cell) {
  const int cy = cell / p.nx, cx = cell - cy * p.nx;
  CellRect r;
  r.cl = __dsub_rn(__dadd_rn(p.gx0, __dmul_rn((double)cx, p.cell)), 0.05);
  r.cb = __dsub_rn(__dadd_rn(p.gy0, __dmul_rn((double)cy, p.cell)), 0.05);
  r.cr = __dadd_rn(__dadd_rn(r.cl, p.cell), 0.1);
  r.ct = __dadd_rn(__dadd_rn(r.cb, p.cell), 0.1);
  return r;
}

// Pass 1's filter of edge e for the cell: true and the lower bound d - rs if e is a candidate.
__device__ bool cell_candidate(const RayListDev& p, const CellRect& c, int e, double& lb) {
  const double eps = 1e-2, rs = p.rs, L = p.L;
  const double* hb = p.hull_bb + 4 * p.ehull[e];
  const double dx = dmax(dmax(__dsub_rn(hb[0], c.cr), __dsub_rn(c.cl, hb[2])), 0.0);
  const double dy = dmax(dmax(__dsub_rn(hb[1], c.ct), __dsub_rn(c.cb, hb[3])), 0.0);
  const double reach = __dadd_rn(L, rs);
  if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) > __dmul_rn(reach, reach)) return false;
  const double cxs[4] = {c.cl, c.cr, c.cr, c.cl}, cys[4] = {c.cb, c.cb, c.ct, c.ct};
  const double bx = p.vert[2 * e], by = p.vert[2 * e + 1], nx = p.normal[2 * e], ny = p.normal[2 * e + 1];
  const double nnx = p.nn[2 * e], nny = p.nn[2 * e + 1], ax = p.a[2 * e], ay = p.a[2 * e + 1];
  // (3) some corner in front of plane e or of the next plane
  double pd = -1e300, pdn = -1e300;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double ox = __dsub_rn(cxs[k], bx), oy = __dsub_rn(cys[k], by);
    pd = dmax(pd, __dadd_rn(__dmul_rn(ox, nx), __dmul_rn(oy, ny)));
    pdn = dmax(pdn, __dadd_rn(__dmul_rn(ox, nnx), __dmul_rn(oy, nny)));
  }
  if (!(pd > -eps || pdn > -eps)) return false;
  // Euclidean distance rectangle <-> segment AB (0 when they intersect)
  const double abx = __dsub_rn(bx, ax), aby = __dsub_rn(by, ay);
  double l0 = 0.0, l1 = 1.0;
  clip_slab(ax, abx, c.cl, c.cr, l0, l1);
  clip_slab(ay, aby, c.cb, c.ct, l0, l1);
  double d = 0.0;
  if (l0 > l1) {
    d = dmin(point_rect_dist(ax, ay, c.cl, c.cb, c.cr, c.ct), point_rect_dist(bx, by, c.cl, c.cb, c.cr, c.ct));
    const double l2 = dmax(__dadd_rn(__dmul_rn(abx, abx), __dmul_rn(aby, aby)), 1e-300);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      double tt = __dadd_rn(__dmul_rn(__dsub_rn(cxs[k], ax), abx), __dmul_rn(__dsub_rn(cys[k], ay), aby)) / l2;
      tt = dmin(dmax(tt, 0.0), 1.0);
      const double qx = __dsub_rn(cxs[k], __dadd_rn(ax, __dmul_rn(abx, tt)));
      const double qy = __dsub_rn(cys[k], __dadd_rn(ay, __dmul_rn(aby, tt)));
      d = dmin(d, hypot_rn(qx, qy));
    }
  }
  if (__dsub_rn(d, rs) >= L) return false;
  lb = __dsub_rn(d, rs);
  return true;
}

// The ray's projections of the cell rectangle: t along the ray, w across it.
struct RaySpan { double ux, uy, t0, t1, w0, w1; };
__device__ __forceinline__ RaySpan ray_span(const RayListDev& p, const CellRect& c, int i) {
  RaySpan s;
  s.ux = p.u[2 * i]; s.uy = p.u[2 * i + 1];
  const double cxs[4] = {c.cl, c.cr, c.cr, c.cl}, cys[4] = {c.cb, c.cb, c.ct, c.ct};
  s.t0 = 1e300; s.t1 = -1e300; s.w0 = 1e300; s.w1 = -1e300;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double t = __dadd_rn(__dmul_rn(cxs[k], s.ux), __dmul_rn(cys[k], s.uy));
    const double w = __dadd_rn(__dmul_rn(-cxs[k], s.uy), __dmul_rn(cys[k], s.ux));
    s.t0 = dmin(s.t0, t); s.t1 = dmax(s.t1, t); s.w0 = dmin(s.w0, w); s.w1 = dmax(s.w1, w);
  }
  return s;
}

// The list entry of candidate edge e (per-cell lower bound cand_lb) for the ray; false if e is not in the list.
__device__ __forceinline__ bool list_entry(const RayListDev& p, const RaySpan& s, int e, double cand_lb, uint32_t& out) {
  const double rs = p.rs, L = p.L;
  const double nx = p.normal[2 * e], ny = p.normal[2 * e + 1], nnx = p.nn[2 * e], nny = p.nn[2 * e + 1];
  // (2) the ray runs against the edge's normal or the next edge's
  const bool against = (__dadd_rn(__dmul_rn(s.ux, nx), __dmul_rn(s.uy, ny)) < 1e-4) ||
                       (__dadd_rn(__dmul_rn(s.ux, nnx), __dmul_rn(s.uy, nny)) < 1e-4);
  if (!against) return false;
  const double ax = p.a[2 * e], ay = p.a[2 * e + 1], bx = p.vert[2 * e], by = p.vert[2 * e + 1];
  const double tA = __dadd_rn(__dmul_rn(ax, s.ux), __dmul_rn(ay, s.uy)), wA = __dadd_rn(__dmul_rn(-ax, s.uy), __dmul_rn(ay, s.ux));
  const double tB = __dadd_rn(__dmul_rn(bx, s.ux), __dmul_rn(by, s.uy));
  const double wB = __dadd_rn(__dmul_rn(-bx, s.uy), __dmul_rn(by, s.ux));
  double l0 = 0.0, l1 = 1.0;
  const double dt = __dsub_rn(tB, tA);
  clip_slab(tA, dt, __dsub_rn(s.t0, rs), __dadd_rn(__dadd_rn(s.t1, L), rs), l0, l1);   // (1)
  clip_slab(wA, __dsub_rn(wB, wA), __dsub_rn(s.w0, rs), __dadd_rn(s.w1, rs), l0, l1);
  if (l0 > l1) return false;
  const double tmin = dmin(__dadd_rn(tA, __dmul_rn(l0, dt)), __dadd_rn(tA, __dmul_rn(l1, dt)));
  const double lb = dmax(dmax(__dsub_rn(__dsub_rn(tmin, rs), s.t1), cand_lb), 0.0);
  if (lb >= L) return false;
  out = bound_bits(lb) | (uint32_t)e;
  return true;
}

// overflow words of a list of n entries: 0 up to 4 entries; else the 3 in the slot, chunks of 3 + a link while more than
// 4 are left, and a last chunk of at most 4
__device__ __forceinline__ unsigned list_words(unsigned n) {
  if (n <= 4) return 0;
  const unsigned m = n - 3, nf = m <= 4 ? 0 : (m - 4 + 2) / 3;
  return 4 * (nf + 1);
}

}  // namespace rldev

// Pass 1.  WRITE = false: candidates per cell into cand_off[cell]; true: the candidates at cand_off[cell] (scanned).
template <bool WRITE>
__global__ void __launch_bounds__(kRlThreads) cat_ray_list_cand_kernel(const RayListDev p) {
  __shared__ unsigned count;
  const int cells = p.nx * p.ny;
  for (int cell = blockIdx.x; cell < cells; cell += gridDim.x) {
    if (threadIdx.x == 0) count = 0;
    __syncthreads();
    const rldev::CellRect c = rldev::cell_rect(p, cell);
    const unsigned long long base = WRITE ? p.cand_off[cell] : 0;
    for (int e = threadIdx.x; e < p.E; e += blockDim.x) {
      double lb;
      if (!rldev::cell_candidate(p, c, e, lb)) continue;
      const unsigned q = atomicAdd(&count, 1u);
      if (WRITE) { p.cand_e[base + q] = e; p.cand_lb[base + q] = lb; }
    }
    __syncthreads();
    if (!WRITE && threadIdx.x == 0) p.cand_off[cell] = count;
    __syncthreads();
  }
}

// Exclusive scan of n values in place (v[n] = the total), one CTA: a user-facing map has at most a few 10^5 cells.
__global__ void __launch_bounds__(1024) cat_ray_list_scan_kernel(unsigned long long* v, int n) {
  __shared__ unsigned long long part[1024];
  const int t = threadIdx.x, per = (n + 1023) / 1024, b = min(n, t * per), e = min(n, b + per);
  unsigned long long s = 0;
  for (int i = b; i < e; ++i) s += v[i];
  part[t] = s;
  __syncthreads();
  if (t == 0) {
    unsigned long long acc = 0;
    for (int i = 0; i < 1024; ++i) { const unsigned long long x = part[i]; part[i] = acc; acc += x; }
    v[n] = acc;
  }
  __syncthreads();
  unsigned long long acc = part[t];
  for (int i = b; i < e; ++i) { const unsigned long long x = v[i]; v[i] = acc; acc += x; }
}

// Passes 2 and 4: one CTA per cell, one warp per ray.
template <bool FILL>
__global__ void __launch_bounds__(kRlThreads) cat_ray_list_kernel(const RayListDev p) {
  __shared__ int s_e[kRlCandCap];
  __shared__ double s_lb[kRlCandCap];
  __shared__ uint32_t s_sort[kRlThreads / 32][kRlSortCap];
  __shared__ unsigned long long s_words[CAT_MAX_RAYS], s_long[CAT_MAX_RAYS];   // FILL: each ray's offsets in the cell
  __shared__ unsigned long long c_words, c_long;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int cells = p.nx * p.ny, R = p.R;
  for (int cell = blockIdx.x; cell < cells; cell += gridDim.x) {
    const unsigned long long cb = p.cand_off[cell];
    const int nc = (int)(p.cand_off[cell + 1] - cb);
    const bool staged = nc <= kRlCandCap;
    for (int q = threadIdx.x; staged && q < nc; q += blockDim.x) { s_e[q] = p.cand_e[cb + q]; s_lb[q] = p.cand_lb[cb + q]; }
    if (threadIdx.x == 0) {
      c_words = 0; c_long = 0;
      if (FILL) {   // the lists' overflow words and long-list entries in ray order: offsets within the cell
        unsigned long long w = 0, l = 0;
        for (int i = 0; i < R; ++i) {
          const unsigned n = p.n_list[(size_t)cell * R + i];
          s_words[i] = w; s_long[i] = l;
          w += rldev::list_words(n); l += n > (unsigned)kRlSortCap ? n : 0;
        }
      }
    }
    __syncthreads();
    const int* ce = staged ? s_e : p.cand_e + cb;
    const double* cl = staged ? s_lb : p.cand_lb + cb;
    const rldev::CellRect c = rldev::cell_rect(p, cell);
    for (int i = warp; i < R; i += nwarps) {
      const rldev::RaySpan s = rldev::ray_span(p, c, i);
      const size_t li = (size_t)cell * R + i;
      if (!FILL) {
        unsigned n = 0;
        for (int q0 = 0; q0 < nc; q0 += 32) {
          uint32_t v;
          const bool ok = q0 + lane < nc && rldev::list_entry(p, s, ce[q0 + lane], cl[q0 + lane], v);
          n += __popc(__ballot_sync(0xFFFFFFFFu, ok));
        }
        if (lane == 0) {
          p.n_list[li] = n;
          atomicAdd(&c_words, (unsigned long long)rldev::list_words(n));
          if (n > (unsigned)kRlSortCap) atomicAdd(&c_long, (unsigned long long)n);
        }
        continue;
      }
      const unsigned n = p.n_list[li];
      uint32_t* buf = n <= (unsigned)kRlSortCap ? s_sort[warp] : p.long_buf + p.longs[cell] + s_long[i];
      unsigned k = 0;
      for (int q0 = 0; q0 < nc; q0 += 32) {
        uint32_t v = 0;
        const bool ok = q0 + lane < nc && rldev::list_entry(p, s, ce[q0 + lane], cl[q0 + lane], v);
        const unsigned m = __ballot_sync(0xFFFFFFFFu, ok);
        if (ok) buf[k + __popc(m & ((1u << lane) - 1))] = v;
        k += __popc(m);
      }
      __syncwarp();
      // rank each entry among the list's (entries are distinct: each edge appears once) and store it at its word
      uint32_t* slot = p.slots + li * 4;
      const unsigned long long o = 4 + p.words[cell] + s_words[i];   // first overflow word of the list
      const unsigned m = n > 4 ? n - 3 : 0, nf = m <= 4 ? 0 : (m - 4 + 2) / 3;
      for (unsigned j = lane; j < n; j += 32) {
        const uint32_t v = buf[j];
        unsigned r = 0;
        for (unsigned q = 0; q < n; ++q) r += buf[q] < v ? 1u : 0u;
        if (n <= 4 || r < 3) { slot[r] = v; continue; }
        const unsigned qq = r - 3, ch = qq / 3 < nf ? qq / 3 : nf;
        p.ovf[o + 4 * ch + (qq - 3 * ch)] = v;
      }
      if (lane < 4 && n <= 4 && (unsigned)lane >= n) slot[lane] = kRayEnd;
      if (n > 4) {
        if (lane == 0) slot[3] = kRayLink | (uint32_t)o;
        for (unsigned ch = lane; ch < nf; ch += 32) p.ovf[o + 4 * ch + 3] = kRayLink | (uint32_t)(o + 4 * ch + 4);
        const unsigned left = m - 3 * nf;   // entries of the last chunk
        if ((unsigned)lane >= left && lane < 4) p.ovf[o + 4 * nf + lane] = kRayEnd;
      }
      __syncwarp();
    }
    __syncthreads();
    if (!FILL && threadIdx.x == 0) { p.words[cell] = c_words; p.longs[cell] = c_long; }
    if (FILL && cell == 0 && threadIdx.x < 4) p.ovf[threadIdx.x] = kRayEnd;   // the 4 unused words
    __syncthreads();
  }
}
