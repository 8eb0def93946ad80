// render_kernel.cuh — rgb_array frames of many worlds in one launch (cat_render), and the static wall layer of a map
// (cat_renderer_create).  Included by cat_b200.cu.
//
// A frame is render.render_rgb's image, bit for bit: (width, height, 3) uint8, black, then the optional sensor rays,
// then the walls (white), then the agents in index order (cops blue, thieves red).  Every test that decides a pixel is
// evaluated in fp64 in numpy's operation order with __dadd_rn / __dsub_rn / __dmul_rn, so nvcc cannot contract it into
// an FMA that numpy does not do.
//
// One CTA draws a tile of kRenderTX x kRenderTY output pixels of one frame.  y is the contiguous axis of the frame, so
// each of the tile's columns is one run of kRenderTY * 3 bytes in global memory: the CTA builds the columns in shared
// memory, at the same 16-byte phase as their global addresses, and writes them with 16-byte streaming stores.  Before
// the pixels, the CTA works out its frame's A x R ray segments and keeps, in (agent, ray) order, those whose bounding
// box reaches the tile; each pixel walks that list backwards, so the last segment that covers it (numpy's painting
// order) wins, and skips most segments with an fp32 distance test whose margin keeps it conservative.

constexpr int kRenderTX = 8;                          // output columns per tile
constexpr int kRenderTY = 256;                        // output rows per tile
constexpr int kRenderThreads = 256;                   // one thread per row of the tile
constexpr int kRenderChunks = (15 + kRenderTY * 3 + 15) / 16;   // 16-byte chunks a staged column can touch
constexpr int kRenderColBytes = kRenderChunks * 16 + 16;
constexpr int kRenderStageBytes = kRenderTX * kRenderColBytes;
constexpr int kRenderAgentBytes = CAT_MAX_AGENTS * 6 * 8;

// One map of the renderer: its window and its wall layer, a bit per full-resolution pixel (column x, row y is bit y % 32
// of word x * hwords + y / 32).
struct RenderMap {
  const uint32_t* wall;
  int W, H, hwords;
};

struct RenderParams {
  RenderMap maps[CAT_MAX_MAPS];
  int n_maps, A, nc, R;
  const float2* dirs;                 // [R] ray directions (ray_directions())
  long long n_elements;
  const int64_t* world;               // [K] element of frame k, NULL = k
  const int64_t* map_of;              // per element, NULL = map 0
  const unsigned char* pos;           // agent a of element e: float x, y at pos + e * pos_stride + 8 a
  long long pos_stride;
  const unsigned char* ray_dist;      // f16 [A][R] at ray_dist + e * dist_stride, NULL = no rays
  long long dist_stride;
  const unsigned char* ray_type;      // u8 [A][R] at ray_type + e * type_stride
  long long type_stride;
  int d, Wd, Hd, tiles_y, tiles;      // downsample, frame size, tiles per frame column, tiles per frame
  double radius, radius2;             // agent radius and its square as Python computes it (radius ** 2)
  unsigned char* frames;              // u8 [K][Wd][Hd][3]
};

// One ray segment P -> Q of a frame, with the fp64 values of the exact test and fp32 copies for the cheap rejection.
struct RaySeg {
  double px, py, qx, qy, ex, ey, L;
  float fpx, fpy, fex, fey, fL;
  uint32_t rgb;
};

__host__ __device__ constexpr int render_smem_bytes(int n_segs) {
  return kRenderStageBytes + kRenderAgentBytes + n_segs * (int)sizeof(RaySeg) + n_segs * 3;
}

// render_rgb's ray colours by ObjectType; 0 = a type without a colour (not drawn)
__device__ __forceinline__ uint32_t ray_rgb(unsigned t) {
  switch (t) {
    case 0: return 0x606060u;    // wall (96, 96, 96)
    case 1: return 0x00A0FFu;    // cop (0, 160, 255)
    case 2: return 0xFFA000u;    // thief (255, 160, 0)
    case 4: return 0x282828u;    // empty (40, 40, 40)
    default: return 0u;
  }
}

// pixel centre (cx, cy) within 0.5 of segment s: render._on_segment, operation for operation
__device__ __forceinline__ bool on_segment(const RaySeg& s, double cx, double cy) {
  const double wx = __dsub_rn(cx, s.px), wy = __dsub_rn(cy, s.py);
  const double t = __dadd_rn(__dmul_rn(wx, s.ex), __dmul_rn(wy, s.ey));
  if (t <= 0.0) return __dadd_rn(__dmul_rn(wx, wx), __dmul_rn(wy, wy)) <= 0.25;
  if (t >= s.L) {
    const double ux = __dsub_rn(cx, s.qx), uy = __dsub_rn(cy, s.qy);
    return __dadd_rn(__dmul_rn(ux, ux), __dmul_rn(uy, uy)) <= 0.25;
  }
  const double c = __dsub_rn(__dmul_rn(wx, s.ey), __dmul_rn(wy, s.ex));
  return __dmul_rn(c, c) <= __dmul_rn(0.25, s.L);
}

// false only where the pixel centre is farther than 0.5 from the segment's LINE (so from the segment) by more than
// the fp32 error: |w| |e| 1e-5 covers the few roundings of the cross product many times over.
__device__ __forceinline__ bool near_line(const RaySeg& s, float cx, float cy) {
  const float wx = cx - s.fpx, wy = cy - s.fpy;
  const float c = wx * s.fey - wy * s.fex;
  const float m = 0.5f + 1e-5f * (fabsf(wx) + fabsf(wy));
  return c * c <= m * m * s.fL * 1.0001f;
}

__global__ void __launch_bounds__(kRenderThreads) cat_render_kernel(const RenderParams p) {
  extern __shared__ __align__(16) unsigned char rsm[];
  unsigned char* stage = rsm;
  double* agent = reinterpret_cast<double*>(rsm + kRenderStageBytes);   // [A][6]: x, y, box x0, x1, y0, y1
  const int n_segs = p.ray_dist ? p.A * p.R : 0;
  RaySeg* seg = reinterpret_cast<RaySeg*>(rsm + kRenderStageBytes + kRenderAgentBytes);
  uint16_t* list = reinterpret_cast<uint16_t*>(seg + n_segs);
  unsigned char* keep = reinterpret_cast<unsigned char*>(list + n_segs);
  __shared__ long long s_elem;
  __shared__ int s_map, s_nlist;

  const int tid = threadIdx.x;
  const long long k = blockIdx.x / p.tiles;
  const int tile = blockIdx.x - (int)(k * p.tiles);
  const int xo0 = (tile / p.tiles_y) * kRenderTX, yo0 = (tile % p.tiles_y) * kRenderTY;
  const int d = p.d, h = d >> 1;
  if (tid == 0) {
    const long long e = p.world ? p.world[k] : k;
    int m = -1;
    if (e >= 0 && e < p.n_elements) {
      const long long mm = p.map_of ? p.map_of[e] : 0;
      if (mm >= 0 && mm < p.n_maps) m = (int)mm;
    }
    s_elem = e; s_map = m;
  }
  __syncthreads();
  const int m = s_map;
  const long long e = s_elem;
  int W = 0, H = 0, hwords = 0;
  const uint32_t* wall = nullptr;
  if (m >= 0) { W = p.maps[m].W; H = p.maps[m].H; hwords = p.maps[m].hwords; wall = p.maps[m].wall; }
  // the tile's pixel centres at full resolution span [cx0, cx1] x [cy0, cy1]
  const int xl1 = min(kRenderTX, p.Wd - xo0), yl1 = min(kRenderTY, p.Hd - yo0);
  const bool visible = m >= 0 && xo0 * d + h < W && yo0 * d + h < H;

  if (visible) {
    if (tid < p.A) {
      const float* q = reinterpret_cast<const float*>(p.pos + e * p.pos_stride + 8 * tid);
      const double x = (double)q[0], y = (double)q[1], r = p.radius;
      double* a = agent + 6 * tid;
      a[0] = x; a[1] = y;
      a[2] = trunc(__dsub_rn(__dsub_rn(x, r), 1.0)); a[3] = trunc(__dadd_rn(__dadd_rn(x, r), 2.0));
      a[4] = trunc(__dsub_rn(__dsub_rn(y, r), 1.0)); a[5] = trunc(__dadd_rn(__dadd_rn(y, r), 2.0));
    }
    if (n_segs) {
      const double cx0 = xo0 * d + h + 0.5, cx1 = (xo0 + xl1 - 1) * d + h + 0.5;
      const double cy0 = yo0 * d + h + 0.5, cy1 = (yo0 + yl1 - 1) * d + h + 0.5;
      const unsigned char* dist = p.ray_dist + e * p.dist_stride;
      const unsigned char* type = p.ray_type + e * p.type_stride;
      for (int j = tid; j < n_segs; j += kRenderThreads) {
        const int a = j / p.R, i = j - a * p.R;
        const float* q = reinterpret_cast<const float*>(p.pos + e * p.pos_stride + 8 * a);
        const float2 u = p.dirs[i];
        const double len = (double)__half2float(__ushort_as_half(reinterpret_cast<const unsigned short*>(dist)[j]));
        RaySeg s;
        s.fpx = q[0]; s.fpy = q[1];
        s.px = s.fpx; s.py = s.fpy;
        s.qx = __dadd_rn(s.px, __dmul_rn(len, (double)u.x));
        s.qy = __dadd_rn(s.py, __dmul_rn(len, (double)u.y));
        s.ex = __dsub_rn(s.qx, s.px); s.ey = __dsub_rn(s.qy, s.py);
        s.L = __dadd_rn(__dmul_rn(s.ex, s.ex), __dmul_rn(s.ey, s.ey));
        s.fex = (float)s.ex; s.fey = (float)s.ey; s.fL = (float)s.L;
        s.rgb = ray_rgb(type[j]);
        const bool finite = isfinite(s.px) && isfinite(s.py) && isfinite(s.qx) && isfinite(s.qy) && isfinite(s.fL);
        keep[j] = s.rgb != 0u && finite && fmin(s.px, s.qx) - 1.0 <= cx1 && fmax(s.px, s.qx) + 1.0 >= cx0 &&
                  fmin(s.py, s.qy) - 1.0 <= cy1 && fmax(s.py, s.qy) + 1.0 >= cy0;
        seg[j] = s;
      }
    }
  }
  __syncthreads();
  if (visible && n_segs && tid < 32) {   // ordered compaction of the kept segments
    int n = 0;
    for (int b = 0; b < n_segs; b += 32) {
      const bool f = b + tid < n_segs && keep[b + tid];
      const unsigned bal = __ballot_sync(0xffffffffu, f);
      if (f) list[n + __popc(bal & ((1u << tid) - 1u))] = (uint16_t)(b + tid);
      n += __popc(bal);
    }
    if (tid == 0) s_nlist = n;
  }
  __syncthreads();
  const int n_list = (visible && n_segs) ? s_nlist : 0;

  const uintptr_t base = reinterpret_cast<uintptr_t>(p.frames);
  for (int xl = 0; xl < xl1; ++xl) {   // thread tid draws row yo0 + tid of each column
    const int xo = xo0 + xl, yo = yo0 + tid;
    const long long g0 = ((k * p.Wd + xo) * p.Hd + yo0) * 3;
    const int ph = (int)((base + (uintptr_t)g0) & 15);
    if (tid >= yl1) continue;
    uint32_t rgb = 0;
    const int X = xo * d + h, Y = yo * d + h;
    if (visible && X < W && Y < H) {
      const double cx = X + 0.5, cy = Y + 0.5, xd = X, yd = Y;
      bool done = false;
      for (int a = p.A - 1; a >= 0; --a) {
        const double* ag = agent + 6 * a;
        if (xd >= ag[2] && xd < ag[3] && yd >= ag[4] && yd < ag[5]) {
          const double dx = __dsub_rn(cx, ag[0]), dy = __dsub_rn(cy, ag[1]);
          if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= p.radius2) {
            rgb = a < p.nc ? 0x0000FFu : 0xFF0000u;
            done = true;
            break;
          }
        }
      }
      if (!done && ((__ldg(wall + (size_t)X * hwords + (Y >> 5)) >> (Y & 31)) & 1u)) { rgb = 0xFFFFFFu; done = true; }
      if (!done) {
        const float fcx = (float)cx, fcy = (float)cy;
        for (int s = n_list - 1; s >= 0; --s) {
          const RaySeg& sg = seg[list[s]];
          if (near_line(sg, fcx, fcy) && on_segment(sg, cx, cy)) { rgb = sg.rgb; break; }
        }
      }
    }
    unsigned char* px = stage + xl * kRenderColBytes + ph + tid * 3;
    px[0] = (unsigned char)(rgb >> 16); px[1] = (unsigned char)(rgb >> 8); px[2] = (unsigned char)rgb;
  }
  __syncthreads();
  // each staged column to global memory: 16-byte stores, single bytes at a column's unaligned ends
  const int count = yl1 * 3;
  for (int c = tid; c < xl1 * kRenderChunks; c += kRenderThreads) {
    const int xl = c / kRenderChunks, q = c - xl * kRenderChunks;
    const long long g0 = ((k * p.Wd + xo0 + xl) * p.Hd + yo0) * 3;
    const int ph = (int)((base + (uintptr_t)g0) & 15);
    const int lo = 16 * q, hi = lo + 16;
    if (lo >= ph + count) continue;
    const unsigned char* src = stage + xl * kRenderColBytes;
    unsigned char* dst = p.frames + g0 - ph;
    if (lo >= ph && hi <= ph + count) {
      __stcs(reinterpret_cast<uint4*>(dst + lo), *reinterpret_cast<const uint4*>(src + lo));
    } else {
      for (int b = max(lo, ph); b < min(hi, ph + count); ++b) dst[b] = src[b];
    }
  }
}

// The wall layer of one map: a pixel is a wall when its centre passes render_rgb's hull test for a hull whose clip box
// contains it.  One thread per pixel of a column padded to hwords * 32 rows; each warp writes one word.
struct WallHull {
  int e0, e1;           // the hull's edges
  int x0, x1, y0, y1;   // render_rgb's clip box, already clamped to the window
};

__global__ void cat_wall_bits_kernel(const WallHull* hulls, int n_hulls, const double2* vert, const double2* normal, int H,
                                     int hwords, long long n_threads, uint32_t* bits) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= n_threads) return;   // n_threads is a multiple of 32: whole warps leave together
  const int x = (int)(gid / (hwords * 32)), y = (int)(gid % (hwords * 32));
  bool in = false;
  if (y < H) {
    const double cx = x + 0.5, cy = y + 0.5;
    for (int hh = 0; hh < n_hulls && !in; ++hh) {
      const WallHull hl = hulls[hh];
      if (x < hl.x0 || x >= hl.x1 || y < hl.y0 || y >= hl.y1) continue;
      bool inside = true;
      for (int i = hl.e0; i < hl.e1 && inside; ++i) {
        const double2 v = vert[i], n = normal[i];
        inside = __dadd_rn(__dmul_rn(__dsub_rn(cx, v.x), n.x), __dmul_rn(__dsub_rn(cy, v.y), n.y)) <= 1.0;
      }
      in = inside;
    }
  }
  const unsigned b = __ballot_sync(0xffffffffu, in);
  if ((threadIdx.x & 31) == 0) bits[gid >> 5] = b;
}
