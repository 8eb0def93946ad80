// world_kernel.cuh — device side of the fused world step: map blob view, Chipmunk geometry, the sensor-sweep
// rasteriser, observation writers, rewards, the rigid-body step, auto-reset and `cat_world_kernel` itself.
// Included by cat_b200.cu inside its anonymous namespace (one translation unit, one shared library).
#pragma once
#ifndef CAT_WARPS_PER_CTA
#define CAT_WARPS_PER_CTA 8
#endif
#ifndef CAT_MIN_CTAS_PER_SM
#define CAT_MIN_CTAS_PER_SM 4
#endif
constexpr int kWarpsPerCta = CAT_WARPS_PER_CTA;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int kMaxThreads = 1024;   // the host picks 2..32 warps per CTA per environment (pick_launch_shape); 64 registers either way
constexpr int kMinCtasPerSm = CAT_MIN_CTAS_PER_SM;
constexpr int kSlots = CAT_WALL_SLOTS;
constexpr int kNear = CAT_NEAR_SLOTS;   // hulls an origin can be "inside" (alpha = 0 rule) per agent
constexpr uint32_t kEmpty = 0xFFFFFFFFu;

enum { TYPE_WALL = 0, TYPE_COP = 1, TYPE_THIEF = 2, TYPE_EMPTY = 4 };
enum { MODE_STEP = 0, MODE_RESET = 1, MODE_OBSERVE = 2, MODE_INIT = 3 };

#ifdef CAT_STATS   // developer build only (tools/raster_stats.py): rasteriser work counters
__device__ unsigned long long g_stats[8];
#define CAT_COUNT(i, v) atomicAdd(&g_stats[i], (unsigned long long)(v))
// index / capacity assertions of the checked build (tools/bounds_check.py): a violation is COUNTED (g_stats[6], with the
// source line of the last one in g_stats[7]) instead of trapping, so one run reports all of them and the context survives
#define CAT_CHECK(cond) do { if (!(cond)) { atomicAdd(&g_stats[6], 1ull); g_stats[7] = __LINE__; } } while (0)
#else
#define CAT_COUNT(i, v)
#define CAT_CHECK(cond)
#endif

// ------------------------------------------------------------------ shared-memory map blob
struct BlobHeader {
  int32_t n_hulls, n_edges, nx, ny;
  float gx0, gy0, cell, inv_cell;
  int32_t off_edge, off_len, off_hbb, off_heo;
  int32_t off_nextn, off_edgehull, off_conoff, off_conlist;
  int32_t off_dir, off_regoff, off_regions, off_initpos;
  int32_t off_batchbb;
  // the map's tables in global memory (written by the host once they are on the device): with these in the header a
  // CTA's map is fully described by the blob it stages, so the CTAs of one launch can run different maps
  int32_t rg_nx, rg_ny;                     // (cell, ray) candidate-list grid (ray_lists.h)
  uint32_t ray_slot_count;                  // sizes of the two list arrays (checked build only)
  float rg_x0, rg_y0, rg_inv_cell;
  uint32_t ray_ovf_words;
  const uint4* ray_slots;                   // slots [cells * R] of 4 words; nullptr = rasterise
  const uint32_t* ray_ovf;                  // overflow words of the lists
  const int32_t* view_off;                  // per grid cell candidate-edge lists (nullptr = scan all edges)
  const uint16_t* view_edges;
};
static_assert(sizeof(BlobHeader) == 144, "header must stay 16-byte sized");
__device__ __forceinline__ const BlobHeader* blob_header(const unsigned char* blob) {
  return reinterpret_cast<const BlobHeader*>(blob);
}

struct MapView {
  const float4* edge;      // vx, vy, nx, ny  (vertex ending the edge, outward normal)
  const float* edge_len;
  const float4* hull_bb;   // l,b,r,t grown by the wall radius (the shape's bb)
  const uint32_t* hull_eo; // edge offset | count << 16
  const float4* batch_bb;    // bounding box of edges [32b, 32b+32) incl. both end points
  const float2* next_n;      // outward normal of the NEXT edge of the same hull (shares vertex v_i)
  const uint16_t* edge_hull; // hull of each edge
  const uint16_t* con_off;
  const uint16_t* con_list;
  const float4* dir;       // per ray: ux, uy, 1/ux, 1/uy (unit direction and its reciprocals)
  const int32_t* reg_off;
  const float4* regions;
  const float2* init_pos;
  int H, nx, ny;
  float gx0, gy0, cell, inv_cell;
  int n_edges;
};

// Word offsets inside a world's packed state record and byte offsets inside a warp's scratch area — ONE definition,
// evaluated by the host for every environment (into KParams) and at COMPILE TIME by the kernel instantiation for the
// shipped shape, where every offset then is an immediate instead of a constant-bank load + add.
struct Layout {
  int P, nrays, nrays_pad, maxc;
  int o_vel, o_vb, o_tc, o_wkey, o_wjn, o_page, o_pjn, o_sc, o_ep, o_flags, o_near, rec_words;
  int r_bytes, r_off_type, r_off_reward, r_off_flags;
  int rp_bytes, rp_off_reward, rp_off_flags;   // the same record with the types packed 4 to a byte (host-facing path)
  int s_rdist, s_rtype, s_min, s_rcell, s_nearcnt, s_con, s_ccount, s_order, s_best, s_cand, scratch_bytes;
};
__host__ __device__ constexpr int layout_align(int v, int a) { return (v + a - 1) / a * a; }
__host__ __device__ constexpr Layout make_layout(int A, int R) {
  Layout l{};
  l.P = A * (A - 1) / 2; l.nrays = A * R; l.nrays_pad = layout_align(A * R, 32); l.maxc = A * kSlots + l.P;
  l.o_vel = 2 * A; l.o_vb = 4 * A; l.o_tc = 6 * A; l.o_wkey = 8 * A; l.o_wjn = 8 * A + A * kSlots;
  l.o_page = 8 * A + 2 * A * kSlots; l.o_pjn = l.o_page + l.P; l.o_sc = l.o_pjn + l.P; l.o_ep = l.o_sc + 1; l.o_flags = l.o_ep + 1;
  l.o_near = l.o_flags + 1;                                   // u16 [A][kNear]: hulls within ray_r of each body (0xFFFF = none)
  l.rec_words = layout_align(l.o_near + (A * kNear + 1) / 2, 32);
  // the world's output record, staged contiguously (CatRecordLayout): f16 distances | u8 types | f32 rewards | flags
  l.r_off_type = layout_align(l.nrays * 2, 16);
  l.r_off_reward = layout_align(l.r_off_type + l.nrays, 4);
  l.r_off_flags = l.r_off_reward + 4 * A;
  l.r_bytes = layout_align(l.r_off_flags + 3, 16);
  // ... and its host-facing form: the u8 types packed to 2 bits each, in place at the same offset; rewards and flags follow
  l.rp_off_reward = layout_align(l.r_off_type + (l.nrays + 3) / 4, 4);
  l.rp_off_flags = l.rp_off_reward + 4 * A;
  l.rp_bytes = layout_align(l.rp_off_flags + 3, 16);
  int so = l.rec_words * 4;
  l.s_rdist = so; so = layout_align(so + l.r_bytes, 16);
  l.s_rtype = l.s_rdist + l.r_off_type;
  l.s_min = so; so = layout_align(so + CAT_MAX_AGENTS * 4, 16);
  l.s_rcell = so; so = layout_align(so + CAT_MAX_AGENTS * 4, 16);      // (holds the warp's mbarrier)
  l.s_nearcnt = so; so = layout_align(so + CAT_MAX_AGENTS * 4, 16);
  l.s_con = so; so = layout_align(so + l.maxc * 32, 16);
  l.s_ccount = so; so = layout_align(so + CAT_MAX_AGENTS * 4, 16);
  l.s_order = so; so = layout_align(so + l.maxc, 16);
  // per-ray hit keys; with ray lists the same area first holds the rays' 16-byte candidate slots
  l.s_best = so; so = layout_align(so + l.nrays_pad * 16, 16);
  l.s_cand = so; so = layout_align(so + 64 * 2, 16);
  l.scratch_bytes = layout_align(so, 128);
  return l;
}

// inside a function templated on <TM>: a map-dependent value — from the blob header the CTA staged (TM: a mixed-map
// launch, every CTA may run another map) or from the parameters (a single-map launch, constant-bank operands)
#define MAPK(blob, f) (TM ? blob_header(blob)->f : k.f)

template <int TA, int TR> struct FixedLayout { static constexpr Layout v = make_layout(TA ? TA : 1, TR ? TR : 1); };
// inside a function templated on <TA, TR>: the layout value as an immediate (shipped shape) or from the parameters
#define LAY(f) (TA ? FixedLayout<TA, TR>::v.f : k.lay.f)

// One map's share of a launch: CTAs [cta_begin, next entry's cta_begin or gridDim.x) step the worlds
// [world_begin, world_end) of the environment, all of them on the map whose blob they stage.
struct MapSlice {
  const unsigned char* blob;
  int blob_bytes;
  int cta_begin;
  int world_begin, world_end;
};

struct KParams {
  // The map of a single-map launch (the instantiations with TM = false).  A mixed-map launch (TM = true) finds its
  // CTA's blob in `maps` below and every other map-dependent value in that blob's header (BlobHeader).
  const unsigned char* blob;
  int blob_bytes;
  const int32_t* view_off;      // global memory: per grid cell candidate-edge lists (nullptr = scan all edges)
  const uint16_t* view_edges;
  // per (cell, ray) candidate lists (ray_lists.h): slots [cells * R] of 4 words + overflow words; nullptr = rasterise
  const uint4* ray_slots;
  const uint32_t* ray_ovf;
  float rg_x0, rg_y0, rg_inv_cell;
  int rg_nx, rg_ny;
  unsigned int ray_slot_count, ray_ovf_words;   // sizes of the two arrays (checked build only)
  unsigned long long* overflow;  // [2] wall-contact / near-hull slots exceeded (cat_env_overflow_counts)
  float* state;
  int n_worlds;
  int world_begin, world_end;   // the slice of worlds this launch steps (chunked host path); default [0, n_worlds)
  long long gid0;
  int A, nc, R, n_edges;
  int mode;
  Layout lay;      // record offsets (words), per-warp scratch offsets (bytes), output-record offsets: make_layout(A, R)
  int state_dim;
  // constants
  float dt, inv_dt, impulse, inv_mass, agent_r, max_speed, term_r, ray_len, ray_r, wall_r;
  float slop, bias_coef;
  int iterations, persistence, max_steps, stale, auto_reset;
  unsigned long long seed;
  // I/O
  const void* actions[CAT_MAX_AGENTS];
  int actions_kind;
  const uint8_t* reset_mask;
  uint16_t* shared_dist;
  uint8_t* shared_type;
  uint16_t* team_pos;
  float* obs_f32;
  float* state_f32;
  float* hit_point;
  unsigned char* record;          // record output: one r_bytes block per world, record_stride apart
  int record_stride;
  int record_packed;              // types packed 4 to a byte (rp_bytes per world): what crosses PCIe on the host path
  float* critic_f32;
  uint16_t* obs_bf16;
  uint16_t* critic_bf16;
  // The launch's maps, by value (no device table, graph-capturable): entries in increasing cta_begin and world order,
  // together covering [world_begin, world_end).  Read by the TM = true instantiations only; a single-map launch fills
  // one entry that mirrors the fields above.
  int n_maps;
  MapSlice maps[CAT_MAX_MAPS];
  // Final outputs (CatStepIO.final_*): what a world that ends in this step would have emitted with auto_reset = 0.  Set by
  // step launches only and read by the TX = true instantiations only (kernel_for never picks the record-only one for them).
  unsigned char* final_record;    // unpacked record, final_record_stride apart
  int final_record_stride;
  float* final_obs_f32;
  float* final_state_f32;
  float* final_critic_f32;
  // Episode statistics (cat_env_attach_episode_stats), carried by every launch of the environment while attached and read
  // by the TX = true instantiations only (kernel_for never picks the record-only one while ep_acc is set).
  float* ep_acc;                  // [N][A] running returns
  float* ep_return;               // [N][A] return of the episode a world ended in this step
  int32_t* ep_length;             // [N]
  CatEpisodeTotals* ep_totals;    // [n_maps]
  int map_slot0;                  // the environment's map slot of maps[0] (a host-path chunk's table starts at its first map)
  // Per-world parameters (cat_env_attach_world_params), carried like the statistics and read by the TX = true
  // instantiations only (kernel_for never picks the record-only one while wp is set).
  CatWorldParams* wp;                      // [N]
  const CatWorldParamRanges* wp_ranges;    // [n_maps], by map slot like ep_totals; nullptr = never draw
  // Scripted agents (cat_env_attach_scripts), carried like the statistics and read by the TX = true instantiations only
  // (kernel_for never picks the record-only one while script_mode is set).  Both set or both null.
  const uint8_t* script_mode;     // [N][A] CAT_SCRIPT_*
  uint8_t* script_dec;            // [N][A] the controllers' decisions from the last emitted observation
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ MapView make_view(const unsigned char* blob) {
  const BlobHeader* h = reinterpret_cast<const BlobHeader*>(blob);
  MapView m;
  m.edge = reinterpret_cast<const float4*>(blob + h->off_edge);
  m.edge_len = reinterpret_cast<const float*>(blob + h->off_len);
  m.hull_bb = reinterpret_cast<const float4*>(blob + h->off_hbb);
  m.hull_eo = reinterpret_cast<const uint32_t*>(blob + h->off_heo);
  m.next_n = reinterpret_cast<const float2*>(blob + h->off_nextn);
  m.batch_bb = reinterpret_cast<const float4*>(blob + h->off_batchbb);
  m.edge_hull = reinterpret_cast<const uint16_t*>(blob + h->off_edgehull);
  m.con_off = reinterpret_cast<const uint16_t*>(blob + h->off_conoff);
  m.con_list = reinterpret_cast<const uint16_t*>(blob + h->off_conlist);
  m.dir = reinterpret_cast<const float4*>(blob + h->off_dir);
  m.reg_off = reinterpret_cast<const int32_t*>(blob + h->off_regoff);
  m.regions = reinterpret_cast<const float4*>(blob + h->off_regions);
  m.init_pos = reinterpret_cast<const float2*>(blob + h->off_initpos);
  m.H = h->n_hulls; m.nx = h->nx; m.ny = h->ny; m.n_edges = h->n_edges;
  m.gx0 = h->gx0; m.gy0 = h->gy0; m.cell = h->cell; m.inv_cell = h->inv_cell;
  return m;
}

// ------------------------------------------------------------------ geometry (device)

// Closest feature of the raw hull to point p (CircleToPoly's GJK/EPA result for a point):
// d = signed distance (negative inside: least-penetration edge), n = unit vector from p towards
// the hull surface.  Same quantity cpPolyShapePointQuery reports as +-minDist.  Everything is
// evaluated relative to the hull's own vertices so that d keeps ~1e-6 absolute accuracy.
__device__ __noinline__ float3 hull_closest_impl(const float4* __restrict__ edge, uint32_t eo, float px, float py) {
  const int o = eo & 0xFFFF, n = eo >> 16;
  bool inside = true, binterior = false;
  float maxpd = -CUDART_INF_F, mnx = 0.f, mny = 0.f;
  float bestd2 = CUDART_INF_F, bdx = 0.f, bdy = 0.f, benx = 0.f, beny = 0.f, bpd = 0.f;
  float4 pv = edge[o + n - 1];
  float v0x = pv.x, v0y = pv.y;
#pragma unroll 1
  for (int i = 0; i < n; ++i) {
    const float4 e = edge[o + i];
    const float pd = (px - e.x) * e.z + (py - e.y) * e.w;
    if (pd > 0.f) inside = false;
    if (pd > maxpd) { maxpd = pd; mnx = e.z; mny = e.w; }
    const float edx = e.x - v0x, edy = e.y - v0y;
    const float r0x = px - v0x, r0y = py - v0y;
    float t = (r0x * edx + r0y * edy) / (edx * edx + edy * edy);
    const bool interior = (t > 0.f) && (t < 1.f);
    t = fminf(fmaxf(t, 0.f), 1.f);
    const float ddx = r0x - edx * t, ddy = r0y - edy * t;  // p - q
    const float d2 = interior ? pd * pd : ddx * ddx + ddy * ddy;
    if (d2 < bestd2) { bestd2 = d2; bdx = ddx; bdy = ddy; benx = e.z; beny = e.w; binterior = interior; bpd = pd; }
    v0x = e.x; v0y = e.y;
  }
  if (inside) return make_float3(maxpd, -mnx, -mny);
  if (binterior) return make_float3(fabsf(bpd), -benx, -beny);
  const float d = sqrtf(bestd2);
  const float inv = 1.f / (d + 1.17549435e-38f);
  return make_float3(d, -bdx * inv, -bdy * inv);
}

__device__ __forceinline__ void hull_closest(const MapView& m, int h, float px, float py, float& d, float& nx,
                                             float& ny) {
  const float3 r = hull_closest_impl(m.edge, m.hull_eo[h], px, py);
  d = r.x; nx = r.y; ny = r.z;
}

// cpBBSegmentQuery(bb, a, b) < 1: the BB-tree visits a leaf only if the THIN segment enters its bb.
// (idx, idy) = 1 / (b - a) per axis (unused where the delta is exactly zero).
__device__ __forceinline__ bool thin_bb_hit(const float4 bb, float ox, float oy, bool zx, bool zy, float idx,
                                            float idy) {
  float tmin = -CUDART_INF_F, tmax = CUDART_INF_F;
  if (zx) {
    if (ox < bb.x || bb.z < ox) return false;
  } else {
    const float t1 = (bb.x - ox) * idx, t2 = (bb.z - ox) * idx;
    tmin = fminf(t1, t2);
    tmax = fmaxf(t1, t2);
  }
  if (zy) {
    if (oy < bb.y || bb.w < oy) return false;
  } else {
    const float t1 = (bb.y - oy) * idy, t2 = (bb.w - oy) * idy;
    tmin = fmaxf(tmin, fminf(t1, t2));
    tmax = fminf(tmax, fmaxf(t1, t2));
  }
  return (tmin <= tmax) && (0.f <= tmax) && (tmin < 1.f);
}

__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Depth-buffer key of a ray: (float bits of s) << 32 | feature.  Walls: edge * 2 + (1 = bevelled vertex);
// agents: kAgentTag + j — larger than any wall feature, so at equal s the static shape wins, like
// cpSpaceSegmentQueryFirst (static index first, dynamic only if strictly closer).  s = distance along
// the ray of the fat-ray centre at first touch (alpha * L).
constexpr uint32_t kAgentTag = 0x40000000u;
constexpr uint32_t kNoFeature = 0xFFFFFFFFu;
__device__ __forceinline__ unsigned long long make_key(float s, uint32_t feat) {
  return ((unsigned long long)__float_as_uint(s) << 32) | feat;
}

// atan2 to ~1e-4 rad (odd minimax polynomial on [0,1] + octant folding); callers pad their angular
// spans by 2e-3 rad, so this only ever adds a spare (edge, ray) test, never drops one.
__device__ __forceinline__ float fast_atan2(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float a = __fdividef(fminf(ax, ay), fmaxf(fmaxf(ax, ay), 1e-30f));
  const float q = a * a;
  float r = fmaf(fmaf(fmaf(-0.0464964749f, q, 0.15931422f), q, -0.327622764f), q * a, a);
  if (ay > ax) r = 1.57079637f - r;
  if (x < 0.f) r = 3.14159274f - r;
  return copysignf(r, y);
}

// float16(npy_hypotf(dx, dy)) for float16-valued dx, dy: numpy evaluates hypotf (glibc: sqrt in double, rounded to
// float) and then rounds to half.  dx*dx and dy*dy are exact in fp32 (11-bit significands), so
// sqrt.rn.f32(fma(dx, dx, dy*dy)) is within 1.5 fp32 ulp of that float; the two can only round to different
// halves when the low 13 bits sit within 2 ulp of the tie point (or in the half-subnormal range): only then is the
// double-precision path taken (about 6 rays in 10^4).
__device__ __forceinline__ uint16_t half_hypot_bits(float dxh, float dyh) {
  float hyp = __fsqrt_rn(fmaf(dxh, dxh, dyh * dyh));
  const uint32_t low = __float_as_uint(hyp) & 0x1FFFu;
  if ((low - 0x0FFEu <= 4u) || hyp < 6.2e-5f) hyp = (float)sqrt((double)dxh * (double)dxh + (double)dyh * (double)dyh);
  return __half_as_ushort(__float2half_rn(hyp));
}

struct Ray {
  float ox, oy, ux, uy, L;
  bool zx, zy;      // direction component exactly zero (cpBBSegmentQuery special case)
  float idx, idy;   // 1 / (L * u)
};

// One edge of cpPolyShapeSegmentQuery against the ray o + s*u: plane i offset by rsum = wall_r + ray_r
// (accepted inside the edge's tangential extent) and the bevelled vertex v_i as a circle of radius rsum
// (CircleSegmentQuery, perpendicular-offset form of the discriminant).  Returns the smaller s (INF if
// neither is hit; range / nearest checks are the caller's) and which of the two it was.
__device__ __forceinline__ float ray_edge(const float4 e, float len, const Ray& r, float rsum, float rs2, int& kind) {
  const float rx = r.ox - e.x, ry = r.oy - e.y;
  const float d = fmaf(rx, e.z, fmaf(ry, e.w, -rsum));   // a.n - v0.n - rsum
  const float un = fmaf(r.ux, e.z, r.uy * e.w);          // (b.n - a.n) / L
  float s = CUDART_INF_F;
  kind = 0;
  if (d >= 0.f && un < 0.f) {
    const float sp = __fdividef(d, -un);
    const float c = fmaf(e.z, fmaf(sp, r.uy, ry), -e.w * fmaf(sp, r.ux, rx));  // cross(n, P - v_i) in [-len, 0]
    if (c <= 0.f && c >= -len) s = sp;
  }
  const float cp = fmaf(rx, r.uy, -ry * r.ux);
  const float disc = fmaf(-cp, cp, rs2);
  if (disc >= 0.f) {
    const float sc = -fmaf(rx, r.ux, ry * r.uy) - fast_sqrt(disc);
    if (sc >= 0.f && sc < s) { s = sc; kind = 1; }
  }
  return s;
}

// Surface normal of a wall hit (plane: the edge normal; bevel: from the vertex to the ray centre).
__device__ __forceinline__ float2 wall_hit_normal(const MapView& m, uint32_t feat, float s, const Ray& r, float rsum) {
  const float4 e = m.edge[feat >> 1];
  if ((feat & 1u) == 0) return make_float2(e.z, e.w);
  const float inv = 1.f / rsum;
  return make_float2((r.ox - e.x + s * r.ux) * inv, (r.oy - e.y + s * r.uy) * inv);
}

__device__ __forceinline__ Ray make_ray(float ax, float ay, float dx, float dy) {
  Ray r;
  r.ox = ax; r.oy = ay;
  r.L = sqrtf(dx * dx + dy * dy);
  const float inv = r.L > 0.f ? 1.f / r.L : 0.f;
  r.ux = dx * inv; r.uy = dy * inv;
  r.zx = dx == 0.f; r.zy = dy == 0.f;
  r.idx = r.zx ? 0.f : 1.f / dx;
  r.idy = r.zy ? 0.f : 1.f / dy;
  return r;
}

// Thin segment a -> b against the wall hulls h0, h0+32, ... with query radius 0 (capture line of
// sight, base_env.py:536-544): true if any blocks (alpha < 1), including the alpha = 0 rule.
// Rare path (only evaluated for thief-cop pairs closer than the capture radius): not inlined.
__device__ __noinline__ bool los_blocked(const unsigned char* blob, int h0, float ax, float ay, float bx, float by,
                                         float wall_r) {
  const MapView m = make_view(blob);
  const Ray r = make_ray(ax, ay, bx - ax, by - ay);
  bool blocked = false;
#pragma unroll 1
  for (int h = h0; h < m.H && !blocked; h += 32) {
    if (!thin_bb_hit(m.hull_bb[h], ax, ay, r.zx, r.zy, r.idx, r.idy)) continue;
    const float3 c = hull_closest_impl(m.edge, m.hull_eo[h], ax, ay);
    if (c.x - wall_r <= 0.f) { blocked = true; break; }  // start point inside the rounded hull
    if (!(r.L > 0.f)) continue;
    const uint32_t eo = m.hull_eo[h];
#pragma unroll 1
    for (int ei = eo & 0xFFFF, ee = (eo & 0xFFFF) + (eo >> 16); ei < ee && !blocked; ++ei) {
      int kind;
      blocked = ray_edge(m.edge[ei], m.edge_len[ei], r, wall_r, wall_r * wall_r, kind) < r.L;  // alpha < 1
    }
  }
  return blocked;
}

__device__ __forceinline__ int grid_cell(const MapView& m, float x, float y) {
  const float gx = (x - m.gx0) * m.inv_cell, gy = (y - m.gy0) * m.inv_cell;
  if (!(gx >= 0.f && gy >= 0.f && gx < (float)m.nx && gy < (float)m.ny)) return -1;
  return (int)gy * m.nx + (int)gx;
}

// ------------------------------------------------------------------ per-warp world context
struct Warp {
  float* rec;
  uint16_t* rdist;
  uint8_t* rtype;
  uint32_t* minbits;
  uint16_t* near;
  uint32_t* nearcnt;
  float* con;       // contact entries, 8 words each
  uint32_t* ccount; // wall contacts per agent
  uint8_t* order;   // compact solver order
  unsigned long long* best;  // per ray: (float bits of s) << 32 | feature id  — the 1-D depth buffer
  uint16_t* cand;   // candidate edge ids awaiting rasterisation
  float* rew;       // staged rewards [A] and flags {terminated, truncated, winner} of the world's output record
  uint8_t* flg;
  unsigned long long* mbar;   // the warp's own mbarrier: completion of the staged ray slots
  const unsigned char* blob;  // the map blob in shared memory
  int lane;
};

// Rasterise up to 32 candidate edges (cand[0..n)) of one agent into its per-ray depth buffer `best`.
// Lane l owns candidate l and computes the span of ray indices whose thin line can come within rsum of
// the edge (conservative: angle of the offset segment's far end and of the bevel circle, padded); the
// (edge, ray) pairs of all 32 spans are then flattened with a warp scan so that every lane tests one
// pair per iteration regardless of how uneven the spans are.  Not inlined: one compact copy keeps the
// kernel's instruction footprint inside the instruction cache.
__device__ __noinline__ void raster_batch(const unsigned char* blob, unsigned long long* best, const uint16_t* cand,
                                          int n, float ox, float oy, float rsum, float L, int R) {
  const MapView m = make_view(blob);
  const int lane = threadIdx.x & 31;
  const float rs2 = rsum * rsum, inv_L = 1.f / L;
  int e = 0, i0 = 0, cnt = 0;
  if (lane < n) {
    e = cand[lane];
    const float4 ed = m.edge[e];
    const float bx = ed.x - ox, by = ed.y - oy;           // B - o (B = v_i, the vertex ending the edge)
    const float nb2 = bx * bx + by * by;
    if (nb2 <= rs2) { cnt = R; }                           // origin inside the bevel circle: every direction
    else {
      const float thB = fast_atan2(by, bx);
      const float x = fminf(rsum * rsqrtf(nb2), 1.f);
      const float wv = x * fmaf(0.5708f, x * x, 1.f);     // >= asin(x) on [0,1]: half-width of the bevel circle
      float lo = -wv, hi = wv;
      const float pd = -(bx * ed.z + by * ed.w);          // (o - B).n
      if (pd - rsum >= 0.f) {
        // offset segment A'B' (B' lies on the bevel circle, already covered): far end A' = B - len*t + n*rsum
        const float len = m.edge_len[e];
        const float apx = bx + ed.z * rsum + len * ed.w, apy = by + ed.w * rsum - len * ed.z;   // t = (-ny, nx)
        float dA = fast_atan2(apy, apx) - thB;
        dA = dA > CUDART_PI_F ? dA - 2.f * CUDART_PI_F : (dA < -CUDART_PI_F ? dA + 2.f * CUDART_PI_F : dA);
        lo = fminf(lo, dA); hi = fmaxf(hi, dA);
      }
      const float pad = 2e-3f;
      const float inv_dth = (float)R * (0.5f / CUDART_PI_F);
      const int ilo = (int)ceilf((thB + lo - pad) * inv_dth), ihi = (int)floorf((thB + hi + pad) * inv_dth);
      cnt = min(max(ihi - ilo + 1, 0), R);
      i0 = ilo;                                            // |ilo| < 2R
      if (i0 < 0) i0 += R;
      if (i0 < 0) i0 += R;
      if (i0 >= R) i0 -= R;
      if (cnt > 0 && cnt <= 3) {
        // Occlusion: a narrow (far) edge whose every ray already holds a strictly nearer hit cannot win the
        // depth test.  Any hit on this edge or its bevel has s >= dist(origin, raw segment) - rsum.
        const float len = m.edge_len[e];
        const float qa = fmaf(-by, ed.z, bx * ed.w);        // position of o along A->B, relative to B
        const float dq = qa - fminf(fmaxf(qa, -len), 0.f);
        const float smin = fast_sqrt(fmaf(pd, pd, dq * dq)) * 0.9999f - rsum - 1e-3f;
        bool occluded = true;
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          int i = i0 + q;
          if (i >= R) i -= R;
          if (q < cnt) occluded = occluded && __uint_as_float((uint32_t)(best[i] >> 32)) < smin;
        }
        CAT_COUNT(2, 1);
        if (occluded) { cnt = 0; CAT_COUNT(3, 1); }
      }
    }
    CAT_COUNT(0, 1);
    CAT_COUNT(1, cnt);
  }
  int scan = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, scan, d); if (lane >= d) scan += t; }
  const int total = __shfl_sync(0xFFFFFFFFu, scan, 31);
  const int excl = scan - cnt;
#pragma unroll 1
  for (int p0 = 0; p0 < total; p0 += 32) {
    const int p = p0 + lane;
    int l = 0;   // owner = first lane whose inclusive scan exceeds p
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
      const int v = __shfl_sync(0xFFFFFFFFu, scan, l + step - 1);
      if (v <= p) l += step;
    }
    l = min(l, 31);
    const int el = __shfl_sync(0xFFFFFFFFu, e, l), i0l = __shfl_sync(0xFFFFFFFFu, i0, l);
    const int exl = __shfl_sync(0xFFFFFFFFu, excl, l);
    if (p < total) {
      int i = i0l + (p - exl);
      if (i >= R) i -= R;
      CAT_CHECK(i >= 0 && i < R && el >= 0 && el < m.n_edges);
      const float4 dv = m.dir[i];
      Ray r;
      r.ox = ox; r.oy = oy; r.ux = dv.x; r.uy = dv.y; r.L = L;
      r.zx = dv.x == 0.f; r.zy = dv.y == 0.f; r.idx = dv.z * inv_L; r.idy = dv.w * inv_L;
      int kind;
      const float sHit = ray_edge(m.edge[el], m.edge_len[el], r, rsum, rs2, kind);
      if (sHit < L) {
        unsigned long long* slot = &best[i];
        const unsigned long long key = make_key(sHit, (uint32_t)(el * 2 + kind));
        // cpBBTree leaf test: a hull is only ever visited if the THIN ray enters its bb (rarely fails, so
        // it is evaluated only for hits that would win the depth test)
        if (key < *slot && thin_bb_hit(m.hull_bb[m.edge_hull[el]], ox, oy, r.zx, r.zy, r.idx, r.idy)) atomicMin(slot, key);
      }
    }
  }
}

// Candidate generation + rasterisation of one agent's walls into its depth buffer — the any-map path (no
// per-(cell, ray) lists: environments created with ray_list_cell < 0).  lanes = edges: candidates face the origin
// (plane i or the next plane, which share vertex v_i and hence its bevel) and lie within sensor range.  Batches
// of 32 edges (hulls are stored in Morton order, so a batch is compact) are visited NEAR TO FAR: lane b measures
// the distance of batch b's bounding box once, a counting rank orders them, and the walk stops at the first batch
// beyond sensor range; the per-grid-cell static lists (maps.view_lists) shorten the scan when present.
template <bool TM>
__device__ __noinline__ void rasterise_agent(const KParams& k, const unsigned char* blob, unsigned char* scratch, int a,
                                             float ox, float oy) {
  // (scalars, not the Warp struct: a struct passed by reference to an out-of-line function would live in local memory)
  const MapView m = make_view(blob);
  struct { unsigned long long* best; uint16_t* cand; const unsigned char* blob; int lane; } w;
  w.best = reinterpret_cast<unsigned long long*>(scratch + k.lay.s_best);
  w.cand = reinterpret_cast<uint16_t*>(scratch + k.lay.s_cand);
  w.blob = blob; w.lane = threadIdx.x & 31;
  const int R = k.R, lane = w.lane, E = MAPK(blob, n_edges);
  const float L = k.ray_len, rsum = k.wall_r + k.ray_r;
  const float range2 = (L + rsum) * (L + rsum);
  int ncand = 0;
  const int nb = (E + 31) >> 5;
  int vq = 0, vq1 = 0;
  const int vcell = MAPK(blob, view_off) ? grid_cell(m, ox, oy) : -1;
  const bool use_view = vcell >= 0;
  uint32_t vnext = 0xFFFFu;
  if (use_view) {
    vq = __ldg(MAPK(blob, view_off) + vcell); vq1 = __ldg(MAPK(blob, view_off) + vcell + 1);
    if (vq + lane < vq1) vnext = __ldg(MAPK(blob, view_edges) + vq + lane);
  }
  const bool ordered = !use_view && nb <= 32;
  float bdist = CUDART_INF_F;
  int brank = 0;
  if (ordered) {
    if (lane < nb) {
      const float4 bb = m.batch_bb[lane];
      const float ddx = fmaxf(fmaxf(bb.x - ox, ox - bb.z), 0.f), ddy = fmaxf(fmaxf(bb.y - oy, oy - bb.w), 0.f);
      bdist = fmaf(ddx, ddx, ddy * ddy);
    }
#pragma unroll 1
    for (int j = 0; j < nb; ++j) {
      const float dj = __shfl_sync(0xFFFFFFFFu, bdist, j);
      brank += (dj < bdist || (dj == bdist && j < lane)) ? 1 : 0;
    }
  }
#pragma unroll 1
  for (int it = 0; ; ++it) {
    int e;
    if (use_view) {
      if (vq >= vq1) break;
      e = vnext == 0xFFFFu ? E : (int)vnext;
      vq += 32;
      vnext = vq + lane < vq1 ? (uint32_t)__ldg(MAPK(blob, view_edges) + vq + lane) : 0xFFFFu;
    } else {
      if (it >= nb) break;
      int base;
      if (ordered) {
        const int b = __ffs(__ballot_sync(0xFFFFFFFFu, lane < nb && brank == it)) - 1;
        if (__shfl_sync(0xFFFFFFFFu, bdist, b) >= range2) break;   // this and every later batch is out of range
        base = b << 5;
      } else {
        base = it << 5;
        const float4 bb = m.batch_bb[it];
        const float ddx = fmaxf(fmaxf(bb.x - ox, ox - bb.z), 0.f), ddy = fmaxf(fmaxf(bb.y - oy, oy - bb.w), 0.f);
        if (fmaf(ddx, ddx, ddy * ddy) >= range2) continue;
      }
      e = base + lane;
    }
    bool is_cand = false;
    if (e < E) {
      const float4 ed = m.edge[e];
      const float2 nn = m.next_n[e];
      const float rx = ox - ed.x, ry = oy - ed.y;
      const float pd = rx * ed.z + ry * ed.w;
      const float pdn = rx * nn.x + ry * nn.y;
      const float len = m.edge_len[e];
      const float qa = fmaf(ry, ed.z, -rx * ed.w);       // position of o along A->B, relative to B
      const float dq = qa - fminf(fmaxf(qa, -len), 0.f);
      is_cand = (pd > 0.f || pdn > 0.f) && (fmaf(pd, pd, dq * dq) < range2);
    }
    const uint32_t cmask = __ballot_sync(0xFFFFFFFFu, is_cand);
    CAT_CHECK(ncand + __popc(cmask) <= 64);
    if (is_cand) w.cand[ncand + __popc(cmask & ((1u << lane) - 1u))] = (uint16_t)e;
    ncand += __popc(cmask);
    __syncwarp();
    if (ncand >= 32) {
      raster_batch(w.blob, w.best + a * R, w.cand, 32, ox, oy, rsum, L, R);
      __syncwarp();
      uint16_t t = 0;
      if (lane + 32 < ncand) t = w.cand[lane + 32];
      __syncwarp();
      if (lane + 32 < ncand) w.cand[lane] = t;
      ncand -= 32;
      __syncwarp();
    }
  }
  if (ncand > 0) raster_batch(w.blob, w.best + a * R, w.cand, ncand, ox, oy, rsum, L, R);
  __syncwarp();
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
#pragma unroll 1
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"   // %3: suspend-time hint (ns): sleep, do not spin
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity), "r"(4000)
        : "memory");
  }
}

// Per-warp state of the slot staging: which phase of the warp's mbarrier the next wait is for, and whether a
// staging is in flight (a world that ends and re-spawns in one step stages twice before it sweeps once).
struct SlotStage { uint32_t phase; bool pending; };

// Stage the (cell, ray) slots of every ray of the world into shared memory.  The R slots of one agent are
// contiguous in global memory (slot index = cell * R + ray), so each agent is ONE TMA bulk copy (cp.async.bulk,
// 16 R bytes) issued by lane 0 and completing on the warp's own mbarrier — no registers, no per-ray address
// arithmetic — started as early as the positions are known so that the L2 / HBM latency hides behind the
// termination test and the action impulses.  Slot r lands at w.best + 2 r (16-byte stride); the walk later writes
// ray r's result key over the first half of its own slot.
template <int TA, int TR, bool TM>
__device__ __forceinline__ void stage_ray_slots(const KParams& k, const Warp& w, SlotStage& st) {
  const int A = TA ? TA : k.A, R = TR ? TR : k.R, lane = w.lane;
  const float* pos = w.rec;
  const uint32_t bar = smem_u32(w.mbar);
  if (st.pending) { mbar_wait(bar, st.phase); st.phase ^= 1u; }
  int base = -1;   // outside the grid: farther than the sensor reach from every wall
  if (lane < A) {
    const float gx = (pos[2 * lane] - MAPK(w.blob, rg_x0)) * MAPK(w.blob, rg_inv_cell), gy = (pos[2 * lane + 1] - MAPK(w.blob, rg_y0)) * MAPK(w.blob, rg_inv_cell);
    if (gx >= 0.f && gy >= 0.f && gx < (float)MAPK(w.blob, rg_nx) && gy < (float)MAPK(w.blob, rg_ny)) base = ((int)gy * MAPK(w.blob, rg_nx) + (int)gx) * R;
  }
  const uint32_t inside = __ballot_sync(0xFFFFFFFFu, base >= 0);   // (also orders the previous world's reads of the slot area)
  if (lane == 0) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy accesses of the area before the async-proxy writes
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(__popc(inside) * R * 16) : "memory");
  }
#pragma unroll 1
  for (int a = 0; a < A; ++a) {
    const int ba = __shfl_sync(0xFFFFFFFFu, base, a);
    uint4* dst = reinterpret_cast<uint4*>(w.best) + a * R;
    if (ba >= 0) {
      CAT_CHECK((unsigned)(ba + R) <= MAPK(w.blob, ray_slot_count) && (a + 1) * R * 16 <= LAY(nrays_pad) * 16);
      if (lane == 0)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                     "l"(MAPK(w.blob, ray_slots) + ba), "r"(R * 16), "r"(bar)
                     : "memory");
    } else {
#pragma unroll 1
      for (int i = lane; i < R; i += 32) dst[i] = make_uint4(kRayEnd, kRayEnd, kRayEnd, kRayEnd);
    }
  }
  st.pending = true;
}

// Wall hits of EVERY ray of the world from the per-(cell, ray) candidate lists (ray_lists.h).
//
// lanes = rays, assigned dynamically: a lane walks its ray's list nearest bound first — one exact
// cpPolyShapeSegmentQuery edge test per iteration — until the hit it holds is nearer than the next entry's lower
// bound, then publishes the hit (over its own slot) and takes the next ray nobody has taken.  No candidate
// generation, no angular spans, no scan / search, no atomics: the work per ray is the 1-3 edges its fat ray can
// actually meet before its first hit.
//   The BB-tree leaf rule (a hull counts only if the THIN ray enters its bounding box) is checked once, on the
// winner; if it fails (a grazing fat ray) the list is walked again with the rule applied to every hit.
//   Hit key = (float bits of s, feature): smaller s first, then smaller feature — the order of the rasteriser's
// 64-bit atomicMin, so both paths pick the same hit bit for bit.
template <int TA, int TR, bool TM>
__device__ __forceinline__ void sweep_lists(const KParams& k, const MapView& m, const Warp& w, SlotStage& st) {
  const int A = TA ? TA : k.A, R = TR ? TR : k.R, nrays = A * R, lane = w.lane;
  const float L = k.ray_len, rsum = k.wall_r + k.ray_r, rs2 = rsum * rsum, inv_L = 1.f / k.ray_len;
  const float inv_R = 1.f / (float)R;
  const float* pos = w.rec;
  uint4* slots = reinterpret_cast<uint4*>(w.best);
  mbar_wait(smem_u32(w.mbar), st.phase);   // the staged slots have landed
  st.phase ^= 1u; st.pending = false;
  __syncwarp();
  const uint32_t kLbits = __float_as_uint(L);
  const uint32_t lt = (1u << lane) - 1u;
  int cur = lane < nrays ? lane : -1;
  int next = 32;                       // warp-uniform: first ray nobody has taken yet
  uint32_t e0 = kRayEnd, e1 = kRayEnd, e2 = kRayEnd, e3 = kRayEnd;
  bool strict = false;
  float ox = 0.f, oy = 0.f, ux = 0.f, uy = 0.f;
  int ci = 0;
  uint32_t bs = kLbits, bf = kNoFeature;   // the hit held: float bits of s, feature
  auto start_ray = [&](int ray) {
    int a = 0;
    if (TA) {
#pragma unroll
      for (int j = 1; j < (TA ? TA : 1); ++j) a += ray >= j * R ? 1 : 0;
    } else a = __float2int_rz(((float)ray + 0.5f) * inv_R);
    ci = ray - a * R;
    const float2 o = *reinterpret_cast<const float2*>(pos + 2 * a);
    ox = o.x; oy = o.y;
    const float2 dv = *reinterpret_cast<const float2*>(m.dir + ci);
    ux = dv.x; uy = dv.y;
    const uint4 sl = slots[ray];
    e0 = sl.x; e1 = sl.y; e2 = sl.z; e3 = sl.w;
    // (no prefetch of the overflow chunk a long list continues in: the 64-bit address arithmetic at every ray start cost
    //  more than the L1 hit saved — 183 -> 175 us on agh-map x 16384 without it)
    bs = kLbits; bf = kNoFeature;
  };
  if (cur >= 0) start_ray(cur);
#pragma unroll 1
  while (__any_sync(0xFFFFFFFFu, cur >= 0)) {
    bool fin = false;
    if (cur >= 0) {
      uint32_t ent = e0;
      if (__builtin_expect((int)ent < 0, 0)) {   // link: the list continues in a chunk of the overflow array
        // (TM: the pointer is read here, on the rare path, so no register holds it across the walk)
        CAT_CHECK((ent & 0x7FFFFFFFu) + 4u <= MAPK(w.blob, ray_ovf_words) && ((ent & 3u) == 0u));
        const uint4 c = __ldg(reinterpret_cast<const uint4*>(MAPK(w.blob, ray_ovf) + (ent & 0x7FFFFFFFu)));
        ent = c.x; e1 = c.y; e2 = c.z; e3 = c.w;
      }
      e0 = e1; e1 = e2; e2 = e3; e3 = kRayEnd;
      if (__uint_as_float(bs) < __uint_as_float(ent & 0xFFFF0000u)) fin = true;   // (an empty list: its first entry is the end mark)
      else {
        const uint32_t el = ent & 0xFFFFu;
        CAT_CHECK((int)el < MAPK(w.blob, n_edges) && cur < nrays);
        Ray r;
        r.ox = ox; r.oy = oy; r.ux = ux; r.uy = uy; r.L = L;
        int kind;
        const float sHit = ray_edge(m.edge[el], m.edge_len[el], r, rsum, rs2, kind);
        CAT_COUNT(4, 1);
        const uint32_t sb = __float_as_uint(sHit), feat = el * 2u + (uint32_t)kind;
        if (sHit < L && (sb < bs || (sb == bs && feat < bf))) {
          bool ok = true;
          if (strict) {
            const float4 dv = m.dir[ci];
            ok = thin_bb_hit(m.hull_bb[m.edge_hull[el]], ox, oy, dv.x == 0.f, dv.y == 0.f, dv.z * inv_L, dv.w * inv_L);
          }
          if (ok) { bs = sb; bf = feat; }
        }
        // nothing nearer can follow once the hit held is closer than the next entry's lower bound (a link reads as negative)
        fin = __uint_as_float(bs) < __uint_as_float(e0 & 0xFFFF0000u);
      }
    }
#ifdef CAT_STATS
    if (lane == 0) CAT_COUNT(5, 1);
#endif
    if (__any_sync(0xFFFFFFFFu, fin)) {
      bool take = false;
      if (fin) {
        bool redo = false;
        if (!strict && bf != kNoFeature) {   // cpBBTree leaf rule on the winner
          // a point of the thin ray well inside the hull's box means the thin ray enters it — decided by 4 compares; only
          // grazing rays pay for the exact slab test.  The probe point lies rsum + 0.5 beyond the centre's position at
          // first touch: at the touch the centre is still rsum away from the surface, i.e. OUTSIDE the box of a thin wall
          // (the 3-unit walls of squarinth / lbirinth / grandbyrinth), and at up to 65 degrees of incidence the probe
          // lands inside it.
          const float4 bb = m.hull_bb[m.edge_hull[bf >> 1]];
          const float sp = __uint_as_float(bs) + (rsum + 0.5f), px = fmaf(sp, ux, ox), py = fmaf(sp, uy, oy);
          if (!(sp <= L && px > bb.x + 0.05f && px < bb.z - 0.05f && py > bb.y + 0.05f && py < bb.w - 0.05f)) {
            const float4 dv = m.dir[ci];
            redo = !thin_bb_hit(bb, ox, oy, dv.x == 0.f, dv.y == 0.f, dv.z * inv_L, dv.w * inv_L);
          }
        }
        if (redo) {                    // grazing fat ray: walk the list again, leaf rule on every hit
          start_ray(cur);
          strict = true;
        } else {
          *reinterpret_cast<uint2*>(slots + cur) = make_uint2(bf, bs);   // = make_key(s, feature)
          strict = false;
          take = true;
        }
      }
      const uint32_t tmask = __ballot_sync(0xFFFFFFFFu, take);
      if (take) {
        cur = next + __popc(tmask & lt);
        if (cur >= nrays) cur = -1;
        else start_ray(cur);
      }
      next += __popc(tmask);
    }
  }
  __syncwarp();
}

// Sensor sweep of every agent of one world (entity.py:159-220) into shared memory.
//
// Wall hits first, into the per-ray buffer w.best (key = distance bits << 32 | feature): from the per-(cell, ray)
// candidate lists (sweep_lists, lanes = rays) or, without lists, by rasterising the edges in view into a 1-D depth
// buffer per agent (rasterise_agent, lanes = edges then (edge, ray) pairs).  Then, lanes = rays: the other agents'
// circles and the alpha = 0 rules are merged in, and the hit point goes through the float16 chain.
template <int TA, int TR, bool TL, bool TX, bool TM>
__device__ __forceinline__ void observe_world(const KParams& k, const MapView& m, const Warp& w, long long world, bool staged,
                                              SlotStage& st) {
  const int A = TA ? TA : k.A, R = TR ? TR : k.R, lane = w.lane;
  const bool lists = TL || MAPK(w.blob, ray_slots) != nullptr;   // TL: an instantiation without the rasteriser
  if (lists && !staged) stage_ray_slots<TA, TR, TM>(k, w, st);
  const float* pos = w.rec;
  const float* tc = w.rec + LAY(o_tc);
  const uint32_t flags = reinterpret_cast<const uint32_t*>(w.rec)[LAY(o_flags)];
  const float L = k.ray_len, rsum = k.wall_r + k.ray_r, inv_L = 1.f / k.ray_len;
  const float reach = k.agent_r + k.ray_r, reach2 = reach * reach, inv_reach = 1.f / reach;
  // per agent: hulls whose rounded surface is within ray_r of the origin -> alpha = 0 candidates.  The list is
  // part of the state record: the physics step that moved the body already measured its distance to every hull
  // in contact reach and stored it; it is recomputed here only after a re-spawn / set_state (flag bit set).
  if (lane < A) {
    uint32_t cnt = 0;
    if ((flags >> lane) & 1u) {
#pragma unroll 1
      for (int q = 0; q < kNear; ++q) w.near[lane * kNear + q] = 0xFFFFu;
      const float px = pos[2 * lane], py = pos[2 * lane + 1];
      const int cell = grid_cell(m, px, py);
      if (cell >= 0) {
        for (int q = m.con_off[cell]; q < m.con_off[cell + 1]; ++q) {
          const int h = m.con_list[q];
          const float4 bb = m.hull_bb[h];  // already grown by wall_r: cheap reject before the exact distance
          if (px < bb.x - k.ray_r || px > bb.z + k.ray_r || py < bb.y - k.ray_r || py > bb.w + k.ray_r) continue;
          float d, nx, ny;
          hull_closest(m, h, px, py, d, nx, ny);
          if (d - k.wall_r <= k.ray_r) {
            if (cnt < kNear) w.near[lane * kNear + cnt++] = (uint16_t)h;
            else atomicAdd(k.overflow + 1, 1ull);
          }
        }
      }
    } else {
#pragma unroll 1
      for (int q = 0; q < kNear; ++q) cnt += w.near[lane * kNear + q] != 0xFFFFu ? 1u : 0u;
    }
    w.nearcnt[lane] = cnt;
    w.minbits[lane] = kEmpty;
  }
  __syncwarp();
  if (lane == 0 && flags) reinterpret_cast<uint32_t*>(w.rec)[LAY(o_flags)] = 0u;   // lists are now valid for these positions

  if (lists) sweep_lists<TA, TR, TM>(k, m, w, st);
  const int kstride = lists ? 2 : 1;   // the list walk leaves ray r's key in the first half of its 16-byte slot

  const int nsub = (R + 31) >> 5;
#pragma unroll 1
  for (int a = 0; a < A; ++a) {
    // ---- warp-uniform, per agent
    const float ox = pos[2 * a], oy = pos[2 * a + 1];
    const uint32_t ncnt = w.nearcnt[a];
    int zero_agent = -1;   // first other agent whose circle is within ray_r of the origin (alpha = 0)
    for (int j = A - 1; j >= 0; --j) {
      if (j == a) continue;
      const float ddx = ox - tc[2 * j], ddy = oy - tc[2 * j + 1];
      if (ddx * ddx + ddy * ddy <= reach2) zero_agent = j;
    }

    if (!lists) {
      // ---- (1) clear the depth buffer (the dynamic shapes and the alpha = 0 rules are merged in step 3)
#pragma unroll 1
      for (int i = lane; i < R; i += 32) w.best[a * R + i] = make_key(L, kNoFeature);
      __syncwarp();
      // ---- (2) rasterise the walls in view
      rasterise_agent<TM>(k, w.blob, reinterpret_cast<unsigned char*>(w.rec), a, ox, oy);
    }

    // the other agents' cached centres relative to this origin, compacted (the candidate queue is free now)
    float4* others = reinterpret_cast<float4*>(w.cand);
    if (lane < A && lane != a)
      others[lane < a ? lane : lane - 1] = make_float4(ox - tc[2 * lane], oy - tc[2 * lane + 1], __uint_as_float(kAgentTag + lane), 0.f);
    __syncwarp();

    // ---- (3) lanes = rays: entity.py:200-215 — hit point, float16 chain at each of its rounding points, type
    const float oxh = __half2float(__float2half_rn(ox)), oyh = __half2float(__float2half_rn(oy));
    const int want = (a < k.nc) ? TYPE_THIEF : TYPE_COP;
#pragma unroll 1
    for (int sub = 0; sub < nsub; ++sub) {
      const int i = sub * 32 + lane;
      if (i < R) {
        const int r = a * R + i;
        const float4 dv = m.dir[i];
        unsigned long long key = w.best[r * kstride];     // nearest wall hit
        {
          Ray rq;
          rq.ox = ox; rq.oy = oy; rq.ux = dv.x; rq.uy = dv.y; rq.L = L;
          rq.zx = dv.x == 0.f; rq.zy = dv.y == 0.f; rq.idx = dv.z * inv_L; rq.idy = dv.w * inv_L;
          // dynamic shapes: the other agents' cached centres (keys order walls before agents at equal s)
          if (zero_agent >= 0) key = min(key, make_key(0.f, kAgentTag + zero_agent));
          else {
#pragma unroll 1
            for (int q = 0; q < A - 1; ++q) {   // CircleSegmentQuery against a cached agent centre, perpendicular-offset form
              const float4 o4 = others[q];
              const float cp = fmaf(o4.x, dv.y, -o4.y * dv.x);
              const float disc = fmaf(-cp, cp, reach2);
              if (disc >= 0.f) {
                const float sc = -fmaf(o4.x, dv.x, o4.y * dv.y) - fast_sqrt(disc);
                if (sc >= 0.f && sc < L) key = min(key, make_key(sc, __float_as_uint(o4.z)));
              }
            }
          }
          // static shapes with the origin inside their reach: alpha = 0, but only if the thin ray enters the bb
#pragma unroll 1
          for (uint32_t q = 0; q < ncnt; ++q) {
            const int h = w.near[a * kNear + q];
            if (thin_bb_hit(m.hull_bb[h], ox, oy, rq.zx, rq.zy, rq.idx, rq.idy)) key = min(key, make_key(0.f, 0u));
          }
        }
        const uint32_t feat = (uint32_t)key;
        const float sHit = __uint_as_float((uint32_t)(key >> 32));
        uint16_t dbits;
        uint8_t type;
        float hx = fmaf(L, dv.x, ox), hy = fmaf(L, dv.y, oy);   // ray end: reported when nothing is hit or alpha = 0
        if (feat == kNoFeature) {
          dbits = __half_as_ushort(__float2half_rn(L));
          type = TYPE_EMPTY;
        } else {
          const bool is_agent = feat >= kAgentTag;
          if (sHit > 0.f) {
            float2 n;
            if (!is_agent) {
              Ray rr; rr.ox = ox; rr.oy = oy; rr.ux = dv.x; rr.uy = dv.y;
              n = wall_hit_normal(m, feat, sHit, rr, rsum);
            } else {
              const int j = (int)(feat - kAgentTag);
              n = make_float2((ox - tc[2 * j] + sHit * dv.x) * inv_reach, (oy - tc[2 * j + 1] + sHit * dv.y) * inv_reach);
            }
            hx = ox + sHit * dv.x - n.x * k.ray_r; hy = oy + sHit * dv.y - n.y * k.ray_r;
          }
          const float pxh = __half2float(__float2half_rn(hx)), pyh = __half2float(__float2half_rn(hy));
          const float dxh = __half2float(__float2half_rn(pxh - oxh));
          const float dyh = __half2float(__float2half_rn(pyh - oyh));
          dbits = half_hypot_bits(dxh, dyh);
          type = !is_agent ? TYPE_WALL : ((int)(feat - kAgentTag) >= k.nc ? TYPE_THIEF : TYPE_COP);
          // rewards need the nearest opponent seen by this agent (cop.py:66-70, thief.py:60-63)
          if (type == want) atomicMin(&w.minbits[a], (uint32_t)dbits);
        }
        CAT_CHECK(r < LAY(nrays) && (feat == kNoFeature || feat >= kAgentTag || (int)(feat >> 1) < MAPK(w.blob, n_edges)));
        w.rdist[r] = dbits;
        w.rtype[r] = type;
        if (TX && k.hit_point) {
          float2* hp = reinterpret_cast<float2*>(k.hit_point) + (size_t)world * LAY(nrays) + r;
          *hp = make_float2(hx, hy);
        }
      }
    }
    __syncwarp();   // `others` aliases the candidate queue of the next agent
  }
  __syncwarp();
}

__device__ __forceinline__ uint16_t f32_to_bf16_bits(float v) {   // round to nearest even
  const uint32_t u = __float_as_uint(v);
  return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
}

// Optional learner-facing layouts (what skrl's wrapper would build on the host): per-agent flattened observation,
// the flattened centralised-critic state, the critic's 4-channel ray block (lstm_value_net.py:122-137), and bf16
// copies.  Only called when the caller asked for them; kept out of line so the native-dtype fast path stays small.
// `o`: the destination — the step's own arrays, or the final-output arrays of a world that ends (write_final_outputs).
struct FlatOut {
  float* obs_f32;
  uint16_t* obs_bf16;
  float* critic_f32;
  uint16_t* critic_bf16;
  float* state_f32;
};
__device__ __noinline__ void write_flat_layouts(const KParams& k, const FlatOut o, const uint16_t* rdist, const uint8_t* rtype,
                                                const float* pos, long long world) {
  const int A = k.A, R = k.R, lane = threadIdx.x & 31;
  if (o.obs_f32 || o.obs_bf16) {  // [A][N][2R]: [distance | object_type] as skrl flattens the Dict (keys sorted)
#pragma unroll 1
    for (int a = 0; a < A; ++a) {
      const size_t off = ((size_t)a * k.n_worlds + world) * (2 * R);
#pragma unroll 1
      for (int i = lane; i < 2 * R; i += 32) {
        const float v = i < R ? __half2float(__ushort_as_half(rdist[a * R + i])) : (float)rtype[a * R + i - R];
        if (o.obs_f32) o.obs_f32[off + i] = v;
        if (o.obs_bf16) o.obs_bf16[off + i] = f32_to_bf16_bits(v);
      }
    }
  }
  if (o.critic_f32 || o.critic_bf16) {
    // LSTMValue's channel stack, cut from the FIRST agent's block of env.state() (SURVEY.md C-8):
    // [own_obj_types | own_distances | object_type_shared | distance_shared] of cop_0; shared = first non-EMPTY of the cops
    const size_t off = (size_t)world * 4 * R;
#pragma unroll 1
    for (int i = lane; i < 4 * R; i += 32) {
      const int ch = i / R, ri = i - ch * R;
      float v;
      if (ch == 0) v = (float)rtype[ri];
      else if (ch == 1) v = __half2float(__ushort_as_half(rdist[ri]));
      else {
        uint8_t t = TYPE_EMPTY;
        uint16_t d = 0;
#pragma unroll 1
        for (int b = 0; b < k.nc; ++b)
          if (t == TYPE_EMPTY) { t = rtype[b * R + ri]; d = rdist[b * R + ri]; }
        v = ch == 2 ? (float)t : __half2float(__ushort_as_half(d));
      }
      if (o.critic_f32) o.critic_f32[off + i] = v;
      if (o.critic_bf16) o.critic_bf16[off + i] = f32_to_bf16_bits(v);
    }
  }
  if (o.state_f32) {
    // env.state(): per agent [distance_shared | object_type_shared | own_distances | own_obj_types | team_positions]
    float* dst = o.state_f32 + (size_t)world * k.state_dim;
    int base = 0;
#pragma unroll 1
    for (int a = 0; a < A; ++a) {
      const int team = a < k.nc ? 0 : 1;
      const int a0 = team == 0 ? 0 : k.nc, a1 = team == 0 ? k.nc : A;
      const int blk = 4 * R + 2 * (a1 - a0);
#pragma unroll 1
      for (int i = lane; i < blk; i += 32) {
        float v;
        if (i < 2 * R) {
          const int ri = i < R ? i : i - R;
          uint8_t t = TYPE_EMPTY;
          uint16_t d = 0;
#pragma unroll 1
          for (int b = a0; b < a1; ++b)
            if (t == TYPE_EMPTY) { t = rtype[b * R + ri]; d = rdist[b * R + ri]; }
          v = i < R ? __half2float(__ushort_as_half(d)) : (float)t;
        } else if (i < 3 * R) v = __half2float(__ushort_as_half(rdist[a * R + i - 2 * R]));
        else if (i < 4 * R) v = (float)rtype[a * R + i - 3 * R];
        else v = __half2float(__float2half_rn(pos[2 * a0 + (i - 4 * R)]));
        dst[base + i] = v;
      }
      base += blk;
    }
  }
}

// Write the optional outputs of one world from shared memory (coalesced).  The record goes last, by write_record: its
// packed form rewrites the staged types in place.
template <int TA, int TR>
__device__ __forceinline__ void write_optional_outputs(const KParams& k, const Warp& w, long long world) {
  const int A = TA ? TA : k.A, R = TR ? TR : k.R, lane = w.lane;
  const float* pos = w.rec;
  if (k.team_pos) {  // observation_spaces.py:92-95
#pragma unroll 1
    for (int i = lane; i < 2 * A; i += 32)
      k.team_pos[(size_t)world * 2 * A + i] = __half_as_ushort(__float2half_rn(pos[i]));
  }
  // observation_spaces.py:97-121 net effect: first non-EMPTY (type, distance) in team order
  if (k.shared_dist || k.shared_type) {
#pragma unroll 1
    for (int team = 0; team < 2; ++team) {
      const int a0 = team == 0 ? 0 : k.nc, a1 = team == 0 ? k.nc : A;
#pragma unroll 1
      for (int i = lane; i < R; i += 32) {
        uint8_t t = TYPE_EMPTY;
        uint16_t d = 0;
#pragma unroll 1
        for (int a = a0; a < a1; ++a)
          if (t == TYPE_EMPTY) { t = w.rtype[a * R + i]; d = w.rdist[a * R + i]; }
        if (k.shared_dist) k.shared_dist[((size_t)world * 2 + team) * R + i] = d;
        if (k.shared_type) k.shared_type[((size_t)world * 2 + team) * R + i] = t;
      }
    }
  }
  if (k.obs_f32 || k.state_f32 || k.critic_f32 || k.obs_bf16 || k.critic_bf16)
    write_flat_layouts(k, FlatOut{k.obs_f32, k.obs_bf16, k.critic_f32, k.critic_bf16, k.state_f32}, w.rdist, w.rtype, pos, world);
}

// The staged record of one world to the step's record output, or (FINAL) to the final record, which is never packed.
template <int TA, int TR, bool FINAL>
__device__ __forceinline__ void write_record(const KParams& k, const Warp& w, long long world) {
  const int A = TA ? TA : k.A, R = TR ? TR : k.R, lane = w.lane, nrays = A * R;
  {
    // one record per world, staged contiguously: [f16 distance | u8 type | f32 reward | flags], 16-byte stores
    unsigned char* stage = reinterpret_cast<unsigned char*>(w.rdist);
    int n16 = LAY(r_bytes) >> 4;
    if (!FINAL && k.record_packed) {
      // host-facing form (CatRecordLayout.type_bits == 2): 16 staged u8 types -> one 32-bit word, written back over the
      // start of the type area (each round reads its 512 source bytes before any lane writes: the 128 bytes a round
      // writes lie inside source bytes an earlier or the same round has read); rewards and flags move up behind them.
      // Codes: wall 0, cop 1, thief 2, empty (TYPE_EMPTY = 4) 3.
      const float rw = lane < A ? w.rew[lane] : 0.f;
      const uint32_t fl = (uint32_t)w.flg[0] | ((uint32_t)w.flg[1] << 8) | ((uint32_t)w.flg[2] << 16);
      const int nw = (nrays + 15) >> 4;
      CAT_CHECK(LAY(r_off_type) + 16 * nw <= LAY(r_bytes) && LAY(rp_bytes) <= LAY(r_bytes) && LAY(r_off_type) + 4 * nw == LAY(rp_off_reward));
#pragma unroll 1
      for (int i0 = 0; i0 < nw; i0 += 32) {
        const int i = i0 + lane;
        uint32_t pk = 0u;
        if (i < nw) {
          const uint4 t = reinterpret_cast<const uint4*>(w.rtype)[i];
          const uint32_t v[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t c = (v[j] & 0x03030303u) | (((v[j] >> 2) & 0x01010101u) * 3u);
            pk |= ((c | (c >> 6) | (c >> 12) | (c >> 18)) & 0xFFu) << (8 * j);
          }
          const int left = nrays - 16 * i;                 // the last word: bits beyond the world's rays stay zero
          if (left < 16) pk &= (1u << (2 * left)) - 1u;
        }
        __syncwarp();
        if (i < nw) reinterpret_cast<uint32_t*>(w.rtype)[i] = pk;
      }
      __syncwarp();
      // behind the packed types: zero up to the end of the packed record, then rewards and flags
#pragma unroll 1
      for (int i = (LAY(r_off_type) >> 2) + nw + lane; i < (LAY(rp_bytes) >> 2); i += 32) reinterpret_cast<uint32_t*>(stage)[i] = 0u;
      __syncwarp();
      if (lane < A) reinterpret_cast<float*>(stage + LAY(rp_off_reward))[lane] = rw;
      if (lane == 0) *reinterpret_cast<uint32_t*>(stage + LAY(rp_off_flags)) = fl;
      __syncwarp();
      n16 = LAY(rp_bytes) >> 4;
    }
    uint4* dst = reinterpret_cast<uint4*>(FINAL ? k.final_record + (size_t)world * k.final_record_stride
                                                    : k.record + (size_t)world * k.record_stride);
    const uint4* src = reinterpret_cast<const uint4*>(stage);
#pragma unroll 1
    for (int i = lane; i < n16; i += 32) dst[i] = src[i];
    if (!FINAL && k.record_packed) {
      // the staged record's own tail (rewards / flags / padding behind the u8 types) held packed-form bytes: restore
      // what the next world expects there — zero padding (its rewards, flags and types are rewritten every step)
      __syncwarp();
#pragma unroll 1
      for (int i = (LAY(r_off_type) >> 2) + lane; i < (LAY(r_bytes) >> 2); i += 32) reinterpret_cast<uint32_t*>(stage)[i] = 0u;
      __syncwarp();
    }
  }
}

// TX = false: the instantiation for launches that ask for the record and nothing else (the host picks it per launch) —
// none of the optional outputs above is compiled in.
template <int TA, int TR, bool TX>
__device__ __forceinline__ void write_observation(const KParams& k, const Warp& w, long long world) {
  if (TX) write_optional_outputs<TA, TR>(k, w, world);
  if (TX ? k.record != nullptr : true) write_record<TA, TR, false>(k, w, world);
}

// A world that ends in this step: its terminal observation, rewards and flags (staged, pre-physics) to the final outputs —
// the record and flat layouts the step would write with auto_reset = 0.
template <int TA, int TR>
__device__ __forceinline__ void write_final_outputs(const KParams& k, const Warp& w, long long world) {
  if (k.final_record) write_record<TA, TR, true>(k, w, world);
  if (k.final_obs_f32 || k.final_state_f32 || k.final_critic_f32)
    write_flat_layouts(k, FlatOut{k.final_obs_f32, nullptr, k.final_critic_f32, nullptr, k.final_state_f32}, w.rdist, w.rtype,
                       w.rec, world);
}

// cop.py:49-75 / thief.py:48-69 in fp32 from the f16 distance (SURVEY.md C-3).
__device__ __forceinline__ float agent_reward(const KParams& k, int a, uint32_t minbits, bool captured, bool timeout) {
  const bool is_cop = a < k.nc;
  if (captured) return is_cop ? 1.f : -1.f;
  if (timeout) return is_cop ? -1.f : 1.f;
  const bool seen = minbits != kEmpty;
  const float d = seen ? __half2float(__ushort_as_half((uint16_t)minbits)) : 0.f;
  if (is_cop) return seen ? (-0.02f + 1.5f * expf(-d / 50.f)) : -0.04f;
  return seen ? tanhf((d - 100.f) / 50.f) / 10.f : 0.15f;
}

// cpSpaceStep(dt) for one world, state in shared memory (SURVEY.md A.2-A.6).
template <int TA, int TR>
__device__ __forceinline__ void physics_world(const KParams& k, const MapView& m, const Warp& w) {
  const int A = TA ? TA : k.A, P = LAY(P), lane = w.lane;
  float* pos = w.rec;
  float* vel = w.rec + LAY(o_vel);
  float* vb = w.rec + LAY(o_vb);
  float* tc = w.rec + LAY(o_tc);
  uint32_t* wkey = reinterpret_cast<uint32_t*>(w.rec + LAY(o_wkey));
  float* wjn = w.rec + LAY(o_wjn);
  uint32_t* page = reinterpret_cast<uint32_t*>(w.rec + LAY(o_page));
  float* pjn = w.rec + LAY(o_pjn);
  const float rsum_w = k.agent_r + k.wall_r;

  // (1) cpBodyUpdatePosition, (2) shape caches
  if (lane < 2 * A) {
    const float p = pos[lane] + (vel[lane] + vb[lane]) * k.dt;
    pos[lane] = p; tc[lane] = p; vb[lane] = 0.f;
  }
  __syncwarp();

  // (3) narrow phase.  Entry: {nx, ny, bias, jn, jBias, nMass, meta, slot}
  // (3a) lanes = (agent, hull of the agent's grid cell) pairs: bounding-box reject + closest feature, all
  //      pairs of the world in one pass; hits are staged per agent in list order ({nx, ny, d, hull}).
  {
    int q0 = 0, len = 0;
    if (lane < A) {
      const int cell = grid_cell(m, pos[2 * lane], pos[2 * lane + 1]);
      if (cell >= 0) { q0 = m.con_off[cell]; len = m.con_off[cell + 1] - q0; }
      w.ccount[lane] = 0;
      w.nearcnt[lane] = 0;
    }
    if (lane < A * kNear) w.near[lane] = 0xFFFFu;   // next step's alpha = 0 candidates (hulls within ray_r of the new position)
    int incl = len;   // inclusive scan over the (at most 8) agent lanes
#pragma unroll
    for (int d = 1; d < CAT_MAX_AGENTS; d <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= d) incl += t; }
    const int total = __shfl_sync(0xFFFFFFFFu, incl, A - 1);
    __syncwarp();
    if (total == 0) {
      // Free flight, the common case away from walls: no hull within contact reach of any agent's cell.  If, besides,
      // no agent pair touches and no arbiter is cached from earlier steps, the rest of cpSpaceStep (arbiter look-up and
      // ageing, warm start, the impulse iterations) has nothing to do: leave with the flags it would have set.
      bool busy = false;
      if (lane < A * kSlots) busy = wkey[lane] != kEmpty;
      if (lane < P) {
        int i = 0, rem = lane;
#pragma unroll 1
        while (rem >= A - 1 - i) { rem -= A - 1 - i; ++i; }
        const int j = i + 1 + rem;
        const float dx = pos[2 * j] - pos[2 * i], dy = pos[2 * j + 1] - pos[2 * i + 1], mind = 2.f * k.agent_r;
        busy = busy || page[lane] != kEmpty || dx * dx + dy * dy < mind * mind;
      }
      if (!__any_sync(0xFFFFFFFFu, busy)) {
        if (lane == 0) reinterpret_cast<uint32_t*>(w.rec)[LAY(o_flags)] = 0u;
        __syncwarp();
        return;
      }
    }
#pragma unroll 1
    for (int p0 = 0; p0 < total; p0 += 32) {
      const int p = p0 + lane;
      int a = 0;
#pragma unroll 1
      for (int j = 0; j < A - 1; ++j) a += (p >= __shfl_sync(0xFFFFFFFFu, incl, j)) ? 1 : 0;
      const int q0a = __shfl_sync(0xFFFFFFFFu, q0, a), excl = __shfl_sync(0xFFFFFFFFu, incl - len, a);
      bool hit = false;
      float d = 0.f, nx = 0.f, ny = 0.f;
      int h = 0;
      if (p < total) {
        h = m.con_list[q0a + (p - excl)];
        const float px = pos[2 * a], py = pos[2 * a + 1];
        const float4 bb = m.hull_bb[h];  // QueryReject: the shape bbs must overlap (hull bb already grown by wall_r)
        if (!(px + k.agent_r < bb.x || bb.z < px - k.agent_r || py + k.agent_r < bb.y || bb.w < py - k.agent_r)) {
          hull_closest(m, h, px, py, d, nx, ny);
          hit = d <= rsum_w;  // CircleToPoly: d <= r_circle + r_poly
        }
      }
      const uint32_t hits = __ballot_sync(0xFFFFFFFFu, hit);
      const uint32_t same = __match_any_sync(0xFFFFFFFFu, a);
      const bool isnear = hit && (d - k.wall_r <= k.ray_r);
      const uint32_t nears = __ballot_sync(0xFFFFFFFFu, isnear);
      if (isnear) {
        const uint32_t rank = w.nearcnt[a] + __popc(nears & same & ((1u << lane) - 1u));
        if (rank < (uint32_t)kNear) w.near[a * kNear + rank] = (uint16_t)h;
        else atomicAdd(k.overflow + 1, 1ull);   // never silent: cat_env_overflow_counts
      }
      if (hit) {
        const uint32_t rank = w.ccount[a] + __popc(hits & same & ((1u << lane) - 1u));
        if (rank < (uint32_t)kSlots) {
          CAT_CHECK(a >= 0 && a < A && (a * kSlots + (int)rank) < LAY(maxc) && h >= 0 && h < m.H);
          float* c = w.con + (a * kSlots + rank) * 8;
          c[0] = nx; c[1] = ny; c[2] = d;
          reinterpret_cast<uint32_t*>(c)[7] = (uint32_t)h;
        } else atomicAdd(k.overflow, 1ull);       // a contact beyond CAT_WALL_SLOTS: counted, the world diverges from the uncapped solver
      }
      __syncwarp();
      if (hit && (hits & same & ((1u << lane) - 1u)) == 0) w.ccount[a] += __popc(hits & same);   // first hit lane of each agent
      if (isnear && (nears & same & ((1u << lane) - 1u)) == 0) w.nearcnt[a] += __popc(nears & same);
      __syncwarp();
    }
  }
  // (3b) lanes = agents: arbiter cache look-up for the staged contacts, in list order (cpArbiterUpdate)
  if (lane < A) {
    const uint32_t nstaged = min(w.ccount[lane], (uint32_t)kSlots);
    uint32_t cnt = 0, used = 0;
#pragma unroll 1
    for (uint32_t idx = 0; idx < nstaged; ++idx) {
      float* cs = w.con + (lane * kSlots + idx) * 8;
      const float nx = cs[0], ny = cs[1], d = cs[2];
      const int h = (int)reinterpret_cast<uint32_t*>(cs)[7];
      // reuse the cached arbiter of this (agent, hull) pair if any
      int slot = -1;
#pragma unroll 1
      for (int s = 0; s < kSlots; ++s)
        if (wkey[lane * kSlots + s] != kEmpty && (wkey[lane * kSlots + s] & 0xFFFF) == (uint32_t)h) slot = s;
      float jn0 = 0.f;
      bool first = true;
      if (slot >= 0) {
        jn0 = wjn[lane * kSlots + slot];
        first = (wkey[lane * kSlots + slot] >> 16) != 0;  // used in the previous step -> not first
      } else {
        // free slot, else the oldest slot not used this step
        uint32_t oldest = 0;
#pragma unroll 1
        for (int s = 0; s < kSlots; ++s) {
          if (used & (1u << s)) continue;
          const uint32_t key = wkey[lane * kSlots + s];
          const uint32_t age = key == kEmpty ? 0x10000u : (key >> 16) + 1u;
          if (age > oldest) { oldest = age; slot = s; }
        }
      }
      if (slot >= 0) {
        used |= 1u << slot;
        wkey[lane * kSlots + slot] = (uint32_t)h;  // age 0 = used this step
        float* c = w.con + (lane * kSlots + cnt) * 8;   // cnt <= idx: never overwrites an unread staged entry
        c[0] = nx; c[1] = ny;
        c[2] = -k.bias_coef * fminf(0.f, (d - rsum_w) + k.slop) * k.inv_dt;  // cpArbiterPreStep
        c[3] = jn0; c[4] = 0.f; c[5] = 1.f / k.inv_mass;
        reinterpret_cast<uint32_t*>(c)[6] = (uint32_t)lane | (0xFFu << 8) | (first ? 1u << 16 : 0u);
        reinterpret_cast<uint32_t*>(c)[7] = (uint32_t)(lane * kSlots + slot);
        ++cnt;
      }
    }
    // cpSpaceArbiterSetFilter: arbiters not used this step age; dropped at collision_persistence
#pragma unroll 1
    for (int s = 0; s < kSlots; ++s) {
      if (used & (1u << s)) continue;
      const uint32_t key = wkey[lane * kSlots + s];
      if (key == kEmpty) continue;
      const uint32_t age = (key >> 16) + 1u;
      if ((int)age >= k.persistence) { wkey[lane * kSlots + s] = kEmpty; wjn[lane * kSlots + s] = 0.f; }
      else wkey[lane * kSlots + s] = (key & 0xFFFF) | (age << 16);
    }
    w.ccount[lane] = cnt;
  }
  if (lane == 0) reinterpret_cast<uint32_t*>(w.rec)[LAY(o_flags)] = 0u;   // the stored near lists are valid for the new positions
  uint32_t pair_hit = 0;
  if (lane < P) {
    // pair index -> (i, j), i-major
    int i = 0, rem = lane;
#pragma unroll 1
    while (rem >= A - 1 - i) { rem -= A - 1 - i; ++i; }
    const int j = i + 1 + rem;
    const float dx = pos[2 * j] - pos[2 * i], dy = pos[2 * j + 1] - pos[2 * i + 1];
    const float mind = 2.f * k.agent_r, dsq = dx * dx + dy * dy;
    const uint32_t age = page[lane];
    if (dsq < mind * mind) {  // CircleToCircle (strict)
      const float dist = sqrtf(dsq);
      float* c = w.con + (A * kSlots + lane) * 8;
      const float invd = dist > 0.f ? 1.f / dist : 0.f;
      c[0] = dist > 0.f ? dx * invd : 1.f;
      c[1] = dy * invd;
      c[2] = -k.bias_coef * fminf(0.f, (dist - mind) + k.slop) * k.inv_dt;
      c[3] = age != kEmpty ? pjn[lane] : 0.f;
      c[4] = 0.f; c[5] = 1.f / (2.f * k.inv_mass);
      reinterpret_cast<uint32_t*>(c)[6] = (uint32_t)i | ((uint32_t)j << 8) | (age != 0 ? 1u << 16 : 0u);
      reinterpret_cast<uint32_t*>(c)[7] = (uint32_t)lane;
      page[lane] = 0;
      pair_hit = 1;
    } else if (age != kEmpty) {
      const uint32_t na = age + 1u;
      if ((int)na >= k.persistence) { page[lane] = kEmpty; pjn[lane] = 0.f; } else page[lane] = na;
    }
  }
  const uint32_t pair_mask = __ballot_sync(0xFFFFFFFFu, pair_hit != 0);
  __syncwarp();

  // (7) warm start + (8) sequential impulses.
  // An iteration that changes no accumulated impulse leaves v / v_bias untouched too, so every later
  // iteration would recompute exactly the same zeros: stopping there is bit-identical to running all of them.
  if (pair_mask == 0) {
    // No agent-agent contact: the wall contacts of different agents touch disjoint state, so their
    // sequential-impulse sweeps are independent -> lane a solves agent a, velocities in registers.
    const uint32_t n = lane < A ? w.ccount[lane] : 0u;
    if (n > 0) {
      const float minv = k.inv_mass;
      float* cbase = w.con + lane * kSlots * 8;
      float vx = vel[2 * lane], vy = vel[2 * lane + 1], bx = vb[2 * lane], by = vb[2 * lane + 1];
#pragma unroll 1
      for (uint32_t q = 0; q < n; ++q) {  // cpArbiterApplyCachedImpulse (dt_coef = 1)
        const float* c = cbase + q * 8;
        if (reinterpret_cast<const uint32_t*>(c)[6] & (1u << 16)) continue;  // first contact: nothing applied
        vx -= c[0] * c[3] * minv; vy -= c[1] * c[3] * minv;
      }
#pragma unroll 1
      for (int it = 0; it < k.iterations; ++it) {
        bool changed = false;
#pragma unroll 1
        for (uint32_t q = 0; q < n; ++q) {  // cpArbiterApplyImpulse against a static body, e = 0, u = 0
          float* c = cbase + q * 8;
          const float nx = c[0], ny = c[1], nMass = c[5];
          const float vbn = (-bx) * nx + (-by) * ny;
          const float vrn = (-vx) * nx + (-vy) * ny;
          const float jbnOld = c[4], jnOld = c[3];
          const float jBias = fmaxf(jbnOld + (c[2] - vbn) * nMass, 0.f);
          const float jnAcc = fmaxf(jnOld - vrn * nMass, 0.f);
          c[4] = jBias; c[3] = jnAcc;
          const float jb = (jBias - jbnOld) * minv, j = (jnAcc - jnOld) * minv;
          bx -= nx * jb; by -= ny * jb;
          vx -= nx * j; vy -= ny * j;
          changed |= (jb != 0.f) | (j != 0.f);
        }
        if (!changed) break;
      }
      vel[2 * lane] = vx; vel[2 * lane + 1] = vy; vb[2 * lane] = bx; vb[2 * lane + 1] = by;
#pragma unroll 1
      for (uint32_t q = 0; q < n; ++q) {  // persist jnAcc in the arbiter cache
        const float* c = cbase + q * 8;
        wjn[reinterpret_cast<const uint32_t*>(c)[7]] = c[3];
      }
    }
  } else if (lane == 0) {
    // Agent-agent contacts couple the bodies: one fixed global order (wall contacts agent-major, then pairs), lane 0
    int n = 0;
#pragma unroll 1
    for (int a = 0; a < A; ++a)
#pragma unroll 1
      for (uint32_t q = 0; q < w.ccount[a]; ++q) w.order[n++] = (uint8_t)(a * kSlots + q);
#pragma unroll 1
    for (int p = 0; p < P; ++p)
      if (pair_mask & (1u << p)) w.order[n++] = (uint8_t)(A * kSlots + p);
    const float minv = k.inv_mass;
#pragma unroll 1
    for (int q = 0; q < n; ++q) {  // cpArbiterApplyCachedImpulse (dt_coef = 1)
      float* c = w.con + w.order[q] * 8;
      const uint32_t meta = reinterpret_cast<uint32_t*>(c)[6];
      if (meta & (1u << 16)) continue;  // first contact: nothing applied
      const int a = meta & 0xFF, b = (meta >> 8) & 0xFF;
      const float jx = c[0] * c[3] * minv, jy = c[1] * c[3] * minv;
      vel[2 * a] -= jx; vel[2 * a + 1] -= jy;
      if (b != 0xFF) { vel[2 * b] += jx; vel[2 * b + 1] += jy; }
    }
#pragma unroll 1
    for (int it = 0; it < k.iterations; ++it) {
      bool changed = false;
#pragma unroll 1
      for (int q = 0; q < n; ++q) {  // cpArbiterApplyImpulse, e = 0, u = 0
        float* c = w.con + w.order[q] * 8;
        const uint32_t meta = reinterpret_cast<uint32_t*>(c)[6];
        const int a = meta & 0xFF, b = (meta >> 8) & 0xFF;
        const float nx = c[0], ny = c[1], nMass = c[5];
        float vbx = -vb[2 * a], vby = -vb[2 * a + 1], vrx = -vel[2 * a], vry = -vel[2 * a + 1];
        if (b != 0xFF) { vbx += vb[2 * b]; vby += vb[2 * b + 1]; vrx += vel[2 * b]; vry += vel[2 * b + 1]; }
        const float vbn = vbx * nx + vby * ny;
        const float vrn = vrx * nx + vry * ny;
        const float jbnOld = c[4];
        const float jBias = fmaxf(jbnOld + (c[2] - vbn) * nMass, 0.f);
        const float jnOld = c[3];
        const float jnAcc = fmaxf(jnOld - vrn * nMass, 0.f);
        c[4] = jBias; c[3] = jnAcc;
        const float jb = (jBias - jbnOld) * minv, j = (jnAcc - jnOld) * minv;
        vb[2 * a] -= nx * jb; vb[2 * a + 1] -= ny * jb;
        vel[2 * a] -= nx * j; vel[2 * a + 1] -= ny * j;
        if (b != 0xFF) {
          vb[2 * b] += nx * jb; vb[2 * b + 1] += ny * jb;
          vel[2 * b] += nx * j; vel[2 * b + 1] += ny * j;
        }
        changed |= (jb != 0.f) | (j != 0.f);
      }
      if (!changed) break;
    }
#pragma unroll 1
    for (int q = 0; q < n; ++q) {  // persist jnAcc in the arbiter cache
      const float* c = w.con + w.order[q] * 8;
      const uint32_t meta = reinterpret_cast<const uint32_t*>(c)[6];
      const uint32_t slot = reinterpret_cast<const uint32_t*>(c)[7];
      if (((meta >> 8) & 0xFF) == 0xFF) wjn[slot] = c[3]; else pjn[slot] = c[3];
    }
  }
  __syncwarp();
}

// BaseEnv.reset for one world (base_env.py:313-350, _get_non_colliding_position :123-166).
__device__ __forceinline__ void reset_world(const KParams& k, const MapView& m, const Warp& w, long long world) {
  const int A = k.A, lane = w.lane;
  float* pos = w.rec;
  float* vel = w.rec + k.lay.o_vel;
  float* tc = w.rec + k.lay.o_tc;
  uint32_t* ep = reinterpret_cast<uint32_t*>(w.rec + k.lay.o_ep);
  const uint32_t episode = *ep + 1u;
  // With pymunk's stale shape cache (A.10) every candidate is tested against the centres the OTHER agents had
  // before this reset, so the A spawns are independent and run on A lanes at once.  With the cache kept fresh
  // (stale_shape_cache = 0) agent j must see the new positions of agents i < j (base_env.py:313-332 resets them
  // in order): one round per agent, the accepted position published before the next round.
  const int rounds = k.stale ? 1 : A;
#pragma unroll 1
  for (int round = 0; round < rounds; ++round) {
    float nx_ = 0.f, ny_ = 0.f;
    const bool mine = lane < A && (k.stale || lane == round);
    if (mine) {
      const int r0 = m.reg_off[lane], nr = m.reg_off[lane + 1] - r0;
      if (nr > 0) {
        const unsigned long long gid = (unsigned long long)(k.gid0 + world);
        const uint32_t idx = cat_spawn_region_index(k.seed, gid, episode, (uint32_t)lane, (uint32_t)nr);
        const float4 reg = m.regions[r0 + (int)idx];
        nx_ = reg.x + reg.z / 2.f; ny_ = reg.y + reg.w / 2.f;  // base_env.py:163-166 fallback
#pragma unroll 1
        for (uint32_t t = 0; t < 20; ++t) {
          float ux, uy;
          cat_spawn_uniforms(k.seed, gid, episode, (uint32_t)lane, t, &ux, &uy);
          const float px = fmaf(reg.z, ux, reg.x), py = fmaf(reg.w, uy, reg.y);
          // point_query_nearest(pos, 5, ray_filter): any shape with distance < 5
          bool blocked = false;
          const int cell = grid_cell(m, px, py);
          if (cell >= 0) {
#pragma unroll 1
            for (int q = m.con_off[cell]; q < m.con_off[cell + 1] && !blocked; ++q) {
              float d, ax, ay;
              hull_closest(m, m.con_list[q], px, py, d, ax, ay);
              if (d - k.wall_r < k.agent_r) blocked = true;
            }
          }
#pragma unroll 1
          for (int j = 0; j < A && !blocked; ++j) {
            if (j == lane) continue;
            const float dx = px - tc[2 * j], dy = py - tc[2 * j + 1];
            if (sqrtf(dx * dx + dy * dy) - k.agent_r < k.agent_r) blocked = true;
          }
          if (!blocked) { nx_ = px; ny_ = py; break; }
        }
      } else {
        const float2 ip = m.init_pos[lane];  // base_env.py:328-332 -> Entity.reset() default
        nx_ = ip.x; ny_ = ip.y;
      }
    }
    __syncwarp();  // every lane has finished reading the centres of this round
    if (mine) {
      pos[2 * lane] = nx_; pos[2 * lane + 1] = ny_;       // entity.py:154-156
      vel[2 * lane] = 0.f; vel[2 * lane + 1] = 0.f;        // entity.py:157
      if (!k.stale) { tc[2 * lane] = nx_; tc[2 * lane + 1] = ny_; }
    }
    __syncwarp();
  }
  if (lane == 0) {
    *ep = episode;
    reinterpret_cast<int32_t*>(w.rec)[k.lay.o_sc] = 0;  // base_env.py:350
    reinterpret_cast<uint32_t*>(w.rec)[k.lay.o_flags] = 0xFFu;  // re-spawned bodies may sit next to a wall
  }
  __syncwarp();
}

// A re-spawned world's fresh parameters (cat_env_attach_world_params), when its map slot draws: one lane makes the two
// Philox calls of cat_param_draws, keyed by the new episode number reset_world has just stored, and writes the entry.
// The entry is next read by the world's next step.
__device__ __forceinline__ void draw_world_params(const KParams& k, const Warp& w, long long world, int mi) {
  if (w.lane != 0) return;
  const CatWorldParamRanges* r = k.wp_ranges + k.map_slot0 + mi;
  if (!r->draw) return;
  const uint32_t episode = reinterpret_cast<const uint32_t*>(w.rec)[k.lay.o_ep];
  uint32_t u[6];
  cat_param_draws(k.seed, (unsigned long long)(k.gid0 + world), episode, u);
  CatWorldParams p;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    p.unit_velocity[t] = cat_param_float(u[t], r->lo.unit_velocity[t], r->hi.unit_velocity[t]);
    p.max_speed[t] = cat_param_float(u[2 + t], r->lo.max_speed[t], r->hi.max_speed[t]);
  }
  p.termination_radius = cat_param_float(u[4], r->lo.termination_radius, r->hi.termination_radius);
  p.max_step_count = cat_param_int(u[5], r->lo.max_step_count, r->hi.max_step_count);
  k.wp[world] = p;
}

// Scripted agents (cat_env_attach_scripts): the three controllers' next actions from the observation the warp has
// staged and is about to emit, one byte per agent (random | chase << 2 | evade << 4, cat_b200.h).  Lanes are rays: for
// each agent an argmin of (d << 16 | i) over the rays that see its target, by warp reduction; lane a then owns agent a's
// decision (four axis-ray reads for evade, one Philox call).  Kept out of line, like los_blocked, so that it stays off
// the register budget of the full-output kernels.  Reads the staged record only; the caller syncs the warp after it.
__device__ __noinline__ void write_script_decisions(uint8_t* dec, const uint16_t* rdist, const uint8_t* rtype,
                                                    unsigned long long seed, unsigned long long gid, uint32_t episode,
                                                    uint32_t step_count, int lane, int A, int nc, int R) {
  uint32_t mine = kEmpty;   // lane a: the (d << 16 | i) key of the closest target agent a sees
#pragma unroll 1
  for (int a = 0; a < A; ++a) {
    const uint8_t target = a < nc ? TYPE_THIEF : TYPE_COP;
    uint32_t best = kEmpty;
#pragma unroll 1
    for (int i = lane; i < R; i += 32)
      if (rtype[a * R + i] == target) best = min(best, (uint32_t)rdist[a * R + i] << 16 | (uint32_t)i);
    best = __reduce_min_sync(0xFFFFFFFFu, best);
    if (lane == a) mine = best;
  }
  if (lane >= A) return;
  const int a = lane;
  const uint32_t rnd = cat_script_random(seed, gid, episode, step_count, (uint32_t)a);
  uint32_t chase = rnd, evade = rnd;
  if (mine != kEmpty) {
    constexpr uint32_t kAct = 2u | 1u << 2 | 0u << 4 | 3u << 6;   // ACT[q] = (kAct >> 2 q) & 3: +x, +y, -x, -y
    const uint8_t target = a < nc ? TYPE_THIEF : TYPE_COP;
    const int qs = ((8 * (int)(mine & 0xFFFFu) + R) / (2 * R)) & 3;
    chase = (kAct >> (2 * qs)) & 3u;
    int best_q = 0;
    uint32_t best_c = 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int q = (qs + (t == 0 ? 2 : t == 1 ? 1 : 3)) & 3;
      const int j = ((q * R + 2) / 4) % R;
      const uint32_t c = rtype[a * R + j] == target ? 0u : (uint32_t)rdist[a * R + j];
      if (t == 0 || c > best_c) { best_c = c; best_q = q; }
    }
    evade = (kAct >> (2 * best_q)) & 3u;
  }
  dec[a] = (uint8_t)(rnd | chase << 2 | evade << 4);
}

// Order-preserving u32 key of an fp32 value (CatEpisodeTotals): sign bit clear -> bits | 0x80000000, set -> ~bits.
// Non-zero for every non-NaN value, and so is its complement, so 0 stays "empty" for both the maximum and the minimum.
__device__ __forceinline__ uint32_t ep_key(float v) {
  const uint32_t b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// Episode statistics of one stepped world (cat_env_attach_episode_stats), once its rewards are staged: lanes < A add
// their agent's emitted reward to the running return (acc, loaded by the caller); a world that ends publishes the episode's
// return and length and adds it to the totals of its map slot, and its running return restarts at zero.
template <int TA, int TR>
__device__ __forceinline__ void episode_stats(const KParams& k, const Warp& w, long long world, int mi, float acc, bool done,
                                              bool captured) {
  const int A = TA ? TA : k.A, lane = w.lane;
  CatEpisodeTotals* t = k.ep_totals ? k.ep_totals + k.map_slot0 + mi : nullptr;
  if (lane < A) {
    const size_t i = (size_t)world * A + lane;
    const float ret = acc + w.rew[lane];   // one fp32 add: cumulative_rewards += rewards
    k.ep_acc[i] = done ? 0.f : ret;
    if (done) {
      if (k.ep_return) k.ep_return[i] = ret;
      if (t) {
        const double r = (double)ret;
        atomicAdd(&t->return_sum[lane], r);
        atomicAdd(&t->return_sq_sum[lane], r * r);   // exact: a float's square fits a double
        const uint32_t key = ep_key(ret);
        atomicMax(&t->return_max_key[lane], key);
        atomicMax(&t->return_min_key[lane], ~key);
      }
    }
  }
  if (done && lane == 0) {
    const int32_t len = reinterpret_cast<const int32_t*>(w.rec)[LAY(o_sc)];   // the step_count this step reached
    if (k.ep_length) k.ep_length[world] = len;
    if (t) {
      atomicAdd(reinterpret_cast<unsigned long long*>(&t->episodes), 1ull);
      atomicAdd(reinterpret_cast<unsigned long long*>(captured ? &t->captures : &t->timeouts), 1ull);
      atomicAdd(reinterpret_cast<unsigned long long*>(&t->length_sum), (unsigned long long)(uint32_t)len);
      atomicMax(&t->length_max_key, (uint32_t)len);
      atomicMax(&t->length_min_key, ~(uint32_t)len);
    }
  }
}

// TA / TR: agents per world and rays per agent as compile-time constants (the 2 cops + 1 thief x 90 rays of every
// shipped map: <3, 90>), or 0 = read them from the parameters (any other configuration: <0, 0>).  TL: the environment
// has ray lists (the default) — the instantiation carries no rasteriser code at all.  TX = false: a STEP launch that wants the
// output record only — none of the optional outputs (shared observations, team positions, fp32 / bf16 layouts, hit
// points) and none of the init / reset / observe launch modes is compiled in.  TM: a mixed-map environment — each CTA
// looks its map up in the launch's map table and reads the map-dependent values from the blob header it staged; the
// single-map instantiations (TM = false) take them from the parameters, at no register cost (a run-time table lookup
// in every instantiation raised the spills of three of the four, by up to 148 bytes of loads).
template <int TA, int TR, bool TL, bool TX, bool TM>
__global__ void __launch_bounds__(kMaxThreads, 1) cat_world_kernel(const __grid_constant__ KParams k) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) unsigned long long mbar;
  __shared__ int next_slot;   // the CTA's world queue (below)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mode = TX ? k.mode : (int)MODE_STEP;   // the record-only instantiation serves step launches only (kernel_for)

  // The CTA's map: the last entry of the launch's map table whose first CTA is at or below this one (at most
  // CAT_MAX_MAPS - 1 uniform compares).  Inside its map's share of the launch the CTA numbers itself and its worlds
  // exactly as a launch of that map alone would.
  int mi = 0;
  if (TM) {
#pragma unroll
    for (int i = 1; i < CAT_MAX_MAPS; ++i) mi += (i < k.n_maps && (int)blockIdx.x >= k.maps[i].cta_begin) ? 1 : 0;
  }
  const unsigned char* map_blob_m = k.maps[mi].blob;
  const int map_blob_bytes_m = k.maps[mi].blob_bytes;
  // the CTA's share of the launch: its map's group of CTAs and worlds (TM), or the whole launch — a single-map
  // instantiation reads these straight from the parameters and special registers, as it always has
  const unsigned cta_m = blockIdx.x - (unsigned)k.maps[mi].cta_begin;   // (unsigned, like blockIdx.x)
  const unsigned n_cta_m = (unsigned)((mi + 1 < k.n_maps ? k.maps[mi + 1].cta_begin : (int)gridDim.x) - k.maps[mi].cta_begin);
  const int world_begin_m = k.maps[mi].world_begin, world_end_m = k.maps[mi].world_end;
#define MAP_BLOB (TM ? map_blob_m : k.blob)
#define MAP_BLOB_BYTES (TM ? map_blob_bytes_m : k.blob_bytes)
#define CTA_IDX (TM ? cta_m : blockIdx.x)
#define CTA_CNT (TM ? n_cta_m : gridDim.x)
#define W_BEGIN (TM ? world_begin_m : k.world_begin)
#define W_END (TM ? world_end_m : k.world_end)

  // Stage the map once per CTA: one elected thread issues a TMA bulk copy (cp.async.bulk ->
  // UBLKCP) that completes on an mbarrier; everyone else waits on the barrier's phase.
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    next_slot = (int)(blockDim.x >> 5);   // slots 0 .. warps-1 are the warps' first worlds
  }
  __syncthreads();
  if (tid == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(MAP_BLOB_BYTES)
                 : "memory");
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem)),
        "l"(MAP_BLOB), "r"(MAP_BLOB_BYTES), "r"(smem_u32(&mbar))
        : "memory");
  }
  // Programmatic dependent launch (the host launches with programmatic stream serialisation): everything above — CTA
  // scheduling, barrier set-up, the copy of the map, which no kernel ever writes — may run while the previous launch
  // in the stream (the previous step) is still draining; nothing it wrote is touched before this wait returns.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // Prefetch this warp's first record while the map copy is in flight (with one world per warp, the usual case
  // at a few thousand worlds, both latencies would otherwise add up on the critical path).
  const bool one_wave_launch = (long long)CTA_CNT * (blockDim.x >> 5) >= W_END - W_BEGIN;
  const long long first_world = one_wave_launch ? W_BEGIN + (long long)CTA_IDX * (blockDim.x >> 5) + warp
                                                : W_BEGIN + CTA_IDX + (long long)warp * CTA_CNT;
  const bool prefetched = LAY(rec_words) <= 64 && mode != MODE_INIT && first_world < W_END;
  float pf0 = 0.f, pf1 = 0.f;
  if (prefetched) {
    const float* g = k.state + (size_t)first_world * LAY(rec_words);
    if (lane < LAY(rec_words)) pf0 = g[lane];
    if (lane + 32 < LAY(rec_words)) pf1 = g[lane + 32];
  }
  {
    uint32_t done = 0;
#pragma unroll 1
    while (!done) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(smem_u32(&mbar)), "r"(0)
          : "memory");
    }
  }
  const MapView m = make_view(smem);

  unsigned char* scratch = smem + ((MAP_BLOB_BYTES + 127) & ~127) + (size_t)warp * LAY(scratch_bytes);
  Warp w;
  w.rec = reinterpret_cast<float*>(scratch);
  w.rdist = reinterpret_cast<uint16_t*>(scratch + LAY(s_rdist));
  w.rtype = reinterpret_cast<uint8_t*>(scratch + LAY(s_rtype));
  w.minbits = reinterpret_cast<uint32_t*>(scratch + LAY(s_min));
  w.near = reinterpret_cast<uint16_t*>(w.rec + LAY(o_near));   // lives in the state record
  w.nearcnt = reinterpret_cast<uint32_t*>(scratch + LAY(s_nearcnt));
  w.con = reinterpret_cast<float*>(scratch + LAY(s_con));
  w.ccount = reinterpret_cast<uint32_t*>(scratch + LAY(s_ccount));
  w.order = reinterpret_cast<uint8_t*>(scratch + LAY(s_order));
  w.best = reinterpret_cast<unsigned long long*>(scratch + LAY(s_best));
  w.cand = reinterpret_cast<uint16_t*>(scratch + LAY(s_cand));
  w.rew = reinterpret_cast<float*>(scratch + LAY(s_rdist) + LAY(r_off_reward));
  w.flg = reinterpret_cast<uint8_t*>(scratch + LAY(s_rdist) + LAY(r_off_flags));
  w.mbar = reinterpret_cast<unsigned long long*>(scratch + LAY(s_rcell));
  w.blob = smem;
  w.lane = lane;
  SlotStage slot_stage{0u, false};
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(w.mbar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  // the padding of the staged output record is shipped by the 16-byte store paths: keep it zero
  for (int i = lane; i < (LAY(r_bytes) >> 2); i += 32) reinterpret_cast<uint32_t*>(w.rdist)[i] = 0u;
  __syncwarp();
  const int A = TA ? TA : k.A;
  // Worlds to warps.  CTA c owns the worlds c, c + G, c + 2 G, ... of its map's share of the launch (G = that share's CTAs): every SM gets the same
  // number of worlds to within one, whatever the world count — with contiguous blocks of `warps` worlds per CTA and round,
  // 16384 worlds on 148 x 32 warps left 80 SMs with three rounds and 68 with four: the SMs were busy 77 % of the launch
  // (ncu sm__cycles_active / elapsed, profiles/r2_notes.md).  Inside the CTA the warps draw their next world from a
  // shared counter when they finish one (slot s = the CTA's s-th world), so a warp that met cheap worlds takes more of
  // them and the CTA's last round is spread over all its warps' leftovers instead of pinned to the first few.
  auto next_world_slot = [&]() {
    int s_ = 0;
    if (lane == 0) s_ = atomicAdd(&next_slot, 1);
    return __shfl_sync(0xFFFFFFFFu, s_, 0);
  };
  // (a launch with a warp for every world keeps the contiguous numbering: neighbouring records stay in one CTA)
  const int wpc = blockDim.x >> 5;
  const bool one_wave = one_wave_launch;
#pragma unroll 1
  for (int slot = warp;; slot = next_world_slot()) {
    if (one_wave && slot >= wpc) break;
    const long long world = one_wave ? W_BEGIN + (long long)CTA_IDX * wpc + slot
                                     : W_BEGIN + CTA_IDX + (long long)slot * CTA_CNT;
    if (world >= W_END) break;
    float* grec = k.state + (size_t)world * LAY(rec_words);
    int32_t* reci = reinterpret_cast<int32_t*>(w.rec);

    if (mode == MODE_INIT) {  // fresh environment (entity.py:115,124): agents at map positions
#pragma unroll 1
      for (int i = lane; i < LAY(rec_words); i += 32) {
        float v = 0.f;
        if (i < 2 * A) v = (i & 1) ? m.init_pos[i >> 1].y : m.init_pos[i >> 1].x;
        else if (i >= LAY(o_tc) && i < LAY(o_tc) + 2 * A) { const int q = i - LAY(o_tc); v = (q & 1) ? m.init_pos[q >> 1].y : m.init_pos[q >> 1].x; }
        else if ((i >= LAY(o_wkey) && i < LAY(o_wkey) + A * kSlots) || (i >= LAY(o_page) && i < LAY(o_page) + LAY(P))) v = __uint_as_float(kEmpty);
        else if (i == LAY(o_flags)) v = __uint_as_float(0xFFu);
        grec[i] = v;
      }
      if (TX && k.ep_acc && lane < A) k.ep_acc[(size_t)world * A + lane] = 0.f;   // no episode is running yet
      if (TX && k.script_mode && lane < A) k.script_dec[(size_t)world * A + lane] = 0;   // nothing observed yet
      continue;
    }
    if (mode == MODE_RESET && k.reset_mask && !k.reset_mask[world]) continue;
    // Episode statistics: a reset drops the running returns (it never counts an episode); a step loads them here, next
    // to the record, so that the load's latency hides behind the sensor sweep.
    const bool ep_on = TX && k.ep_acc != nullptr;
    float ep_acc = 0.f;
    if (ep_on && lane < A) {
      if (mode == MODE_STEP) ep_acc = k.ep_acc[(size_t)world * A + lane];
      else if (mode == MODE_RESET) k.ep_acc[(size_t)world * A + lane] = 0.f;
    }
    // Per-world parameters of a step, loaded here for the same reason: lanes < A take their team's thrust and top
    // speed, every lane the capture radius and time limit (one broadcast load each).  The record-only instantiation
    // reads the parameters where it always has (WORLD_PARAM): hoisted to here, they changed its SASS and stack frame.
    float impulse = 0.f, max_speed = 0.f, term_r = 0.f;
    int max_steps = 0;
#define WORLD_PARAM(local, field) (TX ? local : k.field)
    if (TX) { impulse = k.impulse; max_speed = k.max_speed; term_r = k.term_r; max_steps = k.max_steps; }
    if (TX && k.wp && mode == MODE_STEP) {
      const CatWorldParams* e = k.wp + world;
      const int team = lane < k.nc ? 0 : 1;
      if (lane < A) { impulse = e->unit_velocity[team]; max_speed = e->max_speed[team]; }
      term_r = e->termination_radius;
      max_steps = e->max_step_count;
    }

    if (prefetched && world == first_world) {
      if (lane < LAY(rec_words)) w.rec[lane] = pf0;
      if (lane + 32 < LAY(rec_words)) w.rec[lane + 32] = pf1;
    } else {
#pragma unroll 1
      for (int i = lane; i < LAY(rec_words); i += 32) w.rec[i] = grec[i];
    }
    __syncwarp();

    bool do_step = mode == MODE_STEP, do_reset = mode == MODE_RESET;
    bool captured = false, timeout = false;
    // the sensor sweep reads the PRE-step positions, which are known now: start fetching the rays' candidate slots
    bool staged = false;
    if (do_step && (TL || MAPK(smem, ray_slots))) { stage_ray_slots<TA, TR, TM>(k, w, slot_stage); staged = true; }
    if (do_step) {  // ---------------- base_env.py:354-383 ----------------
      const float* pos = w.rec;
      float* vel = w.rec + LAY(o_vel);
      const int step_count = reci[LAY(o_sc)] + 1;  // :372
      __syncwarp();
      if (lane == 0) reci[LAY(o_sc)] = step_count;
      // _termination_criterion (:521-554): thief-major; LOS blocked by walls only; dist < radius (strict)
#pragma unroll 1
      for (int t = k.nc; t < A && !captured; ++t)
#pragma unroll 1
        for (int c = 0; c < k.nc && !captured; ++c) {
          const float tx = pos[2 * t], ty = pos[2 * t + 1], cx = pos[2 * c], cy = pos[2 * c + 1];
          const float dx = tx - cx, dy = ty - cy;
          if (dx * dx + dy * dy < WORLD_PARAM(term_r, term_r) * WORLD_PARAM(term_r, term_r)) {
            const bool blocked = los_blocked(smem, lane, tx, ty, cx, cy, k.wall_r);
            if (!__any_sync(0xFFFFFFFFu, blocked)) captured = true;
          }
        }
      timeout = !captured && step_count >= WORLD_PARAM(max_steps, max_steps);
      // Entity._perform_action (entity.py:126-134)
      if (lane < A) {
        int act;
        const size_t ai = (size_t)world * A + lane;
        if (k.actions_kind == 0) act = reinterpret_cast<const uint8_t*>(k.actions[0])[ai];
        else if (k.actions_kind == 1) act = reinterpret_cast<const int32_t*>(k.actions[0])[ai];
        else if (k.actions_kind == 2) act = (int)reinterpret_cast<const long long*>(k.actions[0])[ai];
        else act = (int)reinterpret_cast<const long long*>(k.actions[lane])[world];
        if (TX && k.script_mode) {   // a scripted agent: its controller's decision from the last emitted observation
          const int sm = k.script_mode[ai];
          if (sm) act = (k.script_dec[ai] >> (2 * (sm - 1))) & 3;
        }
        float fx = 0.f, fy = 0.f;
        if (act == 0) fx = -WORLD_PARAM(impulse, impulse); else if (act == 1) fy = WORLD_PARAM(impulse, impulse);
        else if (act == 2) fx = WORLD_PARAM(impulse, impulse); else if (act == 3) fy = -WORLD_PARAM(impulse, impulse);
        float vx = vel[2 * lane] + fx * k.inv_mass, vy = vel[2 * lane + 1] + fy * k.inv_mass;
        const float sp = sqrtf(vx * vx + vy * vy);
        if (sp > WORLD_PARAM(max_speed, max_speed)) {
          vx = vx / sp * WORLD_PARAM(max_speed, max_speed); vy = vy / sp * WORLD_PARAM(max_speed, max_speed);
        }
        vel[2 * lane] = vx; vel[2 * lane + 1] = vy;
      }
      __syncwarp();
    }

    // One call site each for the sensor sweep, the output writer, the physics and the re-spawn:
    //   STEP    : observe -> rewards/flags -> (write) -> physics -> [done: reset -> observe -> write]
    //   RESET   : reset -> observe -> write
    //   OBSERVE : observe -> write
#pragma unroll 1
    for (;;) {
      if (do_reset) {
        reset_world(k, m, w, world);
        if (TX && k.wp_ranges) draw_world_params(k, w, world, mi);
        do_reset = false; staged = false;
      }
      // entity.py:143 — observation of the pre-physics state (SURVEY.md C-1).  A world that ends on this step and
      // is re-spawned in it emits the NEW episode's observation (C-10) and a terminal reward that does not depend
      // on what is seen, so its terminal sensor sweep would be thrown away unless the launch asks for final outputs:
      // skip it then.  With one world per warp the launch lasts as long as its slowest warp, and a second sweep made
      // every finishing world that warp.
      const bool ends = do_step && (captured || timeout);
      const bool final_out = TX && ends && (k.final_record || k.final_obs_f32 || k.final_state_f32 || k.final_critic_f32);
      // (TX = false keeps the test spelled out: written through `ends`, ptxas schedules the record-only kernel, which
      // never writes final outputs, differently — DESIGN.md §2.2)
      if (TX ? !(ends && k.auto_reset) || final_out : !(do_step && (captured || timeout) && k.auto_reset))
        observe_world<TA, TR, TL, TX, TM>(k, m, w, world, staged, slot_stage);
      bool again = false;
      if (do_step) {
        if (lane < A) w.rew[lane] = agent_reward(k, lane, w.minbits[lane], captured, timeout);
        const bool done = captured || timeout;
        if (lane == 0) {
          w.flg[0] = done ? 1 : 0;                                      // terminated, entity.py:146
          w.flg[1] = timeout ? 1 : 0;                                   // truncated, base_env.py:397
          w.flg[2] = (uint8_t)(done ? (captured ? 0 : 1) : -1);         // winner
        }
        again = done && k.auto_reset;  // SURVEY.md C-10: emit the observation of the re-spawned state instead
        if (ep_on) episode_stats<TA, TR>(k, w, world, mi, ep_acc, done, captured);
      } else if (mode != MODE_STEP) {
        if (lane < A) w.rew[lane] = 0.f;
        if (lane == 0) { w.flg[0] = 0; w.flg[1] = 0; w.flg[2] = 0xFF; }
      }
      __syncwarp();
      if (final_out) write_final_outputs<TA, TR>(k, w, world);
      if (!again) {
        // the controllers decide on the observation this launch emits (before write_observation: the packed record
        // form rewrites the staged types); observe launches leave the decisions alone
        if (TX && k.script_mode && mode != MODE_OBSERVE) {
          const uint32_t* recu = reinterpret_cast<const uint32_t*>(w.rec);
          write_script_decisions(k.script_dec + (size_t)world * A, w.rdist, w.rtype, k.seed,
                                 (unsigned long long)(k.gid0 + world), recu[LAY(o_ep)], recu[LAY(o_sc)], lane, A, k.nc,
                                 TR ? TR : k.R);
          __syncwarp();
        }
        write_observation<TA, TR, TX>(k, w, world);
      }
      __syncwarp();
      if (do_step) {
        physics_world<TA, TR>(k, m, w);  // base_env.py:392
        do_step = false;
        if (again) { do_reset = true; continue; }
      }
      break;
    }
    if (mode != MODE_OBSERVE) {
#pragma unroll 1
      for (int i = lane; i < LAY(rec_words); i += 32) grec[i] = w.rec[i];
    }
    __syncwarp();
  }
}
#undef MAP_BLOB
#undef MAP_BLOB_BYTES
#undef CTA_IDX
#undef CTA_CNT
#undef W_BEGIN
#undef W_END
#undef WORLD_PARAM

