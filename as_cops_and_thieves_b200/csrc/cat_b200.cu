// cat_b200.cu — hand-written sm_100a kernels + C ABI for the batched cops-and-thieves step.
//
// One warp owns one world for one lockstep transition (persistent CTAs loop over worlds):
//   state record (coalesced) -> termination test -> action impulses -> 90-ray sensor sweep per
//   agent (the wall edges, staged in shared memory by one TMA bulk copy per CTA, are RASTERISED into
//   a per-agent 1-D depth buffer: lanes = candidate edges, then lanes = (edge, ray) pairs) ->
//   float16 observation chain -> rewards -> team-shared merge -> rigid-body step (position integrate,
//   circle-hull / circle-circle contacts, warm start, sequential impulses) -> auto-reset (Philox) ->
//   outputs + state record (coalesced).  Plus the MAPPO GAE / advantage-normalisation kernels.
//
// Restates /root/reference/src/environments/base_env.py:354-413,521-554,286-352,
// /root/reference/src/agents/entity.py:126-241, cop.py:49-75, thief.py:48-69,
// /root/reference/src/environments/observation_spaces.py:67-131 and the Chipmunk2D 7.0.3
// routines they call (cpSpaceStep, cpArbiterPreStep/ApplyImpulse, CircleToPoly, CircleToCircle,
// cpShapeSegmentQuery, cpPolyShapeSegmentQuery, CircleSegmentQuery, cpBBSegmentQuery) in fp32,
// origin-relative so that ray distances keep ~1e-5 absolute accuracy at coordinates ~1e3.
//
// No CPU fallback, no Triton, no tensor cores (the step is instruction-issue bound, GAE is HBM bound; DESIGN.md §3).

#include <cuda.h>            // CUtensorMap types only: the encoder is fetched through cudaGetDriverEntryPoint, libcuda is not linked
#include <cudaTypedefs.h>    // PFN_cuTensorMapEncodeTiled
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/cat_b200.h"
#include "../../include/cat_philox.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return fail(CAT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
  } while (0)

#include "ray_lists.h"
#include "ray_lists_kernel.cuh"
#include "world_kernel.cuh"
#include "state_view.cuh"
#include "gae_kernels.cuh"
#include "render_kernel.cuh"

inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

// Every ABI entry runs with the environment's device current and restores the caller's device on return.
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
    if (prev != device) ok = cudaSetDevice(device) == cudaSuccess;
    if (prev == device) prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define DEVICE_SCOPE(env)                                                                    \
  DeviceGuard _guard((env)->device);                                                          \
  if (!_guard.ok) return fail(CAT_ERR_CUDA, "cudaSetDevice(" + std::to_string((env)->device) + ") failed")

}  // namespace

// ------------------------------------------------------------------ host side / C ABI
typedef void (*WorldKernel)(const KParams);
struct LaunchShape { int threads, smem, grid; };

// The (cell, ray) candidate lists depend on the map and the sensor parameters only: environments created on the same
// device for the same map share ONE copy (reference-counted; built and uploaded by the first, freed with the last) — ten
// environments on agh-map hold 120 MB of lists, not 1.2 GB, and creating the second one skips the second-long build.
struct SharedRayLists {
  std::vector<unsigned char> key;   // device, sensor parameters, grid rule and every map array the builder reads
  uint4* slots_dev = nullptr;
  uint32_t* ovf_dev = nullptr;
  RayListGrid g{};
  size_t slot_words = 0, ovf_words = 0;
  int refs = 0;
};
static std::mutex g_ray_lists_mutex;
static std::vector<SharedRayLists*> g_ray_lists;

static void ray_lists_release(SharedRayLists* sh) {
  if (!sh) return;
  std::lock_guard<std::mutex> lock(g_ray_lists_mutex);
  if (--sh->refs > 0) return;
  g_ray_lists.erase(std::remove(g_ray_lists.begin(), g_ray_lists.end(), sh), g_ray_lists.end());
  if (sh->slots_dev) cudaFree(sh->slots_dev);
  if (sh->ovf_dev) cudaFree(sh->ovf_dev);
  delete sh;
}

// One map of an environment: its staged blob, its view lists and its share of the (cell, ray) lists.  Map m owns the
// worlds [world_begin, world_begin + n_worlds) of the environment.
struct EnvMap {
  unsigned char* blob_dev = nullptr;
  int blob_bytes = 0;
  BlobHeader header{};                   // the header of the uploaded blob: the map's one device description
  int32_t* view_off_dev = nullptr;
  uint16_t* view_edges_dev = nullptr;
  SharedRayLists* ray_lists = nullptr;   // shared with the other environments of this map on this device
  int world_begin = 0, n_worlds = 0;
};

struct CatEnv {
  std::vector<std::pair<int, LaunchShape>> shape_cache;   // launch shape per world count (the chunked host path asks every step)
  WorldKernel kernel = nullptr;        // every output the ABI offers
  WorldKernel kernel_record = nullptr; // record output only (launches that ask for nothing else)
  int device = 0;
  int n_worlds = 0;
  std::vector<EnvMap> maps;            // 1 .. CAT_MAX_MAPS, in world order
  unsigned long long* overflow_dev = nullptr;
  CatRecordLayout rec{}, rec_packed{};
  KParams kp{};                        // with the map table of a full-environment launch
  CatEnvInfo info{};
  int smem_bytes = 0;
  int grid = 0;
  int threads = kThreads;
  int blob_bytes = 0, max_optin = 0, n_sm = 0;   // blob_bytes: the largest of the maps' blobs (swappable: the capacity)
  // cat_env_create_swappable: every map's blob is allocated at blob_bytes and the mixed-map kernels run, so that
  // cat_env_set_map changes neither the launch shape nor the KParams of a captured launch
  bool swappable = false;
  CatParams params{};
  // chunked host path: a second stream for the device-to-host copies and one event per chunk
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> chunk_events;
  cudaEvent_t copies_done = nullptr;
};

// the kernel instantiation an environment runs (fixed at creation): agents / rays as compile-time constants for the
// shipped shape, the any-shape instantiation otherwise (CAT_GENERIC_KERNEL=1 at creation forces it: test knob); the
// mixed-map instantiations (multi) for an environment of several maps
template <bool TM>
static WorldKernel pick_world_kernel_t(int A, int R, bool lists, bool extras) {
  const char* e = getenv("CAT_GENERIC_KERNEL");
  const bool generic = e && e[0] == '1';
  if (A == 3 && R == 90 && !generic) {
    if (lists) return extras ? cat_world_kernel<3, 90, true, true, TM> : cat_world_kernel<3, 90, true, false, TM>;
    return cat_world_kernel<3, 90, false, true, TM>;
  }
  return cat_world_kernel<0, 0, false, true, TM>;
}
static WorldKernel pick_world_kernel(int A, int R, bool lists, bool extras, bool multi) {
  return multi ? pick_world_kernel_t<true>(A, R, lists, extras) : pick_world_kernel_t<false>(A, R, lists, extras);
}

static bool pick_launch_shape(CatEnv* env, int n_worlds, LaunchShape* out) {
  for (const auto& kv : env->shape_cache)
    if (kv.first == n_worlds) { *out = kv.second; return true; }
  long long best_score = -1;
  int wpc_max = kMaxThreads / 32;
  if (const char* e = getenv("CAT_MAX_WARPS_PER_CTA")) { const int v = atoi(e); if (v >= 2 && v < wpc_max) wpc_max = v; }   // tuning knob
  for (int wpc = wpc_max; wpc >= 2; --wpc) {   // any warp count: 4096 worlds = 586 CTAs of 7 warps = 28 warps per SM
    const int smem = align_up(env->blob_bytes, 128) + wpc * env->kp.lay.scratch_bytes;
    if (smem > env->max_optin) continue;
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, env->kernel, wpc * 32, smem) != cudaSuccess || occ < 1) continue;
    const int need = (n_worlds + wpc - 1) / wpc;
    const bool one_wave = need <= env->n_sm * occ;
    // one wave: fewest warps on the fullest SM; persistent: most resident warps per SM
    const int key = one_wave ? 4096 - ((need + env->n_sm - 1) / env->n_sm) * wpc : occ * wpc;
    const long long score = ((long long)(one_wave ? 1 : 0) << 40) + ((long long)key << 8) + wpc;
    if (score > best_score) {
      best_score = score;
      out->threads = wpc * 32; out->smem = smem; out->grid = one_wave ? need : env->n_sm * occ;
    }
  }
  if (const char* e = getenv("CAT_MAX_GRID")) { const int v = atoi(e); if (v >= 1 && v < out->grid) out->grid = v; }   // tuning knob
  if (best_score >= 0 && env->shape_cache.size() < 64) env->shape_cache.emplace_back(n_worlds, *out);
  return best_score >= 0;
}

// Fill the map table of a launch that steps the worlds [w0, w1) of the environment with `grid` CTAs of `wpc` warps and
// return the grid to launch.  The CTAs are split between the maps with worlds in the range: a one-wave grid (a warp for
// every world) gives each map the CTAs its worlds need, so every map's share stays one wave; a persistent grid is split
// in proportion to the worlds, at least one CTA per map (raised to one CTA per map if it is smaller).  With one map the
// grid is returned unchanged.
static int fill_map_table(const CatEnv* env, KParams& k, int w0, int w1, int grid, int wpc) {
  int len[CAT_MAX_MAPS], ctas[CAT_MAX_MAPS];
  int n = 0;
  k.map_slot0 = -1;
  for (const EnvMap& m : env->maps) {
    const int b = std::max(w0, m.world_begin), e = std::min(w1, m.world_begin + m.n_worlds);
    if (b >= e) continue;
    if (k.map_slot0 < 0) k.map_slot0 = (int)(&m - env->maps.data());   // the maps of [w0, w1) are consecutive slots
    MapSlice& sl = k.maps[n];
    sl.blob = m.blob_dev; sl.blob_bytes = m.blob_bytes; sl.world_begin = b; sl.world_end = e;
    len[n++] = e - b;
  }
  k.n_maps = n;
  k.world_begin = w0; k.world_end = w1;
  const long long total = (long long)w1 - w0;
  if ((long long)grid * wpc >= total) {
    grid = 0;
    for (int i = 0; i < n; ++i) { ctas[i] = (len[i] + wpc - 1) / wpc; grid += ctas[i]; }
  } else {
    grid = std::max(grid, n);
    int used = 0;
    for (int i = 0; i < n; ++i) { ctas[i] = std::max(1, (int)((long long)grid * len[i] / total)); used += ctas[i]; }
    while (used > grid) {          // the minimum of one CTA pushed the sum over: take from the map with the most
      int j = 0;
      for (int i = 1; i < n; ++i) if (ctas[i] > ctas[j]) j = i;
      --ctas[j]; --used;
    }
    while (used < grid) {          // rounding left CTAs over: give each to the map with the most worlds per CTA
      int j = 0;
      for (int i = 1; i < n; ++i) if ((long long)len[i] * ctas[j] > (long long)len[j] * ctas[i]) j = i;
      ++ctas[j]; ++used;
    }
  }
  int c = 0;
  for (int i = 0; i < n; ++i) { k.maps[i].cta_begin = c; c += ctas[i]; }
  return grid;
}

// Launch with programmatic stream serialisation: the kernel's CTAs may be scheduled while the previous kernel in the
// stream drains; the kernels call griddepcontrol.wait before they touch global memory (gae_kernels.cuh).
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  static const int allowed = [] { const char* e = getenv("CAT_PDL"); return (e && e[0] == '0') ? 0 : 1; }();
  attr[0].val.programmaticStreamSerializationAllowed = allowed;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// One run of the device list builder (ray_lists_kernel.cuh) on the current device: size() uploads the map and runs the
// counting passes, fill() writes the lists into the caller's arrays of slot_words / ovf_words words.  Synchronous; the
// temporary arrays are freed with the object.
struct RayListDeviceBuild {
  RayListSetup su;
  RayListDev p{};
  size_t slot_words = 0, ovf_words = 0;
  std::vector<void*> allocs;
  int grid = 1;
  ~RayListDeviceBuild() { for (void* a : allocs) cudaFree(a); }

  template <typename T> cudaError_t alloc(T** ptr, size_t n) {
    void* v = nullptr;
    const cudaError_t e = cudaMalloc(&v, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) { allocs.push_back(v); *ptr = static_cast<T*>(v); }
    return e;
  }
  template <typename T> cudaError_t upload(const T** ptr, const T* src, size_t n) {
    T* d = nullptr;
    cudaError_t e = alloc(&d, n);
    if (e == cudaSuccess && n) e = cudaMemcpy(d, src, n * sizeof(T), cudaMemcpyHostToDevice);
    *ptr = d;
    return e;
  }
  unsigned long long total(const unsigned long long* scanned, int n, cudaError_t* e) {
    unsigned long long v = 0;
    if (*e == cudaSuccess) *e = cudaMemcpy(&v, scanned + n, sizeof(v), cudaMemcpyDeviceToHost);
    return v;
  }

  int size(const CatMapDesc* map, int R, double L, double rsum, double cell) {
    ray_list_setup(map, R, L, rsum, cell, &su);
    const int H = map->n_hulls, E = map->n_edges, cells = su.g.nx * su.g.ny;
    if ((long long)su.g.nx * su.g.ny * R * 4 > 0x7FFFFFFFll) return fail(CAT_ERR_LIMIT, "ray-list grid too large");
    p.H = H; p.E = E; p.R = R; p.nx = su.g.nx; p.ny = su.g.ny;
    p.gx0 = su.gx0; p.gy0 = su.gy0; p.cell = su.cell; p.L = su.L; p.rs = su.rs;
    std::vector<double> a(2 * (size_t)E), nn(2 * (size_t)E), u(2 * (size_t)R);
    std::vector<int32_t> ehull(E);
    for (int e = 0; e < E; ++e) { a[2 * e] = su.ax[e]; a[2 * e + 1] = su.ay[e]; nn[2 * e] = su.nnx[e]; nn[2 * e + 1] = su.nny[e]; }
    for (int h = 0; h < H; ++h) for (int e = map->hull_off[h]; e < map->hull_off[h + 1]; ++e) ehull[e] = h;
    for (int i = 0; i < R; ++i) { u[2 * i] = su.ux[i]; u[2 * i + 1] = su.uy[i]; }
    grid = std::min(cells, 4096);
    cudaError_t e = upload(&p.vert, map->vert, 2 * (size_t)E);
    if (e == cudaSuccess) e = upload(&p.normal, map->normal, 2 * (size_t)E);
    if (e == cudaSuccess) e = upload(&p.a, a.data(), a.size());
    if (e == cudaSuccess) e = upload(&p.nn, nn.data(), nn.size());
    if (e == cudaSuccess) e = upload(&p.hull_bb, map->hull_bb, 4 * (size_t)H);
    if (e == cudaSuccess) e = upload(&p.ehull, ehull.data(), ehull.size());
    if (e == cudaSuccess) e = upload(&p.u, u.data(), u.size());
    if (e == cudaSuccess) e = alloc(&p.cand_off, cells + 1);
    if (e == cudaSuccess) { cat_ray_list_cand_kernel<false><<<grid, kRlThreads>>>(p); e = cudaGetLastError(); }
    if (e == cudaSuccess) { cat_ray_list_scan_kernel<<<1, 1024>>>(p.cand_off, cells); e = cudaGetLastError(); }
    const unsigned long long n_cand = total(p.cand_off, cells, &e);
    if (e == cudaSuccess) e = alloc(&p.cand_e, n_cand);
    if (e == cudaSuccess) e = alloc(&p.cand_lb, n_cand);
    if (e == cudaSuccess) { cat_ray_list_cand_kernel<true><<<grid, kRlThreads>>>(p); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = alloc(&p.n_list, (size_t)cells * R);
    if (e == cudaSuccess) e = alloc(&p.words, cells + 1);
    if (e == cudaSuccess) e = alloc(&p.longs, cells + 1);
    if (e == cudaSuccess) { cat_ray_list_kernel<false><<<grid, kRlThreads>>>(p); e = cudaGetLastError(); }
    if (e == cudaSuccess) { cat_ray_list_scan_kernel<<<1, 1024>>>(p.words, cells); e = cudaGetLastError(); }
    if (e == cudaSuccess) { cat_ray_list_scan_kernel<<<1, 1024>>>(p.longs, cells); e = cudaGetLastError(); }
    const unsigned long long n_words = total(p.words, cells, &e), n_long = total(p.longs, cells, &e);
    if (e == cudaSuccess) e = alloc(&p.long_buf, n_long);
    if (e != cudaSuccess) return fail(CAT_ERR_CUDA, std::string("ray lists (device build): ") + cudaGetErrorString(e));
    if (4 + n_words > 0x7FFFFFFFull) return fail(CAT_ERR_LIMIT, "ray-list overflow array too large for 31-bit links");
    slot_words = (size_t)cells * R * 4;
    ovf_words = 4 + (size_t)n_words;
    return CAT_OK;
  }

  int fill(uint32_t* slots_dev, uint32_t* ovf_dev) {
    p.slots = slots_dev; p.ovf = ovf_dev;
    cat_ray_list_kernel<true><<<grid, kRlThreads>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    return e == cudaSuccess ? CAT_OK : fail(CAT_ERR_CUDA, std::string("ray lists (device build): ") + cudaGetErrorString(e));
  }
};

extern "C" {

#ifdef CAT_STATS
int cat_debug_stats(unsigned long long* out8, int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out8, g_stats, sizeof(g_stats));
  if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_stats, z, sizeof(z)); }
  return 0;
}
#endif

int cat_abi_version(void) { return CAT_ABI_VERSION; }
const char* cat_last_error(void) { return g_last_error.c_str(); }

// Everything cat_env_create checks of one map, before any CUDA call (testable without a device).
static int check_map(const CatMapDesc* map, const CatParams* pr) {
  const int A = map->n_cops + map->n_thieves, R = pr->n_rays, H = map->n_hulls, E = map->n_edges;
  if (map->n_cops < 1 || map->n_thieves < 1) return fail(CAT_ERR_INVALID, "need at least one cop and one thief");
  if (A > CAT_MAX_AGENTS) return fail(CAT_ERR_LIMIT, "too many agents (CAT_MAX_AGENTS)");
  if (R < 2 || R > CAT_MAX_RAYS) return fail(CAT_ERR_LIMIT, "n_rays out of range (2..CAT_MAX_RAYS)");
  if (H < 1 || H > 65535 || E > 65535) return fail(CAT_ERR_LIMIT, "hull/edge count out of range");
  const int ncell = map->nx * map->ny;
  if (ncell < 1 || map->con_cell_off[ncell] > 65535)
    return fail(CAT_ERR_LIMIT, "grid lists too long for 16-bit offsets");
  for (int h = 0; h < H; ++h)
    if (map->hull_off[h + 1] - map->hull_off[h] > 65535) return fail(CAT_ERR_LIMIT, "hull too large");
  if (!(pr->dt > 0.0)) return fail(CAT_ERR_INVALID, "dt must be > 0");
  const int P = A * (A - 1) / 2;
  if (P > 32) return fail(CAT_ERR_LIMIT, "too many agent pairs for one warp");
  return CAT_OK;
}

// The fp32 ray directions of every consumer (the step's blob, the renderer, cat_ray_directions): out[2 i], out[2 i + 1]
// = cos, sin of i 2 pi / R (entity.py:182 linspace(0, 2pi, R, endpoint=False)).
static void ray_directions(int R, float* out) {
  const double step = (2.0 * M_PI) / (double)R;
  for (int i = 0; i < R; ++i) { out[2 * i] = (float)cos(i * step); out[2 * i + 1] = (float)sin(i * step); }
}

// The shared-memory blob of one map (BlobHeader + arrays).  The header's global-memory table pointers are left zero:
// the caller fills them in once the tables are on the device.
static std::vector<unsigned char> build_blob(const CatMapDesc* map, const CatParams* pr) {
  const int A = map->n_cops + map->n_thieves, R = pr->n_rays, H = map->n_hulls, E = map->n_edges;
  const int ncell = map->nx * map->ny;
  // ---- blob
  const int nreg = map->region_off[A];
  BlobHeader hd{};
  int off = sizeof(BlobHeader);
  auto take = [&](int bytes) { int o = off; off = align_up(off + bytes, 16); return o; };
  hd.n_hulls = H; hd.n_edges = E; hd.nx = map->nx; hd.ny = map->ny;
  hd.gx0 = (float)map->grid_x0; hd.gy0 = (float)map->grid_y0; hd.cell = (float)map->cell;
  hd.inv_cell = (float)(1.0 / map->cell);
  hd.off_edge = take(E * 16);
  hd.off_len = take(E * 4);
  hd.off_hbb = take(H * 16);
  hd.off_heo = take(H * 4);
  hd.off_nextn = take(E * 8);
  hd.off_edgehull = take(E * 2 + 2);
  hd.off_conoff = take((ncell + 1) * 2);
  hd.off_conlist = take(map->con_cell_off[ncell] * 2 + 2);
  hd.off_dir = take(R * 16);
  hd.off_regoff = take((A + 1) * 4);
  hd.off_regions = take((nreg > 0 ? nreg : 1) * 16);
  hd.off_initpos = take(A * 8);
  hd.off_batchbb = take(((E + 31) / 32) * 16);
  const int blob_bytes = align_up(off, 16);
  std::vector<unsigned char> blob(blob_bytes, 0);
  memcpy(blob.data(), &hd, sizeof(hd));
  {
    float* e = reinterpret_cast<float*>(blob.data() + hd.off_edge);
    float* l = reinterpret_cast<float*>(blob.data() + hd.off_len);
    for (int i = 0; i < E; ++i) {
      e[4 * i + 0] = (float)map->vert[2 * i]; e[4 * i + 1] = (float)map->vert[2 * i + 1];
      e[4 * i + 2] = (float)map->normal[2 * i]; e[4 * i + 3] = (float)map->normal[2 * i + 1];
      l[i] = (float)map->edge_len[i];
    }
    float* bb = reinterpret_cast<float*>(blob.data() + hd.off_hbb);
    uint32_t* eo = reinterpret_cast<uint32_t*>(blob.data() + hd.off_heo);
    for (int h = 0; h < H; ++h) {
      // shape bb = raw hull bb grown by the wall radius; rounded outwards so fp32 never shrinks it
      bb[4 * h + 0] = nextafterf((float)(map->hull_bb[4 * h + 0] - pr->wall_radius), -INFINITY);
      bb[4 * h + 1] = nextafterf((float)(map->hull_bb[4 * h + 1] - pr->wall_radius), -INFINITY);
      bb[4 * h + 2] = nextafterf((float)(map->hull_bb[4 * h + 2] + pr->wall_radius), INFINITY);
      bb[4 * h + 3] = nextafterf((float)(map->hull_bb[4 * h + 3] + pr->wall_radius), INFINITY);
      eo[h] = (uint32_t)map->hull_off[h] | ((uint32_t)(map->hull_off[h + 1] - map->hull_off[h]) << 16);
    }
    uint16_t* co = reinterpret_cast<uint16_t*>(blob.data() + hd.off_conoff);
    for (int c = 0; c <= ncell; ++c) co[c] = (uint16_t)map->con_cell_off[c];
    uint16_t* eh = reinterpret_cast<uint16_t*>(blob.data() + hd.off_edgehull);
    float* nn = reinterpret_cast<float*>(blob.data() + hd.off_nextn);
    for (int h = 0; h < H; ++h) {
      const int o = map->hull_off[h], e = map->hull_off[h + 1];
      for (int i = o; i < e; ++i) {
        const int nx_ = (i + 1 < e) ? i + 1 : o;
        eh[i] = (uint16_t)h;
        nn[2 * i] = (float)map->normal[2 * nx_]; nn[2 * i + 1] = (float)map->normal[2 * nx_ + 1];
      }
    }
    uint16_t* cl = reinterpret_cast<uint16_t*>(blob.data() + hd.off_conlist);
    for (int i = 0; i < map->con_cell_off[ncell]; ++i) cl[i] = (uint16_t)map->con_cell_hulls[i];
    float* dir = reinterpret_cast<float*>(blob.data() + hd.off_dir);
    std::vector<float> u(2 * R);
    ray_directions(R, u.data());
    for (int i = 0; i < R; ++i) {
      const float ux = u[2 * i], uy = u[2 * i + 1];
      dir[4 * i] = ux; dir[4 * i + 1] = uy;
      dir[4 * i + 2] = ux != 0.f ? 1.f / ux : 0.f; dir[4 * i + 3] = uy != 0.f ? 1.f / uy : 0.f;
    }
    int32_t* rg = reinterpret_cast<int32_t*>(blob.data() + hd.off_regoff);
    for (int a = 0; a <= A; ++a) rg[a] = map->region_off[a];
    float* rr = reinterpret_cast<float*>(blob.data() + hd.off_regions);
    for (int i = 0; i < nreg * 4; ++i) rr[i] = (float)map->regions[i];
    float* bbb = reinterpret_cast<float*>(blob.data() + hd.off_batchbb);
    for (int b = 0; b * 32 < E; ++b) {
      float l = INFINITY, bo = INFINITY, r = -INFINITY, t = -INFINITY;
      for (int i = b * 32; i < E && i < b * 32 + 32; ++i) {
        // edge i spans vert[prev(i)] -> vert[i]; prev = i - 1 within the hull, else the hull's last vertex
        int h = 0;
        while (map->hull_off[h + 1] <= i) ++h;
        const int pi = (i > map->hull_off[h]) ? i - 1 : map->hull_off[h + 1] - 1;
        const int idx[2] = {i, pi};
        for (int q = 0; q < 2; ++q) {
          const float x = (float)map->vert[2 * idx[q]], y = (float)map->vert[2 * idx[q] + 1];
          l = fminf(l, x); r = fmaxf(r, x); bo = fminf(bo, y); t = fmaxf(t, y);
        }
      }
      bbb[4 * b + 0] = nextafterf(l, -INFINITY); bbb[4 * b + 1] = nextafterf(bo, -INFINITY);
      bbb[4 * b + 2] = nextafterf(r, INFINITY); bbb[4 * b + 3] = nextafterf(t, INFINITY);
    }
    float* ip = reinterpret_cast<float*>(blob.data() + hd.off_initpos);
    for (int i = 0; i < 2 * A; ++i) ip[i] = (float)map->init_pos[i];
  }

  return blob;
}

// The per-(cell, ray) candidate lists of one map on one device: found in the cache or built (on the device), and cached.
static int acquire_ray_lists(const CatMapDesc* map, const CatParams* pr, int device, SharedRayLists** out) {
  const int R = pr->n_rays, H = map->n_hulls, E = map->n_edges;
  const double rsum = pr->wall_radius + pr->ray_radius;
  // key: everything build_ray_lists reads
  std::vector<unsigned char> key;
  auto put = [&key](const void* p, size_t n) { const unsigned char* b = static_cast<const unsigned char*>(p); key.insert(key.end(), b, b + n); };
  const char* knob_cells = getenv("CAT_RAY_LIST_CELLS");
  const char* knob_min = getenv("CAT_RAY_LIST_MIN_CELL");
  const double head[6] = {(double)device, (double)R, pr->ray_length, rsum, pr->ray_list_cell,
                          (knob_cells ? atof(knob_cells) : 0.0) * 4096.0 + (knob_min ? atof(knob_min) : 0.0)};
  put(head, sizeof(head));
  put(&H, sizeof(H)); put(&E, sizeof(E));
  put(map->hull_off, sizeof(int32_t) * (H + 1));
  put(map->vert, sizeof(double) * 2 * E);
  put(map->normal, sizeof(double) * 2 * E);
  put(map->hull_bb, sizeof(double) * 4 * H);
  std::lock_guard<std::mutex> lock(g_ray_lists_mutex);
  SharedRayLists* sh = nullptr;
  for (SharedRayLists* c : g_ray_lists)
    if (c->key == key) { sh = c; break; }
  if (!sh) {
    RayListDeviceBuild b;
    int rc = b.size(map, R, pr->ray_length, rsum, pr->ray_list_cell);
    if (rc != CAT_OK) return rc;
    sh = new SharedRayLists();
    sh->g = b.su.g; sh->slot_words = b.slot_words; sh->ovf_words = b.ovf_words;
    const cudaError_t e1 = cudaMalloc(&sh->slots_dev, b.slot_words * 4);
    const cudaError_t e2 = e1 == cudaSuccess ? cudaMalloc(&sh->ovf_dev, b.ovf_words * 4) : e1;
    rc = e2 == cudaSuccess ? b.fill(reinterpret_cast<uint32_t*>(sh->slots_dev), sh->ovf_dev)
                           : fail(CAT_ERR_CUDA, std::string("ray lists: ") + cudaGetErrorString(e2));
    if (rc != CAT_OK) {
      if (sh->slots_dev) cudaFree(sh->slots_dev);
      if (sh->ovf_dev) cudaFree(sh->ovf_dev);
      delete sh;
      return rc;
    }
    sh->key.swap(key);
    g_ray_lists.push_back(sh);
  }
  ++sh->refs;
  *out = sh;
  return CAT_OK;
}

#define UPLOAD_TRY(expr, what)                                                                              \
  do {                                                                                                      \
    cudaError_t _e = (expr);                                                                                \
    if (_e != cudaSuccess) return fail(CAT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(_e));    \
  } while (0)

// Everything of one map but its blob allocation: its view lists and its share of the (cell, ray) lists go into `em`, and
// `blob` receives the blob whose header (also kept in em.header) points at them.  On failure whatever was allocated is
// left in `em` for release_map_tables.
static int prepare_map(const CatMapDesc* md, const CatParams* pr, int device, EnvMap& em, std::vector<unsigned char>& blob) {
  blob = build_blob(md, pr);
  BlobHeader& hd = em.header;
  memcpy(&hd, blob.data(), sizeof(hd));
  const int E = md->n_edges, ncell = md->nx * md->ny;
  // per-cell candidate lists (optional; valid only if they were built for at least this sensor range)
  // Worth it only when the full scan is long: the lists live in global memory (two dependent loads per sweep,
  // cold after an L2 flush), and a map of a few dozen edges is scanned in one or two batches anyway.
  if (md->view_cell_off && md->view_cell_edges && E >= 96 &&
      md->view_range >= pr->ray_length + pr->wall_radius + pr->ray_radius) {
    const int n_list = md->view_cell_off[ncell];
    std::vector<uint16_t> ve((size_t)(n_list > 0 ? n_list : 1));
    for (int i = 0; i < n_list; ++i) ve[i] = (uint16_t)md->view_cell_edges[i];
    UPLOAD_TRY(cudaMalloc(&em.view_off_dev, sizeof(int32_t) * (ncell + 1)), "cudaMalloc(view lists)");
    UPLOAD_TRY(cudaMalloc(&em.view_edges_dev, sizeof(uint16_t) * ve.size()), "cudaMalloc(view lists)");
    UPLOAD_TRY(cudaMemcpy(em.view_off_dev, md->view_cell_off, sizeof(int32_t) * (ncell + 1), cudaMemcpyHostToDevice), "cudaMemcpy(view lists)");
    UPLOAD_TRY(cudaMemcpy(em.view_edges_dev, ve.data(), sizeof(uint16_t) * ve.size(), cudaMemcpyHostToDevice), "cudaMemcpy(view lists)");
    hd.view_off = em.view_off_dev; hd.view_edges = em.view_edges_dev;
  }
  // per-(cell, ray) candidate lists of the sensor sweep (ray_lists.h), built from the map description
  if (!(pr->ray_list_cell < 0.0)) {
    const int rc = acquire_ray_lists(md, pr, device, &em.ray_lists);
    if (rc != CAT_OK) return rc;
    const SharedRayLists* sh = em.ray_lists;
    hd.ray_slots = sh->slots_dev; hd.ray_ovf = sh->ovf_dev;
    hd.ray_slot_count = (unsigned)(sh->slot_words / 4); hd.ray_ovf_words = (unsigned)sh->ovf_words;
    hd.rg_x0 = sh->g.x0; hd.rg_y0 = sh->g.y0; hd.rg_inv_cell = sh->g.inv_cell; hd.rg_nx = sh->g.nx; hd.rg_ny = sh->g.ny;
  }
  memcpy(blob.data(), &hd, sizeof(hd));
  return CAT_OK;
}

// The view lists and the (cell, ray) lists of `em` (not its blob).
static void release_map_tables(EnvMap& em) {
  if (em.view_off_dev) cudaFree(em.view_off_dev);
  if (em.view_edges_dev) cudaFree(em.view_edges_dev);
  ray_lists_release(em.ray_lists);
  em.view_off_dev = nullptr; em.view_edges_dev = nullptr; em.ray_lists = nullptr;
}

// Upload one map into `em`: prepare_map, then its blob in an allocation of `capacity` bytes (0: the blob's size) with a
// zeroed tail.  On failure whatever was allocated is left in `em` for cat_env_destroy.
static int upload_map(const CatMapDesc* md, const CatParams* pr, int device, int capacity, EnvMap& em) {
  std::vector<unsigned char> blob;
  const int rc = prepare_map(md, pr, device, em, blob);
  if (rc != CAT_OK) return rc;
  em.blob_bytes = capacity > 0 ? capacity : (int)blob.size();
  UPLOAD_TRY(cudaMalloc(&em.blob_dev, em.blob_bytes), "cudaMalloc(map blob)");
  UPLOAD_TRY(cudaMemcpy(em.blob_dev, blob.data(), blob.size(), cudaMemcpyHostToDevice), "cudaMemcpy(map blob)");
  if (em.blob_bytes > (int)blob.size())
    UPLOAD_TRY(cudaMemset(em.blob_dev + blob.size(), 0, em.blob_bytes - blob.size()), "cudaMemset(map blob)");
  return CAT_OK;
}
#undef UPLOAD_TRY

// Map m's own figures in `inf`: its worlds, hulls, edges, blob, CTAs of a full launch and (cell, ray) lists.
static void map_info(const CatEnv* env, int m, CatEnvInfo& inf) {
  const EnvMap& em = env->maps[m];
  const SharedRayLists* sh = em.ray_lists;
  inf.n_worlds = em.n_worlds; inf.n_hulls = em.header.n_hulls; inf.n_edges = em.header.n_edges; inf.map_blob_bytes = em.blob_bytes;
  inf.grid = (m + 1 < env->kp.n_maps ? env->kp.maps[m + 1].cta_begin : env->grid) - env->kp.maps[m].cta_begin;
  inf.ray_list_nx = em.header.rg_nx; inf.ray_list_ny = em.header.rg_ny; inf.ray_list_cells = inf.ray_list_nx * inf.ray_list_ny;
  inf.ray_list_cell = sh ? sh->g.cell : 0.f;
  inf.ray_list_bytes = sh ? (int64_t)(sh->slot_words + sh->ovf_words) * 4 : 0;
}

// The environment's figures: map 0's, then the totals over the maps (worlds, list bytes, the largest blob, the grid).
static void env_info(CatEnv* env) {
  const KParams& k = env->kp;
  CatEnvInfo& inf = env->info;
  map_info(env, 0, inf);
  for (int m = 1; m < (int)env->maps.size(); ++m) { CatEnvInfo other{}; map_info(env, m, other); inf.ray_list_bytes += other.ray_list_bytes; }
  inf.n_worlds = env->n_worlds; inf.n_agents = k.A; inf.n_cops = k.nc; inf.n_thieves = k.A - k.nc;
  inf.n_rays = k.R; inf.state_dim = k.state_dim; inf.record_words = k.lay.rec_words;
  inf.map_blob_bytes = env->blob_bytes; inf.smem_bytes_per_cta = env->smem_bytes; inf.warps_per_cta = env->threads / 32;
  inf.grid = env->grid; inf.n_pairs = k.lay.P;
}

static int create_env(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map, const CatParams* pr,
                      int64_t gid0, int32_t device, int blob_capacity, CatEnv** out);

// Map 0's values in the launch parameters: what a single-map launch reads (a mixed-map launch reads each map's from its
// blob header).  Refreshed when map 0 is replaced, so they never point at released lists.
static void set_map0_params(CatEnv* env) {
  KParams& k = env->kp;
  const EnvMap& em = env->maps[0];
  const BlobHeader& h = em.header;
  k.blob = em.blob_dev; k.blob_bytes = em.blob_bytes;
  k.view_off = h.view_off; k.view_edges = h.view_edges;
  k.ray_slots = h.ray_slots; k.ray_ovf = h.ray_ovf; k.ray_slot_count = h.ray_slot_count; k.ray_ovf_words = h.ray_ovf_words;
  k.rg_x0 = h.rg_x0; k.rg_y0 = h.rg_y0; k.rg_inv_cell = h.rg_inv_cell; k.rg_nx = h.rg_nx; k.rg_ny = h.rg_ny;
  k.n_edges = h.n_edges;
}

int cat_env_create(const CatMapDesc* map, const CatParams* pr, int32_t n_worlds, int64_t gid0, int32_t device,
                   CatEnv** out) {
  if (!map || !pr || !out) return fail(CAT_ERR_INVALID, "null argument");
  return cat_env_create_multi(map, 1, &n_worlds, pr, gid0, device, out);
}

int cat_env_create_multi(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map, const CatParams* pr,
                         int64_t gid0, int32_t device, CatEnv** out) {
  return create_env(maps, n_maps, worlds_per_map, pr, gid0, device, 0, out);
}

int cat_map_blob_bytes(const CatMapDesc* map, const CatParams* pr, int32_t* bytes) {
  if (!map || !pr || !bytes) return fail(CAT_ERR_INVALID, "null argument");
  const int rc = check_map(map, pr);
  if (rc != CAT_OK) return rc;
  *bytes = (int32_t)build_blob(map, pr).size();
  return CAT_OK;
}

// 227 KB: the largest dynamic shared memory a block of an sm_100 device can opt in to
static constexpr int kMaxBlobCapacity = 227 * 1024;

int cat_env_create_swappable(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map, const CatParams* pr,
                             int32_t blob_capacity, int64_t gid0, int32_t device, CatEnv** out) {
  if (!maps || !worlds_per_map || !pr || !out) return fail(CAT_ERR_INVALID, "null argument");
  *out = nullptr;
  if (pr->ray_list_cell < 0.0) return fail(CAT_ERR_INVALID, "a swappable environment needs ray lists (ray_list_cell >= 0)");
  // the step kernel stages the blob with one cp.async.bulk of blob_bytes, which must be a multiple of 16; and no blob
  // can exceed a block's shared memory (create_env checks the device's own limit before it allocates anything)
  if (blob_capacity < 16 || blob_capacity % 16) return fail(CAT_ERR_INVALID, "blob_capacity must be a positive multiple of 16");
  if (blob_capacity > kMaxBlobCapacity) return fail(CAT_ERR_LIMIT, "blob_capacity exceeds a block's shared memory");
  return create_env(maps, n_maps, worlds_per_map, pr, gid0, device, blob_capacity, out);
}

// cat_env_create_multi, and with blob_capacity > 0 cat_env_create_swappable
static int create_env(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map, const CatParams* pr,
                      int64_t gid0, int32_t device, int blob_capacity, CatEnv** out) {
  if (!maps || !worlds_per_map || !pr || !out) return fail(CAT_ERR_INVALID, "null argument");
  *out = nullptr;
  if (n_maps < 1) return fail(CAT_ERR_INVALID, "n_maps must be >= 1");
  if (n_maps > CAT_MAX_MAPS) return fail(CAT_ERR_LIMIT, "too many maps (CAT_MAX_MAPS)");
  long long total = 0;
  for (int m = 0; m < n_maps; ++m) {
    if (worlds_per_map[m] < 1) return fail(CAT_ERR_INVALID, "n_worlds must be >= 1");
    const int rc = check_map(&maps[m], pr);
    if (rc != CAT_OK) return rc;
    if (maps[m].n_cops != maps[0].n_cops || maps[m].n_thieves != maps[0].n_thieves)
      return fail(CAT_ERR_INVALID, "every map of an environment needs the same numbers of cops and thieves");
    if (blob_capacity > 0 && (int)build_blob(&maps[m], pr).size() > blob_capacity)
      return fail(CAT_ERR_LIMIT, "map blob larger than blob_capacity");
    total += worlds_per_map[m];
  }
  if (total > 0x7FFFFFFFll) return fail(CAT_ERR_LIMIT, "too many worlds");
  const CatMapDesc* map = &maps[0];   // agents, rays and constants are the same for every map
  const int n_worlds = (int)total;
  const int A = map->n_cops + map->n_thieves, R = pr->n_rays;
  CatEnv* env = new CatEnv();
  env->device = device;
  env->n_worlds = n_worlds;
  env->swappable = blob_capacity > 0;
  env->params = *pr;
  DeviceGuard guard(device);
  if (!guard.ok) { delete env; return fail(CAT_ERR_CUDA, "cudaSetDevice(" + std::to_string(device) + ") failed (no CUDA device?)"); }
  if (blob_capacity > 0) {   // the capacity must leave room for two warps' scratch on this device, checked before any allocation
    int optin = 0;
    if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess) {
      delete env;
      return fail(CAT_ERR_CUDA, "cudaDeviceGetAttribute(cudaDevAttrMaxSharedMemoryPerBlockOptin) failed");
    }
    if ((long long)align_up(blob_capacity, 128) + 2LL * make_layout(A, R).scratch_bytes > optin) {
      delete env;
      return fail(CAT_ERR_LIMIT, "blob_capacity leaves no launch shape (shared memory per block: " + std::to_string(optin) + " B)");
    }
  }
  // every failure below goes through cat_env_destroy: nothing allocated so far is leaked
#define CREATE_TRY(expr, what)                                                                              \
  do {                                                                                                      \
    cudaError_t _e = (expr);                                                                                \
    if (_e != cudaSuccess) { cat_env_destroy(env); return fail(CAT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(_e)); } \
  } while (0)
  CREATE_TRY(cudaMalloc(&env->overflow_dev, 2 * sizeof(unsigned long long)), "cudaMalloc(overflow counters)");
  CREATE_TRY(cudaMemset(env->overflow_dev, 0, 2 * sizeof(unsigned long long)), "cudaMemset(overflow counters)");
  env->maps.resize(n_maps);
  for (int m = 0, w0 = 0; m < n_maps; w0 += worlds_per_map[m], ++m) {
    EnvMap& em = env->maps[m];
    em.world_begin = w0; em.n_worlds = worlds_per_map[m];
    const int rc = upload_map(&maps[m], pr, device, blob_capacity, em);
    if (rc != CAT_OK) { cat_env_destroy(env); return rc; }
    env->blob_bytes = std::max(env->blob_bytes, em.blob_bytes);
  }

  KParams& k = env->kp;
  set_map0_params(env);
  k.overflow = env->overflow_dev;
  k.n_worlds = n_worlds; k.gid0 = gid0;
  k.A = A; k.nc = map->n_cops; k.R = R;
  k.lay = make_layout(A, R);          // record / scratch / output-record offsets (world_kernel.cuh)
  CatRecordLayout& rc = env->rec;
  rc.off_dist = 0; rc.off_type = k.lay.r_off_type; rc.off_reward = k.lay.r_off_reward;
  rc.off_terminated = k.lay.r_off_flags; rc.off_truncated = k.lay.r_off_flags + 1; rc.off_winner = k.lay.r_off_flags + 2;
  rc.bytes = k.lay.r_bytes; rc.type_bits = 8;
  CatRecordLayout& rp = env->rec_packed;   // the host-facing form: types packed 4 to a byte
  rp.off_dist = 0; rp.off_type = k.lay.r_off_type; rp.off_reward = k.lay.rp_off_reward;
  rp.off_terminated = k.lay.rp_off_flags; rp.off_truncated = k.lay.rp_off_flags + 1; rp.off_winner = k.lay.rp_off_flags + 2;
  rp.bytes = k.lay.rp_bytes; rp.type_bits = 2;
  k.state_dim = 0;
  for (int a = 0; a < A; ++a) k.state_dim += 4 * R + 2 * (a < map->n_cops ? map->n_cops : map->n_thieves);
  k.dt = (float)pr->dt; k.inv_dt = (float)(1.0 / pr->dt);
  k.impulse = (float)pr->unit_velocity; k.inv_mass = (float)(1.0 / pr->unit_mass);
  k.agent_r = (float)pr->unit_size; k.max_speed = (float)pr->max_speed; k.term_r = (float)pr->termination_radius;
  k.ray_len = (float)pr->ray_length; k.ray_r = (float)pr->ray_radius; k.wall_r = (float)pr->wall_radius;
  k.slop = (float)pr->collision_slop; k.bias_coef = (float)(1.0 - pow(pr->collision_bias, pr->dt));
  k.iterations = pr->iterations; k.persistence = pr->collision_persistence; k.max_steps = pr->max_step_count;
  k.stale = pr->stale_shape_cache; k.auto_reset = pr->auto_reset; k.seed = pr->seed;

  // Launch shape.  A warp owns a world, so with few worlds (one resident wave) the step takes as long as the
  // SM holding the most warps: smaller CTAs spread N warps more evenly over the SMs (4096 worlds = 27.7 warps per
  // SM: 8-warp CTAs put 32 on some SMs, 4-warp CTAs at most 28).  With many worlds the grid is persistent and the
  // shape with the most resident warps wins (ties: the larger CTA, fewer copies of the map).
  int max_optin = 0, n_sm = 0;
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
  const int smem_max = align_up(env->blob_bytes, 128) + 2 * k.lay.scratch_bytes;
  if (smem_max > max_optin) {
    cat_env_destroy(env);
    return fail(CAT_ERR_LIMIT, "map does not fit in shared memory (" + std::to_string(smem_max) + " B)");
  }
  // The attribute belongs to the FUNCTION (per device), not to this environment: always raise it to the device
  // maximum, so creating an environment for a smaller map never lowers the cap of one that is still alive.
  cudaFuncAttributes fattr{};
  env->kernel = pick_world_kernel(A, R, k.ray_slots != nullptr, true, n_maps > 1 || env->swappable);
  env->kernel_record = pick_world_kernel(A, R, k.ray_slots != nullptr, false, n_maps > 1 || env->swappable);
  CREATE_TRY(cudaFuncGetAttributes(&fattr, env->kernel), "cudaFuncGetAttributes");
  max_optin -= (int)fattr.sharedSizeBytes;      // the opt-in limit covers static + dynamic shared memory
  CREATE_TRY(cudaFuncSetAttribute(env->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin), "cudaFuncSetAttribute");
  if (env->kernel_record != env->kernel)
    CREATE_TRY(cudaFuncSetAttribute(env->kernel_record, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin), "cudaFuncSetAttribute");
  env->max_optin = max_optin; env->n_sm = n_sm;
  LaunchShape shp;
  if (!pick_launch_shape(env, n_worlds, &shp)) { cat_env_destroy(env); return fail(CAT_ERR_CUDA, "occupancy query failed"); }
  env->threads = shp.threads; env->smem_bytes = shp.smem;
  env->grid = fill_map_table(env, k, 0, n_worlds, shp.grid, shp.threads / 32);   // the table every full launch uses

  env_info(env);
#undef CREATE_TRY
  *out = env;
  return CAT_OK;
}

int cat_env_destroy(CatEnv* env) {
  if (!env) return CAT_OK;
  DeviceGuard guard(env->device);
  for (EnvMap& m : env->maps) {
    if (m.blob_dev) cudaFree(m.blob_dev);
    release_map_tables(m);
  }
  if (env->overflow_dev) cudaFree(env->overflow_dev);
  for (cudaEvent_t e : env->chunk_events) cudaEventDestroy(e);
  if (env->copies_done) cudaEventDestroy(env->copies_done);
  if (env->copy_stream) cudaStreamDestroy(env->copy_stream);
  delete env;
  return CAT_OK;
}

int cat_env_info(const CatEnv* env, CatEnvInfo* info) {
  if (!env || !info) return fail(CAT_ERR_INVALID, "null argument");
  *info = env->info;
  return CAT_OK;
}

int cat_env_map_info(const CatEnv* env, int32_t map, CatEnvInfo* info) {
  if (!env || !info) return fail(CAT_ERR_INVALID, "null argument");
  if (map < 0 || map >= (int)env->maps.size()) return fail(CAT_ERR_INVALID, "map index out of range");
  CatEnvInfo inf = env->info;
  map_info(env, map, inf);
  *info = inf;
  return CAT_OK;
}

int cat_env_set_map(CatEnv* env, int32_t m, const CatMapDesc* desc, void* stream) {
  if (!env || !desc) return fail(CAT_ERR_INVALID, "null argument");
  if (!env->swappable) return fail(CAT_ERR_INVALID, "the environment was not created by cat_env_create_swappable");
  if (m < 0 || m >= (int)env->maps.size()) return fail(CAT_ERR_INVALID, "map index out of range");
  const CatParams* pr = &env->params;
  int rc = check_map(desc, pr);
  if (rc != CAT_OK) return rc;
  if (desc->n_cops != env->kp.nc || desc->n_cops + desc->n_thieves != env->kp.A)
    return fail(CAT_ERR_INVALID, "the new map needs the environment's numbers of cops and thieves");
  if ((int)build_blob(desc, pr).size() > env->blob_bytes) return fail(CAT_ERR_LIMIT, "map blob larger than the environment's blob_capacity");
  DEVICE_SCOPE(env);
  // build everything new first: on failure the environment keeps its old map
  EnvMap fresh;
  std::vector<unsigned char> blob;
  rc = prepare_map(desc, pr, env->device, fresh, blob);
  if (rc != CAT_OK) { release_map_tables(fresh); return rc; }
  // a step in flight may still be staging the old blob (before griddepcontrol.wait): nothing is overwritten before it ends
  cudaError_t e = cudaDeviceSynchronize();
  EnvMap& em = env->maps[m];
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(em.blob_dev, blob.data(), blob.size(), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && em.blob_bytes > (int)blob.size()) e = cudaMemsetAsync(em.blob_dev + blob.size(), 0, em.blob_bytes - blob.size(), s);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { release_map_tables(fresh); return fail(CAT_ERR_CUDA, std::string("cat_env_set_map: ") + cudaGetErrorString(e)); }
  release_map_tables(em);
  em.view_off_dev = fresh.view_off_dev; em.view_edges_dev = fresh.view_edges_dev; em.ray_lists = fresh.ray_lists;
  em.header = fresh.header;
  if (m == 0) set_map0_params(env);
  env_info(env);
  return CAT_OK;
}

int cat_ray_lists_device(const CatMapDesc* map, int32_t n_rays, double ray_length, double rsum, double cell, double grid_out[5],
                         uint32_t* slots_dev, int64_t* n_slot_words, uint32_t* ovf_dev, int64_t* n_ovf_words, int32_t device) {
  if (!map || !grid_out || !n_slot_words || !n_ovf_words) return fail(CAT_ERR_INVALID, "null argument");
  if (n_rays < 2 || n_rays > CAT_MAX_RAYS || map->n_hulls < 1 || map->n_edges > 65535) return fail(CAT_ERR_LIMIT, "ray / hull / edge count out of range");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(CAT_ERR_CUDA, "cudaSetDevice(" + std::to_string(device) + ") failed (no CUDA device?)");
  RayListDeviceBuild b;
  int rc = b.size(map, n_rays, ray_length, rsum, cell);
  if (rc != CAT_OK) return rc;
  const RayListGrid& g = b.su.g;
  grid_out[0] = g.x0; grid_out[1] = g.y0; grid_out[2] = g.cell; grid_out[3] = g.nx; grid_out[4] = g.ny;
  if (slots_dev && ovf_dev) {
    if (*n_slot_words < (int64_t)b.slot_words || *n_ovf_words < (int64_t)b.ovf_words) return fail(CAT_ERR_INVALID, "buffers too small");
    rc = b.fill(slots_dev, ovf_dev);
    if (rc != CAT_OK) return rc;
  }
  *n_slot_words = (int64_t)b.slot_words; *n_ovf_words = (int64_t)b.ovf_words;
  return CAT_OK;
}

int cat_ray_lists_host(const CatMapDesc* map, int32_t n_rays, double ray_length, double rsum, double cell, double grid_out[5],
                       uint32_t* slots, int64_t* n_slot_words, uint32_t* ovf, int64_t* n_ovf_words) {
  if (!map || !grid_out || !n_slot_words || !n_ovf_words) return fail(CAT_ERR_INVALID, "null argument");
  if (n_rays < 2 || n_rays > CAT_MAX_RAYS || map->n_hulls < 1 || map->n_edges > 65535) return fail(CAT_ERR_LIMIT, "ray / hull / edge count out of range");
  RayLists rl;
  build_ray_lists(map, n_rays, ray_length, rsum, cell, &rl);
  grid_out[0] = rl.g.x0; grid_out[1] = rl.g.y0; grid_out[2] = rl.g.cell; grid_out[3] = rl.g.nx; grid_out[4] = rl.g.ny;
  if (slots && ovf) {
    if (*n_slot_words < (int64_t)rl.slots.size() || *n_ovf_words < (int64_t)rl.ovf.size()) return fail(CAT_ERR_INVALID, "buffers too small");
    memcpy(slots, rl.slots.data(), rl.slots.size() * 4);
    memcpy(ovf, rl.ovf.data(), rl.ovf.size() * 4);
  }
  *n_slot_words = (int64_t)rl.slots.size(); *n_ovf_words = (int64_t)rl.ovf.size();
  return CAT_OK;
}

int cat_env_record_layout(const CatEnv* env, CatRecordLayout* layout) {
  if (!env || !layout) return fail(CAT_ERR_INVALID, "null argument");
  *layout = env->rec;
  return CAT_OK;
}

int cat_env_packed_record_layout(const CatEnv* env, CatRecordLayout* layout) {
  if (!env || !layout) return fail(CAT_ERR_INVALID, "null argument");
  *layout = env->rec_packed;
  return CAT_OK;
}

int cat_env_overflow_counts(CatEnv* env, uint64_t out[2], int32_t reset) {
  if (!env || !out) return fail(CAT_ERR_INVALID, "null argument");
  DEVICE_SCOPE(env);
  CUDA_TRY(cudaDeviceSynchronize());
  unsigned long long v[2] = {0, 0};
  CUDA_TRY(cudaMemcpy(v, env->overflow_dev, sizeof(v), cudaMemcpyDeviceToHost));
  out[0] = v[0]; out[1] = v[1];
  if (reset) CUDA_TRY(cudaMemset(env->overflow_dev, 0, sizeof(v)));
  return CAT_OK;
}

int cat_env_set_seed(CatEnv* env, uint64_t seed) {
  if (!env) return fail(CAT_ERR_INVALID, "null env");
  env->kp.seed = seed;
  return CAT_OK;
}

size_t cat_env_state_bytes(const CatEnv* env) {
  return env ? (size_t)env->n_worlds * env->kp.lay.rec_words * 4 : 0;
}

static int prepare(CatEnv* env, void* state_dev, const CatStepIO* io, int mode, KParams* out) {
  if (!env || !state_dev) return fail(CAT_ERR_INVALID, "null env/state");
  KParams k = env->kp;
  k.state = reinterpret_cast<float*>(state_dev);
  k.mode = mode;
  if (io) {
    if (mode == MODE_STEP) {
      if (!io->actions) return fail(CAT_ERR_INVALID, "step needs actions");
      if (io->actions_kind < 0 || io->actions_kind > 3) return fail(CAT_ERR_INVALID, "bad actions_kind");
      k.actions_kind = io->actions_kind;
      if (io->actions_kind == 3) for (int a = 0; a < k.A; ++a) k.actions[a] = reinterpret_cast<const void* const*>(io->actions)[a];
      else k.actions[0] = io->actions;
    }
    k.reset_mask = io->reset_mask;
    k.shared_dist = io->shared_dist; k.shared_type = io->shared_type;
    k.team_pos = io->team_pos; k.obs_f32 = io->obs_f32; k.state_f32 = io->state_f32; k.hit_point = io->hit_point;
    k.critic_f32 = io->critic_f32; k.obs_bf16 = io->obs_bf16; k.critic_bf16 = io->critic_bf16;
    if (io->record) {
      k.record = reinterpret_cast<unsigned char*>(io->record);
      k.record_packed = io->record_packed_types ? 1 : 0;
      const int rec_bytes = k.record_packed ? k.lay.rp_bytes : k.lay.r_bytes;
      k.record_stride = io->record_world_stride ? io->record_world_stride : rec_bytes;
      if ((reinterpret_cast<uintptr_t>(io->record) & 15) || (k.record_stride & 15) || k.record_stride < rec_bytes)
        return fail(CAT_ERR_INVALID, "record output must be 16-byte aligned with a world stride that is a multiple of 16 and >= CatRecordLayout.bytes");
    }
    if (mode == MODE_STEP) {   // final outputs: step launches only (reset / observe share the caller's CatStepIO)
      if (io->final_record) {
        k.final_record = reinterpret_cast<unsigned char*>(io->final_record);
        k.final_record_stride = io->final_record_world_stride ? io->final_record_world_stride : k.lay.r_bytes;
        if ((reinterpret_cast<uintptr_t>(io->final_record) & 15) || (k.final_record_stride & 15) || k.final_record_stride < k.lay.r_bytes)
          return fail(CAT_ERR_INVALID, "final_record must be 16-byte aligned with a world stride that is a multiple of 16 and >= CatRecordLayout.bytes");
      }
      k.final_obs_f32 = io->final_obs_f32; k.final_state_f32 = io->final_state_f32; k.final_critic_f32 = io->final_critic_f32;
    }
  } else if (mode == MODE_STEP) {
    return fail(CAT_ERR_INVALID, "step needs a CatStepIO");
  }
  *out = k;
  return CAT_OK;
}

// the instantiation for this launch: the record-only one for a step whose record is all it writes (no final outputs)
static WorldKernel kernel_for(const CatEnv* env, const KParams& k) {
  const bool record_only = k.mode == MODE_STEP && k.record && !k.shared_dist && !k.shared_type && !k.team_pos && !k.obs_f32 && !k.state_f32 &&
                           !k.hit_point && !k.critic_f32 && !k.obs_bf16 && !k.critic_bf16 &&
                           !k.final_record && !k.final_obs_f32 && !k.final_state_f32 && !k.final_critic_f32 && !k.ep_acc && !k.wp &&
                           !k.script_mode;
  return record_only ? env->kernel_record : env->kernel;
}

// The statistics live in env->kp, which every launch (prepare) starts from.
int cat_env_attach_episode_stats(CatEnv* env, const CatEpisodeStatsIO* io) {
  if (!env) return fail(CAT_ERR_INVALID, "null env");
  if (!io) {
    env->kp.ep_acc = nullptr; env->kp.ep_return = nullptr; env->kp.ep_length = nullptr; env->kp.ep_totals = nullptr;
    return CAT_OK;
  }
  if (!io->acc) return fail(CAT_ERR_INVALID, "episode statistics need acc");
  if (((reinterpret_cast<uintptr_t>(io->acc) | reinterpret_cast<uintptr_t>(io->episode_return) |
        reinterpret_cast<uintptr_t>(io->episode_length)) & 3) || (reinterpret_cast<uintptr_t>(io->totals) & 7))
    return fail(CAT_ERR_INVALID, "episode statistics: acc / episode_return / episode_length must be 4-byte aligned, totals 8-byte aligned");
  env->kp.ep_acc = io->acc; env->kp.ep_return = io->episode_return; env->kp.ep_length = io->episode_length;
  env->kp.ep_totals = io->totals;
  return CAT_OK;
}

// Like the statistics, the table lives in env->kp.
int cat_env_attach_world_params(CatEnv* env, const CatWorldParamsIO* io) {
  if (!env) return fail(CAT_ERR_INVALID, "null env");
  if (!io) {
    env->kp.wp = nullptr; env->kp.wp_ranges = nullptr;
    return CAT_OK;
  }
  if (!io->params) return fail(CAT_ERR_INVALID, "world parameters need params");
  if ((reinterpret_cast<uintptr_t>(io->params) | reinterpret_cast<uintptr_t>(io->ranges)) & 3)
    return fail(CAT_ERR_INVALID, "world parameters: params / ranges must be 4-byte aligned");
  env->kp.wp = io->params; env->kp.wp_ranges = io->ranges;
  return CAT_OK;
}

// Like the statistics, the tables live in env->kp.
int cat_env_attach_scripts(CatEnv* env, const CatScriptIO* io) {
  if (!env) return fail(CAT_ERR_INVALID, "null env");
  if (!io) {
    env->kp.script_mode = nullptr; env->kp.script_dec = nullptr;
    return CAT_OK;
  }
  if (!io->mode || !io->decisions) return fail(CAT_ERR_INVALID, "scripts need mode and decisions");
  env->kp.script_mode = io->mode; env->kp.script_dec = io->decisions;
  return CAT_OK;
}

static int launch(CatEnv* env, void* state_dev, const CatStepIO* io, int mode, void* stream) {
  KParams k;
  const int rc = prepare(env, state_dev, io, mode, &k);
  if (rc != CAT_OK) return rc;
  DEVICE_SCOPE(env);
  CUDA_TRY(launch_pdl(kernel_for(env, k), env->grid, env->threads, (size_t)env->smem_bytes, reinterpret_cast<cudaStream_t>(stream), k));
  return CAT_OK;
}

int cat_env_init_state(CatEnv* env, void* state_dev, void* stream) { return launch(env, state_dev, nullptr, MODE_INIT, stream); }
int cat_env_reset(CatEnv* env, void* state_dev, const CatStepIO* io, void* stream) { return launch(env, state_dev, io, MODE_RESET, stream); }
int cat_env_step(CatEnv* env, void* state_dev, const CatStepIO* io, void* stream) { return launch(env, state_dev, io, MODE_STEP, stream); }
int cat_env_observe(CatEnv* env, void* state_dev, const CatStepIO* io, void* stream) { return launch(env, state_dev, io, MODE_OBSERVE, stream); }

// BaseEnv.step for a caller whose buffers are pinned HOST memory, pipelined: the worlds are stepped in
// `n_chunks` consecutive launches on `stream`, each writing its worlds' output RECORDS into `records_dev`; as
// soon as a chunk's launch has finished, its block of records moves to `records_host` with ONE cudaMemcpyAsync on
// an internal copy stream (DMA engine, full PCIe rate) while the next chunk computes.  `stream` finally waits for
// the copies, so one cudaStreamSynchronize(stream) by the caller makes every result visible.
int cat_env_step_host(CatEnv* env, void* state_dev, const uint8_t* host_actions, void* records_dev, void* records_host,
                      int32_t record_world_stride, int32_t packed_types, int32_t n_chunks, void* stream_) {
  if (!env || !host_actions || !records_dev || !records_host) return fail(CAT_ERR_INVALID, "null argument");
  const int N = env->n_worlds;
  if (n_chunks < 1) n_chunks = 1;
  if (n_chunks > N) n_chunks = N;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  DEVICE_SCOPE(env);
  if (!env->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&env->copy_stream, cudaStreamNonBlocking));
  if (!env->copies_done) CUDA_TRY(cudaEventCreateWithFlags(&env->copies_done, cudaEventDisableTiming));
  while ((int)env->chunk_events.size() < n_chunks) {
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    env->chunk_events.push_back(e);
  }
  CatStepIO io{};
  io.actions = host_actions; io.actions_kind = 0;
  io.record = records_dev; io.record_world_stride = record_world_stride; io.record_packed_types = packed_types;
  KParams k;
  const int rc = prepare(env, state_dev, &io, MODE_STEP, &k);
  if (rc != CAT_OK) return rc;
  const size_t stride = (size_t)k.record_stride;
  const int per = ((N + n_chunks - 1) / n_chunks + 7) / 8 * 8;   // worlds per chunk, a multiple of the CTA's 8 warps
  int c = 0;
  for (int w0 = 0; w0 < N; w0 += per, ++c) {
    const int w1 = w0 + per < N ? w0 + per : N, n = w1 - w0;
    LaunchShape shp;
    if (!pick_launch_shape(env, n, &shp)) return fail(CAT_ERR_CUDA, "occupancy query failed");
    const int grid = fill_map_table(env, k, w0, w1, shp.grid, shp.threads / 32);   // (a chunk may span several maps)
    CUDA_TRY(launch_pdl(kernel_for(env, k), grid, shp.threads, (size_t)shp.smem, stream, k));
    CUDA_TRY(cudaEventRecord(env->chunk_events[c], stream));
    CUDA_TRY(cudaStreamWaitEvent(env->copy_stream, env->chunk_events[c], 0));
    CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(records_host) + (size_t)w0 * stride, static_cast<const char*>(records_dev) + (size_t)w0 * stride,
                             (size_t)n * stride, cudaMemcpyDeviceToHost, env->copy_stream));
  }
  CUDA_TRY(cudaEventRecord(env->copies_done, env->copy_stream));
  CUDA_TRY(cudaStreamWaitEvent(stream, env->copies_done, 0));
  return CAT_OK;
}

static int state_view(CatEnv* env, void* state_dev, const CatStateView* view, int set, void* stream) {
  if (!env || !state_dev || !view) return fail(CAT_ERR_INVALID, "null argument");
  const KParams& k = env->kp;
  ViewParams p{};
  p.state = reinterpret_cast<float*>(state_dev);
  p.rec_words = k.lay.rec_words; p.n_worlds = k.n_worlds; p.A = k.A; p.P = k.lay.P;
  p.o_vel = k.lay.o_vel; p.o_vb = k.lay.o_vb; p.o_tc = k.lay.o_tc; p.o_wkey = k.lay.o_wkey; p.o_wjn = k.lay.o_wjn;
  p.o_page = k.lay.o_page; p.o_pjn = k.lay.o_pjn; p.o_sc = k.lay.o_sc; p.o_ep = k.lay.o_ep; p.o_flags = k.lay.o_flags;
  p.v = *view; p.set = set;
  DEVICE_SCOPE(env);
  const int threads = 128, blocks = (k.n_worlds + threads - 1) / threads;
  cat_state_view_kernel<<<blocks, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  CUDA_TRY(cudaGetLastError());
  return CAT_OK;
}

int cat_env_get_state(CatEnv* env, const void* state_dev, const CatStateView* view, void* stream) {
  return state_view(env, const_cast<void*>(state_dev), view, 0, stream);
}
int cat_env_set_state(CatEnv* env, void* state_dev, const CatStateView* view, void* stream) {
  return state_view(env, state_dev, view, 1, stream);
}

// ---- tensor maps for the TMA-fed GAE kernel
static PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

static bool gae_tma_usable(const void* r, const void* d, const void* v, int M) {
  const char* env = getenv("CAT_GAE_TMA");   // opt-out (A/B against the register-pipelined kernel); a libc table look-up, ~50 ns
  if (env && env[0] == '0') return false;
  if (M % 16 != 0) return false;                                           // u8 row stride must be a multiple of 16 bytes
  if ((reinterpret_cast<uintptr_t>(r) | reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(v)) & 15) return false;
  return tensor_map_encoder() != nullptr;
}

static bool encode_2d(CUtensorMap* tm, CUtensorMapDataType dt, const void* ptr, int M, int T, int elem) {
  const cuuint64_t dims[2] = {(cuuint64_t)M, (cuuint64_t)T};
  const cuuint64_t strides[1] = {(cuuint64_t)M * elem};
  const cuuint32_t box[2] = {(cuuint32_t)kTmaCols, (cuuint32_t)kTmaRows};
  const cuuint32_t estr[2] = {1, 1};
  return tensor_map_encoder()(tm, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int cat_gae(const float* rewards, const uint8_t* dones, const float* values, const float* last_values, float* returns,
            float* advantages, double* stats_dev, int32_t T, int32_t M, float gamma, float lam, void* stream) {
  if (!rewards || !dones || !values || !last_values || !returns || !advantages || !stats_dev)
    return fail(CAT_ERR_INVALID, "null argument");
  if (T < 1 || M < 1) return fail(CAT_ERR_INVALID, "T and M must be >= 1");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int threads = kGaeCols * kGaeSegs, blocks = (M + kGaeCols - 1) / kGaeCols;
  const bool idx32 = (long long)(T + kTmaRows) * M < (1ll << 31);
  if (gae_tma_usable(rewards, dones, values, M)) {
    // TMA-fed variant: tensor maps over (M, T) for r, V (fp32) and done (u8), box 64 columns x 32 steps
    CUtensorMap tm_r, tm_v, tm_d;
    if (encode_2d(&tm_r, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rewards, M, T, 4) && encode_2d(&tm_v, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, values, M, T, 4) &&
        encode_2d(&tm_d, CU_TENSOR_MAP_DATA_TYPE_UINT8, dones, M, T, 1)) {
      const int smem = kTmaStages * kTmaStageBytes, tblocks = (M + kTmaCols - 1) / kTmaCols;
      // the shared-memory opt-in is a per-function, per-device attribute: set once per device, not per call
      static bool attr_set[64] = {false};
      int devid = 0;
      CUDA_TRY(cudaGetDevice(&devid));
      if (devid < 0 || devid >= 64 || !attr_set[devid]) {
        CUDA_TRY(cudaFuncSetAttribute(cat_gae_tma_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        CUDA_TRY(cudaFuncSetAttribute(cat_gae_tma_kernel<size_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (devid >= 0 && devid < 64) attr_set[devid] = true;
      }
      if (idx32)
        CUDA_TRY(launch_pdl(cat_gae_tma_kernel<uint32_t>, tblocks, kTmaCols * kTmaSegs, smem, s, tm_r, tm_v, tm_d, last_values, returns, advantages, stats_dev, T, M, gamma, lam));
      else
        CUDA_TRY(launch_pdl(cat_gae_tma_kernel<size_t>, tblocks, kTmaCols * kTmaSegs, smem, s, tm_r, tm_v, tm_d, last_values, returns, advantages, stats_dev, T, M, gamma, lam));
      CUDA_TRY(cudaGetLastError());
      return CAT_OK;
    }
  }
  if (idx32)
    CUDA_TRY(launch_pdl(cat_gae_kernel<uint32_t>, blocks, threads, 0, s, rewards, dones, values, last_values, returns, advantages, stats_dev, T, M, gamma, lam));
  else
    CUDA_TRY(launch_pdl(cat_gae_kernel<size_t>, blocks, threads, 0, s, rewards, dones, values, last_values, returns, advantages, stats_dev, T, M, gamma, lam));
  CUDA_TRY(cudaGetLastError());
  return CAT_OK;
}

int cat_adv_normalize(float* advantages, int64_t n, const double* stats_dev, int64_t count, void* stream) {
  if (!advantages || !stats_dev) return fail(CAT_ERR_INVALID, "null argument");
  if (n < 1 || count < 1) return fail(CAT_ERR_INVALID, "n and count must be >= 1");
  if ((reinterpret_cast<uintptr_t>(advantages) & 15) != 0) return fail(CAT_ERR_INVALID, "advantages must be 16-byte aligned");
  const int threads = 256;
  long long blocks = (n / 4 + threads - 1) / threads;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 16) blocks = 148 * 16;
  CUDA_TRY(launch_pdl(cat_adv_normalize_kernel, (int)blocks, threads, 0, reinterpret_cast<cudaStream_t>(stream), advantages, (long long)n, stats_dev, (long long)count));
  CUDA_TRY(cudaGetLastError());
  return CAT_OK;
}


// ---- renderer (render_kernel.cuh)
struct CatRenderer {
  int device = 0, n_maps = 0, A = 0, nc = 0, R = 0, Wmax = 0, Hmax = 0;
  RenderMap maps[CAT_MAX_MAPS] = {};
  float2* dirs_dev = nullptr;
};

int cat_renderer_destroy(CatRenderer* r) {
  if (!r) return CAT_OK;
  DeviceGuard guard(r->device);
  for (int m = 0; m < r->n_maps; ++m)
    if (r->maps[m].wall) cudaFree(const_cast<uint32_t*>(r->maps[m].wall));
  if (r->dirs_dev) cudaFree(r->dirs_dev);
  delete r;
  return CAT_OK;
}

// Map m's wall layer: the hulls go to the device in fp64 (with render_rgb's clip boxes), one kernel sets the bits.
static int build_wall_layer(const CatMapDesc* md, int W, int H, RenderMap& rm) {
  const int nh = md->n_hulls, ne = md->n_edges;
  rm.W = W; rm.H = H; rm.hwords = (H + 31) / 32;
  std::vector<WallHull> hulls(nh > 0 ? nh : 1);
  for (int h = 0; h < nh; ++h) {
    const double* bb = md->hull_bb + 4 * h;   // l, b, r, t; render_rgb: [max(0, floor(l - 1)), min(W, ceil(r + 1) + 1))
    auto lo = [](double v) { return (int)std::max(0.0, std::min(1e9, floor(v - 1.0))); };
    auto hi = [](double v, int n) { return (int)std::min((double)n, std::max(-1.0, ceil(v + 1.0) + 1.0)); };
    hulls[h] = WallHull{md->hull_off[h], md->hull_off[h + 1], lo(bb[0]), hi(bb[2], W), lo(bb[1]), hi(bb[3], H)};
  }
  const size_t words = (size_t)W * rm.hwords;
  WallHull* hulls_dev = nullptr;
  double2 *vert_dev = nullptr, *normal_dev = nullptr;
  uint32_t* bits = nullptr;
  cudaError_t e = cudaMalloc(&bits, words * 4);
  if (e == cudaSuccess) rm.wall = bits;
  if (e == cudaSuccess) e = cudaMalloc(&hulls_dev, sizeof(WallHull) * hulls.size());
  if (e == cudaSuccess) e = cudaMalloc(&vert_dev, sizeof(double2) * (ne > 0 ? ne : 1));
  if (e == cudaSuccess) e = cudaMalloc(&normal_dev, sizeof(double2) * (ne > 0 ? ne : 1));
  if (e == cudaSuccess) e = cudaMemcpy(hulls_dev, hulls.data(), sizeof(WallHull) * hulls.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && ne > 0) e = cudaMemcpy(vert_dev, md->vert, sizeof(double2) * ne, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && ne > 0) e = cudaMemcpy(normal_dev, md->normal, sizeof(double2) * ne, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    const long long n = (long long)words * 32;
    cat_wall_bits_kernel<<<(unsigned)((n + 255) / 256), 256>>>(hulls_dev, nh, vert_dev, normal_dev, H, rm.hwords, n, bits);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (hulls_dev) cudaFree(hulls_dev);
  if (vert_dev) cudaFree(vert_dev);
  if (normal_dev) cudaFree(normal_dev);
  return e == cudaSuccess ? CAT_OK : fail(CAT_ERR_CUDA, std::string("renderer wall layer: ") + cudaGetErrorString(e));
}

int cat_renderer_create(const CatMapDesc* maps, const int32_t* windows, int32_t n_maps, int32_t n_rays, int32_t device,
                        CatRenderer** out) {
  if (!maps || !windows || !out) return fail(CAT_ERR_INVALID, "null argument");
  *out = nullptr;
  if (n_maps < 1) return fail(CAT_ERR_INVALID, "n_maps must be >= 1");
  if (n_maps > CAT_MAX_MAPS) return fail(CAT_ERR_LIMIT, "too many maps (CAT_MAX_MAPS)");
  if (n_rays < 2 || n_rays > CAT_MAX_RAYS) return fail(CAT_ERR_LIMIT, "n_rays out of range (2..CAT_MAX_RAYS)");
  for (int m = 0; m < n_maps; ++m) {
    const CatMapDesc& md = maps[m];
    if (windows[2 * m] < 1 || windows[2 * m] > 8192 || windows[2 * m + 1] < 1 || windows[2 * m + 1] > 8192)
      return fail(CAT_ERR_INVALID, "window sides must be in 1..8192");
    if (md.n_cops < 1 || md.n_thieves < 1) return fail(CAT_ERR_INVALID, "need at least one cop and one thief");
    if (md.n_cops + md.n_thieves > CAT_MAX_AGENTS) return fail(CAT_ERR_LIMIT, "too many agents (CAT_MAX_AGENTS)");
    if (md.n_cops != maps[0].n_cops || md.n_thieves != maps[0].n_thieves)
      return fail(CAT_ERR_INVALID, "every map of a renderer needs the same numbers of cops and thieves");
    if (md.n_hulls < 0 || md.n_edges < 0) return fail(CAT_ERR_INVALID, "negative hull / edge count");
    if (md.n_hulls > 0 && (!md.hull_off || !md.vert || !md.normal || !md.hull_bb)) return fail(CAT_ERR_INVALID, "null hull array");
  }
  CatRenderer* r = new CatRenderer();
  r->device = device; r->n_maps = n_maps; r->nc = maps[0].n_cops; r->A = maps[0].n_cops + maps[0].n_thieves; r->R = n_rays;
  DeviceGuard guard(device);
  if (!guard.ok) { delete r; return fail(CAT_ERR_CUDA, "cudaSetDevice(" + std::to_string(device) + ") failed (no CUDA device?)"); }
  for (int m = 0; m < n_maps; ++m) {
    r->Wmax = std::max(r->Wmax, (int)windows[2 * m]); r->Hmax = std::max(r->Hmax, (int)windows[2 * m + 1]);
    const int rc = build_wall_layer(&maps[m], windows[2 * m], windows[2 * m + 1], r->maps[m]);
    if (rc != CAT_OK) { cat_renderer_destroy(r); return rc; }
  }
  std::vector<float> u(2 * n_rays);
  ray_directions(n_rays, u.data());
  cudaError_t e = cudaMalloc(&r->dirs_dev, sizeof(float2) * n_rays);
  if (e == cudaSuccess) e = cudaMemcpy(r->dirs_dev, u.data(), sizeof(float2) * n_rays, cudaMemcpyHostToDevice);
  // the largest frame table any renderer needs (CAT_MAX_AGENTS x CAT_MAX_RAYS segments); a per-function attribute
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(cat_render_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, render_smem_bytes(CAT_MAX_AGENTS * CAT_MAX_RAYS));
  if (e != cudaSuccess) { cat_renderer_destroy(r); return fail(CAT_ERR_CUDA, std::string("cat_renderer_create: ") + cudaGetErrorString(e)); }
  *out = r;
  return CAT_OK;
}

static int frame_size(const CatRenderer* r, int d, int* w, int* h) {
  if (d < 1) return fail(CAT_ERR_INVALID, "downsample must be >= 1");
  *w = (r->Wmax - d / 2 + d - 1) / d; *h = (r->Hmax - d / 2 + d - 1) / d;
  if (*w < 1 || *h < 1) return fail(CAT_ERR_INVALID, "downsample leaves an empty frame");
  return CAT_OK;
}

int cat_renderer_frame_size(const CatRenderer* r, int32_t downsample, int32_t* w, int32_t* h) {
  if (!r || !w || !h) return fail(CAT_ERR_INVALID, "null argument");
  return frame_size(r, downsample, w, h);
}

int cat_ray_directions(int32_t n_rays, float* out) {
  if (!out) return fail(CAT_ERR_INVALID, "null argument");
  if (n_rays < 2 || n_rays > CAT_MAX_RAYS) return fail(CAT_ERR_LIMIT, "n_rays out of range (2..CAT_MAX_RAYS)");
  ray_directions(n_rays, out);
  return CAT_OK;
}

int cat_render(const CatRenderer* r, const CatRenderIO* io, void* stream) {
  if (!r || !io) return fail(CAT_ERR_INVALID, "null argument");
  if (io->n_frames < 0) return fail(CAT_ERR_INVALID, "n_frames must be >= 0");
  if (io->n_elements < 0) return fail(CAT_ERR_INVALID, "n_elements must be >= 0");
  if (io->downsample < 1) return fail(CAT_ERR_INVALID, "downsample must be >= 1");
  if (!io->pos || !io->frames) return fail(CAT_ERR_INVALID, "null pos / frames");
  if ((reinterpret_cast<uintptr_t>(io->pos) & 3) || (io->pos_stride & 3))
    return fail(CAT_ERR_INVALID, "pos must be 4-byte aligned with a stride that is a multiple of 4");
  if (!io->ray_dist != !io->ray_type) return fail(CAT_ERR_INVALID, "ray_dist and ray_type go together");
  if (io->ray_dist && ((reinterpret_cast<uintptr_t>(io->ray_dist) & 1) || (io->ray_dist_stride & 1)))
    return fail(CAT_ERR_INVALID, "ray_dist must be 2-byte aligned with an even stride");
  if (!(io->agent_radius >= 0.0) || !isfinite(io->agent_radius)) return fail(CAT_ERR_INVALID, "agent_radius must be finite and >= 0");
  // the checks that need the renderer's figures
  const int A = r->A, R = r->R;
  if (io->pos_stride < 8 * A) return fail(CAT_ERR_INVALID, "pos stride smaller than 8 * n_agents");
  if (io->ray_dist && (io->ray_dist_stride < 2LL * A * R || io->ray_type_stride < (long long)A * R))
    return fail(CAT_ERR_INVALID, "ray strides smaller than one element's block");
  RenderParams p{};
  const int rc = frame_size(r, io->downsample, &p.Wd, &p.Hd);
  if (rc != CAT_OK) return rc;
  p.tiles_y = (p.Hd + kRenderTY - 1) / kRenderTY;
  p.tiles = (p.Wd + kRenderTX - 1) / kRenderTX * p.tiles_y;
  if ((long long)io->n_frames * p.tiles > 0x7FFFFFFFLL) return fail(CAT_ERR_LIMIT, "too many frames for one launch");
  if (io->n_frames == 0) return CAT_OK;
  for (int m = 0; m < r->n_maps; ++m) p.maps[m] = r->maps[m];
  p.n_maps = r->n_maps; p.A = A; p.nc = r->nc; p.R = R; p.dirs = r->dirs_dev;
  p.n_elements = io->n_elements; p.world = io->world; p.map_of = io->map_of;
  p.pos = static_cast<const unsigned char*>(io->pos); p.pos_stride = io->pos_stride;
  p.ray_dist = static_cast<const unsigned char*>(io->ray_dist); p.dist_stride = io->ray_dist_stride;
  p.ray_type = static_cast<const unsigned char*>(io->ray_type); p.type_stride = io->ray_type_stride;
  p.d = io->downsample; p.radius = io->agent_radius; p.radius2 = pow(io->agent_radius, 2.0);
  p.frames = io->frames;
  DEVICE_SCOPE(r);
  const int smem = render_smem_bytes(io->ray_dist ? A * R : 0);
  cat_render_kernel<<<(unsigned)((long long)io->n_frames * p.tiles), kRenderThreads, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  CUDA_TRY(cudaGetLastError());
  return CAT_OK;
}

}  // extern "C"
