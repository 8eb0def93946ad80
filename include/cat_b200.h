/* cat_b200 — C ABI of the B200-native batched cops-and-thieves environment step.
 *
 * The reference (Hevagog/as-cops-and-thieves) is pure Python over pymunk's CFFI; it has no FFI
 * seam of its own.  Each entry point below replaces the reference call(s) named beside it; the
 * Python class that mirrors the reference's PettingZoo / skrl surface
 * (as_cops_and_thieves_b200/env.py) is the only caller.  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; every `*_dev` / device pointer is CUDA device memory owned by the caller
 *     (PyTorch tensors); the library owns only the staged map constants inside CatEnv;
 *   - all work is enqueued on the caller's stream (`stream` = cudaStream_t as void*), no internal
 *     synchronisation, CUDA-graph capturable; one CatEnv per GPU / rank; not thread-safe per CatEnv;
 *   - return 0 on success, negative CatStatus on failure; never throws, never exits;
 *     cat_last_error() returns a thread-local message for the last failure;
 *   - there is NO CPU fallback: every compute entry point fails with CAT_ERR_CUDA without a GPU.
 *
 * Layouts (N worlds, A = n_cops + n_thieves agents ordered cops then thieves
 * [base_env.py:91-96], R rays).  Fields of each world's output record (CatStepIO.record, CatRecordLayout):
 *   distance  f16 [A][R]      entity.py:200-210   (float16 chain reproduced bit-for-bit)
 *   type      u8  [A][R]      entity.py:222-241   (WALL 0, COP 1, THIEF 2, EMPTY 4)
 *   reward    f32 [A]         cop.py:49-75, thief.py:48-69
 *   terminated u8             captured or timed out (entity.py:146)
 *   truncated  u8             timed out (base_env.py:397)
 *   winner     i8             -1 none, 0 cop, 1 thief (base_env.py:399-411)
 * Optional caller arrays:
 *   shared_dist f16 [N][2][R], shared_type u8 [N][2][R]   observation_spaces.py:97-121 (team 0 cops, 1 thieves)
 *   team_pos  f16 [N][A][2]   observation_spaces.py:92-95
 *   obs_f32   f32 [A][N][2R]  per-agent obs as skrl flattens it: [distance | object_type]
 *   state_f32 f32 [N][S]      env.state() as skrl flattens it, S = sum_a (4R + 2*team_size(a))
 *   hit_point f32 [N][A][R][2] pre-quantisation hit point (parity/debug)
 */
#ifndef CAT_B200_H
#define CAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAT_ABI_VERSION 9
#define CAT_MAX_AGENTS 8
#define CAT_MAX_RAYS 128
#define CAT_MAX_MAPS 8 /* maps of one environment (cat_env_create_multi) */
#define CAT_WALL_SLOTS 4 /* cached wall arbiters / simultaneous wall contacts kept per agent; a 5th is counted by
                            cat_env_overflow_counts, never dropped silently */
#define CAT_NEAR_SLOTS 4 /* hulls whose reach can contain a ray origin (alpha = 0 rule) kept per agent; same rule */

typedef enum {
  CAT_OK = 0,
  CAT_ERR_INVALID = -1, /* bad argument */
  CAT_ERR_CUDA = -2,    /* CUDA runtime error (incl. no device) */
  CAT_ERR_LIMIT = -3,   /* map / agent / ray count exceeds a compiled limit */
} CatStatus;

/* Host-side description of one compiled map (what maps.compile_map() yields; replaces
 * Map.populate_space + pymunk.Poly hulls, /root/reference/src/maps/map.py:119-128). */
typedef struct {
  int32_t n_hulls, n_edges;
  const int32_t* hull_off; /* [H+1] */
  const double* vert;      /* [E][2] hull vertices, CCW; edge i runs vert[i-1] -> vert[i] */
  const double* normal;    /* [E][2] outward unit normals */
  const double* edge_len;  /* [E] */
  const double* hull_bb;   /* [H][4] l,b,r,t of the raw hull */
  int32_t n_cops, n_thieves;
  const double* init_pos;    /* [A][2] */
  const int32_t* region_off; /* [A+1] */
  const double* regions;     /* [n_regions][4] x,y,w,h */
  double grid_x0, grid_y0, cell; /* uniform grid used by contact / spawn / start-inside lookups */
  int32_t nx, ny;
  const int32_t* con_cell_off;   /* [nx*ny+1] hulls within contact reach of each cell */
  const int32_t* con_cell_hulls;
  /* Optional (NULL = scan every edge): per grid cell, the edges that can be sensor candidates for some origin
   * inside the cell (facing it and within view_range), nearest first — maps.view_lists().  A conservative
   * superset: the kernel still applies the exact per-origin test to every listed edge, so results do not
   * depend on these lists; they only shorten the candidate scan.  Ignored unless
   * view_range >= ray_length + wall_radius + ray_radius. */
  const int32_t* view_cell_off;   /* [nx*ny+1] */
  const int32_t* view_cell_edges; /* edge ids (< 65535) */
  double view_range;
} CatMapDesc;

/* pyproject.toml:12-19 [tool.physical-params], entity.py:84-86, Chipmunk space defaults, SimpleEnv defaults */
typedef struct {
  double dt;              /* simple_env.py:20 (1/60) */
  int32_t max_step_count; /* simple_env.py:19 (400) */
  double unit_velocity, unit_mass, unit_size, max_speed, termination_radius;
  double ray_length, ray_radius, wall_radius;
  int32_t n_rays;
  int32_t iterations; /* cpSpace iterations (10) */
  double collision_slop, collision_bias;
  int32_t collision_persistence;
  int32_t stale_shape_cache; /* 1 = pymunk behaviour: reset leaves the query centres of the shapes stale (SURVEY.md A.10) */
  int32_t auto_reset;        /* 1 = done worlds are re-spawned inside the step and emit the reset observation */
  uint64_t seed;
  /* Sensor-sweep acceleration (never changes a result, tests/test_parity_gpu.py::test_candidate_lists_do_not_change_results):
   * the library builds, per cell of a uniform grid over the walls' reach and per ray index, the list of edges that
   * ray can touch from any origin in the cell, nearest first.  ray_list_cell = edge length of those cells in map
   * units; 0 = choose automatically (about 65536 cells, not below 6 units: 60-120 MB of lists); < 0 = no lists: every sweep rasterises
   * the map's edges into the per-agent depth buffer (the slower, any-map path). */
  double ray_list_cell;
} CatParams;

typedef struct {
  /* input (step only) */
  const void* actions;   /* kind 0: u8 [N][A]; 1: i32 [N][A]; 2: i64 [N][A]; 3: HOST array of A device pointers to i64 [N] */
  int32_t actions_kind;
  /* input (reset only): u8 [N] device mask, NULL = every world */
  const uint8_t* reset_mask;
  /* outputs — device pointers, any may be NULL */
  uint16_t* shared_dist;
  uint8_t* shared_type;
  uint16_t* team_pos;
  float* obs_f32;
  float* state_f32;
  float* hit_point;
  /* RECORD OUTPUT: one contiguous record per world, CatRecordLayout below —
   *   [ f16 distance A*R | pad to 16 | u8 type A*R | pad to 4 | f32 reward A | u8 terminated | u8 truncated | i8 winner | pad to 16 ]
   * written with 16-byte stores (device memory or mapped pinned host memory).  One world = one block, so a host-facing
   * caller moves a range of worlds with ONE copy.  NULL = no record: the launch writes only the optional outputs it is
   * given.  record must be 16-byte aligned and record_world_stride a multiple of 16 that is >= CatRecordLayout.bytes
   * (0 = exactly that). */
  void* record;
  int32_t record_world_stride;
  /* critic front end (lstm_value_net.py:122-137): the 4 ray channels LSTMValue cuts from the first agent's block of
   * env.state(), in the order it stacks them — [own_obj_types | own_distances | object_type_shared | distance_shared]
   * of cop_0 — f32 [N][4][R] */
  float* critic_f32;
  /* bf16 copies of obs_f32 ([A][N][2R]) and critic_f32 ([N][4][R]) for mixed-precision learners (optional) */
  uint16_t* obs_bf16;
  uint16_t* critic_bf16;
  /* != 0: `record` takes the PACKED form of the record (cat_env_packed_record_layout; types at 2 bits each, 640 B
   * instead of 832 B per world for 3 agents x 90 rays) — the form meant to cross PCIe on the host-facing path. */
  int32_t record_packed_types;
  /* FINAL OUTPUTS (step launches only; cat_env_reset / cat_env_observe ignore them).  For every world that ENDS in the
   * step (terminated: captured or timed out) they receive what that step would have emitted with auto_reset = 0: the
   * observation of the pre-physics positions with the terminal rewards, terminated, truncated and winner — bit for bit
   * the record / obs_f32 / state_f32 / critic_f32 of an auto_reset = 0 twin.  With auto_reset = 1 the normal outputs
   * of such a world hold the re-spawned episode's observation, so this is the only place its last observation appears
   * (gymnasium's final_observation: truncated episodes can be bootstrapped from V(s_final)).  The entries of worlds
   * that do not end are left untouched.  Any may be NULL; a step with none set costs nothing extra.
   *   final_record: the unpacked record (cat_env_record_layout), the alignment and stride rules of `record`
   *   final_obs_f32 / final_state_f32 / final_critic_f32: the layouts of obs_f32 / state_f32 / critic_f32 */
  void* final_record;
  int32_t final_record_world_stride;
  float* final_obs_f32;
  float* final_state_f32;
  float* final_critic_f32;
} CatStepIO;

/* EPISODE STATISTICS (cat_env_attach_episode_stats): the step kernel keeps each world's running return and reports
 * every episode that ends, per world and summed per map, at the cost of a few stores and atomics of the worlds that end.
 *
 * Semantics.  While statistics are attached, every step launch adds each agent's emitted fp32 reward to the world's
 * running return, acc = acc + reward (one fp32 add: bit for bit a cumulative_rewards += rewards on the same rewards).
 * A world ENDS in a step when it reports terminated (captured or timed out); for such a world the kernel writes the
 * episode's return per agent and its length (the step_count the step reached: steps since the world's last reset) to
 * episode_return / episode_length, adds the episode to the totals of its map, and zeroes acc.  The per-world entries
 * of other worlds are left untouched: valid where terminated, as the final outputs.  A reset never counts an episode:
 * cat_env_reset zeroes acc of the worlds it resets, cat_env_init_state zeroes every acc; cat_env_set_state does not
 * touch acc (a length follows whatever step_count it sets).  auto_reset = 0 follows the same rules.  cat_env_observe
 * ignores the statistics.
 *
 * Totals are indexed by the world's map slot (0 for a single-map environment, the slot of cat_env_create_multi /
 * _swappable otherwise); a zero-filled CatEpisodeTotals is the empty state.  Every field is updated by atomicAdd or
 * atomicMax only.  Minima and maxima are u32 keys under atomicMax: the maximum is stored as an order-preserving key of
 * the value, the minimum as the key's complement, so 0 = "no episode yet".  For lengths the key is the length itself;
 * for an fp32 return r with bits b, key = b | 0x80000000 if its sign bit is clear and ~b if it is set, which is
 * non-zero for every non-NaN value.  Counts, length sums and the minima and maxima are exact; the f64 sums depend on
 * the order in which the atomics land, so they may differ between runs in the last bits. */
typedef struct {
  uint64_t episodes;                            /* episodes that ended */
  uint64_t captures;                            /* ... by capture (cop win) */
  uint64_t timeouts;                            /* ... by timeout (thief win) */
  uint64_t length_sum;
  uint32_t length_min_key;                      /* ~min(length) */
  uint32_t length_max_key;                      /* max(length) */
  double return_sum[CAT_MAX_AGENTS];            /* per agent, sum of episode returns */
  double return_sq_sum[CAT_MAX_AGENTS];         /* per agent, sum of squared episode returns */
  uint32_t return_min_key[CAT_MAX_AGENTS];      /* ~key(min return) */
  uint32_t return_max_key[CAT_MAX_AGENTS];      /* key(max return) */
} CatEpisodeTotals;

/* caller-owned device pointers (N worlds, A agents) */
typedef struct {
  float* acc;                  /* f32 [N][A] running returns; required, zeroed by the caller before it is attached */
  float* episode_return;       /* f32 [N][A] return of the episode a world ended in its last step; optional */
  int32_t* episode_length;     /* i32 [N] its length; optional */
  CatEpisodeTotals* totals;    /* [n_maps] per map slot; optional */
} CatEpisodeStatsIO;

/* PER-WORLD PHYSICS PARAMETERS (cat_env_attach_world_params): each world reads its thrust and top speed per team, its
 * capture radius and its time limit from a caller-owned table instead of CatParams.
 *
 * Semantics.  While a table is attached, every step, reset and host-path chunk reads world w's entry params[w] in
 * place of CatParams.unit_velocity, .max_speed, .termination_radius and .max_step_count.  Agent a uses team
 * t = (a < n_cops ? 0 : 1): its action adds unit_velocity[t] * (1 / unit_mass) to its velocity (fp32, mass stays
 * environment-wide) and clamps the speed to max_speed[t].  The capture test is dist^2 < termination_radius^2 and the
 * timeout step_count >= max_step_count.
 *
 * Domain randomisation.  With ranges attached and ranges[slot].draw != 0 for the world's map slot, every re-spawn of
 * the world (cat_env_reset, the in-kernel auto-reset, and so the resets after cat_env_set_map) writes a fresh draw
 * into params[w]; the step in which a world ends used its old entry, the new one applies from its next step on.
 * cat_env_init_state never draws, and with draw == 0 or no ranges the resets leave the table alone (the caller writes
 * it: curriculum).  The draw is cat_param_draws (cat_philox.h) of (seed, gid, the new episode number): independent of
 * sharding, chunking and launch shape.  lo == hi pins a field.
 *
 * The kernel does not validate the table: it expects finite values, thrust >= 0, top speeds > 0, radius >= 0,
 * max_step_count >= 1 and lo <= hi (the Python setters check these). */
typedef struct {
  float unit_velocity[2];       /* impulse of one action: [0] cops, [1] thieves */
  float max_speed[2];           /* [0] cops, [1] thieves */
  float termination_radius;
  int32_t max_step_count;
} CatWorldParams;

typedef struct {
  CatWorldParams lo, hi;        /* floats fmaf(hi - lo, u, lo) with u in [0, 1), max_step_count in [lo, hi] */
  int32_t draw;                 /* 0: re-spawns leave the table alone */
} CatWorldParamRanges;

/* caller-owned device pointers, 4-byte aligned */
typedef struct {
  CatWorldParams* params;              /* [N] one entry per world; required */
  const CatWorldParamRanges* ranges;   /* [n_maps] one entry per map slot; optional */
} CatWorldParamsIO;

/* SCRIPTED AGENTS (cat_env_attach_scripts): built-in controllers that act for chosen agents inside the step kernel, as
 * fixed opponents and as a yardstick that does not move when the learner changes.
 *
 * Modes.  mode[w][a] selects what agent a of world w does at a step:
 *   CAT_SCRIPT_NONE    the caller's action, exactly as without scripts;
 *   CAT_SCRIPT_RANDOM  a uniform draw (cat_script_random, cat_philox.h);
 *   CAT_SCRIPT_CHASE   move along the axis nearest to the closest opponent the agent sees, otherwise random;
 *   CAT_SCRIPT_EVADE   move away from the closest opponent it sees, towards open space, otherwise random.
 * Values above 3 are undefined: the kernel does not validate the table (the Python setters do).
 *
 * Decisions.  A policy picks its next action from the observation the last launch emitted, and a controller sees
 * exactly that observation: the launch that emits a world's observation also writes, into decisions[w][a], the action
 * each controller would take next, random in bits 0-1, chase in bits 2-3 and evade in bits 4-5.  All three are stored,
 * so a mode may change between steps (in place, graph-safe) and the next step still acts on the latest observation.
 * A step uses (decisions[w][a] >> 2 (mode - 1)) & 3 for every agent whose mode is non-zero and does not read the
 * caller's action for it.
 *   - Step launches (every cat_env_step_host chunk included) and reset launches (so the resets after cat_env_set_map)
 *     write the decisions of every world whose observation they emit, from that observation: a world that auto-resets
 *     decides from its re-spawned observation; final outputs are never used.
 *   - cat_env_init_state zeroes every entry.  cat_env_observe and cat_env_set_state leave them alone (observing into
 *     another buffer, as the renderer does, must not change what the next step does).
 *
 * Controllers.  Agent a reads only its own observation, the f16 distance bits d[i] and types ty[i] of its rays
 * i < R.  Its target type is THIEF (2) for a cop and COP (1) for a thief.  Integer rules only:
 *   quadrant of ray i   q(i) = ((8 i + R) / (2 R)) mod 4, i.e. round(4 i / R) with halves going up;
 *   action of quadrant  ACT = {2 (+x), 1 (+y), 0 (-x), 3 (-y)};  axis ray of quadrant q: j(q) = ((q R + 2) / 4) mod R;
 *   seen                some ray has ty[i] == target; i* = the ray with the smallest (d[i], i), d compared as u16 bits;
 *   random              cat_script_random(seed, gid, episode, step_count, a), episode and step_count being the world's
 *                       values when the observation is emitted (0 and the new episode right after a re-spawn);
 *   chase               seen: ACT[q(i*)]; otherwise random;
 *   evade               seen: with q* = q(i*), score the quadrants (q*+2, q*+1, q*+3) mod 4 in that order by
 *                       c(q) = (ty[j(q)] == target ? 0 : d[j(q)]) and take ACT of the first with the strictly largest
 *                       score; otherwise random. */
#define CAT_SCRIPT_NONE 0
#define CAT_SCRIPT_RANDOM 1
#define CAT_SCRIPT_CHASE 2
#define CAT_SCRIPT_EVADE 3

/* caller-owned device pointers, both required */
typedef struct {
  const uint8_t* mode;          /* u8 [N][A] CAT_SCRIPT_* per agent */
  uint8_t* decisions;           /* u8 [N][A] the controllers' next actions, written by the kernel */
} CatScriptIO;

/* byte offsets inside one world's output record (cat_env_record_layout / cat_env_packed_record_layout) */
typedef struct {
  int32_t bytes;        /* record size = default world stride (multiple of 16) */
  int32_t off_dist;     /* f16 [A][R] */
  int32_t off_type;     /* type_bits == 8: u8 [A][R], ObjectType values (0 wall, 1 cop, 2 thief, 4 empty);
                         * type_bits == 2: ray r = a * R + i of the world is bits 2 (r % 4) .. + 1 of byte r / 4,
                         *   codes 0 wall, 1 cop, 2 thief, 3 empty */
  int32_t off_reward;   /* f32 [A] */
  int32_t off_terminated, off_truncated, off_winner; /* u8, u8, i8 */
  int32_t type_bits;    /* 8 or 2 */
} CatRecordLayout;

typedef struct {
  int32_t n_worlds, n_agents, n_cops, n_thieves, n_rays, n_hulls, n_edges;
  int32_t state_dim;          /* S of state_f32 */
  int32_t record_words;       /* 4-byte words per world in the packed state buffer */
  int32_t map_blob_bytes;     /* bytes staged into shared memory per CTA */
  int32_t smem_bytes_per_cta;
  int32_t warps_per_cta;
  int32_t grid;               /* CTAs launched by cat_env_step (cat_env_map_info: those of them that step the map) */
  int32_t n_pairs;
  int32_t ray_list_cells;     /* cells of the (cell, ray) candidate-list grid, 0 = lists disabled */
  int32_t ray_list_nx, ray_list_ny;
  float ray_list_cell;
  int64_t ray_list_bytes;     /* device bytes held by the lists (slots + overflow) */
} CatEnvInfo;

/* SoA view of the world state for get/set (device pointers; any may be NULL = skip). */
typedef struct {
  float* pos;          /* [N][A][2] */
  float* vel;          /* [N][A][2] */
  float* vbias;        /* [N][A][2] */
  float* tc;           /* [N][A][2] cached shape centres the queries see */
  int32_t* step_count; /* [N] */
  uint32_t* episode;   /* [N] */
  int32_t* wall_hull;  /* [N][A][CAT_WALL_SLOTS] hull id, -1 empty */
  int32_t* wall_age;   /* [N][A][CAT_WALL_SLOTS] */
  float* wall_jn;      /* [N][A][CAT_WALL_SLOTS] */
  int32_t* pair_age;   /* [N][P] pairs (i<j) in i-major order, -1 empty */
  float* pair_jn;      /* [N][P] */
} CatStateView;

typedef struct CatEnv CatEnv;

int cat_abi_version(void);
const char* cat_last_error(void);

/* BaseEnv.__init__ (base_env.py:51-121): stage the map, fix the constants.  gid0 = global id of
 * this rank's world 0 (spawn RNG is keyed by global world id). */
int cat_env_create(const CatMapDesc* map, const CatParams* params, int32_t n_worlds, int64_t gid0,
                   int32_t device, CatEnv** out);
/* One environment whose worlds run on several maps (mixed-map training), stepped by one launch per call: map m owns
 * the worlds [off_m, off_m + worlds_per_map[m]), off_m = the sum of the counts before it, and world i of the
 * environment is the same world as world i - off_m of a cat_env_create environment of map m with gid0 + off_m.
 * Every map must have the same numbers of cops and thieves (the rays and constants come from `params`, so the
 * observation, state and record layouts are the same for every map).  Each map's (cell, ray) lists are shared with
 * every other environment of that map on the device.  Returns CAT_ERR_INVALID for null pointers, n_maps < 1, a
 * count < 1 or maps with different agent counts, and CAT_ERR_LIMIT for n_maps > CAT_MAX_MAPS; the arguments are
 * checked before any CUDA call.  cat_env_create(map, params, n, gid0, device, out) is this call with one map.
 * Every other entry point works on such an environment as on a single-map one. */
int cat_env_create_multi(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map,
                         const CatParams* params, int64_t gid0, int32_t device, CatEnv** out);
/* A cat_env_create_multi environment whose maps can be replaced later (cat_env_set_map), e.g. to cycle a training run
 * through procedurally generated layouts without re-creating the environment, its buffers or a captured CUDA graph.
 * It differs from cat_env_create_multi in three ways:
 *   - it always runs the mixed-map kernels, even with one map: they read every map-dependent value (list pointers and
 *     grid, counts) from the blob each CTA stages, never from the launch parameters a captured graph keeps;
 *   - every map's blob is allocated once at blob_capacity bytes, and CatEnvInfo.map_blob_bytes and the launch shape
 *     are those of the capacity, so replacing a map changes neither.  blob_capacity must be a positive multiple of 16
 *     (the kernel stages the blob with one bulk copy of that size; CAT_ERR_INVALID otherwise) and >= every creation
 *     map's cat_map_blob_bytes; CAT_ERR_LIMIT if it is smaller, larger than 227 KB, or leaves no launch shape in the
 *     device's shared memory (checked before anything is allocated);
 *   - it needs (cell, ray) lists: params->ray_list_cell < 0 returns CAT_ERR_INVALID.
 * Every other argument and result is cat_env_create_multi's. */
int cat_env_create_swappable(const CatMapDesc* maps, int32_t n_maps, const int32_t* worlds_per_map,
                             const CatParams* params, int32_t blob_capacity, int64_t gid0, int32_t device, CatEnv** out);
/* Replace map m of a swappable environment by `desc` (same numbers of cops and thieves).  Checked before any CUDA call:
 * CAT_ERR_INVALID if the environment is not swappable, m is out of range, desc is NULL or its agent counts differ;
 * CAT_ERR_LIMIT if its blob (cat_map_blob_bytes) exceeds the environment's blob_capacity.  The new view lists and
 * (cell, ray) lists are built first (the lists on the device, shared through the same cache as at creation); only then is
 * the blob copied into the existing allocation, its tail zeroed, and the old map's lists released.  On any failure the
 * environment stays on its old map.
 * Ordering: a step kernel stages its map's blob before it waits on the previous kernel (programmatic dependent launch),
 * so this call synchronises the DEVICE before it overwrites anything and again before it returns.  It may allocate and is
 * not graph-capturable; a graph captured before it stays valid and steps the new map on its next replay.
 * World state is not touched: the worlds of map m still hold positions on the old map and MUST be reset
 * (cat_env_reset with a mask of those worlds) before the next step. */
int cat_env_set_map(CatEnv* env, int32_t m, const CatMapDesc* desc, void* stream);
/* host only: the bytes of the shared-memory blob of this map with these parameters (what blob_capacity must cover);
 * the map is checked as cat_env_create checks it */
int cat_map_blob_bytes(const CatMapDesc* map, const CatParams* params, int32_t* bytes);
int cat_env_destroy(CatEnv* env);
/* n_worlds: every world of the environment; ray_list_bytes: the sum over its maps; map_blob_bytes: the largest blob;
 * the other map-dependent fields (n_hulls, n_edges, ray_list_cells/nx/ny/cell) describe map 0 */
int cat_env_info(const CatEnv* env, CatEnvInfo* info);
/* the same figures for map `map` of the environment alone (n_worlds = that map's worlds, grid = its CTAs of a step) */
int cat_env_map_info(const CatEnv* env, int32_t map, CatEnvInfo* info);
int cat_env_record_layout(const CatEnv* env, CatRecordLayout* layout);
/* the record with CatStepIO.record_packed_types != 0 (what cat_env_step_host moves when packed_types != 0) */
int cat_env_packed_record_layout(const CatEnv* env, CatRecordLayout* layout);
/* Fixed-capacity bookkeeping that the reference (Chipmunk) does not have: out[0] = wall contacts beyond
 * CAT_WALL_SLOTS per agent, out[1] = near hulls beyond CAT_NEAR_SLOTS per agent, summed over every launch since
 * creation (or since the last call with reset != 0).  Synchronises the device.  Zero means no world ever diverged
 * from the uncapped algorithm for this reason. */
int cat_env_overflow_counts(CatEnv* env, uint64_t out[2], int32_t reset);
/* reset(seed=...) (base_env.py:307-311): re-key the spawn RNG of this environment */
int cat_env_set_seed(CatEnv* env, uint64_t seed);
/* bytes of the caller-owned packed state buffer (`state_dev` below) */
size_t cat_env_state_bytes(const CatEnv* env);

/* fresh-environment state: agents at their map positions (entity.py:115), nothing cached */
int cat_env_init_state(CatEnv* env, void* state_dev, void* stream);
/* BaseEnv.reset (base_env.py:286-352) for the masked worlds */
int cat_env_reset(CatEnv* env, void* state_dev, const CatStepIO* io, void* stream);
/* BaseEnv.step (base_env.py:354-413) for every world, one launch */
int cat_env_step(CatEnv* env, void* state_dev, const CatStepIO* io, void* stream);
/* BaseEnv.step for a caller whose buffers live in pinned HOST memory (the reference's own calling convention:
 * numpy in, numpy out), pipelined: the worlds are stepped in n_chunks consecutive launches on `stream` that write
 * record output (CatRecordLayout, stride record_world_stride) into `records_dev`; as soon as a chunk's launch has
 * finished its block of records is moved to `records_host` (pinned) with ONE cudaMemcpyAsync on an internal copy
 * stream while the next chunk computes.  host_actions: u8 [N][A] in pinned host memory, read by the kernel
 * directly.  `stream` waits for the copies: one cudaStreamSynchronize(stream) makes every result visible.
 * packed_types != 0: the records have the packed form (cat_env_packed_record_layout) — 23 % fewer bytes over PCIe. */
int cat_env_step_host(CatEnv* env, void* state_dev, const uint8_t* host_actions, void* records_dev,
                      void* records_host, int32_t record_world_stride, int32_t packed_types, int32_t n_chunks,
                      void* stream);
/* Entity.get_observation + get_shared_observations of the current state (entity.py:159-220,
 * observation_spaces.py:67-131) without stepping */
int cat_env_observe(CatEnv* env, void* state_dev, const CatStepIO* io, void* stream);
/* Attach episode statistics (CatEpisodeStatsIO above) to an environment, or detach them with io = NULL.  Host only, no
 * CUDA call: the pointers are stored, and every later launch of the environment (step, reset, init and the chunks of
 * cat_env_step_host) carries them; such launches run the full-output kernel.  CAT_ERR_INVALID for a null env, outputs
 * without acc, or a misaligned pointer (4 bytes for the arrays, 8 for totals); nothing is stored then.  A CUDA graph
 * captured before this call keeps the parameters its launches were captured with. */
int cat_env_attach_episode_stats(CatEnv* env, const CatEpisodeStatsIO* io);
/* Attach a per-world parameter table (CatWorldParamsIO above), or detach it with io = NULL.  Host only, no CUDA call,
 * like cat_env_attach_episode_stats: every later launch carries the pointers and runs the full-output kernel.
 * CAT_ERR_INVALID for a null env, a missing params pointer or a pointer that is not 4-byte aligned; nothing is stored
 * then.  The table's contents are not checked. */
int cat_env_attach_world_params(CatEnv* env, const CatWorldParamsIO* io);
/* Attach scripted agents (CatScriptIO above), or detach them with io = NULL.  Host only, no CUDA call, like
 * cat_env_attach_episode_stats: every later launch carries the pointers and runs the full-output kernel.
 * CAT_ERR_INVALID for a null env or a missing pointer; nothing is stored then.  The modes are not checked. */
int cat_env_attach_scripts(CatEnv* env, const CatScriptIO* io);
/* parity-test access to the hidden state */
int cat_env_get_state(CatEnv* env, const void* state_dev, const CatStateView* view, void* stream);
int cat_env_set_state(CatEnv* env, void* state_dev, const CatStateView* view, void* stream);

/* Inspection / test entry point (host only, needs no GPU): the per-(cell, ray) candidate lists cat_env_create builds for
 * this map and these sensor parameters, from the host reference builder (csrc/ray_lists.h).  grid_out = {x0, y0, cell, nx, ny}.  Call with slots = ovf =
 * NULL to get the sizes (in 32-bit words) in n_slot_words / n_ovf_words, then again with buffers of those sizes.
 * slot[(cell * n_rays + ray) * 4 .. +4]: entries (bf16 bits of the lower bound of the hit distance << 16 | edge id),
 * 0x7F80FFFF = end, bit 31 = link to a 4-word chunk of ovf (word offset in the low 31 bits). */
int cat_ray_lists_host(const CatMapDesc* map, int32_t n_rays, double ray_length, double rsum, double cell,
                       double grid_out[5], uint32_t* slots, int64_t* n_slot_words, uint32_t* ovf, int64_t* n_ovf_words);
/* The same lists built on device `device` by the builder every environment uses (csrc/ray_lists_kernel.cuh): the same
 * words as cat_ray_lists_host, into DEVICE buffers slots / ovf, with the same two-call sizing protocol.  Synchronises the
 * device; CAT_ERR_CUDA without one. */
int cat_ray_lists_device(const CatMapDesc* map, int32_t n_rays, double ray_length, double rsum, double cell,
                         double grid_out[5], uint32_t* slots, int64_t* n_slot_words, uint32_t* ovf, int64_t* n_ovf_words,
                         int32_t device);

/* skrl MAPPO._update GAE (SURVEY.md a-10; call site agent_learning_utils.py:198-199).
 * rewards/values [T][M] f32, dones [T][M] u8, last_values [M]; returns/advantages [T][M].
 * stats_dev: CAT_GAE_STATS_DOUBLES (6) doubles = { slot0[2], slot1[2], u64 calls, u64 ticket }, ZEROED BY THE CALLER
 * ONCE when it allocates them and then owned by cat_gae.  After a call, {sum(adv), sum(adv^2)} of that call are in slot
 * (calls & 1), i.e. stats_dev[2 * (calls & 1) .. + 2]; the other slot is zero and takes the next call's sums (so no memset
 * runs in front of the kernel and no CTA waits on a counter at its end: csrc/gae_kernels.cuh).  Calls that share a
 * stats buffer must be ordered (same stream).  Both kernels are launched with programmatic stream serialisation — their
 * prologues overlap the previous kernel's tail (environment CAT_PDL=0 turns that off).
 * Runs the TMA-fed kernel when M % 16 == 0 and the three input arrays are 16-byte aligned, the register-pipelined
 * kernel otherwise (environment CAT_GAE_TMA=0 forces the latter); both give the same results to fp32 rounding. */
#define CAT_GAE_STATS_DOUBLES 6
int cat_gae(const float* rewards, const uint8_t* dones, const float* values, const float* last_values,
            float* returns, float* advantages, double* stats_dev, int32_t T, int32_t M, float gamma,
            float lam, void* stream);
/* advantages = (advantages - mean) / (std + 1e-8) with mean/std (unbiased) from stats over `count` samples.  stats_dev
 * has cat_gae's layout (pass the buffer cat_gae filled).  For a global normalisation across ranks, all-reduce the sums and
 * the count and pass a zeroed CAT_GAE_STATS_DOUBLES buffer with the reduced sums in [0..1] (calls = 0 selects slot 0). */
int cat_adv_normalize(float* advantages, int64_t n, const double* stats_dev, int64_t count, void* stream);

/* ---- Renderer: rgb_array frames of many worlds in one launch (python: render.Renderer, CatWorlds.render_frames).
 * A renderer needs no CatEnv, so recorded trajectories can be drawn after their environment is gone.  A frame is the
 * image render.render_rgb(cmap, pos, agent_radius, rays) returns, bit for bit: u8 [W][H][3] (the layout of
 * pygame.surfarray.array3d), layers from first to last: black; the sensor rays when asked for (by ray type: wall
 * (96, 96, 96), cop (0, 160, 255), thief (255, 160, 0), empty (40, 40, 40); a pixel is on ray i of agent a when its
 * centre is within 0.5 of the segment from the agent's position P to P + dist[a][i] * direction[i], and a later
 * (a, i) wins); walls (white); the agents in index order, cops (0, 0, 255), thieves (255, 0, 0).  A frame is
 * (largest window width, largest window height) of the renderer's maps; pixels outside the frame's own map's window
 * are zero.  With downsample d the frame is frame_1[d/2::d, d/2::d]: (W - d/2 + d - 1) / d by (H - d/2 + d - 1) / d. */
typedef struct CatRenderer CatRenderer;

typedef struct {
  int32_t n_frames;          /* K */
  const int64_t* world;      /* device [K]: the element frame k shows; NULL = k.  An id outside [0, n_elements) gives
                                an all-zero frame, as does an element whose map_of is not a map of the renderer */
  int64_t n_elements;
  const int64_t* map_of;     /* device, the map of every element (CatWorlds.map_index); NULL = map 0 */
  const void* pos;           /* device: agent a of element e is the fp32 (x, y) at pos + e * pos_stride + 8 a (4-byte
                                aligned) — the packed state buffer holds them in words 0 .. 2A-1 of each record */
  int64_t pos_stride;        /* bytes, a multiple of 4, >= 8 A */
  const void* ray_dist;      /* optional (NULL = no rays): f16 [A][R] at ray_dist + e * ray_dist_stride (2-byte aligned) */
  int64_t ray_dist_stride;   /* bytes, even, >= 2 A R */
  const void* ray_type;      /* u8 [A][R] ObjectType at ray_type + e * ray_type_stride; given with ray_dist */
  int64_t ray_type_stride;   /* bytes, >= A R */
  int32_t downsample;        /* >= 1 */
  double agent_radius;       /* finite, >= 0 */
  uint8_t* frames;           /* device u8 [K][W'][H'][3], cat_renderer_frame_size; indexed with 64-bit offsets */
} CatRenderIO;

/* windows: [n_maps][2] window (width, height) of each map, sides in 1..8192.  Every map needs the same numbers of cops
 * and thieves; n_rays in 2..CAT_MAX_RAYS.  The arguments are checked before any CUDA call.  Builds each map's wall
 * layer (a bit per pixel) on the device and synchronises: call it outside graph capture. */
int cat_renderer_create(const CatMapDesc* maps, const int32_t* windows, int32_t n_maps, int32_t n_rays, int32_t device,
                        CatRenderer** out);
int cat_renderer_destroy(CatRenderer* renderer);
/* host only: the frame size (W', H') at this downsample */
int cat_renderer_frame_size(const CatRenderer* renderer, int32_t downsample, int32_t* w, int32_t* h);
/* K frames, one launch on `stream`: no allocation, no synchronisation, CUDA-graph capturable */
int cat_render(const CatRenderer* renderer, const CatRenderIO* io, void* stream);
/* host only: the fp32 ray directions the step and the renderer use, out[2 i] = (float)cos(i 2 pi / R),
 * out[2 i + 1] = (float)sin(i 2 pi / R) */
int cat_ray_directions(int32_t n_rays, float* out);

/* Environment variables the library reads (tuning / test knobs; none is needed for normal use, results never depend on them):
 *   CAT_GENERIC_KERNEL=1       cat_env_create: run the any-shape instantiation <0, 0> even for 3 agents x 90 rays (tests)
 *   CAT_MAX_WARPS_PER_CTA=n    pick_launch_shape: cap the warps per CTA (2..32)
 *   CAT_MAX_GRID=n             pick_launch_shape: cap the CTAs of a launch
 *   CAT_RAY_LIST_CELLS=n       automatic list grid: target cell count (default 65536)
 *   CAT_RAY_LIST_MIN_CELL=x    automatic list grid: smallest cell (default 6 units)
 *   CAT_PDL=0                  launch without programmatic stream serialisation (read once per process)
 *   CAT_GAE_TMA=0              cat_gae: use the register-pipelined kernel for every shape
 * Python side: CAT_B200_LIB=path loads another build of this library (profiling / checked builds under variants/). */

#ifdef __cplusplus
}
#endif
#endif /* CAT_B200_H */
