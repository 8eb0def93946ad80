/* Philox4x32-10 counter-based RNG (Salmon et al., SC'11; Random123 reference constants).
 *
 * Shared by the CUDA kernels and the host code so that spawn sampling is a pure function of
 * (seed, global world id, episode, agent, try) — independent of how worlds are sharded over GPUs.
 * Replaces the reference's mix of numpy Generator + unseeded python `random`
 * (/root/reference/src/environments/base_env.py:144, /root/reference/src/utils/map_utils.py:9-10),
 * which cannot be reproduced (SURVEY.md C-7).
 */
#ifndef CAT_PHILOX_H
#define CAT_PHILOX_H

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define CAT_HD __host__ __device__ __forceinline__
#else
#define CAT_HD static inline
#endif

#define CAT_PHILOX_M0 0xD2511F53u
#define CAT_PHILOX_M1 0xCD9E8D57u
#define CAT_PHILOX_W0 0x9E3779B9u
#define CAT_PHILOX_W1 0xBB67AE85u

typedef struct { uint32_t v[4]; } cat_u32x4;

CAT_HD cat_u32x4 cat_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                   uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)CAT_PHILOX_M0 * c0;
    uint64_t p1 = (uint64_t)CAT_PHILOX_M1 * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += CAT_PHILOX_W0; k1 += CAT_PHILOX_W1;
  }
  cat_u32x4 out;
  out.v[0] = c0; out.v[1] = c1; out.v[2] = c2; out.v[3] = c3;
  return out;
}

/* 24-bit uniform in [0,1): exactly representable in fp32, so fp32 (GPU) and fp64 (oracle) agree. */
CAT_HD float cat_u01_24(uint32_t bits) { return (float)(bits >> 8) * (1.0f / 16777216.0f); }

/* Spawn stream layout (one Philox call each):
 *   region pick : counter = (gid_lo, gid_hi, episode, agent<<8 | 0)      -> word 0, idx = mulhi(w0, n_regions)
 *   try t (0..) : counter = (gid_lo, gid_hi, episode, agent<<8 | (t+1))  -> x from word 0, y from word 1
 *   key = (seed_lo, seed_hi)
 */
CAT_HD uint32_t cat_spawn_region_index(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t agent,
                                       uint32_t n_regions) {
  cat_u32x4 r = cat_philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), episode, agent << 8,
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
  return (uint32_t)(((uint64_t)r.v[0] * (uint64_t)n_regions) >> 32);
}

CAT_HD void cat_spawn_uniforms(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t agent,
                               uint32_t attempt, float* ux, float* uy) {
  cat_u32x4 r = cat_philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), episode,
                                  (agent << 8) | (attempt + 1u),
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
  *ux = cat_u01_24(r.v[0]);
  *uy = cat_u01_24(r.v[1]);
}

/* Per-world parameter draws (CatWorldParams, cat_b200.h), at each re-spawn:
 *   call j (0, 1) : counter = (gid_lo, gid_hi, episode, 0xFF00 | j)
 *   fields 0..3 (unit_velocity[0..1], max_speed[0..1]) take the words of call 0, fields 4..5 (termination_radius,
 *   max_step_count) the first two words of call 1.  Spawns use agent << 8 | try with agent < 8, so the two streams
 *   never share a counter.
 * words[6] receives the six words; cat_param_float / cat_param_int map one to its range. */
CAT_HD void cat_param_draws(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t words[6]) {
  for (uint32_t j = 0; j < 2; ++j) {
    cat_u32x4 r = cat_philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), episode, 0xFF00u | j,
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    for (int i = 0; i < 4 && 4 * (int)j + i < 6; ++i) words[4 * j + i] = r.v[i];
  }
}

/* a float field: uniform on [lo, hi) before the fp32 rounding, which can reach hi (one fma: the GPU and the oracle
 * agree bit for bit) */
CAT_HD float cat_param_float(uint32_t word, float lo, float hi) { return fmaf(hi - lo, cat_u01_24(word), lo); }

/* an integer field in [lo, hi] */
CAT_HD int32_t cat_param_int(uint32_t word, int32_t lo, int32_t hi) {
  return lo + (int32_t)(((uint64_t)word * (uint64_t)(uint32_t)(hi - lo + 1)) >> 32);
}

/* The random controller's next action (CAT_SCRIPT_RANDOM, cat_b200.h) for agent a (< 8) of a world whose observation
 * is emitted at (episode, step_count):
 *   counter = (gid_lo, gid_hi, episode, 0x80000000 | (step_count & 0x0FFFFFFF) << 3 | a)  -> mulhi(word 0, 4)
 * Bit 31 keeps this stream apart from the spawn stream (agent << 8 | try, below 0x800) and from the parameter draws
 * (0xFF00 | j), so attaching scripts moves neither spawns nor parameter draws. */
CAT_HD uint32_t cat_script_random(uint64_t seed, uint64_t gid, uint32_t episode, uint32_t step_count, uint32_t a) {
  cat_u32x4 r = cat_philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), episode,
                                  0x80000000u | (step_count & 0x0FFFFFFFu) << 3 | a,
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
  return (uint32_t)(((uint64_t)r.v[0] * 4u) >> 32);
}

#endif /* CAT_PHILOX_H */
