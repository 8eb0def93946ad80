"""Numpy reference of the step kernel's scripted controllers (include/cat_b200.h, "SCRIPTED AGENTS"): integer rules on
one agent's own observation, and cat_script_random over the oracle's Philox.  ``decide_numpy`` gives the decision byte
the kernel writes (random | chase << 2 | evade << 4); ``decisions_of_record`` applies it to every agent of every world
of an emitted record."""
import numpy as np

from oracle import cat_oracle as co

ACT = (2, 1, 0, 3)          # quadrant 0 +x, 1 +y, 2 -x, 3 -y (entity.py:77-82)
TYPE_COP, TYPE_THIEF = 1, 2


def quadrant(i: int, R: int) -> int:
    """round(4 i / R) mod 4, halves going up."""
    return ((8 * i + R) // (2 * R)) % 4


def axis_ray(q: int, R: int) -> int:
    return ((q * R + 2) // 4) % R


def script_counter(step_count: int, a: int) -> int:
    """The fourth counter word of cat_script_random."""
    return 0x80000000 | ((step_count & 0x0FFFFFFF) << 3) | a


def random_action(seed: int, gid: int, episode: int, step_count: int, a: int) -> int:
    w = co.philox([gid & 0xFFFFFFFF, gid >> 32, episode & 0xFFFFFFFF, script_counter(step_count, a)],
                  [seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF])
    return int((int(w[0]) * 4) >> 32)


def decide_numpy(d_bits, types, is_cop: bool, seed: int, gid: int, episode: int, step_count: int, a: int, R: int) -> int:
    """The decision byte of agent ``a`` from its own rays: ``d_bits`` the f16 distance bits (uint16 [R]) and ``types``
    the ray types (uint8 [R])."""
    d = np.asarray(d_bits, dtype=np.uint16).astype(np.int64)
    ty = np.asarray(types, dtype=np.uint8)
    target = TYPE_THIEF if is_cop else TYPE_COP
    rnd = random_action(seed, gid, episode, step_count, a)
    seen = np.nonzero(ty[:R] == target)[0]
    if len(seen) == 0:
        return rnd | rnd << 2 | rnd << 4
    i_star = min(seen, key=lambda i: (int(d[i]), int(i)))
    qs = quadrant(int(i_star), R)
    chase = ACT[qs]
    best_q, best_c = None, -1
    for q in ((qs + 2) % 4, (qs + 1) % 4, (qs + 3) % 4):
        j = axis_ray(q, R)
        c = 0 if ty[j] == target else int(d[j])
        if c > best_c:
            best_q, best_c = q, c
    evade = ACT[best_q]
    return rnd | chase << 2 | evade << 4


def decisions_of_record(dist_bits, types, n_cops: int, seed: int, gid0: int, episode, step_count, worlds=None):
    """(N, A) uint8 decisions of an emitted record: ``dist_bits`` (N, A, R) uint16, ``types`` (N, A, R) uint8,
    ``episode`` / ``step_count`` (N,) the worlds' values; ``worlds`` restricts to those indices (others zero)."""
    dist_bits, types = np.asarray(dist_bits), np.asarray(types)
    N, A, R = types.shape
    out = np.zeros((N, A), np.uint8)
    for n in (range(N) if worlds is None else worlds):
        for a in range(A):
            out[n, a] = decide_numpy(dist_bits[n, a], types[n, a], a < n_cops, seed, gid0 + n, int(episode[n]) & 0xFFFFFFFF,
                                     int(step_count[n]), a, R)
    return out
