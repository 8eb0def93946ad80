"""The CPU oracle with a per-world parameter table (test infrastructure).

``TableOracle`` steps worlds whose thrust and top speed per team, capture radius and time limit come from a table
(``world_params.PARAMS_DTYPE``, one entry per world), as the step kernel does while a table is attached.  It is built
from unmodified oracle calls:

* the action (``Entity._perform_action``, cat_oracle.c's ``orc_step``) is applied here in fp64 with the world's team
  values, the fp32 entries widened to double, with the same operations in the same order;
* then ``orc_step`` of an oracle created with the world's capture radius and time limit, zero thrust and an infinite
  top speed runs the rest of the step: its own action adds a signed zero and never clamps, and the termination test,
  observation, rewards, physics and auto-reset are the oracle's.  Worlds with equal radius and time limit are stepped
  together, in runs of consecutive worlds (so that every world keeps its global id);
* a re-spawn of a world whose ranges draw (``ranges``, one ``world_params.RANGES_DTYPE`` entry) writes
  ``draws_numpy`` of the new episode into its entry.

``draws_numpy`` re-implements ``cat_param_draws`` (cat_philox.h) from ``orc_philox``.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from as_cops_and_thieves_b200 import world_params as wparams
from oracle import cat_oracle as co
from oracle.cat_oracle import Oracle, OracleOut, OracleState

_STATE_FIELDS = ("pos", "vel", "vbias", "tc", "step_count", "episode", "wall_jn", "wall_age", "pair_jn", "pair_age")
_OUT_FIELDS = ("obs_dist", "obs_type", "hit_point", "hit_alpha", "reward", "terminated", "truncated", "winner",
               "shared_dist", "shared_type", "team_pos")


def draws_numpy(seed: int, gid: int, episode: int, r: np.ndarray) -> np.ndarray:
    """cat_param_draws + the field mapping, from orc_philox.  The float fields are exact in fp64 before their one
    rounding to fp32 when (hi - lo) has few significant bits (the ranges the tests use), so this is fmaf bit for bit."""
    k = [seed & 0xFFFFFFFF, seed >> 32]
    words = np.concatenate([co.philox([gid & 0xFFFFFFFF, gid >> 32, episode, 0xFF00 | j], k) for j in (0, 1)])[:6]
    u = (words >> np.uint32(8)).astype(np.float64) / 16777216.0
    out = np.zeros((), wparams.PARAMS_DTYPE)
    lo, hi = r["lo"], r["hi"]

    def f(i, a, b):
        return np.float32(np.float64(np.float32(b - a)) * u[i] + np.float64(a))
    for t in range(2):
        out["unit_velocity"][t] = f(t, lo["unit_velocity"][t], hi["unit_velocity"][t])
        out["max_speed"][t] = f(2 + t, lo["max_speed"][t], hi["max_speed"][t])
    out["termination_radius"] = f(4, lo["termination_radius"], hi["termination_radius"])
    n = int(hi["max_step_count"]) - int(lo["max_step_count"]) + 1
    out["max_step_count"] = int(lo["max_step_count"]) + ((int(words[5]) * n) >> 32)
    return out


def table_of(n: int, **params) -> np.ndarray:
    """(n,) entries holding ``EnvParams`` values (plus ``params``) for both teams."""
    from as_cops_and_thieves_b200.params import EnvParams
    t = np.zeros(n, wparams.PARAMS_DTYPE)
    t[:] = wparams.defaults(dict(EnvParams().as_dict(), **params))
    return t


def _view(cls, src, fields, i, j, **extra):
    """A sub-state / sub-output of worlds [i, j) whose arrays are views of ``src``'s: the oracle writes through them."""
    v = cls.__new__(cls)
    for name in fields:
        setattr(v, name, getattr(src, name)[i:j])
    for k, x in extra.items():
        setattr(v, k, x)
    return v


class TableOracle:
    """One map + parameter set, stepped with a per-world table: ``table`` (N,) ``PARAMS_DTYPE``, given per call or set
    on the object.  Resets draw into the table when ``ranges`` draws."""

    def __init__(self, cmap, ranges: Optional[np.ndarray] = None, **params):
        self.base = Oracle(cmap, **params)
        self.cmap, self.ranges, self.table = cmap, ranges, None
        self._by_key = {}

    def __getattr__(self, name):          # params, A, H, R, observe, segment_query_first, ...
        return getattr(self.base, name)

    def _oracle(self, radius: float, max_steps: int) -> Oracle:
        key = (radius, max_steps)
        if key not in self._by_key:
            p = dict(self.base.params, unit_velocity=0.0, max_speed=float("inf"), termination_radius=radius,
                     max_step_count=max_steps)
            self._by_key[key] = Oracle(self.cmap, **p)
        return self._by_key[key]

    def _draw(self, st: OracleState, table: np.ndarray, worlds: np.ndarray) -> None:
        if self.ranges is None or not int(self.ranges["draw"]):
            return
        for w in worlds:
            table[w] = draws_numpy(int(self.base.params["seed"]), st.gid0 + int(w), int(st.episode[w]), self.ranges)

    def reset(self, st: OracleState, mask: Optional[np.ndarray] = None, out: Optional[OracleOut] = None,
              table: Optional[np.ndarray] = None) -> OracleOut:
        table = self.table if table is None else table
        out = self.base.reset(st, mask, out)
        self._draw(st, table, np.arange(st.N) if mask is None else np.flatnonzero(mask))
        return out

    def step(self, st: OracleState, actions: np.ndarray, out: Optional[OracleOut] = None,
             table: Optional[np.ndarray] = None) -> OracleOut:
        table = self.table if table is None else table
        assert table is not None and table.dtype == wparams.PARAMS_DTYPE and table.shape == (st.N,)
        out = out or self.base.new_out(st.N)
        a = np.ascontiguousarray(actions, np.int32)
        A, nc, mass = self.base.A, self.cmap.n_cops, float(self.base.params["unit_mass"])
        team = (np.arange(A) >= nc).astype(int)
        # Entity._perform_action (entity.py:126-134) as orc_step does it, with the world's team values
        s = table["unit_velocity"].astype(np.float64)[:, team]
        vmax = table["max_speed"].astype(np.float64)[:, team]
        fx = np.where(a == 0, -s, np.where(a == 2, s, 0.0))
        fy = np.where(a == 1, s, np.where(a == 3, -s, 0.0))
        vx = st.vel[..., 0] + fx / mass
        vy = st.vel[..., 1] + fy / mass
        sp = np.sqrt(vx * vx + vy * vy)
        over = sp > vmax
        q = np.where(over, sp, 1.0)                  # (the clamped worlds divide by their own speed, as orc_step does)
        st.vel[..., 0] = np.where(over, vx / q * vmax, vx)
        st.vel[..., 1] = np.where(over, vy / q * vmax, vy)
        # the rest of the step, by runs of consecutive worlds sharing radius and time limit
        keys = list(zip(table["termination_radius"].astype(np.float64).tolist(), table["max_step_count"].tolist()))
        i = 0
        while i < st.N:
            j = i + 1
            while j < st.N and keys[j] == keys[i]:
                j += 1
            sub = _view(OracleState, st, _STATE_FIELDS, i, j, N=j - i, A=st.A, H=st.H, gid0=st.gid0 + i)
            sub_out = _view(OracleOut, out, _OUT_FIELDS, i, j)
            self._oracle(*keys[i]).step(sub, a[i:j], sub_out)
            i = j
        if int(self.base.params["auto_reset"]):
            self._draw(st, table, np.flatnonzero(out.terminated))
        return out
