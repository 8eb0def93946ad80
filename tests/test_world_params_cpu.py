"""Per-world physics parameters without a GPU: the numpy views of the tables against their C structs (whose layout
test_abi.py checks with every struct's), argument checks of cat_env_attach_world_params, the Python-side validation, cat_param_draws against a numpy re-implementation over
orc_philox, and the table-driven oracle (world_params_reference.TableOracle): bit for bit the oracle where the table
holds the oracle's parameters, and its known answers for per-team top speeds, capture radius, time limit and draws."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
from scipy import stats

import parity_utils as pu
from as_cops_and_thieves_b200 import _lib, world_params as wparams
from as_cops_and_thieves_b200.maps import compile_map
from as_cops_and_thieves_b200.params import EnvParams
from oracle import cat_oracle as co
from world_params_reference import TableOracle, draws_numpy, table_of

ROOT = Path(__file__).resolve().parents[1]
P_FIELDS = ("unit_velocity", "max_speed", "termination_radius", "max_step_count")
M, _ = pu.load_analytic()
CMAP = compile_map(M, name="analytic")     # agents cop_0, cop_1 (no spawn region), thief_0; open floor around (500, 400)


def _probe(tmp_path, body: str, includes=("cat_b200.h",)) -> list:
    src = tmp_path / "probe.c"
    inc = "\n".join(f'#include "{h}"' for h in includes)
    src.write_text(f"#include <stdio.h>\n#include <stddef.h>\n#include <stdalign.h>\n{inc}\nint main(void) {{\n{body}\nreturn 0;\n}}\n")
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", "-std=gnu11", "-ffp-contract=off", "-I", str(ROOT / "include"), str(src), "-o", str(exe),
                    "-lm"], check=True)
    return subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()


def test_table_dtypes_match_the_structs():
    W, R = _lib.CatWorldParams, _lib.CatWorldParamRanges
    assert C.sizeof(W) == 24 and C.sizeof(R) == 52
    assert wparams.PARAMS_DTYPE.itemsize == 24 and wparams.RANGES_DTYPE.itemsize == 52
    assert all(wparams.PARAMS_DTYPE.fields[f][1] == getattr(W, f).offset for f in P_FIELDS)


def test_attach_checks_the_environment_first():
    assert "cat_env_attach_world_params" in _lib.EXPORTS
    L = _lib.load()
    io = _lib.CatWorldParamsIO()
    assert L.cat_env_attach_world_params(None, C.byref(io)) == -1
    assert b"null env" in L.cat_last_error()
    assert L.cat_env_attach_world_params(None, None) == -1


@pytest.mark.parametrize("field,value", [
    ("unit_velocity", -1.0), ("unit_velocity", float("nan")), ("max_speed", 0.0), ("max_speed", float("inf")),
    ("termination_radius", -0.5), ("max_step_count", 0), ("max_step_count", 2.5), ("max_step_count", 2 ** 31),
    ("mass", 1.0), ("max_speed", "fast")])
def test_values_are_checked(field, value):
    with pytest.raises(ValueError):
        wparams.check_values(field, value)


def test_teams_and_ranges_are_checked():
    p = EnvParams().as_dict()
    with pytest.raises(ValueError, match="unknown team"):
        list(wparams.per_team("max_speed", {"robber": 1.0}))
    with pytest.raises(ValueError, match="not a per-team"):
        list(wparams.per_team("termination_radius", {"cop": 1.0}))
    with pytest.raises(ValueError, match="lo"):
        wparams.ranges_entry({"termination_radius": (25, 15)}, p)
    with pytest.raises(ValueError):
        wparams.ranges_entry({"max_speed": (0, 10)}, p)
    with pytest.raises(ValueError):
        wparams.ranges_entry({"max_step_count": (1, 2, 3)}, p)
    with pytest.raises(ValueError):
        wparams.per_slot([None], 2)
    for bad in ("max_speed.thief", "max_speed=a:b", "max_speed=1:2:3", "max_speed.robber=1:2", "max_speed=2:1",
                "max_step_count=0:5"):
        with pytest.raises(ValueError):
            wparams.parse_cli(bad)


def test_spec_pins_what_it_does_not_name():
    p = EnvParams().as_dict()
    e = wparams.ranges_entry({"max_speed": {"thief": (125, 175)}, "termination_radius": (15, 25), "max_step_count": 400}, p)
    assert e["draw"] == 1
    assert list(e["lo"]["max_speed"]) == [125, 125] and list(e["hi"]["max_speed"]) == [125, 175]
    assert list(e["lo"]["unit_velocity"]) == [10, 10] and list(e["hi"]["unit_velocity"]) == [10, 10]
    assert (e["lo"]["termination_radius"], e["hi"]["termination_radius"]) == (15, 25)
    assert e["lo"]["max_step_count"] == e["hi"]["max_step_count"] == 400
    assert wparams.parse_cli("max_speed.thief=125:175, termination_radius=15:25,max_step_count=300:500") == \
        {"max_speed": {"thief": (125.0, 175.0)}, "termination_radius": (15.0, 25.0), "max_step_count": (300, 500)}
    d = wparams.defaults(p)
    assert d["max_step_count"] == 400 and d["termination_radius"] == np.float32(20.0)


# ---------------------------------------------------------------------------------------------- cat_param_draws
RANGES = wparams.ranges_entry({"unit_velocity": {"cop": (8, 12), "thief": (9.5, 10.5)}, "max_speed": (100, 150),
                               "termination_radius": (15, 25), "max_step_count": (3, 5)}, EnvParams().as_dict())


def test_param_draws_match_numpy(tmp_path):
    cases = [(0, 0, 1), (7, 5, 1), (2 ** 40 + 3, 2 ** 33 + 17, 9), (0xFFFFFFFFFFFFFFFF, 123456, 0xFFFFFFFF)]
    r = RANGES
    lines = []
    for seed, gid, ep in cases:
        lines.append(f"""{{ uint32_t u[6]; cat_param_draws({seed}ull, {gid}ull, {ep}u, u);
  printf("%u %u %u %u %u %u ", u[0], u[1], u[2], u[3], u[4], u[5]);
  float f[5]; int32_t n;
  f[0] = cat_param_float(u[0], {r['lo']['unit_velocity'][0]}f, {r['hi']['unit_velocity'][0]}f);
  f[1] = cat_param_float(u[1], {r['lo']['unit_velocity'][1]}f, {r['hi']['unit_velocity'][1]}f);
  f[2] = cat_param_float(u[2], {r['lo']['max_speed'][0]}f, {r['hi']['max_speed'][0]}f);
  f[3] = cat_param_float(u[3], {r['lo']['max_speed'][1]}f, {r['hi']['max_speed'][1]}f);
  f[4] = cat_param_float(u[4], {r['lo']['termination_radius']}f, {r['hi']['termination_radius']}f);
  n = cat_param_int(u[5], {r['lo']['max_step_count']}, {r['hi']['max_step_count']});
  for (int i = 0; i < 5; ++i) {{ union {{ float f; uint32_t u; }} b; b.f = f[i]; printf("%u ", b.u); }}
  printf("%d\\n", n); }}""")
    got = np.array(_probe(tmp_path, "\n".join(lines), includes=("cat_philox.h",)), np.int64).reshape(len(cases), 12)
    for (seed, gid, ep), row in zip(cases, got):
        k = [seed & 0xFFFFFFFF, seed >> 32]
        want_words = np.concatenate([co.philox([gid & 0xFFFFFFFF, gid >> 32, ep, 0xFF00 | j], k) for j in (0, 1)])[:6]
        assert list(row[:6]) == [int(w) for w in want_words]
        d = draws_numpy(seed, gid, ep, r)
        want = np.array([d["unit_velocity"][0], d["unit_velocity"][1], d["max_speed"][0], d["max_speed"][1],
                         d["termination_radius"]], np.float32).view(np.uint32)
        assert list(row[6:11]) == [int(x) for x in want]
        assert row[11] == d["max_step_count"]


def test_param_draws_cover_their_ranges_uniformly():
    r = RANGES
    d = np.array([draws_numpy(3, g, 1 + g % 7, r) for g in range(4000)])
    for f, t in (("unit_velocity", 0), ("unit_velocity", 1), ("max_speed", 0), ("max_speed", 1)):
        lo, hi = float(r["lo"][f][t]), float(r["hi"][f][t])
        v = d[f][:, t].astype(np.float64)
        assert (v >= lo).all() and (v <= hi).all()
        assert stats.kstest(v, "uniform", args=(lo, hi - lo)).pvalue > 1e-3, f
    v = d["termination_radius"].astype(np.float64)
    assert (v >= 15).all() and (v <= 25).all()
    assert stats.kstest(v, "uniform", args=(15, 10)).pvalue > 1e-3
    n = d["max_step_count"]
    assert set(np.unique(n)) == {3, 4, 5}, "both integer endpoints are reachable"
    assert stats.chisquare(np.bincount(n - 3)).pvalue > 1e-3
    # the two teams and the two calls are different streams
    assert not np.array_equal(d["max_speed"][:, 0], d["max_speed"][:, 1])


def test_param_counters_are_disjoint_from_the_spawn_stream():
    spawn = {(agent << 8) | t for agent in range(8) for t in range(21)}     # region pick (t = 0) and tries 1..20
    assert not spawn & {0xFF00, 0xFF01}


# ---------------------------------------------------------------------------------------------- the oracle with a table
OUT_KEYS = ("obs_dist", "obs_type", "reward", "terminated", "truncated", "winner")


def _run(orc, st, steps, rng, **kw):
    outs = []
    for _ in range(steps):
        o = orc.step(st, rng.integers(0, 4, (st.N, orc.A)), **kw)
        outs.append({k: getattr(o, k).copy() for k in OUT_KEYS})
    return outs


X = dict(unit_velocity=12.0, max_speed=140.0, termination_radius=25.0, max_step_count=60)


@pytest.mark.parametrize("params", [{}, X])
def test_table_oracle_is_bit_identical_to_the_oracle(params):
    """A table holding X steps exactly as the oracle created with X (X = the defaults, then other values), auto-resets
    included; the table never changes without ranges."""
    cm = pu.named_cmap("squarinth")
    ref, orc = co.Oracle(cm, seed=3, **params), TableOracle(cm, seed=3)
    s0, s1 = ref.new_state(48), orc.new_state(48)
    ref.reset(s0), orc.reset(s1, table=table_of(48))
    table = table_of(48, **params)
    before = table.copy()
    o0 = _run(ref, s0, 410, np.random.default_rng(1))
    o1 = _run(orc, s1, 410, np.random.default_rng(1), table=table)
    for t, (x, y) in enumerate(zip(o0, o1)):
        for k in OUT_KEYS:
            assert np.array_equal(x[k], y[k]), (t, k)
    for k in ("pos", "vel", "vbias", "tc", "step_count", "episode", "wall_jn", "pair_jn"):
        assert np.array_equal(getattr(s0, k), getattr(s1, k)), k
    assert np.array_equal(table, before)
    assert s0.episode.max() > 1, "no auto-reset happened"


def test_table_oracle_steps_each_world_with_its_own_entry():
    """Worlds alternating between two entries step as the oracle created with each entry steps them (same global
    ids): the runs of equal radius and time limit keep every world's id."""
    cm = pu.named_cmap("squarinth")
    N, gid0 = 40, 77
    table = table_of(N)
    table[1::2] = table_of(1, **X)[0]
    orc = TableOracle(cm, seed=3)
    st = orc.new_state(N, gid0=gid0)
    orc.reset(st, table=table)
    o = _run(orc, st, 150, np.random.default_rng(2), table=table)
    rng = np.random.default_rng(2)                                    # the actions _run drew
    acts = [rng.integers(0, 4, (N, 3)) for _ in range(150)]
    for params, worlds in (({}, range(0, N, 2)), (X, range(1, N, 2))):
        ref = co.Oracle(cm, seed=3, **params)
        for w in worlds:
            r = ref.new_state(1, gid0=gid0 + w)
            ref.reset(r)
            for t in range(150):
                out = ref.step(r, acts[t][w:w + 1])
                for k in OUT_KEYS:
                    assert np.array_equal(getattr(out, k)[0], o[t][k][w]), (w, t, k)
            assert np.array_equal(r.pos[0], st.pos[w]) and r.episode[0] == st.episode[w]
    assert st.episode.max() > 1


def test_team_top_speeds():
    orc = TableOracle(CMAP, auto_reset=0)
    st = orc.new_state(1)
    st.pos[0] = [[400.0, 300.0], [400.0, 500.0], [400.0, 400.0]]     # cop_0, cop_1, thief_0: 100 apart
    st.tc[0] = st.pos[0]
    table = table_of(1)
    table["max_speed"][0] = [125.0, 150.0]
    for _ in range(25):
        out = orc.step(st, np.array([[2, 2, 2]], np.int32), table=table)   # +x: free flight
    assert not out.terminated[0]
    np.testing.assert_allclose(st.vel[0, :, 0], [125.0, 125.0, 150.0], rtol=0, atol=1e-9)
    np.testing.assert_allclose(st.vel[0, :, 1], 0.0, atol=1e-9)


@pytest.mark.parametrize("dist,captured", [(25.0, True), (35.0, False)])
def test_capture_radius(dist, captured):
    orc = TableOracle(CMAP, auto_reset=0)
    for table, want in ((table_of(1, termination_radius=30.0), captured), (table_of(1), False)):   # default radius 20
        st = orc.new_state(1)
        st.pos[0] = [[500.0, 400.0], [200.0, 700.0], [500.0 + dist, 400.0]]
        st.tc[0] = st.pos[0]
        out = orc.step(st, np.array([[4, 4, 4]], np.int32), table=table)
        assert bool(out.terminated[0]) == want and out.winner[0] == (0 if want else -1)


def test_time_limit():
    orc = TableOracle(CMAP, auto_reset=0)
    st = orc.new_state(3)
    for w in range(3):
        st.pos[w] = [[400.0, 300.0], [400.0, 400.0], [400.0, 500.0]]
    st.tc[:] = st.pos
    table = table_of(3)
    table["max_step_count"] = [1, 7, 12]
    first = np.full(3, -1)
    for i in range(1, 13):
        out = orc.step(st, np.full((3, 3), 4, np.int32), table=table)
        first[(first < 0) & (out.truncated == 1)] = i
    assert list(first) == [1, 7, 12]


def test_resets_draw_from_the_ranges():
    cm = pu.named_cmap("squarinth")
    ranges = RANGES.copy()
    orc, twin = TableOracle(cm, seed=5, ranges=ranges), co.Oracle(cm, seed=5)
    st, st2 = orc.new_state(32, gid0=1000), twin.new_state(32, gid0=1000)
    table = table_of(32)
    orc.reset(st, table=table), twin.reset(st2)
    for w in range(32):
        assert table[w].tobytes() == draws_numpy(5, 1000 + w, int(st.episode[w]), ranges).tobytes()
    assert np.array_equal(st.pos, st2.pos), "spawns do not depend on the draws"
    prev = table.copy()
    rng = np.random.default_rng(0)
    for _ in range(12):                                               # time limits 3..5: every world ends
        out = orc.step(st, rng.integers(0, 4, (32, 3)), table=table)
        ended = out.terminated.astype(bool)
        changed = table != prev
        assert not changed[~ended].any() and changed[ended].all()
        for w in np.flatnonzero(ended):
            assert table[w].tobytes() == draws_numpy(5, 1000 + w, int(st.episode[w]), ranges).tobytes()
        prev = table.copy()
    assert st.episode.min() > 2
    ranges["draw"] = 0
    keep = table.copy()
    TableOracle(cm, seed=5, ranges=ranges).reset(st, table=table)
    assert np.array_equal(table, keep), "draw = 0 leaves the table alone"
