"""Per-world physics parameters in the step kernel, on the GPU.

A table of the environment's own values changes nothing: an environment with it steps bit for bit like a twin without
it, on every kernel and launch shape and with mixed maps, final outputs and episode statistics.  A constant table X
steps like a twin created with X.  Asymmetric and per-world tables match the oracle given the same table.  Draws equal
the host's cat_param_draws whatever the sharding, chunking or launch shape, per map slot, only where a world
re-spawns, and never move a spawn.  In-place updates reach a captured graph; set_map, state_dict and the learner's
rollout graph work with the table."""
import numpy as np
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200 import world_params as wparams
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner
from as_cops_and_thieves_b200.maps import compile_map, generate_maze, load_named_map
from as_cops_and_thieves_b200.worlds import CatWorlds
from world_params_reference import TableOracle, draws_numpy

pytestmark = pytest.mark.gpu

FLAT = ("obs_f32", "state_f32", "critic_f32")
# ranges whose float draws the numpy reference reproduces bit for bit ((hi - lo) has few significant bits)
SPEC = {"unit_velocity": {"cop": (8, 12), "thief": (9.5, 10.5)}, "max_speed": {"cop": (110, 130), "thief": (125, 175)},
        "termination_radius": (15, 25), "max_step_count": (20, 60)}
SPEC2 = {"max_speed": (60, 80), "termination_radius": (30, 34), "max_step_count": (70, 90)}


def _bits(t):
    return t.contiguous().view(torch.int32)


def _check_same(S, T, what):
    assert torch.equal(S.state, T.state), f"{what}: state"
    assert torch.equal(S._out, T._out), f"{what}: records"
    if S._final_out is not None:
        assert torch.equal(S._final_out, T._final_out), f"{what}: final records"
    for name in FLAT + tuple("final_" + f for f in FLAT):
        a, b = getattr(S, name, None), getattr(T, name, None)
        if a is not None and b is not None:
            assert torch.equal(_bits(a), _bits(b)), f"{what}: {name}"


def _table_np(env):
    return env._wp.cpu().numpy().copy().view(wparams.PARAMS_DTYPE).reshape(-1)


def _expected_draws(env, ranges_by_world, episodes):
    out = np.zeros(env.n_worlds, wparams.PARAMS_DTYPE)
    for w in range(env.n_worlds):
        out[w] = draws_numpy(int(env.params["seed"]), env.gid0 + w, int(episodes[w]), ranges_by_world(w))
    return out


def _lockstep(cuda_device, cmaps, counts, steps=300, s_kw=None, t_kw=None, s_params=None, **kw):
    """S: a table (set to s_params, default the environment's values, no draws); T: no table, created with s_params."""
    kw = dict(device=cuda_device, gid0=11, seed=5, want_critic=True, max_step_count=40, **kw)
    S = CatWorlds(cmaps, counts, want_world_params=True, **(s_kw or {}), **kw)
    T = CatWorlds(cmaps, counts, **(t_kw or s_kw or {}), **dict(kw, **(s_params or {})))
    if s_params:
        S.set_world_params(**s_params)
    table = S._wp.clone()
    N = S.n_worlds
    for e in (S, T):
        e.reset()
    g = torch.Generator().manual_seed(7)
    ended = 0
    for t in range(steps):
        a = torch.randint(0, 4, (N, S.A), dtype=torch.uint8, generator=g).to(cuda_device)
        for e in (S, T):
            e.step(a)
        _check_same(S, T, f"step {t}")
        ended += int(T.terminated.sum())
    assert torch.equal(S._wp, table), "without draws the table never changes"
    assert ended > 0 and int((T.winner == 1).sum()) + int((T.winner == 0).sum()) > 0
    for e in (S, T):
        e.close()
    return S, T


SHAPES = {"one_wave": 4096, "persistent": 12000}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kernel", ["shipped", "generic", "raster"])
def test_default_table_is_bit_identical(cuda_device, monkeypatch, kernel, shape):
    kw = {}
    if kernel == "generic":
        monkeypatch.setenv("CAT_GENERIC_KERNEL", "1")
    if kernel == "raster":
        kw["ray_list_cell"] = -1.0
    _lockstep(cuda_device, pu.named_cmap("agh-map", free_spawn=True), SHAPES[shape], **kw)


def test_default_table_mixed_maps_final_outputs_and_statistics(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    S, _ = _lockstep(cuda_device, cmaps, (1, 37, 4096), s_kw=dict(want_final=True, want_episode_stats=True))
    assert S.episode_acc is not None


@pytest.mark.parametrize("X", [dict(unit_velocity=12.0, max_speed=140.0, termination_radius=25.0, max_step_count=30),
                               dict(unit_velocity=8.0, max_speed=100.0, termination_radius=12.5, max_step_count=7),
                               dict(unit_velocity=10.0, max_speed=125.0, termination_radius=20.0, max_step_count=400)])
def test_constant_table_equals_a_twin_created_with_it(cuda_device, X):
    _lockstep(cuda_device, pu.named_cmap("squarinth", free_spawn=True), 4096, steps=120, s_params=X)


@pytest.mark.parametrize("name,free,N,gaps", [("squarinth", False, 4096, (0, 49, 150)), ("agh-map", True, 1024, (0, 49, 150))])
def test_asymmetric_per_world_tables_match_the_oracle(cuda_device, name, free, N, gaps):
    from test_parity_gpu import _acts, _compare_transition
    cmap = pu.named_cmap(name, free_spawn=free)
    cw = CatWorlds(cmap, N, device=cuda_device, want_hits=True, seed=7, want_world_params=True)
    g = torch.Generator(device=cuda_device).manual_seed(3)
    u = lambda lo, hi: lo + (hi - lo) * torch.rand(N, device=cuda_device, generator=g)   # noqa: E731
    cw.set_world_params(unit_velocity={"cop": u(8, 12), "thief": u(9, 11)}, max_speed={"cop": u(110, 130), "thief": u(130, 170)},
                        termination_radius=u(15, 25), max_step_count=torch.randint(120, 400, (N,), device=cuda_device,
                                                                                     generator=g))
    orc = TableOracle(cmap, seed=7)
    orc.table = _table_np(cw)                    # no ranges: the table stays as set
    rng = np.random.default_rng(123)
    cw.reset()
    for gap in gaps:
        for _ in range(gap):
            cw.step(_acts(rng, N, cw.A, cw.device)[1])
        _compare_transition(cw, orc, rng, f"world-params {name}@+{gap}")
    st = cw.get_state()
    v = st["vel"].norm(dim=-1)
    wp = cw.world_params()
    assert bool((v[:, 2] <= wp["max_speed"][:, 1] * (1 + 1e-6)).all()) and bool((v[:, :2] <= wp["max_speed"][:, :1] * (1 + 1e-6)).all())
    cw.close()


def test_draws_match_the_host_across_sharding_shapes_and_chunks(cuda_device):
    cmap = pu.named_cmap("squarinth", free_spawn=True)
    kw = dict(device=cuda_device, seed=9, param_ranges=SPEC)
    big = CatWorlds(cmap, 12000, gid0=0, **kw)              # persistent launch
    small = CatWorlds(cmap, 4096, gid0=0, **kw)             # one wave
    shard = CatWorlds(cmap, 2048, gid0=2048, **kw)          # worlds 2048.. of the others
    host = CatWorlds(cmap, 4096, gid0=0, **kw)              # host path, 4 chunks
    twin = CatWorlds(cmap, 4096, gid0=0, device=cuda_device, seed=9)     # no table: spawns only
    r = wparams.ranges_entry(SPEC, big.params)
    init = _table_np(small)
    assert np.array_equal(init, np.tile(wparams.defaults(small.params), 4096)), "init_state never draws"
    for e in (big, small, shard, host, twin):
        e.reset()
    assert torch.equal(small.get_state()["pos"], twin.get_state()["pos"]), "spawns do not depend on the draws"
    ep = small.get_state()["episode"].cpu().numpy()
    assert np.array_equal(_table_np(small), _expected_draws(small, lambda w: r, ep))
    g = torch.Generator().manual_seed(1)
    prev = _table_np(small)
    for t in range(90):
        a = torch.randint(0, 4, (12000, 3), dtype=torch.uint8, generator=g)
        big.step(a.to(cuda_device))
        small.step(a[:4096].to(cuda_device))
        shard.step(a[2048:4096].to(cuda_device))
        host.step_host(a[:4096].contiguous().pin_memory(), mode="pipelined", chunks=4)
        torch.cuda.synchronize()
        cur = _table_np(small)
        assert np.array_equal(_table_np(big)[:4096], cur), t
        assert np.array_equal(_table_np(shard), cur[2048:]), t
        assert np.array_equal(_table_np(host), cur), t
        ended = small.terminated.cpu().numpy().astype(bool)
        changed = (cur != prev)
        assert not changed[~ended].any(), f"step {t}: an entry changed without a re-spawn"
        if ended.any():
            ep = small.get_state()["episode"].cpu().numpy()
            idx = np.flatnonzero(ended)
            want = np.array([draws_numpy(9, int(w), int(ep[w]), r) for w in idx], wparams.PARAMS_DTYPE)
            assert np.array_equal(cur[idx], want), t
        prev = cur
    assert int(small.get_state()["episode"].min()) >= 2
    for e in (big, small, shard, host, twin):
        e.close()


def test_pinned_draws_keep_spawns_and_dynamics(cuda_device):
    """Ranges pinned to the environment's values with draw on: every re-spawn rewrites the entry with the same values,
    and the environment steps bit for bit like a twin without a table."""
    cmap = pu.named_cmap("agh-map", free_spawn=True)
    S = CatWorlds(cmap, 4096, device=cuda_device, seed=4, max_step_count=30, param_ranges={})
    T = CatWorlds(cmap, 4096, device=cuda_device, seed=4, max_step_count=30)
    assert int(S.param_ranges()["draw"].min()) == 1
    for e in (S, T):
        e.reset()
    g = torch.Generator().manual_seed(2)
    for t in range(100):
        a = torch.randint(0, 4, (4096, 3), dtype=torch.uint8, generator=g).to(cuda_device)
        for e in (S, T):
            e.step(a)
        _check_same(S, T, f"step {t}")
    assert np.array_equal(_table_np(S), np.tile(wparams.defaults(S.params), 4096))
    for e in (S, T):
        e.close()


def test_each_map_slot_draws_from_its_own_ranges(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    env = CatWorlds(cmaps, (1000, 1500, 700), device=cuda_device, seed=3, gid0=5, param_ranges=[SPEC, SPEC2, None])
    env.set_world_params(mask=env.map_index == 2, termination_radius=5.0, max_step_count=30)   # ends by timeouts only
    kept = _table_np(env)[env.map_index.cpu().numpy() == 2].copy()
    env.reset()
    g = torch.Generator().manual_seed(8)
    for _ in range(100):
        env.step(torch.randint(0, 4, (env.n_worlds, 3), dtype=torch.uint8, generator=g).to(cuda_device))
    torch.cuda.synchronize()
    mi = env.map_index.cpu().numpy()
    ranges = [wparams.ranges_entry(SPEC, env.params), wparams.ranges_entry(SPEC2, env.params)]
    ep = env.get_state()["episode"].cpu().numpy()
    tab = _table_np(env)
    for w in range(env.n_worlds):
        if mi[w] < 2:
            assert tab[w].tobytes() == draws_numpy(3, 5 + w, int(ep[w]), ranges[mi[w]]).tobytes(), w
    assert np.array_equal(tab[mi == 2], kept), "draw = 0 leaves the table untouched"
    assert (ep[mi == 2] > 1).any()
    env.close()


def test_graph_replays_pick_up_new_ranges_and_set_map_draws(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map")]
    G = CatWorlds(cmaps, (2048, 2048), device=cuda_device, seed=2, param_ranges=SPEC, swappable_maps=True,
                  want_final=True, want_episode_stats=True)
    N = G.n_worlds
    G.reset()
    acts = torch.zeros((N, 3), dtype=torch.uint8, device=cuda_device)
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        G.step(acts)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        G.step(acts)
    torch.cuda.synchronize()
    G.set_param_ranges(slot=1, **SPEC2)
    r2 = wparams.ranges_entry(SPEC2, G.params)
    g = torch.Generator().manual_seed(1)
    ended = 0
    for t in range(100):
        acts.copy_(torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g))
        graph.replay()
        torch.cuda.synchronize()
        done = G.terminated.cpu().numpy().astype(bool) & (G.map_index.cpu().numpy() == 1)
        if done.any():
            ep = G.get_state()["episode"].cpu().numpy()
            tab = _table_np(G)
            for w in np.flatnonzero(done):
                assert tab[w].tobytes() == draws_numpy(2, int(w), int(ep[w]), r2).tobytes(), (t, w)
            ended += int(done.sum())
    assert ended > 0
    assert G.episode_totals_raw()["episodes"].sum() > 0
    mask = G.set_map(0, compile_map(generate_maze(4)))
    r1 = wparams.ranges_entry(SPEC, G.params)
    ep = G.get_state()["episode"].cpu().numpy()
    tab = _table_np(G)
    for w in np.flatnonzero(mask.cpu().numpy()):
        assert tab[w].tobytes() == draws_numpy(2, int(w), int(ep[w]), r1).tobytes(), w
    G.close()


def test_state_dict_round_trips_the_table(cuda_device):
    env = CatWorlds(pu.named_cmap("squarinth"), 256, device=cuda_device, seed=1, param_ranges=SPEC)
    env.reset()
    sd = env.state_dict()
    env.set_world_params(termination_radius=3.0, max_speed={"thief": 99.0})
    env.set_param_ranges(slot=0, draw=False)
    env.load_state_dict(sd)
    assert torch.equal(env._wp, sd["world_params"]) and torch.equal(env._wp_ranges, sd["param_ranges"])
    assert int(env.param_ranges()["draw"][0]) == 1
    with pytest.raises(ValueError):
        env.set_world_params(max_speed=torch.zeros(256, device=cuda_device))
    with pytest.raises(ValueError):
        env.set_world_params(termination_radius={"cop": 3.0})
    assert torch.equal(env._wp, sd["world_params"]), "a failed call writes nothing"
    env.close()


def test_batched_env_and_learner_rollout_graph(cuda_device):
    env = BatchedCopsThievesEnv(load_named_map("squarinth"), 256, device=cuda_device, seed=6, max_step_count=20,
                                randomize={"max_speed": {"thief": (125, 175)}, "max_step_count": (10, 30)},
                                episode_statistics=True)
    spaces = {a: env.observation_space(a) for a in env.possible_agents}
    cfg = MAPPOConfig(rollouts=32, model="lstm", random_timesteps=0, learning_starts=0, cuda_graph=True,
                      opponent_freeze_duration=0, policy_freeze_duration=0)
    lrn = MAPPOLearner(env, cfg, seed=0)
    for _ in range(3):                       # eager warm-up, capture + replay, replay
        lrn.collect()
    wp = env.world_params()
    assert float(wp["max_speed"][:, 1].min()) >= 125 and float(wp["max_speed"][:, 1].max()) <= 175
    assert bool((wp["max_speed"][:, 0] == 125).all()) and len(torch.unique(wp["max_speed"][:, 1])) > 10
    assert int(wp["max_step_count"].min()) >= 10 and int(wp["max_step_count"].max()) <= 30
    assert env.episode_statistics()["episodes"] > 0
    assert {a: env.observation_space(a) for a in env.possible_agents} == spaces
    env.set_randomization(None)
    before = env.world_params()["max_speed"].clone()
    env.reset()
    assert torch.equal(env.world_params()["max_speed"], before)
    env.set_world_params(termination_radius=30.0)
    assert bool((env.world_params()["termination_radius"] == 30.0).all())
    env.close()
