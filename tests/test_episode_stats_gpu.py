"""Episode statistics from the step kernel, on the GPU.

An environment with statistics (S) is stepped in lockstep with a twin without them (T).  Every step S's state, records
and flat layouts equal T's bit for bit (statistics change nothing else), and a torch tally built from T's outputs
(``acc = acc + reward``; steps since the last reset) gives, on the worlds that ended, S's ``episode_return`` bit for bit
and its ``episode_length``; the entries of the other worlds are untouched.  At the end the per-map totals match the
tally: counts, length sum, minima and maxima exactly, the f64 return sums to rounding.  The same holds on every kernel
and launch shape, for mixed maps, another agent / ray shape, with final outputs, without auto-reset, across resets and
map swaps, under graph capture, on the host path, through ``BatchedCopsThievesEnv`` and inside the learner's rollout
graph."""
import ctypes as C

import numpy as np
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200 import _lib, episodes
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner
from as_cops_and_thieves_b200.maps import generate_maze, compile_map, load_named_map
from as_cops_and_thieves_b200.worlds import CatWorlds

pytestmark = pytest.mark.gpu

FLAT = ("obs_f32", "state_f32", "critic_f32")


def _bits(t):
    return t.contiguous().view(torch.int32)


class Tally:
    """The statistics recomputed with torch ops from an environment's own outputs."""

    def __init__(self, env, auto_reset=True):
        N, A, dev = env.n_worlds, env.A, env.device
        self.acc = torch.zeros((N, A), dtype=torch.float32, device=dev)
        self.since = torch.zeros(N, dtype=torch.int32, device=dev)
        self.map_index, self.n_maps, self.A, self.auto_reset = env.map_index, len(env.cmaps), A, auto_reset
        self.ended = []        # (map, returns, length, captured) of every episode, per step

    def step(self, reward, terminated, truncated):
        self.acc = self.acc + reward
        self.since += 1
        done = terminated.bool()
        ret, ln = self.acc[done].clone(), self.since[done].clone()
        self.ended.append((self.map_index[done].cpu(), ret.cpu(), ln.cpu(), (done & ~truncated.bool())[done].cpu()))
        self.acc[done] = 0.0
        if self.auto_reset:
            self.since[done] = 0
        return done, ret, ln

    def reset(self, mask=None):
        mask = torch.ones_like(self.since, dtype=torch.bool) if mask is None else mask.bool()
        self.acc[mask] = 0.0
        self.since[mask] = 0

    def episodes(self):
        m, r, n, c = (torch.cat([e[i] for e in self.ended]) for i in range(4))
        return m.numpy(), r.numpy(), n.numpy().astype(np.int64), c.numpy()


def _check_totals(env, tally, raw=None):
    raw = env.episode_totals_raw() if raw is None else raw
    m, r, n, c = tally.episodes()
    assert len(raw) == tally.n_maps
    for s in range(tally.n_maps):
        sel = m == s
        t = raw[s]
        assert int(t["episodes"]) == int(sel.sum()), s
        assert int(t["captures"]) == int(c[sel].sum()) and int(t["timeouts"]) == int((~c[sel]).sum()), s
        assert int(t["length_sum"]) == int(n[sel].sum()), s
        if not sel.any():
            assert t["length_max_key"] == 0 and t["length_min_key"] == 0 and not t["return_max_key"].any()
            continue
        assert int(t["length_max_key"]) == n[sel].max() and int(~np.uint32(t["length_min_key"])) == n[sel].min(), s
        A = tally.A
        rs = r[sel].astype(np.float64)
        assert np.array_equal(episodes.key_value(t["return_max_key"][:A]), r[sel].max(axis=0)), s
        assert np.array_equal(episodes.key_value(~t["return_min_key"][:A]), r[sel].min(axis=0)), s
        assert np.allclose(t["return_sum"][:A], rs.sum(axis=0), rtol=1e-12, atol=1e-9), s
        assert np.allclose(t["return_sq_sum"][:A], (rs * rs).sum(axis=0), rtol=1e-12, atol=1e-9), s
        assert not t["return_sum"][A:].any() and not t["return_max_key"][A:].any()
    return int(c.sum()), int((~c).sum())


def _check_same(S, T, what):
    assert torch.equal(S.state, T.state), f"{what}: state"
    assert torch.equal(S._out, T._out), f"{what}: records"
    if S._final_out is not None and T._final_out is not None:
        assert torch.equal(S._final_out, T._final_out), f"{what}: final records"
    for name in FLAT + tuple("final_" + f for f in FLAT):
        a, b = getattr(S, name, None), getattr(T, name, None)
        if a is not None and b is not None:
            assert torch.equal(_bits(a), _bits(b)), f"{what}: {name}"


def _lockstep(cuda_device, cmaps, counts, steps=210, auto_reset=1, s_kw=None, seed=5, **kw):
    kw = dict(device=cuda_device, gid0=11, seed=seed, want_critic=True, max_step_count=40, auto_reset=auto_reset, **kw)
    S = CatWorlds(cmaps, counts, want_episode_stats=True, **(s_kw or {}), **kw)
    T = CatWorlds(cmaps, counts, **(s_kw or {}), **kw)
    N = S.n_worlds
    for e in (S, T):
        e.reset()
    tally = Tally(S, auto_reset=bool(auto_reset))
    g = torch.Generator().manual_seed(7)
    for t in range(steps):
        a = torch.randint(0, 4, (N, S.A), dtype=torch.uint8, generator=g).to(cuda_device)
        r0, l0 = S.episode_return.clone(), S.episode_length.clone()
        for e in (S, T):
            e.step(a)
        _check_same(S, T, f"step {t}")
        done, ret, ln = tally.step(T.reward, T.terminated, T.truncated)
        assert torch.equal(_bits(S.episode_return[done]), _bits(ret)), f"step {t}: episode_return"
        assert torch.equal(S.episode_length[done], ln), f"step {t}: episode_length"
        assert torch.equal(_bits(S.episode_return[~done]), _bits(r0[~done])), f"step {t}: return of a world that did not end"
        assert torch.equal(S.episode_length[~done], l0[~done]), f"step {t}: length of a world that did not end"
        assert torch.equal(_bits(S.episode_acc), _bits(tally.acc)), f"step {t}: running returns"
    captures, timeouts = _check_totals(S, tally)
    assert captures > 0 and timeouts > 0, f"both kinds of ending must occur: {captures} captures, {timeouts} timeouts"
    assert S.overflow_counts() == (0, 0)
    for e in (S, T):
        e.close()


SHAPES = {"one_wave": 4096, "persistent": 12000}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kernel", ["shipped", "generic", "raster"])
@pytest.mark.parametrize("name", ["squarinth", "agh-map"])
def test_statistics_equal_a_tally_of_the_twin(cuda_device, monkeypatch, name, kernel, shape):
    kw = {}
    if kernel == "generic":
        monkeypatch.setenv("CAT_GENERIC_KERNEL", "1")
    if kernel == "raster":
        kw["ray_list_cell"] = -1.0
    _lockstep(cuda_device, pu.named_cmap(name, free_spawn=True), SHAPES[shape], **kw)


def test_statistics_mixed_maps(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    _lockstep(cuda_device, cmaps, (1, 37, 4096))


def test_statistics_other_shape(cuda_device):
    """3 agents x 37 rays: the any-shape instantiation."""
    _lockstep(cuda_device, pu.named_cmap("squarinth", free_spawn=True), 2048, n_rays=37)


def test_statistics_with_final_outputs(cuda_device):
    _lockstep(cuda_device, pu.named_cmap("agh-map", free_spawn=True), 4096, s_kw=dict(want_final=True))


def test_statistics_without_auto_reset(cuda_device):
    """auto_reset = 0: a world that ended keeps reporting terminated, and every such step ends an episode whose length
    is the world's step_count."""
    _lockstep(cuda_device, pu.named_cmap("squarinth", free_spawn=True), 2048, steps=80, auto_reset=0)


def test_attach_validates_its_arguments(cuda_device):
    env = CatWorlds(pu.named_cmap("squarinth"), 64, device=cuda_device, want_episode_stats=True)
    L = env.L
    ok = _lib.CatEpisodeStatsIO(env.episode_acc.data_ptr(), env.episode_return.data_ptr(), env.episode_length.data_ptr(),
                                env._episode_totals.data_ptr())
    for bad in (dict(acc=None), dict(acc=env.episode_acc.data_ptr() + 2), dict(episode_length=env.episode_length.data_ptr() + 1),
                dict(totals=env._episode_totals.data_ptr() + 4)):
        io = _lib.CatEpisodeStatsIO(ok.acc, ok.episode_return, ok.episode_length, ok.totals)
        for k, v in bad.items():
            setattr(io, k, v)
        assert L.cat_env_attach_episode_stats(env._h, C.byref(io)) == -1, bad
    # nothing was stored by the failed calls: a step still updates the buffers attached at creation
    env.reset()
    acts = torch.ones((64, 3), dtype=torch.uint8, device=cuda_device)
    env.step(acts)
    going = ~env.terminated.bool()
    assert bool(going.any())
    assert torch.equal(_bits(env.episode_acc[going]), _bits(0.0 + env.reward[going]))
    # detached: steps leave them alone
    assert L.cat_env_attach_episode_stats(env._h, None) == 0
    before = env.episode_acc.clone()
    env.step(acts)
    torch.cuda.synchronize()
    assert torch.equal(env.episode_acc, before)
    env.close()


def test_resets_and_map_swaps_zero_the_running_returns(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map")]
    kw = dict(device=cuda_device, seed=3, want_critic=True, max_step_count=40)
    S = CatWorlds(cmaps, (1024, 1024), want_episode_stats=True, swappable_maps=True, **kw)
    T = CatWorlds(cmaps, (1024, 1024), swappable_maps=True, **kw)
    N = S.n_worlds
    for e in (S, T):
        e.reset()
    tally = Tally(S)
    g = torch.Generator().manual_seed(4)
    maze = compile_map(generate_maze(2))
    for t in range(120):
        a = torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g).to(cuda_device)
        for e in (S, T):
            e.step(a)
        done, ret, ln = tally.step(T.reward, T.terminated, T.truncated)
        assert torch.equal(_bits(S.episode_return[done]), _bits(ret)) and torch.equal(S.episode_length[done], ln), t
        if t == 30:           # masked reset mid-episode
            mask = torch.rand(N, generator=g).to(cuda_device) < 0.3
            assert bool((tally.acc[mask] != 0).any()), "the reset must drop something"
            for e in (S, T):
                e.reset(mask)
            tally.reset(mask)
        if t == 60:           # every world
            for e in (S, T):
                e.reset()
            tally.reset()
            assert not S.episode_acc.any()
        if t == 90:           # swap map 1: its worlds are reset
            mask = S.set_map(1, maze)
            assert torch.equal(mask, T.set_map(1, maze))
            tally.reset(mask)
            assert not S.episode_acc[mask].any()
        _check_same(S, T, f"step {t}")
        assert torch.equal(_bits(S.episode_acc), _bits(tally.acc)), t
    _check_totals(S, tally)
    for e in (S, T):
        e.close()


def test_graph_replay_equals_eager(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map")]
    kw = dict(device=cuda_device, seed=2, want_critic=True, max_step_count=40, want_episode_stats=True)
    G, E = CatWorlds(cmaps, (512, 3584), **kw), CatWorlds(cmaps, (512, 3584), **kw)
    N = G.n_worlds
    for e in (G, E):
        e.reset()
    acts = torch.zeros((N, 3), dtype=torch.uint8, device=cuda_device)
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):           # warm-up on a side stream, as torch.cuda.graph wants; the twin takes it too
        G.step(acts)
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    E.step(acts)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        G.step(acts)
    torch.cuda.synchronize()
    g = torch.Generator().manual_seed(1)
    ended = 0
    for t in range(30):
        acts.copy_(torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g))
        graph.replay()
        E.step(acts)
        torch.cuda.synchronize()
        done = E.terminated.bool()
        _check_same(G, E, f"replay {t}")
        assert torch.equal(_bits(G.episode_acc), _bits(E.episode_acc)), t
        assert torch.equal(_bits(G.episode_return[done]), _bits(E.episode_return[done])), t
        assert torch.equal(G.episode_length[done], E.episode_length[done]), t
        ended += int(done.sum())
    a, b = G.episode_totals_raw(), E.episode_totals_raw()
    assert ended > 0 and int(b["episodes"].sum()) >= ended
    for f in ("episodes", "captures", "timeouts", "length_sum", "length_min_key", "length_max_key", "return_min_key", "return_max_key"):
        assert np.array_equal(a[f], b[f]), f
    assert np.allclose(a["return_sum"], b["return_sum"], rtol=1e-12, atol=1e-9)
    for e in (G, E):
        e.close()


@pytest.mark.parametrize("mode", ["pipelined", "zero_copy", "staged"])
def test_host_path(cuda_device, mode):
    """Two maps, split so that one of the pipelined path's four chunks spans both and the later ones hold map 1 alone:
    every episode lands in its own map slot."""
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map")]
    kw = dict(device=cuda_device, seed=6, max_step_count=40)
    S = CatWorlds(cmaps, (1536, 2560), want_episode_stats=True, **kw)      # host path with statistics
    P = CatWorlds(cmaps, (1536, 2560), **kw)                                # host path without
    D = CatWorlds(cmaps, (1536, 2560), want_episode_stats=True, **kw)      # device path with
    for e in (S, P, D):
        e.reset()
    g = torch.Generator().manual_seed(3)
    ended = 0
    for t in range(90):
        a = torch.randint(0, 4, (4096, 3), dtype=torch.uint8, generator=g).pin_memory()
        hs = S.step_host(a, mode=mode, chunks=4)
        blob_s = hs["blob"].clone()
        hp = P.step_host(a, mode=mode, chunks=4)
        assert torch.equal(blob_s, hp["blob"]), f"{mode} step {t}: host records"
        D.step(a.to(cuda_device))
        torch.cuda.synchronize()
        assert torch.equal(S.state, D.state), t
        done = D.terminated.bool()
        assert torch.equal(_bits(S.episode_acc), _bits(D.episode_acc)), t
        assert torch.equal(_bits(S.episode_return[done]), _bits(D.episode_return[done])), t
        assert torch.equal(S.episode_length[done], D.episode_length[done]), t
        ended += int(done.sum())
    a, b = S.episode_totals_raw(), D.episode_totals_raw()
    assert ended > 0 and int(a["episodes"].sum()) == ended and (b["episodes"] > 0).all()
    for f in ("episodes", "captures", "timeouts", "length_sum", "length_min_key", "length_max_key", "return_min_key", "return_max_key"):
        assert np.array_equal(a[f], b[f]), f
    assert np.allclose(a["return_sum"], b["return_sum"], rtol=1e-12, atol=1e-9)
    for e in (S, P, D):
        e.close()


def test_batched_env_infos_and_statistics(cuda_device):
    maps = [load_named_map(n) for n in ("squarinth", "agh-map")]
    env = BatchedCopsThievesEnv(maps, 2048, device=cuda_device, seed=4, max_step_count=30, episode_statistics=True)
    plain = BatchedCopsThievesEnv(maps, 2048, device=cuda_device, seed=4, max_step_count=30)
    w = env.worlds
    assert "episode" not in plain.step(torch.zeros((2048, 3), dtype=torch.uint8, device=cuda_device))[4]["cop_0"]
    plain.close()
    env.reset()
    tally = Tally(w)
    g = torch.Generator().manual_seed(8)
    first = None
    for t in range(100):
        acts = {a: torch.randint(0, 4, (2048,), generator=g).to(cuda_device) for a in env.possible_agents}
        out = env.step(acts)
        if first is None:
            first = out
        assert all(x is y for x, y in zip(out, first)), "a step returns the same dict objects"
        obs, rew, term, trunc, infos = out
        done, ret, ln = tally.step(w.reward, w.terminated, w.truncated)
        for i, a in enumerate(env.possible_agents):
            ep = infos[a]["episode"]
            assert ep["r"].shape == (2048,) and ep["r"].data_ptr() == w.episode_return[:, i].data_ptr()
            assert ep["l"] is w.episode_length
            assert torch.equal(_bits(ep["r"][done]), _bits(ret[:, i])), (t, a)
            assert torch.equal(ep["l"][done], ln), (t, a)
    m, r, n, c = tally.episodes()
    st = env.episode_statistics(by_map=True)
    assert st["overall"]["episodes"] == len(m) and st["overall"]["captures"] == int(c.sum())
    assert st["overall"]["length"]["max"] == n.max() and st["overall"]["length"]["mean"] == pytest.approx(n.mean())
    for i, a in enumerate(env.possible_agents):
        q = st["overall"]["returns"][a]
        assert q["min"] == r[:, i].min() and q["max"] == r[:, i].max()
        assert q["mean"] == pytest.approx(r[:, i].astype(np.float64).mean(), rel=1e-9, abs=1e-9)
        assert q["std"] == pytest.approx(r[:, i].astype(np.float64).std(), rel=1e-6, abs=1e-9)
    for s, entry in enumerate(st["maps"]):
        assert entry["map"] == env.map_names[s] and entry["episodes"] == int((m == s).sum())
    flat = env.episode_statistics(reset=True)
    assert flat == st["overall"]
    assert env.episode_statistics()["episodes"] == 0
    env.close()


def test_learner_rollout_graph_counts_every_episode(cuda_device):
    env = BatchedCopsThievesEnv(load_named_map("squarinth"), 256, device=cuda_device, seed=6, max_step_count=20,
                                episode_statistics=True)
    cfg = MAPPOConfig(rollouts=32, model="lstm", random_timesteps=0, learning_starts=0, cuda_graph=True,
                      opponent_freeze_duration=0, policy_freeze_duration=0)
    lrn = MAPPOLearner(env, cfg, seed=0)
    done = 0
    for it in range(3):                       # eager warm-up, capture + replay, replay
        lrn.collect()
        done += int(lrn.mem_done.sum())
        assert env.episode_statistics()["episodes"] == done, it
    assert done > 0
    env.close()
