"""Scripted agents in the step kernel, on the GPU.

Attached with every mode 0, scripts change nothing: an environment steps bit for bit like a twin without them, on every
kernel and launch shape, with mixed maps, without auto-reset, with episode statistics and a world-parameter table.  After
every step and reset the decisions equal scripts_reference applied to the record the launch emitted.  The kernel applies
exactly those decisions: a scripted environment steps like a twin fed them as actions.  observe, set_state and
render_frames leave the decisions alone; modes changed in place reach the next eager step and the next graph replay.
The learner trains only the unscripted agents, evaluate_vs_scripted restores the modes it found, and chasing cops catch
a random thief more often than random cops do."""
import ctypes as C

import numpy as np
import pytest
import torch

import parity_utils as pu
from as_cops_and_thieves_b200 import _lib
from as_cops_and_thieves_b200.env import BatchedCopsThievesEnv
from as_cops_and_thieves_b200.mappo import MAPPOConfig, MAPPOLearner
from as_cops_and_thieves_b200.maps import compile_map, generate_maze, load_named_map
from as_cops_and_thieves_b200.selfplay import evaluate_vs_scripted
from as_cops_and_thieves_b200.worlds import CatWorlds
from scripts_reference import decisions_of_record

pytestmark = pytest.mark.gpu

FLAT = ("obs_f32", "state_f32", "critic_f32")
SHAPES = {"one_wave": 4096, "persistent": 12000}


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


def _kernel_kw(monkeypatch, kernel):
    if kernel == "generic":
        monkeypatch.setenv("CAT_GENERIC_KERNEL", "1")
    return {"ray_list_cell": -1.0} if kernel == "raster" else {}


def _expected(env, dist, types, worlds=None):
    """The decisions scripts_reference gives for the record (dist f16 (N, A, R), types u8 (N, A, R)) and the current
    episode / step counters of every world."""
    st = env.get_state()
    bits = dist.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)
    return decisions_of_record(bits, types.cpu().numpy(), env.n_cops, int(env.params["seed"]), env.gid0,
                               st["episode"].cpu().numpy(), st["step_count"].cpu().numpy(), worlds)


def _check_decisions(env, what, dist=None, types=None, worlds=None):
    torch.cuda.synchronize()
    want = _expected(env, env.obs_dist if dist is None else dist, env.obs_type if types is None else types, worlds)
    got = env.script_decisions.cpu().numpy()
    rows = slice(None) if worlds is None else np.asarray(worlds)
    bad = np.argwhere(got[rows] != want[rows])
    assert len(bad) == 0, f"{what}: {len(bad)} decisions differ, first (row, agent) {bad[:3].tolist()}"


# ---------------------------------------------------------------------------------------------- 1. additive
def _lockstep(cuda_device, cmaps, counts, steps=300, s_kw=None, **kw):
    """S: scripts attached, every mode 0; T: no scripts."""
    kw = dict(device=cuda_device, gid0=11, seed=5, want_critic=True, max_step_count=40, **kw)
    kw.update(s_kw or {})
    S = CatWorlds(cmaps, counts, want_scripts=True, **kw)
    T = CatWorlds(cmaps, counts, **kw)
    N = S.n_worlds
    for e in (S, T):
        e.reset()
    _check_same(S, T, "reset")
    g = torch.Generator().manual_seed(7)
    ended = 0
    for t in range(steps):
        a = torch.randint(0, 4, (N, S.A), dtype=torch.uint8, generator=g).to(cuda_device)
        for e in (S, T):
            e.step(a)
        _check_same(S, T, f"step {t}")
        ended += int(T.terminated.sum())
    assert ended > 0
    assert int(S.script_modes.max()) == 0
    for e in (S, T):
        e.close()


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kernel", ["shipped", "generic", "raster"])
def test_mode_zero_is_bit_identical(cuda_device, monkeypatch, kernel, shape):
    _lockstep(cuda_device, pu.named_cmap("agh-map", free_spawn=True), SHAPES[shape], **_kernel_kw(monkeypatch, kernel))


def test_mode_zero_against_the_record_only_kernel(cuda_device):
    """The twin asks for the record alone, so its steps run the record-only kernel; with scripts attached they cannot."""
    _lockstep(cuda_device, pu.named_cmap("agh-map", free_spawn=True), 4096, steps=150,
              s_kw=dict(want_f32=False, want_shared=False, want_critic=False))


def test_mode_zero_mixed_maps_no_auto_reset_statistics_and_parameters(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    _lockstep(cuda_device, cmaps, (1, 37, 4096), steps=200,
              s_kw=dict(want_final=True, want_episode_stats=True, want_world_params=True))
    _lockstep(cuda_device, cmaps, (100, 37, 900), steps=80, auto_reset=0)


# ---------------------------------------------------------------------------------------------- 2. decisions
@pytest.mark.parametrize("kernel,kw", [("shipped", {}), ("generic", {}), ("raster", {}), ("shipped", {"n_rays": 37})])
def test_decisions_match_the_reference(cuda_device, monkeypatch, kernel, kw):
    kw = dict(kw, **_kernel_kw(monkeypatch, kernel))
    env = CatWorlds(pu.named_cmap("agh-map", free_spawn=True), 300, device=cuda_device, seed=3, gid0=7,
                    max_step_count=25, scripts={2: "evade", 0: "chase"}, **kw)
    assert int(env.script_decisions.max()) == 0, "init_state zeroes the decisions"
    env.reset()
    _check_decisions(env, "reset")
    g = torch.Generator().manual_seed(5)
    for t in range(60):
        env.step(torch.randint(0, 4, (env.n_worlds, env.A), dtype=torch.uint8, generator=g).to(cuda_device))
        _check_decisions(env, f"step {t}")
    assert int(env.get_state()["episode"].min()) >= 2, "every world re-spawned inside a step"
    env.close()


def test_decisions_mixed_maps_auto_reset_off_and_persistent_shape(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map", "labyrinth")]
    env = CatWorlds(cmaps, (1, 37, 200), device=cuda_device, seed=4, max_step_count=20, scripts={1: "random"})
    env.reset()
    _check_decisions(env, "mixed reset")
    for t in range(45):
        env.step(torch.randint(0, 4, (env.n_worlds, env.A), dtype=torch.uint8, device=cuda_device))
        _check_decisions(env, f"mixed step {t}")
    env.close()
    env = CatWorlds(pu.named_cmap("squarinth"), 300, device=cuda_device, seed=4, max_step_count=15, auto_reset=0,
                    want_scripts=True)
    env.reset()
    for t in range(20):                      # the worlds end by step 15 and are never re-spawned
        env.step(torch.randint(0, 4, (env.n_worlds, env.A), dtype=torch.uint8, device=cuda_device))
        _check_decisions(env, f"auto_reset=0 step {t}")
    env.close()
    env = CatWorlds(pu.named_cmap("agh-map", free_spawn=True), 12000, device=cuda_device, seed=8, max_step_count=20,
                    want_scripts=True)
    sample = np.r_[0:200, 5900:6100, 11800:12000]
    env.reset()
    for t in range(25):
        env.step(torch.randint(0, 4, (env.n_worlds, env.A), dtype=torch.uint8, device=cuda_device))
        _check_decisions(env, f"persistent step {t}", worlds=sample)
    env.close()


@pytest.mark.parametrize("mode", ["pipelined", "zero_copy", "staged"])
def test_decisions_from_the_host_path(cuda_device, mode):
    env = CatWorlds(pu.named_cmap("agh-map", free_spawn=True), 2048, device=cuda_device, seed=6, max_step_count=20,
                    scripts={2: "evade"})
    sample = np.r_[0:150, 1900:2048]
    env.reset()
    g = torch.Generator().manual_seed(3)
    for t in range(25):
        h = env.step_host(torch.randint(0, 4, (env.n_worlds, env.A), dtype=torch.uint8, generator=g), mode=mode,
                          chunks=4)
        _check_decisions(env, f"{mode} step {t}", dist=h["obs_dist"], types=h["obs_type"], worlds=sample)
    env.close()


def test_decisions_after_set_map(cuda_device):
    cmaps = [pu.named_cmap(n, free_spawn=True) for n in ("squarinth", "agh-map")]
    env = CatWorlds(cmaps, (150, 150), device=cuda_device, seed=2, swappable_maps=True, scripts={0: "chase"})
    env.reset()
    for _ in range(5):
        env.step(torch.randint(0, 4, (env.n_worlds, env.A), dtype=torch.uint8, device=cuda_device))
    before = env.script_decisions.clone()
    mask = env.set_map(1, compile_map(generate_maze(3)))
    _check_decisions(env, "after set_map")
    keep = ~mask
    assert torch.equal(env.script_decisions[keep], before[keep]), "the other worlds keep their decisions"
    env.step(torch.zeros((env.n_worlds, env.A), dtype=torch.uint8, device=cuda_device))
    _check_decisions(env, "step after set_map")
    env.close()


# ---------------------------------------------------------------------------------------------- 3. the kernel applies them
@pytest.mark.parametrize("spec,half", [({0: "chase", 1: "chase", 2: "evade"}, False), ({0: "random", 1: "random", 2: "random"}, False),
                                       ({0: "chase", 2: "evade"}, True)])
def test_scripted_steps_equal_a_twin_fed_the_decisions(cuda_device, spec, half):
    cmap = pu.named_cmap("agh-map", free_spawn=True)
    N = 2048
    kw = dict(device=cuda_device, seed=12, max_step_count=60, want_critic=True, want_final=True)
    S = CatWorlds(cmap, N, want_scripts=True, **kw)
    T = CatWorlds(cmap, N, **kw)
    mask = torch.arange(N) % 2 == 0 if half else None
    S.set_scripts(spec, mask=mask)
    assert all(S.scripted_in(a) == ("some" if half else "all") for a in spec)
    for e in (S, T):
        e.reset()
    g = torch.Generator().manual_seed(9)
    captures = timeouts = 0
    for t in range(320):
        a = torch.randint(0, 4, (N, S.A), dtype=torch.int64, generator=g).to(cuda_device)
        nxt = S.scripted_actions()
        fed = torch.where(nxt >= 0, nxt, a)
        S.step(a.to(torch.uint8).contiguous())
        T.step(fed.to(torch.uint8).contiguous())
        _check_same(S, T, f"step {t}")
        captures += int(((T.winner == 0) & (T.terminated == 1)).sum())
        timeouts += int(((T.winner == 1) & (T.terminated == 1)).sum())
    assert captures > 0 and timeouts > 0
    for e in (S, T):
        e.close()


# ---------------------------------------------------------------------------------------------- 4. what leaves them alone
def test_observe_set_state_and_render_leave_decisions_alone(cuda_device):
    env = CatWorlds(pu.named_cmap("squarinth"), 256, device=cuda_device, seed=1, scripts={2: "evade"})
    env.reset()
    env.step(torch.randint(0, 4, (256, 3), dtype=torch.uint8, device=cuda_device))
    dec = env.script_decisions.clone()
    env.observe()
    torch.cuda.synchronize()
    assert torch.equal(env.script_decisions, dec), "observe"
    st = env.get_state()
    pos = st["pos"].clone()
    pos[:, :, 0] += 3.0
    env.set_state(pos=pos)
    assert torch.equal(env.script_decisions, dec), "set_state"
    env.render_frames([0, 5], rays=True, downsample=4)
    env.sensor_rays()
    torch.cuda.synchronize()
    assert torch.equal(env.script_decisions, dec), "render_frames / sensor_rays"
    env.close()


# ---------------------------------------------------------------------------------------------- 5. switching modes
def test_modes_changed_in_place_reach_eager_steps_and_graph_replays(cuda_device):
    """G alternates eager steps and replays of a graph captured with every mode 0; twin T, without scripts, is fed the
    decoded decisions of G before each step.  Modes change in place between the steps."""
    cmap = pu.named_cmap("agh-map", free_spawn=True)
    N = 1024
    kw = dict(device=cuda_device, seed=3, max_step_count=50)
    G = CatWorlds(cmap, N, want_scripts=True, **kw)
    T = CatWorlds(cmap, N, **kw)
    G.reset()
    acts = torch.zeros((N, 3), dtype=torch.uint8, device=cuda_device)
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        G.step(acts)                                    # warm-up, eager
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        G.step(acts)
    torch.cuda.synchronize()
    T.state.copy_(G.state)                              # the twin starts from G's state
    g = torch.Generator().manual_seed(4)
    schedule = [({}, None), ({2: "evade"}, None), ({0: "chase", 1: "chase"}, torch.arange(N) < N // 2),
                ({2: "random"}, None), ({0: "none", 1: "none", 2: "none"}, None)]
    eager = False
    for spec, mask in schedule:
        G.set_scripts(spec, mask=mask)
        for t in range(40):
            acts.copy_(torch.randint(0, 4, (N, 3), dtype=torch.uint8, generator=g))
            nxt = G.scripted_actions()
            fed = torch.where(nxt >= 0, nxt, acts.to(torch.int64)).to(torch.uint8).contiguous()
            if eager:
                G.step(acts)
            else:
                graph.replay()
            T.step(fed)
            torch.cuda.synchronize()
            assert torch.equal(G.state, T.state), (spec, t, eager)
            assert torch.equal(G._out, T._out), (spec, t, eager)
            eager = not eager
    for e in (G, T):
        e.close()


# ---------------------------------------------------------------------------------------------- checks of the setters
def test_attach_refuses_missing_pointers_and_setters_validate(cuda_device):
    L = _lib.load()
    env = CatWorlds(pu.named_cmap("squarinth"), 64, device=cuda_device, seed=1)
    modes = torch.zeros((64, 3), dtype=torch.uint8, device=cuda_device)
    for io in (_lib.CatScriptIO(modes.data_ptr(), None), _lib.CatScriptIO(None, modes.data_ptr())):
        assert L.cat_env_attach_scripts(env._h, C.byref(io)) == -1
    assert L.cat_env_attach_scripts(env._h, None) == 0
    env.reset()
    env.step(torch.zeros((64, 3), dtype=torch.uint8, device=cuda_device))
    torch.cuda.synchronize()
    with pytest.raises(_lib.CatError):
        env.set_scripts({0: "chase"})
    env.close()
    env = CatWorlds(pu.named_cmap("squarinth"), 64, device=cuda_device, seed=1, scripts={2: "evade"})
    table = env.script_modes.clone()
    for bad in ({3: "chase"}, {-1: "chase"}, {0: "hide"}, {0: 7}, {"cop_0": "chase"}, {0: "chase", 1: "sneak"}):
        with pytest.raises(ValueError):
            env.set_scripts(bad)
    with pytest.raises(ValueError):
        env.set_scripts({0: "chase"}, mask=torch.ones(63, dtype=torch.bool))
    with pytest.raises(ValueError):
        env.set_script_table(torch.full((64, 3), 4, dtype=torch.uint8))
    assert torch.equal(env.script_modes, table), "a failed call writes nothing"
    assert env.scripted_in(2) == "all" and env.scripted_in(0) == "none"
    env.set_scripts({0: "chase"}, mask=torch.arange(64) < 10)
    assert env.scripted_in(0) == "some" and int(env.script_modes[:10, 0].min()) == 2 and int(env.script_modes[10:, 0].max()) == 0
    sd = env.state_dict()
    env.set_scripts({0: "none", 1: "random"})
    env.load_state_dict(sd)
    assert torch.equal(env.script_modes, sd["script_mode"]) and env.scripted_in(0) == "some" and env.scripted_in(1) == "none"
    env.close()


# ---------------------------------------------------------------------------------------------- 6. learner and evaluation
def test_learner_trains_only_the_unscripted_agents(cuda_device):
    env = BatchedCopsThievesEnv(load_named_map("squarinth"), 256, device=cuda_device, seed=6, max_step_count=30,
                                scripted={"thief_0": "evade"})
    assert env.scripted_agents == ["thief_0"]
    cfg = MAPPOConfig(rollouts=32, model="lstm", random_timesteps=0, learning_starts=0, cuda_graph=True,
                      opponent_freeze_duration=0, policy_freeze_duration=0)
    lrn = MAPPOLearner(env, cfg, seed=0)
    assert lrn.agents == ["cop_0", "cop_1"] and set(lrn.models) == {"cop_0", "cop_1"} and set(lrn.mem) == {"cop_0", "cop_1"}
    for _ in range(3):                       # eager warm-up, capture + replay, replay
        lrn.collect()
    stats = lrn.update()
    assert set(stats) == {"cop_0", "cop_1"} and all(s.minibatches > 0 for s in stats.values())
    # a mapping without the scripted agent steps; with it, the thief's entry is ignored
    obs, rew, term, trunc, infos = env.step({a: torch.zeros(256, dtype=torch.int64, device=cuda_device) for a in lrn.agents})
    assert set(obs) == set(env.possible_agents)
    modes = env.worlds.script_modes.clone()
    rate, per_map = evaluate_vs_scripted(env, lrn, "cop", "evade", n_episodes=1, by_map=True)
    assert 0.0 <= rate <= 1.0 and per_map[0]["episodes"] >= 256
    assert torch.equal(env.worlds.script_modes, modes), "the modes found are restored"
    with pytest.raises(ValueError, match="no models"):
        evaluate_vs_scripted(env, lrn, "thief", "chase", n_episodes=1)
    env.set_scripted({"cop_0": "chase"})
    with pytest.raises(RuntimeError, match="changed"):
        lrn.collect()
    env.set_scripted({"cop_0": "none"})
    lrn.collect()
    env.set_scripted({"thief_0": "none"}, mask=torch.arange(256) < 128)
    with pytest.raises(ValueError, match="some worlds"):
        MAPPOLearner(env, cfg, seed=0)
    env.close()


def test_evaluate_vs_scripted_with_a_full_learner(cuda_device):
    env = BatchedCopsThievesEnv([load_named_map("squarinth"), load_named_map("agh-map")], 512, device=cuda_device, seed=2,
                                max_step_count=25, scripted={})
    assert env.scripted_agents == []
    cfg = MAPPOConfig(rollouts=16, model="mlp", random_timesteps=0, learning_starts=0, cuda_graph=False,
                      opponent_freeze_duration=0, policy_freeze_duration=0)
    lrn = MAPPOLearner(env, cfg, seed=0)
    assert lrn.agents == env.possible_agents
    env.set_scripted({"cop_1": "random"}, mask=torch.arange(512) % 3 == 0)
    modes = env.worlds.script_modes.clone()
    for role, ctl in (("cop", "evade"), ("thief", "chase")):
        rate, per_map = evaluate_vs_scripted(env, lrn, role, ctl, n_episodes=2, by_map=True)
        assert torch.equal(env.worlds.script_modes, modes)
        assert 0.0 <= rate <= 1.0
        n = sum(m["episodes"] for m in per_map)
        assert n >= 2 * 512 and abs(sum(m["rate"] * m["episodes"] for m in per_map) / n - rate) < 1e-9
    cop, thief = (evaluate_vs_scripted(env, lrn, "cop", "random", n_episodes=1),
                  evaluate_vs_scripted(env, lrn, "thief", "random", n_episodes=1))
    assert 0.0 <= cop <= 1.0 and 0.0 <= thief <= 1.0
    env.close()


# ---------------------------------------------------------------------------------------------- 7. behaviour
def test_chasing_cops_catch_a_random_thief_more_often_than_random_cops(cuda_device):
    cmap = pu.named_cmap("squarinth")
    rates = {}
    for cops in ("chase", "random"):
        env = CatWorlds(cmap, 4096, device=cuda_device, seed=21, want_f32=False, want_shared=False,
                        scripts={0: cops, 1: cops, 2: "random"})
        env.reset()
        acts = torch.zeros((4096, 3), dtype=torch.uint8, device=cuda_device)
        captures = torch.zeros((), dtype=torch.int64, device=cuda_device)
        episodes = torch.zeros((), dtype=torch.int64, device=cuda_device)
        for _ in range(2000):
            env.step(acts)
            done = env.terminated == 1
            episodes += done.sum()
            captures += (done & (env.winner == 0)).sum()
        rates[cops] = (int(captures) / max(int(episodes), 1), int(episodes))
        env.close()
    print("capture rate vs a random thief (rate, episodes):", rates)
    assert rates["chase"][1] > 0 and rates["random"][1] > 0
    assert rates["chase"][0] > rates["random"][0], rates
